// 3x3x3 conv for the narrow-N layers (Cout = 32 or 64: 55 % of the network's FLOPs) with shared-memory tap reuse.
//
// Why: with N = 64 the plain implicit GEMM (conv_igemm.cu) needs a fresh 16 KB A tile + 8 KB weight tile per
// 128 tensor-cycles = 192 B/clk/SM, three times what L2 -> SM delivers (~64 B/clk/SM measured): it saturates at ~35 %
// of the tensor peak.  Here one CTA owns a 32(w) x 4(h) x 4(d) output tile = 4 accumulators of 128 voxels, and for a
// fixed w-tap and channel chunk streams the 6 input planes (d0-1 .. d0+4), each ONE TMA box of (4+2) h-lines x 32 w
// = 192 rows.  A plane in shared memory feeds the 3 h-taps by 1024-byte-aligned descriptor offsets (row offset
// dh*32) and the up-to-3 d-taps by accumulating into different output planes; the 9 weight tiles of that w-tap stay
// resident (double-buffered) while the planes stream.  Traffic: (6*24 KB + 72 KB) per 144 MMAs = 47 B/clk/SM.
//
// SS-mode tcgen05.mma reads A (128 x 16 bf16 = 4 KB) from shared memory for every instruction; at N = 64 that is
// 48 cycles of smem reads for 32 cycles of math (measured: 51 cycles per MMA issue, 67 % cap).  The accumulators of
// the four output planes are adjacent in TMEM (64 columns each), and the d-taps of an input plane feed CONSECUTIVE
// output planes, so one instruction with N = 64 * (number of valid d-taps) <= 192 updates up to three accumulators
// from one A read: smem-read cycles == math cycles.  All MMAs accumulate; the epilogue zeroes each accumulator
// (tcgen05.st) after reading it.
//
// Warp roles: 0 MMA issuer (+TMEM), 1-3 plane producers (ring stage s owned by producer s mod 3), 4-6 weight
// producers (one d-tap row each), 7 idle, 8-15 epilogue (two warps per TMEM lane quarter).  Whole-warp uniform loops, elected-lane issue.
#include "common.h"
#include "ptx.cuh"

namespace b2 {

int make_act_tmap(CUtensorMap* map, const void* base, int N, int D, int H, int W, int C, int ld, int coff,
                  int box_c, int bw, int bh, int bd);

struct SlabParams {
  int N, D, H, W;
  int Cin, Cout;       // Cout == BN (32 or 64)
  int n_chunks;
  int tiles_w, tiles_h, tiles_d;
  int stages;          // plane ring depth (multiple of 3)
  int relu;
  int ldy, y_coff;
  __nv_bfloat16* y;
  long long* stat_acc;   // optional [Cout][4] fixed-point statistics accumulators (see conv_igemm.cu, common.h)
  const __nv_bfloat16* stat_r;   // optional: backward statistics (sum dy, sum dy*r)
  const float* bias;             // fp32 [Cout] conv bias of the kBias instantiation, added before ReLU
  long long total_tiles;
};

static constexpr int kSlabThreads = 32 * 16;
static constexpr int kTD = 4;

// kTW x kTH x kTD output tile with kTW * kTH = 128 voxels per plane: 32 x 4 (round 1) or 16 x 8 — the second shape cuts
// the tile-quantisation waste of volumes whose W is not a multiple of 32 (bounding boxes of real cohorts: W = 72 pads to
// 80 instead of 96).  Both keep every h-tap offset (kTW rows) a multiple of the 8-row swizzle atom.
// kBias: layers with a conv bias (a separate instantiation: a run-time test costs the bias-free epilogue registers).
template <int KC, int kTW, bool kBias>
__global__ void __launch_bounds__(kSlabThreads, 1)
conv3d_slab_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                   const SlabParams p) {
  constexpr int kTH = 128 / kTW;
  constexpr int kPlaneRows = kTW * (kTH + 2);
  pdl_wait();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int kRowBytes = KC * 2;
  constexpr int kPlaneBytes = kPlaneRows * kRowBytes;
  const int BN = p.Cout;
  const int tap_bytes = BN * kRowBytes;          // one weight tile
  const int b_bytes = 9 * tap_bytes;             // the 9 (dd, dh) taps of one w-tap
  uint8_t* smem_b = smem;                        // 2 buffers
  uint8_t* smem_p = smem + 2 * (size_t)b_bytes;  // plane ring
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_p + (size_t)p.stages * kPlaneBytes);
  uint64_t* p_full = bars;
  uint64_t* p_empty = bars + p.stages;
  uint64_t* b_full = bars + 2 * p.stages;
  uint64_t* b_empty = b_full + 2;
  uint64_t* tmem_full = b_empty + 2;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  if (warp == 1 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&p_full[s], 1);
      mbar_init(&p_empty[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&b_full[s], 3);
      mbar_init(&b_empty[s], 1);
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], 256);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int tiles_per_n = p.tiles_w * p.tiles_h * p.tiles_d;

  if (warp >= 1 && warp <= 3) {
    // ---------------------------------------------------------------- plane producers
    const int me = warp - 1;
    uint32_t gp = 0;
    for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const int n = (int)(tile / tiles_per_n);
      int t = (int)(tile % tiles_per_n);
      const int w0 = (t % p.tiles_w) * kTW; t /= p.tiles_w;
      const int h0 = (t % p.tiles_h) * kTH;
      const int d0 = (t / p.tiles_h) * kTD;
      for (int ch = 0; ch < p.n_chunks; ++ch)
        for (int dw = -1; dw <= 1; ++dw)
          for (int pl = 0; pl < kTD + 2; ++pl, ++gp) {
            const int stage = (int)(gp % (uint32_t)p.stages);
            if (stage % 3 != me) continue;
            const uint32_t phase = (gp / (uint32_t)p.stages) & 1u;
            mbar_wait(&p_empty[stage], phase ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(&p_full[stage], (uint32_t)kPlaneBytes);
              tma_load_5d(smem_p + (size_t)stage * kPlaneBytes, &tmap_a, &p_full[stage], ch * KC, w0 + dw, h0 - 1,
                          d0 - 1 + pl, n);
            }
            __syncwarp();
          }
    }
    if (warp == 1) pdl_trigger();   // last plane loads issued: the next kernel may be staged
  } else if (warp >= 4 && warp <= 6) {
    // ---------------------------------------------------------------- weight producers (one d-tap row each)
    const int ddi = warp - 4;   // dd + 1
    uint32_t gb = 0;
    for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x)
      for (int ch = 0; ch < p.n_chunks; ++ch)
        for (int dwi = 0; dwi < 3; ++dwi, ++gb) {
          const int bs = (int)(gb & 1u);
          const uint32_t phase = (gb >> 1) & 1u;
          mbar_wait(&b_empty[bs], phase ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&b_full[bs], (uint32_t)(3 * tap_bytes));
            for (int dhi = 0; dhi < 3; ++dhi) {
              const int tap = ddi * 9 + dhi * 3 + dwi;   // PyTorch tap order (kd, kh, kw)
              // buffer layout [dh][dd = +1, 0, -1][co]: the d-taps of one h-tap are consecutive row blocks in the
              // order of the output planes they feed
              tma_load_2d(smem_b + (size_t)bs * b_bytes + (size_t)(dhi * 3 + (2 - ddi)) * tap_bytes, &tmap_b,
                          &b_full[bs], ch * KC, tap * p.Cout);
            }
          }
          __syncwarp();
        }
  } else if (warp == 0) {
    // ---------------------------------------------------------------- MMA issuer
    constexpr uint32_t kLayout = (KC == 64) ? SWZ_128B : (KC == 32 ? SWZ_64B : SWZ_32B);
    constexpr uint32_t kSbo = 8u * kRowBytes;
    const uint64_t desc_hi = make_smem_desc(0, 16, kSbo, kLayout);
    const uint32_t p0 = smem_u32(smem_p) >> 4, b0 = smem_u32(smem_b) >> 4;
    constexpr uint32_t kPlaneStep = kPlaneBytes >> 4;
    constexpr uint32_t kDhStep = (kTW * kRowBytes) >> 4;   // +32 rows
    const uint32_t tap_step = (uint32_t)tap_bytes >> 4, bbuf_step = (uint32_t)b_bytes >> 4;
    const uint32_t idesc1 = make_idesc_bf16(128, (uint32_t)BN, 0, 0);
    const uint32_t idesc2 = make_idesc_bf16(128, (uint32_t)(2 * BN), 0, 0);
    const uint32_t idesc3 = make_idesc_bf16(128, (uint32_t)(3 * BN), 0, 0);
    int ps = 0;
    uint32_t pphase = 0, gb = 0, it = 0;
    for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
      const uint32_t acc = it & 1u;
      mbar_wait(&tmem_empty[acc], (it >> 1) & 1u);   // the epilogue has drained AND zeroed this accumulator set
      tc_fence_after();
      const uint32_t d_base = tmem_base + acc * 256u;
      const int n_groups = p.n_chunks * 3;
      for (int g = 0; g < n_groups; ++g, ++gb) {
        const int bs = (int)(gb & 1u);
        mbar_wait(&b_full[bs], (gb >> 1) & 1u);
        for (int pl = 0; pl < kTD + 2; ++pl) {
          mbar_wait(&p_full[ps], pphase);
          tc_fence_after();
          // input plane pl feeds output planes o = pl-2 (dd=+1), pl-1 (dd=0), pl (dd=-1), clipped to [0, kTD)
          const int o_lo = pl - 2 < 0 ? 0 : pl - 2;
          const int o_hi = pl > kTD - 1 ? kTD - 1 : pl;
          const int nblk = o_hi - o_lo + 1;                 // 1..3 accumulators in one instruction
          const int b_first = o_lo - (pl - 2);              // first row block (dd order +1, 0, -1) that is used
          const uint32_t idesc = nblk == 3 ? idesc3 : (nblk == 2 ? idesc2 : idesc1);
          if (elect_one()) {
            const uint64_t a_plane = desc_hi | (uint64_t)(p0 + (uint32_t)ps * kPlaneStep);
            const uint64_t b_buf = desc_hi | (uint64_t)(b0 + (uint32_t)bs * bbuf_step + (uint32_t)b_first * tap_step);
            const uint32_t d_tmem = d_base + (uint32_t)(o_lo * BN);
#pragma unroll
            for (int dhi = 0; dhi < 3; ++dhi) {
              const uint64_t adesc = a_plane + (uint64_t)(dhi * kDhStep);
              const uint64_t bdesc = b_buf + (uint64_t)(dhi * 3) * tap_step;
#pragma unroll
              for (int k = 0; k < KC / 16; ++k) umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, 1u);
            }
            umma_commit(&p_empty[ps]);
            if (pl == kTD + 1) {
              umma_commit(&b_empty[bs]);
              if (g == n_groups - 1) umma_commit(&tmem_full[acc]);
            }
          }
          __syncwarp();
          if (++ps == p.stages) { ps = 0; pphase ^= 1; }
        }
      }
    }
  } else if (warp >= 8) {
    // ---------------------------------------------------------------- epilogue: 8 warps
    // Warp (q, half): TMEM lane quarter q = warp & 3; with BN = 64 the two halves take the two 32-column chunks of every
    // output plane, with BN = 32 they take the output planes {0, 1} / {2, 3}.  The GroupNorm statistics are accumulated
    // PER THREAD (its row, 32 columns, 2 x 32 fp32 registers) over all tiles of the CTA and reduced across lanes ONCE at
    // the end.  Round 1 ran a 2 x 31-shuffle transposing reduction per chunk, plane and tile in four warps: for the
    // short-K layers (encoders.0.conv2, decoders.2.conv2, every dgrad with fused backward statistics) that epilogue was
    // as long as the main loop — the same launches ran 15-45 us faster without statistics.
    const int q = warp & 3;           // TMEM lane quarter this warp may access
    const int half = (warp - 8) >> 2;
    const int row = q * 32 + lane;    // accumulator row == voxel within the output plane: (h-line, w)
    const int lw = row % kTW, lh = row / kTW;
    const int n_chunks_n = BN / 32;   // 1 or 2
    const int c0 = (n_chunks_n == 2) ? 32 * half : 0;
    const int o_begin = (n_chunks_n == 2) ? 0 : 2 * half, o_end = (n_chunks_n == 2) ? kTD : 2 * half + 2;
    float acc_s[32], acc_q[32];
#pragma unroll
    for (int e = 0; e < 32; ++e) { acc_s[e] = 0.f; acc_q[e] = 0.f; }
    // every MMA accumulates: clear both accumulator sets once, then hand them to the MMA issuer
    for (uint32_t c = 256u * half; c < 256u * half + 256u; c += 32)
      tmem_st32_zero(tmem_base + ((uint32_t)(q * 32) << 16) + c);
    tmem_st_wait();
    tc_fence_before();
    mbar_arrive(&tmem_empty[0]);
    mbar_arrive(&tmem_empty[1]);
    uint32_t it = 0;
    for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
      const int n = (int)(tile / tiles_per_n);
      int t = (int)(tile % tiles_per_n);
      const int w0 = (t % p.tiles_w) * kTW; t /= p.tiles_w;
      const int h0 = (t % p.tiles_h) * kTH;
      const int d0 = (t / p.tiles_h) * kTD;
      const uint32_t acc = it & 1u;
      const int w = w0 + lw, h = h0 + lh;
      mbar_wait(&tmem_full[acc], (it >> 1) & 1u);
      tc_fence_after();
      for (int o = o_begin; o < o_end; ++o) {
        const int d = d0 + o;
        const bool valid = (w < p.W) && (h < p.H) && (d < p.D);
        const size_t vox = (((size_t)n * p.D + d) * p.H + h) * p.W + w;
        const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 256u + (uint32_t)(o * BN + c0);
        uint32_t v[32];
        tmem_ld32(t_addr, v);
        tmem_ld_wait();
        tmem_st32_zero(t_addr);   // ready for the next tile's always-accumulating MMAs
        uint32_t pk[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          float f0 = __uint_as_float(v[2 * e]), f1 = __uint_as_float(v[2 * e + 1]);
          if constexpr (kBias) {
            const float2 b = __ldg(reinterpret_cast<const float2*>(p.bias + c0) + e);
            f0 += b.x;
            f1 += b.y;
          }
          if (p.relu) { f0 = relu_nan(f0); f1 = relu_nan(f1); }
          pk[e] = pack_bf16x2(f0, f1);
        }
        if (valid) {
          uint4* dst = reinterpret_cast<uint4*>(p.y + vox * p.ldy + p.y_coff + c0);
#pragma unroll
          for (int j = 0; j < 4; ++j) dst[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
          if (p.stat_acc != nullptr) {   // statistics of what is STORED (bf16-rounded), this thread's row
            if (p.stat_r != nullptr) {   // backward: sum dy, sum dy * r
              const uint4* rp = reinterpret_cast<const uint4*>(p.stat_r + vox * BN + c0);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const uint4 u = __ldg(rp + j);
                const uint32_t wds[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float g0 = __uint_as_float(pk[4 * j + e] << 16), g1 = __uint_as_float(pk[4 * j + e] & 0xffff0000u);
                  acc_s[8 * j + 2 * e] += g0;
                  acc_s[8 * j + 2 * e + 1] += g1;
                  acc_q[8 * j + 2 * e] = fmaf(g0, __uint_as_float(wds[e] << 16), acc_q[8 * j + 2 * e]);
                  acc_q[8 * j + 2 * e + 1] = fmaf(g1, __uint_as_float(wds[e] & 0xffff0000u), acc_q[8 * j + 2 * e + 1]);
                }
              }
            } else {                     // forward: sum r, sum r^2
#pragma unroll
              for (int e = 0; e < 16; ++e) {
                const float g0 = __uint_as_float(pk[e] << 16), g1 = __uint_as_float(pk[e] & 0xffff0000u);
                acc_s[2 * e] += g0;
                acc_s[2 * e + 1] += g1;
                acc_q[2 * e] = fmaf(g0, g0, acc_q[2 * e]);
                acc_q[2 * e + 1] = fmaf(g1, g1, acc_q[2 * e + 1]);
              }
            }
          }
        }
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&tmem_empty[acc]);
    }
    if (p.stat_acc != nullptr) {
      // one transposing reduction per thread-array: afterwards lane L holds the sums of column c0 + L over this warp's rows
      warp_column_sums(acc_s, lane);
      warp_column_sums(acc_q, lane);
      float2* sbuf = reinterpret_cast<float2*>(smem_p);   // [8 warps][32] in the (now idle) plane ring
      sbuf[(warp - 8) * 32 + lane] = make_float2(acc_s[0], acc_q[0]);
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (warp == 8 || (warp == 12 && n_chunks_n == 2)) {
        // BN = 64: the four warps of a half cover one 32-column chunk; BN = 32: all eight warps cover the same 32 columns
        const int wb = (n_chunks_n == 2) ? 4 * half : 0;
        float2 a = sbuf[(wb + 0) * 32 + lane], b = sbuf[(wb + 1) * 32 + lane];
        float2 cc = sbuf[(wb + 2) * 32 + lane], d = sbuf[(wb + 3) * 32 + lane];
        float ssum = (a.x + b.x) + (cc.x + d.x), qsum = (a.y + b.y) + (cc.y + d.y);
        if (n_chunks_n == 1) {
          a = sbuf[4 * 32 + lane]; b = sbuf[5 * 32 + lane]; cc = sbuf[6 * 32 + lane]; d = sbuf[7 * 32 + lane];
          ssum += (a.x + b.x) + (cc.x + d.x);
          qsum += (a.y + b.y) + (cc.y + d.y);
        }
        stat_atomic_add(p.stat_acc + 4 * (c0 + lane), ssum);
        stat_atomic_add(p.stat_acc + 4 * (c0 + lane) + 2, qsum);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// host: tile shape with the least padding, and whether the slab kernel is worthwhile for this layer.
// Padded voxels cost MMA time; the alternative for these narrow-N layers is the plain implicit GEMM at ~35-45 % of the
// tensor peak against ~85 % here, so the slab kernel wins up to ~1.5x padding.  (Round 1 bailed out above 1.12x with a
// single 32 x 4 x 4 tile: bounding boxes such as 80 x 104 x 72 fell back to the slow path.)
static long long slab_padded(int D, int H, int W, int tw) {
  const int th = 128 / tw;
  return (long long)ceil_div(W, tw) * tw * ceil_div(H, th) * th * ceil_div(D, kTD) * kTD;
}
static int slab_tile_w(int D, int H, int W) { return slab_padded(D, H, W, 16) < slab_padded(D, H, W, 32) ? 16 : 32; }

// Cin: 16 (encoders.0.conv2 of a 32-filter network, one 16-channel chunk) or a multiple of 32 (decoders.2.conv1 of a
// 32-filter network has Cin = 96: three 32-channel chunks).
bool slab_applicable(int N, int D, int H, int W, int Cin, int Cout, int y_is_fp32) {
  if (y_is_fp32) return false;
  if (!(Cout == 32 || Cout == 64)) return false;
  if (!(Cin % 32 == 0 || Cin == 16)) return false;
  const long long padded = slab_padded(D, H, W, slab_tile_w(D, H, W));
  if (padded * 100 > (long long)W * H * D * 150) return false;
  return true;
}

template <int KC, int TW, bool kBias>
static int launch_slab_b(const CUtensorMap& ta, const CUtensorMap& tb, const SlabParams& p, size_t smem_bytes,
                         cudaStream_t stream) {
  long long grid = p.total_tiles < num_sms() ? p.total_tiles : num_sms();
  B2_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab_kernel<KC, TW, kBias>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     227 * 1024));
  B2_LAUNCH((conv3d_slab_kernel<KC, TW, kBias>), (unsigned)grid, kSlabThreads, smem_bytes, stream, ta, tb, p);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}
template <int KC, int TW>
static int launch_slab_t(const CUtensorMap& ta, const CUtensorMap& tb, const SlabParams& p, size_t smem_bytes,
                         cudaStream_t stream) {
  return p.bias ? launch_slab_b<KC, TW, true>(ta, tb, p, smem_bytes, stream)
                : launch_slab_b<KC, TW, false>(ta, tb, p, smem_bytes, stream);
}

int launch_slab(const void* x, int ldx, int x_coff, const void* wpack, void* y, int ldy, int y_coff, int N, int D,
                int H, int W, int Cin, int Cout, int relu, long long* stat_acc, const void* stat_r, const float* bias,
                cudaStream_t stream) {
  SlabParams p;
  p.N = N; p.D = D; p.H = H; p.W = W; p.Cin = Cin; p.Cout = Cout;
  const int KC = (Cin % 64 == 0) ? 64 : (Cin % 32 == 0 ? 32 : 16);
  const int tw = slab_tile_w(D, H, W), th = 128 / tw;
  p.n_chunks = Cin / KC;
  p.tiles_w = ceil_div(W, tw);
  p.tiles_h = ceil_div(H, th);
  p.tiles_d = ceil_div(D, kTD);
  p.relu = relu;
  p.ldy = ldy; p.y_coff = y_coff;
  p.y = reinterpret_cast<__nv_bfloat16*>(y);
  p.total_tiles = (long long)N * p.tiles_w * p.tiles_h * p.tiles_d;
  p.stat_acc = stat_acc;
  p.stat_r = reinterpret_cast<const __nv_bfloat16*>(stat_r);
  p.bias = bias;
  if (stat_acc) B2_REQUIRE(N == 1, "b2_conv3d_igemm_stats: fused statistics need batch 1");
  const int plane_bytes = tw * (th + 2) * KC * 2;
  const int b_bytes = 9 * Cout * KC * 2;
  const int budget = 227 * 1024 - 1024 - 512;
  p.stages = (budget - 2 * b_bytes) / plane_bytes;
  p.stages = (p.stages / 3) * 3;
  if (p.stages > 9) p.stages = 9;
  B2_REQUIRE(p.stages >= 3, "conv3d_slab: tile does not fit shared memory");
  CUtensorMap ta, tb;
  int rc = make_act_tmap(&ta, x, N, D, H, W, Cin, ldx, x_coff, KC, tw, th + 2, 1);
  if (rc) return rc;
  {
    const uint64_t dims[2] = {(uint64_t)Cin, (uint64_t)27 * Cout};
    const uint64_t strides[1] = {(uint64_t)Cin * 2};
    const uint32_t box[2] = {(uint32_t)KC, (uint32_t)Cout};
    rc = encode_tmap_bf16(&tb, wpack, 2, dims, strides, box, KC * 2);
    if (rc) return rc;
  }
  const size_t smem_bytes = 2 * (size_t)b_bytes + (size_t)p.stages * plane_bytes + 1024 + 512;
  if (KC == 64) return tw == 32 ? launch_slab_t<64, 32>(ta, tb, p, smem_bytes, stream)
                                : launch_slab_t<64, 16>(ta, tb, p, smem_bytes, stream);
  if (KC == 32) return tw == 32 ? launch_slab_t<32, 32>(ta, tb, p, smem_bytes, stream)
                                : launch_slab_t<32, 16>(ta, tb, p, smem_bytes, stream);
  return tw == 32 ? launch_slab_t<16, 32>(ta, tb, p, smem_bytes, stream)
                  : launch_slab_t<16, 16>(ta, tb, p, smem_bytes, stream);
}

}  // namespace b2
