// 3x3x3 stride-1 pad-1 Conv3d as an implicit GEMM on tcgen05 (sm_100a).
//
//   out[v, co] = sum_{tap, ci} in[v + off(tap), ci] * Wp[tap][co][ci]          (NDHWC bf16, fp32 accumulate)
//
// fprop and dgrad are the same kernel: dgrad feeds dY as `in` and a flipped/transposed weight pack.
//
// Mapping: M = 128 voxels arranged as a (bw x bh x bd) box, N = BN output channels, K = 27 taps x Cin.
// Per (tap, 64-channel chunk) one TMA 5-D box load brings the shifted 128-voxel x KC-channel A tile
// (out-of-volume voxels are zero-filled by TMA = the conv's zero padding) and one 2-D load brings the
// BN x KC weight tile; both land 128B-swizzled, K-major, and feed tcgen05.mma (128 x BN x 16) with the
// accumulator in TMEM (double-buffered so the epilogue of tile i overlaps the main loop of tile i+1).
// Warp roles: warp 0 MMA issuer (+TMEM owner), warps 1-8 TMA producers, warps 9-12 epilogue.
// Eight producer warps, not one: measured on B200 (tools/micro/tma_bench2.cu) a single thread retires one TMA op
// per ~735 cycles whatever its size (<= 32 KB) and however many are in flight, while ops issued by different warps
// proceed in parallel (1/2/4 warps: 22/45/89 B/clk/SM).  Stage s of the ring is filled by producer pair (s mod 4):
// the even warp of the pair loads the A box, the odd warp the weight tile.
// Round 2: the HALO instantiation (64-channel chunks, one-plane tile boxes) loads each A tile once per (d, w) tap pair
// with an h-halo and takes the three h taps from it by descriptor offsets; see the comment above the kernel.
// 32-filter networks: KC = 16 (32-byte rows, 32B swizzle) for Cin = 16 and the 48-channel split operands of the exact
// path, and N tiles of 16 x odd channels for 16-channel outputs (encoders.0.conv2 dgrad, the exact path's first
// layer) and 48-channel ones (the dgrad shape of a 48-channel input).  16-channel
// activations are not padded to 32: that would double the operand bytes and MMAs of those layers.
#include "common.h"
#include "ptx.cuh"
#include <stdlib.h>

namespace b2 {

struct IgemmParams {
  int N, D, H, W;
  int Cin, Cout;
  int bw, bh, bd;
  int tiles_w, tiles_h, tiles_d;
  int n_tiles_n, BN;
  int KC, n_chunks;
  int stages;
  int stages_b;        // halo variant: depth of the separate weight-tile ring
  int a_bytes, b_bytes;
  int relu;
  int ldy, y_coff;
  __nv_bfloat16* y;
  float* y32;          // optional fp32 output (same indexing, ld = ldy) instead of bf16
  long long* stat_acc;  // optional [Cout][4] fixed-point accumulators (common.h): per-channel sum / sum of squares of the
                        // bf16-rounded outputs (GroupNorm statistics fused into the epilogue; N == 1, one N tile)
  const __nv_bfloat16* stat_r;  // when set, the statistics are (sum dy, sum dy*r) with r = this dense [V][Cout]
                                // tensor: the two per-channel sums GroupNorm backward needs (dgrad launches)
  long long total_tiles;
  // split-K over the 27 taps for layers with fewer tiles than SMs (12x14x12 level): work item = (split, tile);
  // every split writes an fp32 partial tile to y32 + split * split_stride, reduced by conv_splitk_reduce_kernel
  int splits;
  long long split_stride;
  const float* bias;   // optional fp32 [Cout] conv bias (fprop): added to the accumulator before ReLU, the bf16 rounding
                       // and the fused statistics; never set on split-K partials (conv_splitk_reduce_kernel adds it)
};

static constexpr int kProducerPairs = 4;
static constexpr int kThreads = 32 * (1 + 2 * kProducerPairs + 4);
static constexpr int kAccStride = 256;  // TMEM columns between the two accumulators

__device__ __forceinline__ void decode_tile(long long tile, const IgemmParams& p, int& n, int& d0, int& h0,
                                            int& w0, int& n0) {
  const int nt = (int)(tile % p.n_tiles_n);
  long long mt = tile / p.n_tiles_n;
  const int tw = (int)(mt % p.tiles_w);
  mt /= p.tiles_w;
  const int th = (int)(mt % p.tiles_h);
  mt /= p.tiles_h;
  const int td = (int)(mt % p.tiles_d);
  n = (int)(mt / p.tiles_d);
  w0 = tw * p.bw;
  h0 = th * p.bh;
  d0 = td * p.bd;
  n0 = nt * p.BN;
}

// All role loops are executed by the WHOLE warp with warp-uniform control flow and values; only the single
// TMA / tcgen05 instruction is predicated on an elected lane.  (Round-1 finding, tools/timeline_igemm.py: running the
// loops inside `if (lane == 0)` made every descriptor take the R2UR path into the uniform datapath and cost ~140
// cycles per tcgen05.mma issue — the issuing thread, not TMA or the tensor pipe, bounded the kernel at ~900 cycles
// per stage.)
// HALO variant (KC = 64, one-plane tile boxes bw x bh with bw % 8 == 0): the A ring holds tiles with an h-halo —
// bh + 2 lines of bw voxels, one line = bw / 8 whole 1 024-byte swizzle atoms — loaded once per (d, w) tap pair and
// channel chunk; the three h taps read the same tile through descriptors that start one line apart.  A loads drop from 27 to 9 per chunk and tile (the
// plain kernel sits on the L2 -> SM limit: 16 KB of A + BN x 128 B of weights per four MMAs); the weight tiles get a
// ring of their own (one stage per tap and chunk).
template <int KC, bool HALO>
__global__ void __launch_bounds__(kThreads, 1)
conv3d_igemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                    const IgemmParams p) {
  pdl_wait();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int kABytes = HALO ? p.a_bytes : 128 * KC * 2;   // HALO: (bh + 2) lines of bw voxels (runtime)
  const int n_bstages = HALO ? p.stages_b : p.stages;
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + (size_t)p.stages * kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + (size_t)n_bstages * p.b_bytes);
  uint64_t* full = bars;                    // HALO: the A ring's barriers
  uint64_t* empty = bars + p.stages;
  uint64_t* full_b = bars + 2 * p.stages;   // HALO only: the weight ring's barriers
  uint64_t* empty_b = full_b + (HALO ? p.stages_b : 0);
  uint64_t* tmem_full = empty_b + (HALO ? p.stages_b : 0);
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // warp-uniform by construction
  const int lane = threadIdx.x & 31;

  if (warp == 1 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], HALO ? 1 : 2);   // plain: A loader + B loader each arrive with their own expect_tx
      mbar_init(&empty[s], 1);
    }
    if (HALO) {
      for (int s = 0; s < p.stages_b; ++s) {
        mbar_init(&full_b[s], 1);
        mbar_init(&empty_b[s], 1);
      }
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 128);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= 1 && warp <= 2 * kProducerPairs) {
    // ------------------------------------------------------------------ TMA producers
    const int me = (warp - 1) >> 1;
    const bool loads_a = ((warp - 1) & 1) == 0;
    uint32_t gs = 0;  // global stage counter, identical in every producer and in the MMA issuer
    if constexpr (HALO) {
      // item order (shared with the MMA issuer): (dd, dw, chunk) for the A ring, (dd, dw, chunk, dh) for the weights
      for (long long work = blockIdx.x; work < p.total_tiles; work += gridDim.x) {
        int n, d0, h0, w0, n0;
        decode_tile(work, p, n, d0, h0, w0, n0);
        for (int t9 = 0; t9 < 9; ++t9) {
          const int dd = t9 / 3 - 1, dw = t9 % 3 - 1;
          for (int ch = 0; ch < p.n_chunks; ++ch) {
            if (loads_a) {
              if ((int)(gs % kProducerPairs) == me) {
                const int stage = (int)(gs % (uint32_t)p.stages);
                const uint32_t phase = (gs / (uint32_t)p.stages) & 1u;
                mbar_wait(&empty[stage], phase ^ 1);
                if (elect_one()) {
                  mbar_arrive_expect_tx(&full[stage], (uint32_t)kABytes);
                  tma_load_5d(smem_a + (size_t)stage * kABytes, &tmap_a, &full[stage], ch * KC, w0 + dw, h0 - 1,
                              d0 + dd, n);
                }
                __syncwarp();
              }
              ++gs;
            } else {
              for (int j = 0; j < 3; ++j, ++gs) {   // dh = j - 1
                if ((int)(gs % kProducerPairs) != me) continue;
                const int stage = (int)(gs % (uint32_t)p.stages_b);
                const uint32_t phase = (gs / (uint32_t)p.stages_b) & 1u;
                mbar_wait(&empty_b[stage], phase ^ 1);
                if (elect_one()) {
                  mbar_arrive_expect_tx(&full_b[stage], (uint32_t)p.b_bytes);
                  tma_load_2d(smem_b + (size_t)stage * p.b_bytes, &tmap_b, &full_b[stage], ch * KC,
                              ((dd + 1) * 9 + j * 3 + (dw + 1)) * p.Cout + n0);
                }
                __syncwarp();
              }
            }
          }
        }
      }
    } else
    for (long long work = blockIdx.x; work < p.total_tiles * p.splits; work += gridDim.x) {
      int n, d0, h0, w0, n0;
      decode_tile(work % p.total_tiles, p, n, d0, h0, w0, n0);
      const int split = (int)(work / p.total_tiles);
      const int tap_end = 27 * (split + 1) / p.splits;
      for (int tap = 27 * split / p.splits; tap < tap_end; ++tap) {
        const int dd = tap / 9 - 1, dh = (tap / 3) % 3 - 1, dw = tap % 3 - 1;
        for (int ch = 0; ch < p.n_chunks; ++ch, ++gs) {
          if ((int)(gs % kProducerPairs) != me) continue;
          const int stage = (int)(gs % (uint32_t)p.stages);
          const uint32_t phase = (gs / (uint32_t)p.stages) & 1u;
          mbar_wait(&empty[stage], phase ^ 1);
          if (elect_one()) {
            if (loads_a) {
              mbar_arrive_expect_tx(&full[stage], (uint32_t)kABytes);
              tma_load_5d(smem_a + (size_t)stage * kABytes, &tmap_a, &full[stage], ch * KC, w0 + dw, h0 + dh, d0 + dd,
                          n);
            } else {
              mbar_arrive_expect_tx(&full[stage], (uint32_t)p.b_bytes);
              tma_load_2d(smem_b + (size_t)stage * p.b_bytes, &tmap_b, &full[stage], ch * KC, tap * p.Cout + n0);
            }
          }
          __syncwarp();
        }
      }
    }
    if (warp == 1) pdl_trigger();   // this CTA has issued its last loads: the next kernel may be staged
  } else if (warp == 0) {
    // ------------------------------------------------------------------ MMA issuer
    const uint32_t idesc = make_idesc_bf16(128, (uint32_t)p.BN, 0, 0);
    constexpr uint32_t kLayout = (KC == 64) ? SWZ_128B : (KC == 32 ? SWZ_64B : SWZ_32B);
    constexpr uint32_t kSbo = 8u * KC * 2u;
    const uint64_t desc_hi = make_smem_desc(0, 16, kSbo, kLayout);           // everything but the start address
    const uint32_t a0 = smem_u32(smem_a) >> 4, b0 = smem_u32(smem_b) >> 4;   // encoded start addresses of stage 0
    const uint32_t a_step = kABytes >> 4, b_step = (uint32_t)p.b_bytes >> 4;
    int stage = 0;
    uint32_t phase = 0;
    uint32_t it = 0;
    if constexpr (HALO) {
      int sb = 0;
      uint32_t pb = 0;
      const int n_items = 9 * p.n_chunks;
      const uint32_t line_units = (uint32_t)p.bw * 8u;   // one h-line = bw voxels x 128 B, in 16-byte units
      for (long long work = blockIdx.x; work < p.total_tiles; work += gridDim.x, ++it) {
        const uint32_t acc = it & 1u;
        const uint32_t acc_phase = (it >> 1) & 1u;
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * kAccStride;
        for (int i = 0; i < n_items; ++i) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          for (int j = 0; j < 3; ++j) {
            mbar_wait(&full_b[sb], pb);
            tc_fence_after();
            if (elect_one()) {
              // h tap dh = j - 1: output line l reads tile line l + j
              const uint64_t adesc = desc_hi | (uint64_t)(a0 + (uint32_t)stage * a_step + (uint32_t)j * line_units);
              const uint64_t bdesc = desc_hi | (uint64_t)(b0 + (uint32_t)sb * b_step);
#pragma unroll
              for (int k = 0; k < KC / 16; ++k)
                umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (i | j | k) != 0 ? 1u : 0u);
              umma_commit(&empty_b[sb]);
              if (j == 2) {
                umma_commit(&empty[stage]);
                if (i == n_items - 1) umma_commit(&tmem_full[acc]);
              }
            }
            __syncwarp();
            if (++sb == p.stages_b) { sb = 0; pb ^= 1; }
          }
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    } else
    for (long long work = blockIdx.x; work < p.total_tiles * p.splits; work += gridDim.x, ++it) {
      const int split = (int)(work / p.total_tiles);
      const int n_stage_per_tile = (27 * (split + 1) / p.splits - 27 * split / p.splits) * p.n_chunks;
      const uint32_t acc = it & 1u;
      const uint32_t acc_phase = (it >> 1) & 1u;
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * kAccStride;
      for (int ks = 0; ks < n_stage_per_tile; ++ks) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t adesc = desc_hi | (uint64_t)(a0 + (uint32_t)stage * a_step);
          const uint64_t bdesc = desc_hi | (uint64_t)(b0 + (uint32_t)stage * b_step);
#pragma unroll
          for (int k = 0; k < KC / 16; ++k)   // +32 bytes along K inside the swizzle atom = +2 in the encoded address
            umma_bf16(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (ks | k) != 0 ? 1u : 0u);
          umma_commit(&empty[stage]);
          if (ks == n_stage_per_tile - 1) umma_commit(&tmem_full[acc]);
        }
        __syncwarp();
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 9..12)
    const int q = warp & 3;            // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;     // accumulator row == voxel within the box
    const int lw = row % p.bw;
    const int lh = (row / p.bw) % p.bh;
    const int ld = row / (p.bw * p.bh);
    float st_s[8], st_q[8];   // lane L: running sums of channel chunk*32 + L over this warp's rows, all tiles
#pragma unroll
    for (int i = 0; i < 8; ++i) { st_s[i] = 0.f; st_q[i] = 0.f; }
    uint32_t it = 0;
    for (long long work = blockIdx.x; work < p.total_tiles * p.splits; work += gridDim.x, ++it) {
      int n, d0, h0, w0, n0;
      decode_tile(work % p.total_tiles, p, n, d0, h0, w0, n0);
      float* y32 = p.y32 ? p.y32 + (work / p.total_tiles) * p.split_stride : nullptr;
      const uint32_t acc = it & 1u;
      const uint32_t acc_phase = (it >> 1) & 1u;
      const int w = w0 + lw, h = h0 + lh, d = d0 + ld;
      const bool valid = (w < p.W) && (h < p.H) && (d < p.D);
      const size_t vox = (((size_t)n * p.D + d) * p.H + h) * p.W + w;
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * kAccStride;
#pragma unroll
      for (int chunk = 0; chunk < 8; ++chunk) {
        const int c0 = chunk * 32;
        if (c0 >= p.BN) break;
        // 16 in the last chunk when BN = 16 x odd: columns 16..31 are not this tile's.  Only the stores are cut to them;
        // the statistics of those columns land in lanes 16..31 of the column sums, which are never committed.
        const int ncol = p.BN - c0 < 32 ? p.BN - c0 : 32;
        uint32_t v[32];
        tmem_ld32(t_addr + c0, v);
        tmem_ld_wait();
        if (p.bias != nullptr) {   // warp-uniform; columns past ncol (BN = 16 x odd) re-read column 0 and are never used
#pragma unroll
          for (int e = 0; e < 32; ++e)
            v[e] = __float_as_uint(__uint_as_float(v[e]) + __ldg(p.bias + n0 + c0 + (e < ncol ? e : 0)));
        }
        if (p.stat_acc != nullptr) {   // warp-uniform branch
          float xs[32], xq[32];
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            float f = __uint_as_float(v[e]);
            if (p.relu) f = relu_nan(f);
            f = valid ? __bfloat162float(__float2bfloat16_rn(f)) : 0.f;   // statistics of what is stored
            xs[e] = f;
            xq[e] = f * f;
          }
          if (p.stat_r != nullptr) {   // backward statistics: second sum is dy * r
            const uint4* rp = reinterpret_cast<const uint4*>(p.stat_r + vox * p.Cout + n0 + c0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 u = make_uint4(0, 0, 0, 0);
              if (valid) u = __ldg(rp + (j & ((ncol >> 3) - 1)));   // ncol = 16: columns 16..31 re-read 0..15
              const uint32_t wds[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                xq[8 * j + 2 * e] = xs[8 * j + 2 * e] * __uint_as_float(wds[e] << 16);
                xq[8 * j + 2 * e + 1] = xs[8 * j + 2 * e + 1] * __uint_as_float(wds[e] & 0xffff0000u);
              }
            }
          }
          warp_column_sums(xs, lane);
          warp_column_sums(xq, lane);
          st_s[chunk] += xs[0];
          st_q[chunk] += xq[0];
        }
        if (valid) {
          if (y32 != nullptr) {
            float4* dst = reinterpret_cast<float4*>(y32 + vox * p.ldy + p.y_coff + n0 + c0);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              if (4 * j >= ncol) break;
              float4 o;
              o.x = __uint_as_float(v[4 * j + 0]);
              o.y = __uint_as_float(v[4 * j + 1]);
              o.z = __uint_as_float(v[4 * j + 2]);
              o.w = __uint_as_float(v[4 * j + 3]);
              if (p.relu) {
                o.x = relu_nan(o.x); o.y = relu_nan(o.y); o.z = relu_nan(o.z); o.w = relu_nan(o.w);
              }
              dst[j] = o;
            }
          } else {
            uint4* dst = reinterpret_cast<uint4*>(p.y + vox * p.ldy + p.y_coff + n0 + c0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              if (8 * j >= ncol) break;
              float f[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) {
                f[e] = __uint_as_float(v[8 * j + e]);
                if (p.relu) f[e] = relu_nan(f[e]);
              }
              uint4 o;
              o.x = pack_bf16x2(f[0], f[1]);
              o.y = pack_bf16x2(f[2], f[3]);
              o.z = pack_bf16x2(f[4], f[5]);
              o.w = pack_bf16x2(f[6], f[7]);
              dst[j] = o;
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tmem_empty[acc]);
    }
    if (p.stat_acc != nullptr) {
      // combine the four epilogue warps through the (now idle) operand ring, then one exact atomic add per CTA
      float2* sbuf = reinterpret_cast<float2*>(smem_a);   // [4][Cout]
#pragma unroll
      for (int chunk = 0; chunk < 8; ++chunk)
        if (chunk * 32 + lane < p.BN) sbuf[q * p.Cout + chunk * 32 + lane] = make_float2(st_s[chunk], st_q[chunk]);
      asm volatile("bar.sync 1, 128;" ::: "memory");
      for (int c = q * 32 + lane; c < p.Cout; c += 128) {
        const float2 a = sbuf[c], b = sbuf[p.Cout + c], cc = sbuf[2 * p.Cout + c], d = sbuf[3 * p.Cout + c];
        stat_atomic_add(p.stat_acc + 4 * c, (a.x + b.x) + (cc.x + d.x));
        stat_atomic_add(p.stat_acc + 4 * c + 2, (a.y + b.y) + (cc.y + d.y));
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

// ------------------------------------------------------------------------------------------------------------------
// CTA-pair variant (cta_group::2) for the wide layers (BN >= 128, Cin % 64 == 0).
// The one-CTA kernel above needs a 16 KB A tile AND the full BN x 64 weight tile per 128 x BN x 64 MMA group, i.e.
// 94..128 B/clk/SM of L2 -> SM traffic against ~64 B/clk/SM delivered: those layers run at 1150..1300 TFLOP/s.  Here
// two CTAs of a cluster (one TPC) compute TWO adjacent 128-voxel tiles with one 256 x BN x 16 instruction stream issued
// by the leader; each CTA stages only its own A tile and HALF of the weight tile (the tensor cores read both halves
// through the pair's shared memory), so the L2 -> SM weight traffic per SM halves: 62..94 B/clk/SM.
// MEASURED (round 1, profiles/r01_bench_kernels_2cta.txt): correct (all conv parity tests pass) but 20-30 % SLOWER
// than the one-CTA kernel on every wide layer (dec1.conv1 fprop 1203 -> 894, dec0.conv1 fprop 1393 -> 1020, dec2.conv1
// dgrad 1317 -> 1062 TFLOP/s): the partner's half of the weight tile is read over the SM-to-SM path on every MMA, so
// the bytes an SM has to ingest per MMA do not go down, and the pair adds cross-CTA barrier latency.  Kept opt-in
// (B2_2CTA=1) as the starting point for a version that also splits A.
// Barriers: full[s] lives in the leader (4 arrivals: A- and B-loader of each CTA, transaction bytes of all four TMA
// loads); empty[s] / tmem_full[a] exist in both CTAs and are signalled by multicast tcgen05.commit; tmem_empty[a] lives
// in the leader and collects the 2 x 128 epilogue threads of the pair.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
conv3d_igemm2_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                     const IgemmParams p) {
  pdl_prologue();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int KC = 64;
  constexpr int kABytes = 128 * KC * 2;
  const int b_half = p.b_bytes;   // (BN / 2) x KC bf16: this CTA's half of the weight tile
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + (size_t)p.stages * kABytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + (size_t)p.stages * b_half);
  uint64_t* full = bars;
  uint64_t* empty = bars + p.stages;
  uint64_t* tmem_full = bars + 2 * p.stages;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int n_clusters = gridDim.x >> 1, cluster_id = blockIdx.x >> 1;
  const long long m_tiles = p.total_tiles / p.n_tiles_n;
  const long long n_work = ((m_tiles + 1) >> 1) * p.n_tiles_n;   // (pair of M tiles, N tile)

  if (warp == 1 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full[s], 4);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 256);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc_2cta(tmem_slot, 512);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp >= 1 && warp <= 2 * kProducerPairs) {
    // ------------------------------------------------------------------ TMA producers (both CTAs)
    const int me = (warp - 1) >> 1;
    const bool loads_a = ((warp - 1) & 1) == 0;
    uint32_t gs = 0;
    for (long long work = cluster_id; work < n_work; work += n_clusters) {
      long long mt = (work / p.n_tiles_n) * 2 + rank;
      if (mt >= m_tiles) mt = m_tiles - 1;   // odd tile count: the partner re-loads the last tile, stores nothing
      int n, d0, h0, w0, n0;
      decode_tile(mt * p.n_tiles_n + work % p.n_tiles_n, p, n, d0, h0, w0, n0);
      for (int tap = 0; tap < 27; ++tap) {
        const int dd = tap / 9 - 1, dh = (tap / 3) % 3 - 1, dw = tap % 3 - 1;
        for (int ch = 0; ch < p.n_chunks; ++ch, ++gs) {
          if ((int)(gs % kProducerPairs) != me) continue;
          const int stage = (int)(gs % (uint32_t)p.stages);
          const uint32_t phase = (gs / (uint32_t)p.stages) & 1u;
          mbar_wait(&empty[stage], phase ^ 1);
          if (elect_one()) {
            const uint32_t lead_full = mapa_shared(smem_u32(&full[stage]), 0);
            if (loads_a) {
              mbar_arrive_expect_tx_cluster(lead_full, (uint32_t)kABytes);
              tma_load_5d_2sm(smem_a + (size_t)stage * kABytes, &tmap_a, lead_full, ch * KC, w0 + dw, h0 + dh, d0 + dd,
                              n);
            } else {
              mbar_arrive_expect_tx_cluster(lead_full, (uint32_t)b_half);
              tma_load_2d_2sm(smem_b + (size_t)stage * b_half, &tmap_b, lead_full, ch * KC,
                              tap * p.Cout + n0 + (int)rank * (p.BN >> 1));
            }
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 0) {
    if (rank == 0) {
      // ---------------------------------------------------------------- MMA issuer (leader CTA only)
      const uint32_t idesc = make_idesc_bf16(256, (uint32_t)p.BN, 0, 0);
      const uint64_t desc_hi = make_smem_desc(0, 16, 8u * KC * 2u, SWZ_128B);
      const uint32_t a0 = smem_u32(smem_a) >> 4, b0 = smem_u32(smem_b) >> 4;
      const uint32_t a_step = kABytes >> 4, b_step = (uint32_t)b_half >> 4;
      const int n_stage_per_tile = 27 * p.n_chunks;
      int stage = 0;
      uint32_t phase = 0, it = 0;
      for (long long work = cluster_id; work < n_work; work += n_clusters, ++it) {
        const uint32_t acc = it & 1u;
        mbar_wait(&tmem_empty[acc], ((it >> 1) & 1u) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * kAccStride;
        for (int ks = 0; ks < n_stage_per_tile; ++ks) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t adesc = desc_hi | (uint64_t)(a0 + (uint32_t)stage * a_step);
            const uint64_t bdesc = desc_hi | (uint64_t)(b0 + (uint32_t)stage * b_step);
#pragma unroll
            for (int k = 0; k < KC / 16; ++k)
              umma_bf16_2cta(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (ks | k) != 0 ? 1u : 0u);
            umma_commit_2cta(&empty[stage], 3);
            if (ks == n_stage_per_tile - 1) umma_commit_2cta(&tmem_full[acc], 3);
          }
          __syncwarp();
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 9..12, both CTAs)
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const int lw = row % p.bw;
    const int lh = (row / p.bw) % p.bh;
    const int ld = row / (p.bw * p.bh);
    float st_s[8], st_q[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { st_s[i] = 0.f; st_q[i] = 0.f; }
    uint32_t it = 0;
    for (long long work = cluster_id; work < n_work; work += n_clusters, ++it) {
      const long long mt = (work / p.n_tiles_n) * 2 + rank;
      const bool tile_ok = mt < m_tiles;
      int n, d0, h0, w0, n0;
      decode_tile((tile_ok ? mt : m_tiles - 1) * p.n_tiles_n + work % p.n_tiles_n, p, n, d0, h0, w0, n0);
      const uint32_t acc = it & 1u;
      const int w = w0 + lw, h = h0 + lh, d = d0 + ld;
      const bool valid = tile_ok && (w < p.W) && (h < p.H) && (d < p.D);
      const size_t vox = (((size_t)n * p.D + d) * p.H + h) * p.W + w;
      mbar_wait(&tmem_full[acc], (it >> 1) & 1u);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * kAccStride;
#pragma unroll
      for (int chunk = 0; chunk < 8; ++chunk) {
        const int c0 = chunk * 32;
        if (c0 >= p.BN) break;
        uint32_t v[32];
        tmem_ld32(t_addr + c0, v);
        tmem_ld_wait();
        if (p.stat_acc != nullptr) {
          float xs[32], xq[32];
#pragma unroll
          for (int e = 0; e < 32; ++e) {
            float f = __uint_as_float(v[e]);
            if (p.relu) f = relu_nan(f);
            f = valid ? __bfloat162float(__float2bfloat16_rn(f)) : 0.f;
            xs[e] = f;
            xq[e] = f * f;
          }
          if (p.stat_r != nullptr) {
            const uint4* rp = reinterpret_cast<const uint4*>(p.stat_r + vox * p.Cout + n0 + c0);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              uint4 u = make_uint4(0, 0, 0, 0);
              if (valid) u = __ldg(rp + j);
              const uint32_t wds[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                xq[8 * j + 2 * e] = xs[8 * j + 2 * e] * __uint_as_float(wds[e] << 16);
                xq[8 * j + 2 * e + 1] = xs[8 * j + 2 * e + 1] * __uint_as_float(wds[e] & 0xffff0000u);
              }
            }
          }
          warp_column_sums(xs, lane);
          warp_column_sums(xq, lane);
          st_s[chunk] += xs[0];
          st_q[chunk] += xq[0];
        }
        if (valid) {
          uint4* dst = reinterpret_cast<uint4*>(p.y + vox * p.ldy + p.y_coff + n0 + c0);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            float f[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              f[e] = __uint_as_float(v[8 * j + e]);
              if (p.relu) f[e] = relu_nan(f[e]);
            }
            uint4 o;
            o.x = pack_bf16x2(f[0], f[1]);
            o.y = pack_bf16x2(f[2], f[3]);
            o.z = pack_bf16x2(f[4], f[5]);
            o.w = pack_bf16x2(f[6], f[7]);
            dst[j] = o;
          }
        }
      }
      tc_fence_before();
      mbar_arrive_cluster(mapa_shared(smem_u32(&tmem_empty[acc]), 0));   // the leader's MMA issuer owns the pair's TMEM
    }
    if (p.stat_acc != nullptr) {
      // all MMAs that read this CTA's operand ring are complete (tmem_full of the last tile): reuse it as scratch
      float2* sbuf = reinterpret_cast<float2*>(smem_a);   // [4][Cout]
#pragma unroll
      for (int chunk = 0; chunk < 8; ++chunk)
        if (chunk * 32 < p.BN) sbuf[q * p.Cout + chunk * 32 + lane] = make_float2(st_s[chunk], st_q[chunk]);
      asm volatile("bar.sync 1, 128;" ::: "memory");
      for (int c = q * 32 + lane; c < p.Cout; c += 128) {
        const float2 a = sbuf[c], b = sbuf[p.Cout + c], cc = sbuf[2 * p.Cout + c], d = sbuf[3 * p.Cout + c];
        stat_atomic_add(p.stat_acc + 4 * c, (a.x + b.x) + (cc.x + d.x));
        stat_atomic_add(p.stat_acc + 4 * c + 2, (a.y + b.y) + (cc.y + d.y));
      }
    }
  }

  tc_fence_before();
  cluster_sync_all();   // the partner's shared memory and TMEM stay alive until both CTAs are done
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, 512);
  }
}

// out[v, c] = (relu)(sum_s partial[s][v][c] (+ bias[c])) -> bf16 channel window; the partials carry no bias
__global__ void __launch_bounds__(256)
conv_splitk_reduce_kernel(const float* __restrict__ partial, int splits, long long split_stride, long long NV, int C,
                          int relu, __nv_bfloat16* __restrict__ y, int ldy, int y_coff, const float* __restrict__ bias) {
  pdl_prologue();
  const int C4 = C >> 2;
  const long long total = NV * C4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long v = i / C4;
    const int c = (int)(i % C4) * 4;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < splits; ++s) {
      const float4 t = *reinterpret_cast<const float4*>(partial + s * split_stride + v * C + c);
      a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
    }
    if (bias != nullptr) { a.x += bias[c]; a.y += bias[c + 1]; a.z += bias[c + 2]; a.w += bias[c + 3]; }
    if (relu) { a.x = relu_nan(a.x); a.y = relu_nan(a.y); a.z = relu_nan(a.z); a.w = relu_nan(a.w); }
    uint2 o;
    o.x = pack_bf16x2(a.x, a.y);
    o.y = pack_bf16x2(a.z, a.w);
    *reinterpret_cast<uint2*>(y + v * ldy + y_coff + c) = o;
  }
}

// choose the (bw, bh, bd) box with bw*bh*bd == 128 that wastes the fewest padded voxels
static void choose_box(int W, int H, int D, int& bw, int& bh, int& bd) {
  long long best = -1;
  for (int lw = 0; lw <= 7; ++lw)
    for (int lh = 0; lw + lh <= 7; ++lh) {
      const int ld = 7 - lw - lh;
      const int cw = 1 << lw, chh = 1 << lh, cd = 1 << ld;
      const long long cost = (long long)ceil_div(W, cw) * cw * (long long)ceil_div(H, chh) * chh *
                             (long long)ceil_div(D, cd) * cd;
      // tie-break: longer contiguous W runs, then H
      const long long score = cost * 1024 - cw * 8 - chh;
      if (best < 0 || score < best) {
        best = score;
        bw = cw;
        bh = chh;
        bd = cd;
      }
    }
}

bool slab_applicable(int N, int D, int H, int W, int Cin, int Cout, int y_is_fp32);
int launch_slab(const void* x, int ldx, int x_coff, const void* wpack, void* y, int ldy, int y_coff, int N, int D,
                int H, int W, int Cin, int Cout, int relu, long long* stat_acc, const void* stat_r, const float* bias,
                cudaStream_t stream);

int make_act_tmap(CUtensorMap* map, const void* base, int N, int D, int H, int W, int C, int ld, int coff,
                  int box_c, int bw, int bh, int bd) {
  const uint64_t dims[5] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)D, (uint64_t)N};
  const uint64_t e = 2;
  const uint64_t strides[4] = {(uint64_t)ld * e, (uint64_t)W * ld * e, (uint64_t)H * W * ld * e,
                               (uint64_t)D * H * W * ld * e};
  const uint32_t box[5] = {(uint32_t)box_c, (uint32_t)bw, (uint32_t)bh, (uint32_t)bd, 1};
  const __nv_bfloat16* b = reinterpret_cast<const __nv_bfloat16*>(base) + coff;
  return encode_tmap_bf16(map, b, 5, dims, strides, box, box_c * 2);
}

// same 5-D NDHWC channel-window map without shared-memory swizzle (bandwidth kernels that read the box with plain LDS)
int make_act_tmap_plain(CUtensorMap* map, const void* base, int N, int D, int H, int W, int C, int ld, int coff,
                        int box_c, int bw, int bh, int bd) {
  const uint64_t dims[5] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)D, (uint64_t)N};
  const uint64_t e = 2;
  const uint64_t strides[4] = {(uint64_t)ld * e, (uint64_t)W * ld * e, (uint64_t)H * W * ld * e,
                               (uint64_t)D * H * W * ld * e};
  const uint32_t box[5] = {(uint32_t)box_c, (uint32_t)bw, (uint32_t)bh, (uint32_t)bd, 1};
  const __nv_bfloat16* b = reinterpret_cast<const __nv_bfloat16*>(base) + coff;
  return encode_tmap_bf16(map, b, 5, dims, strides, box, 0);
}

}  // namespace b2

using namespace b2;

// See include/unetsulc_b200.h for the contract.
static int conv3d_igemm_impl(const void* x, int ldx, int x_coff, const void* wpack, void* y, int ldy, int y_coff,
                             int y_is_fp32, int N, int D, int H, int W, int Cin, int Cout, int relu,
                             long long* stat_acc, const void* stat_r, void* splitk_workspace,
                             long long splitk_workspace_bytes, const float* bias, cudaStream_t stream) {
  B2_REQUIRE(x && wpack && y, "b2_conv3d_igemm: null pointer");
  B2_REQUIRE(N > 0 && D > 0 && H > 0 && W > 0, "b2_conv3d_igemm: bad shape %dx%dx%dx%d", N, D, H, W);
  B2_REQUIRE(Cin % 16 == 0 && Cin >= 16, "b2_conv3d_igemm: Cin=%d must be a multiple of 16", Cin);
  B2_REQUIRE(Cout % 16 == 0 && Cout >= 16, "b2_conv3d_igemm: Cout=%d must be a multiple of 16", Cout);
  B2_REQUIRE(ldx % 8 == 0 && x_coff % 8 == 0 && ldy % 8 == 0 && y_coff % 8 == 0,
             "b2_conv3d_igemm: channel strides/offsets must be multiples of 8");
  B2_REQUIRE(x_coff + Cin <= ldx && y_coff + Cout <= ldy, "b2_conv3d_igemm: channel window out of range");

  // narrow-N layers at (almost) tile-aligned resolutions: shared-memory tap-reuse kernel (conv_slab.cu)
  static const bool no_slab = getenv("B2_NO_SLAB") != nullptr;
  if (!no_slab && slab_applicable(N, D, H, W, Cin, Cout, y_is_fp32))
    return launch_slab(x, ldx, x_coff, wpack, y, ldy, y_coff, N, D, H, W, Cin, Cout, relu, stat_acc, stat_r, bias,
                       stream);

  IgemmParams p;
  p.N = N; p.D = D; p.H = H; p.W = W; p.Cin = Cin; p.Cout = Cout;
  choose_box(W, H, D, p.bw, p.bh, p.bd);
  p.tiles_w = ceil_div(W, p.bw);
  p.tiles_h = ceil_div(H, p.bh);
  p.tiles_d = ceil_div(D, p.bd);
  // N tile: largest divisor of Cout that is a multiple of 32 and <= 256; for Cout = 16 x odd (16, 48, ...) the largest
  // such divisor that is a multiple of 16 (the epilogue stores the last 16 columns of a 32-column chunk alone)
  int BN = 0;
  for (int c = 256; c >= 32; c -= 32)
    if (Cout % c == 0) { BN = c; break; }
  for (int c = 256; BN == 0 && c >= 16; c -= 16)
    if (Cout % c == 0) BN = c;
  B2_REQUIRE(BN > 0, "b2_conv3d_igemm: no N tile for Cout=%d", Cout);
  p.BN = BN;
  p.n_tiles_n = Cout / BN;
  p.KC = (Cin % 64 == 0) ? 64 : (Cin % 32 == 0 ? 32 : 16);
  p.n_chunks = Cin / p.KC;
  p.a_bytes = 128 * p.KC * 2;
  p.b_bytes = BN * p.KC * 2;
  const int smem_budget = 227 * 1024 - 1024 /*align*/ - 512 /*barriers*/;
  p.stages = smem_budget / (p.a_bytes + p.b_bytes);
  if (p.stages > 12) p.stages = 12;
  // every stage has a fixed producer pair (stage mod kProducerPairs), so that no producer can run two ring
  // phases ahead of the consumer
  p.stages = (p.stages / kProducerPairs) * kProducerPairs;
  B2_REQUIRE(p.stages >= kProducerPairs, "b2_conv3d_igemm: tile does not fit shared memory");
  p.relu = relu;
  p.ldy = ldy; p.y_coff = y_coff;
  p.y = y_is_fp32 ? nullptr : reinterpret_cast<__nv_bfloat16*>(y);
  p.y32 = y_is_fp32 ? reinterpret_cast<float*>(y) : nullptr;
  const int user_ldy = ldy, user_coff = y_coff, user_relu = relu;
  p.total_tiles = (long long)N * p.tiles_d * p.tiles_h * p.tiles_w * p.n_tiles_n;
  p.splits = 1;
  p.split_stride = 0;
  // split-K over taps when the layer has too few tiles to fill the machine (needs a caller-provided fp32 workspace)
  float* splitk_ws = nullptr;
  if (!y_is_fp32 && !stat_acc && splitk_workspace && p.total_tiles * 2 <= num_sms()) {
    int sp = (int)(num_sms() / p.total_tiles);
    if (sp > 9) sp = 9;
    const long long need = (long long)sp * N * D * H * W * Cout * (long long)sizeof(float);
    if (sp >= 2 && need <= splitk_workspace_bytes) {
      p.splits = sp;
      p.split_stride = (long long)N * D * H * W * Cout;
      splitk_ws = reinterpret_cast<float*>(splitk_workspace);
    }
  }
  p.stat_acc = stat_acc;
  p.stat_r = reinterpret_cast<const __nv_bfloat16*>(stat_r);
  p.bias = bias;
  if (stat_acc) {
    B2_REQUIRE(N == 1 && p.n_tiles_n == 1 && !y_is_fp32,
               "b2_conv3d_igemm_stats: fused statistics need batch 1, Cout <= 256 and a bf16 output");
  }

  CUtensorMap ta, tb;
  int rc = make_act_tmap(&ta, x, N, D, H, W, Cin, ldx, x_coff, p.KC, p.bw, p.bh, p.bd);
  if (rc) return rc;
  {
    const uint64_t dims[2] = {(uint64_t)Cin, (uint64_t)27 * Cout};
    const uint64_t strides[1] = {(uint64_t)Cin * 2};
    const uint32_t box[2] = {(uint32_t)p.KC, (uint32_t)BN};
    rc = encode_tmap_bf16(&tb, wpack, 2, dims, strides, box, p.KC * 2);
    if (rc) return rc;
  }
  // wide layers: CTA pairs (each CTA stages half of the weight tile), see conv3d_igemm2_kernel.  Opt-in (B2_2CTA=1):
  // bit-identical results, but measured SLOWER than the one-CTA kernel on B200 in round 1
  // (profiles/r01_bench_kernels_2cta.txt).  Biased launches stay on the one-CTA kernels, whose epilogue adds the bias.
  static const bool no_pairs = getenv("B2_2CTA") == nullptr;
  const long long m_tiles = p.total_tiles / p.n_tiles_n;
  if (!no_pairs && !bias && p.KC == 64 && BN >= 128 && p.splits == 1 && !y_is_fp32 && m_tiles >= 8) {
    p.b_bytes = (BN / 2) * p.KC * 2;
    p.stages = smem_budget / (p.a_bytes + p.b_bytes);
    if (p.stages > 12) p.stages = 12;
    p.stages = (p.stages / kProducerPairs) * kProducerPairs;
    const uint64_t dims[2] = {(uint64_t)Cin, (uint64_t)27 * Cout};
    const uint64_t strides[1] = {(uint64_t)Cin * 2};
    const uint32_t box[2] = {(uint32_t)p.KC, (uint32_t)(BN / 2)};
    rc = encode_tmap_bf16(&tb, wpack, 2, dims, strides, box, p.KC * 2);
    if (rc) return rc;
    const size_t smem2 = (size_t)p.stages * (p.a_bytes + p.b_bytes) + 1024 + 512;
    B2_CHECK_CUDA(cudaFuncSetAttribute(conv3d_igemm2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    const long long n_work = ((m_tiles + 1) / 2) * p.n_tiles_n;
    const long long clusters = n_work < num_sms() / 2 ? n_work : num_sms() / 2;
    B2_LAUNCH(conv3d_igemm2_kernel, (unsigned)(2 * clusters), kThreads, smem2, stream, ta, tb, p);
    B2_CHECK_CUDA(cudaGetLastError());
    return B2_OK;
  }
  // h-halo variant (see the kernel): 64-channel chunks, no split-K, one-plane tile boxes.  B2_IGEMM_HALO = widest N
  // tile that takes it (0: never).  Measured (us, plain -> halo): decoders.2.conv1 dgrad 529 -> 472, decoders.1.conv1
  // fprop 286 -> 275, dgrad 254 -> 247, decoders.1.conv2 105 -> 101, encoders.2.conv2 dgrad 41 -> 36.
  static const int halo_mode = getenv("B2_IGEMM_HALO") ? atoi(getenv("B2_IGEMM_HALO")) : 256;
  if (halo_mode > 0 && p.KC == 64 && p.splits == 1 && BN <= halo_mode) {
    // box with whole swizzle atoms per line (bw % 8 == 0): least padding first, then the smallest halo (largest bh)
    long long best = -1;
    int hbw = 8, hbh = 16;
    for (int cw = 8; cw <= 32; cw *= 2) {
      const int chh = 128 / cw;
      const long long cost = (long long)ceil_div(W, cw) * cw * ceil_div(H, chh) * chh * 64 - chh;
      if (best < 0 || cost < best) { best = cost; hbw = cw; hbh = chh; }
    }
    const int a_halo = (hbh + 2) * hbw * 128;
    int stages_b = (smem_budget - kProducerPairs * a_halo) / p.b_bytes;
    if (stages_b > 12) stages_b = 12;
    stages_b = (stages_b / kProducerPairs) * kProducerPairs;
    if (stages_b >= kProducerPairs) {
      p.bw = hbw; p.bh = hbh; p.bd = 1;
      p.tiles_w = ceil_div(W, p.bw);
      p.tiles_h = ceil_div(H, p.bh);
      p.tiles_d = D;
      p.total_tiles = (long long)N * p.tiles_d * p.tiles_h * p.tiles_w * p.n_tiles_n;
      p.a_bytes = a_halo;
      p.stages = kProducerPairs;
      p.stages_b = stages_b;
      rc = make_act_tmap(&ta, x, N, D, H, W, Cin, ldx, x_coff, p.KC, p.bw, p.bh + 2, p.bd);
      if (rc) return rc;
      const size_t smem_h = (size_t)p.stages * p.a_bytes + (size_t)p.stages_b * p.b_bytes + 1024 + 512;
      const long long grid_h = p.total_tiles < num_sms() ? p.total_tiles : num_sms();
      B2_CHECK_CUDA(cudaFuncSetAttribute((conv3d_igemm_kernel<64, true>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         227 * 1024));
      B2_LAUNCH((conv3d_igemm_kernel<64, true>), (unsigned)grid_h, kThreads, smem_h, stream, ta, tb, p);
      B2_CHECK_CUDA(cudaGetLastError());
      return B2_OK;
    }
  }
  const size_t smem_bytes = (size_t)p.stages * (p.a_bytes + p.b_bytes) + 1024 + 512;
  if (p.splits > 1) {   // partial tiles: dense fp32 [split][voxel][Cout], no ReLU before the reduction
    p.y = nullptr;
    p.y32 = splitk_ws;
    p.ldy = Cout;
    p.y_coff = 0;
    p.relu = 0;
    p.bias = nullptr;
  }
  const long long work_items = p.total_tiles * p.splits;
  long long grid = work_items < num_sms() ? work_items : num_sms();
  if (p.KC == 64) {
    B2_CHECK_CUDA(cudaFuncSetAttribute((conv3d_igemm_kernel<64, false>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       227 * 1024));
    B2_LAUNCH((conv3d_igemm_kernel<64, false>), (unsigned)grid, kThreads, smem_bytes, stream, ta, tb, p);
  } else if (p.KC == 32) {
    B2_CHECK_CUDA(cudaFuncSetAttribute((conv3d_igemm_kernel<32, false>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       227 * 1024));
    B2_LAUNCH((conv3d_igemm_kernel<32, false>), (unsigned)grid, kThreads, smem_bytes, stream, ta, tb, p);
  } else {
    B2_CHECK_CUDA(cudaFuncSetAttribute((conv3d_igemm_kernel<16, false>), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       227 * 1024));
    B2_LAUNCH((conv3d_igemm_kernel<16, false>), (unsigned)grid, kThreads, smem_bytes, stream, ta, tb, p);
  }
  B2_CHECK_CUDA(cudaGetLastError());
  if (p.splits > 1) {
    const long long NV = (long long)N * D * H * W;
    long long rb = (NV * (Cout / 4) + 255) / 256;
    if (rb > num_sms() * 8) rb = num_sms() * 8;
    B2_LAUNCH(conv_splitk_reduce_kernel, (unsigned)rb, 256, 0, stream, splitk_ws, p.splits, p.split_stride, NV, Cout,
                                                                user_relu, reinterpret_cast<__nv_bfloat16*>(y),
                                                                user_ldy, user_coff, bias);
    B2_CHECK_CUDA(cudaGetLastError());
  }
  return B2_OK;
}

// See include/unetsulc_b200.h for the contract.
extern "C" int b2_conv3d_igemm(const void* x, int ldx, int x_coff, const void* wpack, void* y, int ldy, int y_coff,
                               int y_is_fp32, int N, int D, int H, int W, int Cin, int Cout, int relu,
                               cudaStream_t stream) {
  return conv3d_igemm_impl(x, ldx, x_coff, wpack, y, ldy, y_coff, y_is_fp32, N, D, H, W, Cin, Cout, relu, nullptr,
                           nullptr, nullptr, 0, nullptr, stream);
}

// Same as b2_conv3d_igemm with an optional fp32 workspace: layers with fewer than num_SMs/2 output tiles are split
// over the 27 taps (split-K, up to 9 ways) into the workspace and reduced (+ReLU, bf16) by a second kernel.
extern "C" long long b2_conv3d_splitk_workspace_bytes(int N, int D, int H, int W, int Cout) {
  return 9LL * N * D * H * W * Cout * (long long)sizeof(float);
}
extern "C" int b2_conv3d_igemm_splitk(const void* x, int ldx, int x_coff, const void* wpack, void* y, int ldy,
                                      int y_coff, int N, int D, int H, int W, int Cin, int Cout, int relu,
                                      void* workspace, long long workspace_bytes, cudaStream_t stream) {
  return conv3d_igemm_impl(x, ldx, x_coff, wpack, y, ldy, y_coff, 0, N, D, H, W, Cin, Cout, relu, nullptr, nullptr,
                           workspace, workspace_bytes, nullptr, stream);
}

// fprop with the GroupNorm statistics of the stored (bf16-rounded, post-ReLU) output fused into the epilogue.
// stat_acc: int64 [Cout][4] fixed-point accumulators (zero before the launch; see common.h), consumed by
// b2_relu_gn_apply_acc.  Batch 1, Cout <= 256.
extern "C" int b2_conv3d_igemm_stats(const void* x, int ldx, int x_coff, const void* wpack, void* y, int ldy,
                                     int y_coff, int N, int D, int H, int W, int Cin, int Cout, int relu,
                                     long long* stat_acc, cudaStream_t stream) {
  B2_REQUIRE(stat_acc, "b2_conv3d_igemm_stats: null pointer");
  return conv3d_igemm_impl(x, ldx, x_coff, wpack, y, ldy, y_coff, 0, N, D, H, W, Cin, Cout, relu, stat_acc, nullptr,
                           nullptr, 0, nullptr, stream);
}

// dgrad (x = dY, wpack = dgrad pack, output dX written densely) with the GroupNorm-BACKWARD statistics of the layer
// that produced dX's forward tensor fused into the epilogue: per channel sum(dX) and sum(dX * r), r = that layer's
// stored relu(conv) (dense bf16 [V][Cout]).  Same accumulator layout; consumed by b2_relu_gn_bwd_apply_acc.
extern "C" int b2_conv3d_igemm_bstats(const void* x, int ldx, int x_coff, const void* wpack, void* y, int N, int D,
                                      int H, int W, int Cin, int Cout, const void* r, long long* stat_acc,
                                      cudaStream_t stream) {
  B2_REQUIRE(stat_acc && r, "b2_conv3d_igemm_bstats: null pointer");
  return conv3d_igemm_impl(x, ldx, x_coff, wpack, y, Cout, 0, 0, N, D, H, W, Cin, Cout, 0, stat_acc, r, nullptr, 0,
                           nullptr, stream);
}

// fprop of a layer with a conv bias (fp32 [Cout]): the bias joins the fp32 accumulator before ReLU in every path the
// launch can take (slab, plain / h-halo implicit GEMM, the fp32 output, the split-K reduction), so the stored output and
// the fused statistics (stat_acc, optional: batch 1, Cout <= 256) see conv + bias.  splitk_workspace is optional.
extern "C" int b2_conv3d_igemm_bias(const void* x, int ldx, int x_coff, const void* wpack, void* y, int ldy, int y_coff,
                                    int y_is_fp32, int N, int D, int H, int W, int Cin, int Cout, int relu,
                                    const float* bias, long long* stat_acc, void* splitk_workspace,
                                    long long splitk_workspace_bytes, cudaStream_t stream) {
  B2_REQUIRE(bias && (reinterpret_cast<uintptr_t>(bias) & 7) == 0, "b2_conv3d_igemm_bias: bias must be 8-byte aligned");
  return conv3d_igemm_impl(x, ldx, x_coff, wpack, y, ldy, y_coff, y_is_fp32, N, D, H, W, Cin, Cout, relu, stat_acc,
                           nullptr, stat_acc ? nullptr : splitk_workspace, splitk_workspace_bytes, bias, stream);
}
