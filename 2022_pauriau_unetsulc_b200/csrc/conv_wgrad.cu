// Weight gradient of the 3x3x3 stride-1 pad-1 Conv3d on tcgen05 (sm_100a).
//
//   dW[co][ci][tap] = sum_v dY[v, co] * X[v + off(tap), ci]                       (NDHWC bf16, fp32 accumulate)
//
// GEMM view: the reduction (K) runs over voxels, so both operands sit in shared memory "MN-major":
// a TMA box load of 128 voxels x 64 channels lands as [voxel row][128 B of channels], 128B-swizzled, which is
// exactly the canonical MN-major UMMA layout (64-element atoms along M/N at stride LBO, 8-voxel groups along K
// at stride SBO).  A = shifted X tiles ("slots" = (tap, 64-channel chunk); 128/SWC slots stacked along M),
// B = the un-shifted dY tile (N = BN output channels, loaded once per 128-voxel K-step and reused by every
// slot group).  Each CTA owns up to 512/BN accumulators (slot groups) in TMEM and a contiguous range of
// K-steps; partial results go to a fp32 workspace [split][tap][ci][co] and a second kernel reduces the splits
// deterministically into PyTorch's [co][ci][kd][kh][kw] layout.
//
// Round 2 added two planning modes (plan_wgrad): the "dY-halo" mode for Cout <= 128 at one-plane tile boxes — X is
// shifted only in (d, w), the three h taps are three N atoms of ONE dY tile loaded with an h-halo (N = 192 per MMA) —
// and stream-K runs when a uniform K split would leave SMs idle (wgrad_segment).
// 32-filter networks add Cin = 16 slots (32-byte rows, 32B swizzle, 8 slots per 128-row group) and Cout = 32 dY tiles
// (64-byte rows, 64B swizzle; in halo mode three 32-channel atoms, N = 96).
#include "common.h"
#include "ptx.cuh"
#include <stdlib.h>

namespace b2 {

int make_act_tmap(CUtensorMap* map, const void* base, int N, int D, int H, int W, int C, int ld, int coff,
                  int box_c, int bw, int bh, int bd);

struct WgradParams {
  int N, D, H, W;
  int Cin, Cout;
  int bw, bh, bd;
  int tiles_w, tiles_h, tiles_d;
  int SWC, n_cchunks, total_slots, SPG;  // slot width (channels), chunks per tap, slots, slots per group
  int G, gpc, n_gchunks;                 // groups, groups per CTA chunk, number of chunks
  int BN, n_cout_tiles;
  int splits;
  long long ksteps_total;
  int stages_a, n_prod;   // ring depth (a multiple of n_prod) and number of active slot-group producers
  int a_bytes, b_bytes, slot_bytes;
  int halo;        // "dY-halo" mode (BN-channel N tiles read as three h-shifted atoms): see plan_wgrad
  int d_fast;      // K-step order (w, d, h) instead of (w, h, d): see wgrad_tile
  int stages_b;    // depth of the fixed-operand ring (2-4)
  int grid;        // CTAs launched
  int streamk;     // CTAs own equal runs of the column-major (column, K-step) plane: see wgrad_segment
  float* ws;
};

// warp 0: MMA issuer (+TMEM owner); warps 1-4: TMA producers of the slot-group ring (stage s by producer s mod 4);
// warp 5: TMA producer of the dY ring; warps 6-9: epilogue.  (One thread retires only one TMA op per ~735 cycles on
// B200, ops of different warps run in parallel: tools/micro/tma_bench2.cu.)
static constexpr int kWgProducers = 4;
static constexpr int kWgThreads = 32 * (1 + kWgProducers + 1 + 4);

// K-step -> tile origin.  A split owns a contiguous range of K-steps, i.e. a slab of the volume, and re-reads the
// neighbouring planes / lines its shifted boxes touch.  Default order (w, h, d): slabs of whole planes.  Halo mode
// shifts X only in (d, w), so with the order (w, d, h) a split is a band of h-lines through ALL planes: the d +- 1
// planes of one tile are the next tiles of the same CTA (L2 hits) and no X line is fetched by two splits (measured:
// decoders.2.conv2 read 691 MB from DRAM with 59 plane-slabs of 1.6 planes each, 264 MB being the operands).
__device__ __forceinline__ void wgrad_tile(long long t, const WgradParams& p, int& n, int& d0, int& h0, int& w0) {
  w0 = (int)(t % p.tiles_w) * p.bw;
  t /= p.tiles_w;
  if (p.d_fast) {
    d0 = (int)(t % p.tiles_d) * p.bd;
    t /= p.tiles_d;
    h0 = (int)(t % p.tiles_h) * p.bh;
    n = (int)(t / p.tiles_h);
  } else {
    h0 = (int)(t % p.tiles_h) * p.bh;
    t /= p.tiles_h;
    d0 = (int)(t % p.tiles_d) * p.bd;
    n = (int)(t / p.tiles_d);
  }
}

// One unit of work of a CTA: the K-steps [t0, t1) of the group chunk `gchunk` x cout tile `nt`; the partial goes to
// split slice `layer`, zeros to the slices (layer, zero_to).
struct WgSegment {
  int gchunk, nt, layer, zero_to;
  long long t0, t1;
};

// Two ways a 1-D grid covers the (chunk x cout tile) columns x K-steps plane:
//  * uniform splits: CTA = (column, split), every column cut into p.splits equal K ranges;
//  * stream-K (p.streamk; columns > SMs / 2, where a uniform split would leave SMs idle — decoders.0.conv1: 81 columns):
//    the plane is linearised column-major and cut into gridDim.x equal runs; a run touches at most two columns
//    (= two segments, run one after the other), a column collects 2-3 partials in slice order of arrival; the last
//    contributor zero-fills the slices its column does not use.
// (Measured and dropped: CTAs of a short last chunk covering two splits each, to even out the MMA count — they then
// load more bytes per MMA than the others and become the critical path: decoders.2.conv2 245 vs 212 us.)
__device__ __forceinline__ bool wgrad_segment(const WgradParams& p, int sg, WgSegment& s) {
  if (p.streamk) {
    const long long K = p.ksteps_total, total = K * p.n_gchunks * p.n_cout_tiles;
    const long long a = total * blockIdx.x / gridDim.x, b = total * (blockIdx.x + 1) / gridDim.x;
    const long long col0 = a / K, col1 = (b - 1) / K;
    if (sg > (int)(col1 - col0)) return false;
    const long long col = col0 + sg;
    s.t0 = (sg == 0 ? a : col * K) - col * K;
    s.t1 = (b < (col + 1) * K ? b : (col + 1) * K) - col * K;
    s.gchunk = (int)(col % p.n_gchunks);
    s.nt = (int)(col / p.n_gchunks);
    // first CTA whose run holds K-step col*K: the largest j with floor(j * total / grid) <= col * K
    const long long first = ((col * K + 1) * gridDim.x - 1) / total;
    s.layer = (int)(blockIdx.x - first);
    s.zero_to = (b >= (col + 1) * K) ? p.splits : s.layer + 1;
    return true;
  }
  if (sg > 0) return false;
  const int columns = p.n_gchunks * p.n_cout_tiles;
  s.gchunk = (int)blockIdx.x % columns % p.n_gchunks;
  s.nt = (int)blockIdx.x % columns / p.n_gchunks;
  s.layer = (int)blockIdx.x / columns;
  s.zero_to = s.layer + 1;
  s.t0 = p.ksteps_total * s.layer / p.splits;
  s.t1 = p.ksteps_total * s.zero_to / p.splits;
  return true;
}

__global__ void __launch_bounds__(kWgThreads, 1)
conv3d_wgrad_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_dy,
                    const WgradParams p) {
  pdl_wait();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_b = smem;                                          // stages_b x dY tile
  uint8_t* smem_a = smem + (size_t)p.stages_b * p.b_bytes;         // stages_a x slot group
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_a + (size_t)p.stages_a * p.a_bytes);
  uint64_t* full_a = bars;
  uint64_t* empty_a = bars + p.stages_a;
  uint64_t* full_b = bars + 2 * p.stages_a;
  uint64_t* empty_b = full_b + p.stages_b;
  uint64_t* acc_full = empty_b + p.stages_b;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // warp-uniform by construction
  const int lane = threadIdx.x & 31;

  if (warp == 1 && lane == 0) {
    tma_prefetch_desc(&tmap_x);
    tma_prefetch_desc(&tmap_dy);
    for (int s = 0; s < p.stages_a; ++s) {
      mbar_init(&full_a[s], 1);
      mbar_init(&empty_a[s], 1);
    }
    for (int s = 0; s < p.stages_b; ++s) {
      mbar_init(&full_b[s], 1);
      mbar_init(&empty_b[s], 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, 128);   // every epilogue thread arrives once it has read its accumulator rows
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Role loops run on the whole warp with warp-uniform control flow; only the TMA / tcgen05 instruction itself is
  // issued by an elected lane (keeps descriptors and addresses in uniform registers, see conv_igemm.cu).
  WgSegment seg;
  if (warp >= 1 && warp <= kWgProducers) {
    // ---------------------------------------------------------------- producers of the shifted-X slot groups
    const int me = warp - 1;
    uint32_t ga = 0;
    for (int sg = 0; wgrad_segment(p, sg, seg); ++sg) {
      const int g_begin = seg.gchunk * p.gpc, g_end = min(g_begin + p.gpc, p.G);
      for (long long t = seg.t0; t < seg.t1; ++t) {
        int n, d0, h0, w0;
        wgrad_tile(t, p, n, d0, h0, w0);
        for (int g = g_begin; g < g_end; ++g, ++ga) {
          if ((int)(ga % (uint32_t)p.n_prod) != me) continue;   // stage s is always filled by producer s mod n_prod
          const int sa = (int)(ga % (uint32_t)p.stages_a);
          const uint32_t pa = (ga / (uint32_t)p.stages_a) & 1u;
          mbar_wait(&empty_a[sa], pa ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&full_a[sa], (uint32_t)p.a_bytes);
            for (int j = 0; j < p.SPG; ++j) {
              int s = g * p.SPG + j;
              if (s >= p.total_slots) s = p.total_slots - 1;  // padding slot: result discarded
              const int tap = s / p.n_cchunks, cc = s % p.n_cchunks;
              // halo mode: a slot is a (d, w) shift of the shifted operand only (9 per chunk); the three h taps come
              // from the h-halo of the FIXED operand's tile (three N atoms of one MMA)
              const int dd = p.halo ? tap / 3 - 1 : tap / 9 - 1;
              const int dh = p.halo ? 0 : (tap / 3) % 3 - 1;
              const int dw = tap % 3 - 1;
              tma_load_5d(smem_a + (size_t)sa * p.a_bytes + (size_t)j * p.slot_bytes, &tmap_x, &full_a[sa],
                          cc * p.SWC, w0 + dw, h0 + dh, d0 + dd, n);
            }
          }
          __syncwarp();
        }
      }
    }
    if (warp == 1) pdl_trigger();   // last slot loads issued: the next kernel may be staged
  } else if (warp == kWgProducers + 1) {
    // ---------------------------------------------------------------- producer of the dY tiles
    int sb = 0;
    uint32_t pb = 0;
    for (int sg = 0; wgrad_segment(p, sg, seg); ++sg) {
      const int n0 = seg.nt * p.BN;
      for (long long t = seg.t0; t < seg.t1; ++t) {
        int n, d0, h0, w0;
        wgrad_tile(t, p, n, d0, h0, w0);
        mbar_wait(&empty_b[sb], pb ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&full_b[sb], (uint32_t)p.b_bytes);
          if (p.halo) {   // one box with an h-halo: (bh + 2) lines of bw voxels x BN channels, zero-filled outside
            tma_load_5d(smem_b + (size_t)sb * p.b_bytes, &tmap_dy, &full_b[sb], n0, w0, h0 - 1, d0, n);
          } else {   // 64-channel boxes of 128 voxels (one 32-channel box when BN = 32)
            const int box_c = p.BN < 64 ? p.BN : 64;
            for (int j = 0; j < p.BN / box_c; ++j)
              tma_load_5d(smem_b + (size_t)sb * p.b_bytes + (size_t)j * 128 * box_c * 2, &tmap_dy, &full_b[sb],
                          n0 + j * box_c, w0, h0, d0, n);
          }
        }
        __syncwarp();
        if (++sb == p.stages_b) { sb = 0; pb ^= 1; }
      }
    }
  } else if (warp == 0) {
    // halo mode: N = 3 x BN — the three N atoms are the SAME dY tile shifted by -1 / 0 / +1 h-lines (atom stride = one
    // h-line of bw voxel rows), i.e. one MMA accumulates the three h taps of the slot pair: 6 taps per instruction,
    // 10 KB of shared-memory reads for 96 tensor-cycles instead of 6 KB for 32 (BN = 64)
    const uint32_t acc_cols = p.halo ? 3u * (uint32_t)p.BN : (uint32_t)p.BN;
    const uint32_t idesc = make_idesc_bf16(128, acc_cols, 1, 1);
    const uint32_t layout_a = (p.SWC == 64) ? SWZ_128B : (p.SWC == 32 ? SWZ_64B : SWZ_32B);
    const uint32_t row_a = (uint32_t)p.SWC * 2u;
    const uint64_t a_hi = make_smem_desc(0, (uint32_t)p.slot_bytes, 8 * row_a, layout_a);
    // dY rows: 64-channel atoms (128 B, 128B swizzle) or, for BN = 32, one 32-channel atom (64 B, 64B swizzle)
    const uint32_t row_b = p.BN < 64 ? (uint32_t)p.BN * 2u : 128u;
    const uint64_t b_hi = make_smem_desc(0, p.halo ? (uint32_t)p.bw * row_b : 128u * row_b, 8 * row_b,
                                         row_b == 128u ? SWZ_128B : SWZ_64B);
    const uint32_t a0 = smem_u32(smem_a) >> 4, b0 = smem_u32(smem_b) >> 4;
    const uint32_t a_kstep = (16 * row_a) >> 4, b_kstep = (16 * row_b) >> 4;   // encoded advance per K16 (16 voxels)
    int sa = 0, sb = 0;
    uint32_t pa = 0, pb = 0;
    for (int sg = 0; wgrad_segment(p, sg, seg); ++sg) {
      const int g_begin = seg.gchunk * p.gpc, g_end = min(g_begin + p.gpc, p.G);
      if (sg > 0) {   // the accumulators are reused: wait until the epilogue has read the previous segment
        mbar_wait(acc_empty, (uint32_t)(sg - 1) & 1u);
        tc_fence_after();
      }
      for (long long t = seg.t0; t < seg.t1; ++t) {
        mbar_wait(&full_b[sb], pb);
        tc_fence_after();
        const uint64_t bdesc = b_hi | (uint64_t)(b0 + (uint32_t)sb * ((uint32_t)p.b_bytes >> 4));
        for (int g = g_begin; g < g_end; ++g) {
          mbar_wait(&full_a[sa], pa);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t adesc = a_hi | (uint64_t)(a0 + (uint32_t)sa * ((uint32_t)p.a_bytes >> 4));
            const uint32_t d_tmem = tmem_base + (uint32_t)(g - g_begin) * acc_cols;
#pragma unroll
            for (int k = 0; k < 8; ++k)   // 128 voxels = 8 x K16
              umma_bf16(d_tmem, adesc + k * a_kstep, bdesc + k * b_kstep, idesc, (t != seg.t0 || k > 0) ? 1u : 0u);
            umma_commit(&empty_a[sa]);
            if (g == g_end - 1) {
              umma_commit(&empty_b[sb]);
              if (t == seg.t1 - 1) umma_commit(acc_full);
            }
          }
          __syncwarp();
          if (++sa == p.stages_a) { sa = 0; pa ^= 1; }
        }
        if (++sb == p.stages_b) { sb = 0; pb ^= 1; }
      }
    }
  } else {
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const size_t slice4 = (size_t)27 * p.Cin * p.Cout / 4;   // one split slice of the workspace, in float4
    for (int sg = 0; wgrad_segment(p, sg, seg); ++sg) {
      const int g_begin = seg.gchunk * p.gpc, g_end = min(g_begin + p.gpc, p.G);
      const int n0 = seg.nt * p.BN;
      mbar_wait(acc_full, (uint32_t)sg & 1u);
      tc_fence_after();
      for (int g = g_begin; g < g_end; ++g) {
        const int s = g * p.SPG + row / p.SWC;
        const bool valid = s < p.total_slots;
        const int tap = s / p.n_cchunks;
        const int ci = (s % p.n_cchunks) * p.SWC + row % p.SWC;
        const uint32_t acc_cols = p.halo ? 3u * (uint32_t)p.BN : (uint32_t)p.BN;
        const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(g - g_begin) * acc_cols;
        for (int c0 = 0; c0 < (int)acc_cols; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(t_addr + c0, v);
          tmem_ld_wait();
          if (valid) {
            // halo mode: accumulator columns [BN j, BN j + BN) = h tap dh = 1 - j of the slot's (dd, dw) shift
            const int full_tap = p.halo ? (tap / 3) * 9 + (2 - c0 / p.BN) * 3 + tap % 3 : tap;
            const int col = p.halo ? (c0 % p.BN) : c0;
            float4* d4 = reinterpret_cast<float4*>(p.ws + (((size_t)seg.layer * 27 + full_tap) * p.Cin + ci) * p.Cout +
                                                   n0 + col);
#pragma unroll
            for (int j = 0; j < 8; ++j)
              d4[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                  __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
            for (int e = seg.layer + 1; e < seg.zero_to; ++e) {
              d4 += slice4;
#pragma unroll
              for (int j = 0; j < 8; ++j) d4[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(acc_empty);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// dW[co][ci][tap] = sum_s ws[s][tap][ci][co]: block = (32-wide co tile, 8-wide ci tile), all 27 taps; reads run along
// co (128-byte runs), writes run along (ci, tap) (864-byte runs) through a padded shared-memory transpose.
// 27 elements per thread: the loads of 9 elements (x splits) are issued before any is consumed (round 1 walked them one
// dependent load at a time: 28 us for 5.3 M elements, 1.5 TB/s).
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ ws, float* __restrict__ dw, int splits, int Cin, int Cout) {
  pdl_prologue();
  __shared__ float t[32 * 217];
  const int co0 = blockIdx.x * 32, ci0 = blockIdx.y * 8;
  const long long total = 27LL * Cin * Cout;
  const int co = threadIdx.x & 31, ci = (threadIdx.x >> 5) & 7;
  const float* src = ws + ((long long)(ci0 + ci)) * Cout + co0 + co;
  const long long tap_stride = (long long)Cin * Cout;
#pragma unroll
  for (int t0 = 0; t0 < 27; t0 += 9) {
    float acc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] = 0.f;
    for (int s = 0; s < splits; ++s) {
      float v[9];
#pragma unroll
      for (int k = 0; k < 9; ++k) v[k] = __ldcg(src + (long long)s * total + (t0 + k) * tap_stride);
#pragma unroll
      for (int k = 0; k < 9; ++k) acc[k] += v[k];
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) t[co * 217 + ci * 27 + t0 + k] = acc[k];
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 32 * 216; e += 256) {
    const int c = e / 216, r = e % 216;   // r = ci*27 + tap
    dw[((long long)(co0 + c) * Cin + ci0) * 27 + r] = t[c * 217 + r];
  }
}

// small layers (few (co, ci) tiles): one thread per element, all splits summed in registers
__global__ void __launch_bounds__(256)
wgrad_reduce_simple_kernel(const float* __restrict__ ws, float* __restrict__ dw, int splits, int Cin, int Cout) {
  pdl_prologue();
  const long long total = 27LL * Cin * Cout;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    float acc = 0.f;
    int s = 0;
    for (; s + 3 < splits; s += 4)
      acc += (ws[(long long)s * total + i] + ws[(long long)(s + 1) * total + i]) +
             (ws[(long long)(s + 2) * total + i] + ws[(long long)(s + 3) * total + i]);
    for (; s < splits; ++s) acc += ws[(long long)s * total + i];
    const int co = (int)(i % Cout);
    const long long r = i / Cout;
    const int ci = (int)(r % Cin);
    const int tap = (int)(r / Cin);
    dw[((long long)co * Cin + ci) * 27 + tap] = acc;
  }
}

// roles swapped (see b2_conv3d_wgrad): ws[s][tap'][co][ci] with tap' = 26 - tap  ->  dW[co][ci][tap]
__global__ void __launch_bounds__(256)
wgrad_reduce_swapped_kernel(const float* __restrict__ ws, float* __restrict__ dw, int splits, int Cin, int Cout) {
  pdl_prologue();
  const long long total = 27LL * Cin * Cout;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    float acc = 0.f;
    int s = 0;
    for (; s + 3 < splits; s += 4)
      acc += (ws[(long long)s * total + i] + ws[(long long)(s + 1) * total + i]) +
             (ws[(long long)(s + 2) * total + i] + ws[(long long)(s + 3) * total + i]);
    for (; s < splits; ++s) acc += ws[(long long)s * total + i];
    const int ci = (int)(i % Cin);
    const long long r = i / Cin;
    const int co = (int)(r % Cout);
    const int tapf = (int)(r / Cout);
    dw[((long long)co * Cin + ci) * 27 + (26 - tapf)] = acc;
  }
}

// Split reduction for the layers with many splits (37..148 partial tiles per element, ~33 MB of fp32 partials per
// layer).  Round 1 summed all splits of an element in ONE thread: a chain of up to 148 dependent-latency loads per
// thread on only ~200 blocks (14.7 us per launch, 2 TB/s).  Here a block owns 32 consecutive elements and its 8 warps
// take the splits s = warp, warp + 8, ... (coalesced 128-byte rows, 4 loads in flight per thread); the 8 partial sums
// are combined through shared memory in a fixed order: deterministic, 8x the memory-level parallelism.
// swapped = 0: ws[s][tap][ci][co] -> dW[co][ci][tap];  swapped = 1 (roles swapped, see b2_conv3d_wgrad):
// ws[s][26 - tap][co][ci] -> dW[co][ci][tap].
template <int SWAPPED>
__global__ void __launch_bounds__(256)
wgrad_reduce_par_kernel(const float* __restrict__ ws, float* __restrict__ dw, int splits, int Cin, int Cout) {
  pdl_prologue();
  __shared__ float part[8][32];
  const long long total = 27LL * Cin * Cout;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long i = (long long)blockIdx.x * 32 + lane;
  float acc = 0.f;
  if (i < total) {
    int s = warp;
    for (; s + 24 < splits; s += 32)
      acc += (ws[(long long)s * total + i] + ws[(long long)(s + 8) * total + i]) +
             (ws[(long long)(s + 16) * total + i] + ws[(long long)(s + 24) * total + i]);
    for (; s < splits; s += 8) acc += ws[(long long)s * total + i];
  }
  part[warp][lane] = acc;
  __syncthreads();
  if (warp == 0 && i < total) {
    const float r = ((part[0][lane] + part[1][lane]) + (part[2][lane] + part[3][lane])) +
                    ((part[4][lane] + part[5][lane]) + (part[6][lane] + part[7][lane]));
    if (SWAPPED) {
      const int ci = (int)(i % Cin);
      const long long q = i / Cin;
      const int co = (int)(q % Cout);
      const int tapf = (int)(q / Cout);
      dw[((long long)co * Cin + ci) * 27 + (26 - tapf)] = r;
    } else {
      const int co = (int)(i % Cout);
      const long long q = i / Cout;
      const int ci = (int)(q % Cin);
      const int tap = (int)(q / Cin);
      dw[((long long)co * Cin + ci) * 27 + tap] = r;
    }
  }
}

// ---- deferred reduction of SEVERAL layers in one launch --------------------------------------------------------------
// The 13 per-layer reduce launches cost 231 us of a 6.7 ms step (A/B on B200, round 2) although they move little data:
// each is a short, latency-bound kernel between two tensor-core kernels.  b2_conv3d_wgrad_partial leaves the split
// partials of a layer in that layer's own workspace; one launch of this kernel then reduces every pending layer at once
// (at the end of backward, or when a data-parallel gradient bucket closes): one launch latency, the whole GPU busy.
// Per layer: mode 0 = transposing tile (32 co x 8 ci x 27 taps per block; few splits, big tensors), mode 1 = split-parallel
// (32 elements per block, the 8 warps share the splits; many splits, small tensors; also the swapped layout).
static constexpr int kMaxReduceLayers = 16;
struct WgReduceArgs {
  const float* ws[kMaxReduceLayers];
  float* dw[kMaxReduceLayers];
  int splits[kMaxReduceLayers], cin[kMaxReduceLayers], cout[kMaxReduceLayers], mode[kMaxReduceLayers];
  int swapped[kMaxReduceLayers];
  int first_block[kMaxReduceLayers + 1];
  int count;
};

__global__ void __launch_bounds__(256)
wgrad_reduce_multi_kernel(const WgReduceArgs a) {
  pdl_prologue();
  __shared__ float t[32 * 217];
  int l = 0;
  while (l + 1 < a.count && (int)blockIdx.x >= a.first_block[l + 1]) ++l;
  const int b = blockIdx.x - a.first_block[l];
  const float* __restrict__ ws = a.ws[l];
  float* __restrict__ dw = a.dw[l];
  const int splits = a.splits[l], Cin = a.cin[l], Cout = a.cout[l];
  const long long total = 27LL * Cin * Cout;
  if (a.mode[l] == 0) {
    const int co_tiles = Cout / 32;
    const int co0 = (b % co_tiles) * 32, ci0 = (b / co_tiles) * 8;
    const int co = threadIdx.x & 31, ci = (threadIdx.x >> 5) & 7;
    const float* src = ws + ((long long)(ci0 + ci)) * Cout + co0 + co;
    const long long tap_stride = (long long)Cin * Cout;
#pragma unroll
    for (int t0 = 0; t0 < 27; t0 += 9) {
      float acc[9];
#pragma unroll
      for (int k = 0; k < 9; ++k) acc[k] = 0.f;
      for (int s = 0; s < splits; ++s) {
        float v[9];
#pragma unroll
        for (int k = 0; k < 9; ++k) v[k] = __ldcg(src + (long long)s * total + (t0 + k) * tap_stride);
#pragma unroll
        for (int k = 0; k < 9; ++k) acc[k] += v[k];
      }
#pragma unroll
      for (int k = 0; k < 9; ++k) t[co * 217 + ci * 27 + t0 + k] = acc[k];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 32 * 216; e += 256) {
      const int c = e / 216, r = e % 216;   // r = ci*27 + tap
      dw[((long long)(co0 + c) * Cin + ci0) * 27 + r] = t[c * 217 + r];
    }
  } else {
    float (*part)[32] = reinterpret_cast<float (*)[32]>(t);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long i = (long long)b * 32 + lane;
    float acc = 0.f;
    if (i < total) {
      int s = warp;
      for (; s + 24 < splits; s += 32)
        acc += (__ldcg(ws + (long long)s * total + i) + __ldcg(ws + (long long)(s + 8) * total + i)) +
               (__ldcg(ws + (long long)(s + 16) * total + i) + __ldcg(ws + (long long)(s + 24) * total + i));
      for (; s < splits; s += 8) acc += __ldcg(ws + (long long)s * total + i);
    }
    part[warp][lane] = acc;
    __syncthreads();
    if (warp == 0 && i < total) {
      const float r = ((part[0][lane] + part[1][lane]) + (part[2][lane] + part[3][lane])) +
                      ((part[4][lane] + part[5][lane]) + (part[6][lane] + part[7][lane]));
      if (a.swapped[l]) {
        const int ci = (int)(i % Cin);
        const long long q = i / Cin;
        dw[((long long)(int)(q % Cout) * Cin + ci) * 27 + (26 - (int)(q / Cout))] = r;
      } else {
        const int co = (int)(i % Cout);
        const long long q = i / Cout;
        dw[((long long)co * Cin + (int)(q % Cin)) * 27 + (int)(q / Cin)] = r;
      }
    }
  }
}

// Which operand is shifted per tap?  The shifted operand is re-loaded for every tap, the other one once per
// 128-voxel K-step, so shifting the NARROW one and keeping the wide one as the N dimension halves the TMA traffic
// per tensor-cycle when Cout = 64 and Cin >= 128 (decoders.2.conv1: 133 -> 73 B/clk/SM).
static bool wgrad_swap_roles(int Cin, int Cout) { return Cout == 64 && Cin >= 128 && Cin % 64 == 0; }

static void choose_box_w(int W, int H, int D, int& bw, int& bh, int& bd) {
  long long best = -1;
  for (int lw = 0; lw <= 7; ++lw)
    for (int lh = 0; lw + lh <= 7; ++lh) {
      const int ld = 7 - lw - lh;
      const int cw = 1 << lw, chh = 1 << lh, cd = 1 << ld;
      const long long cost = (long long)ceil_div(W, cw) * cw * (long long)ceil_div(H, chh) * chh *
                             (long long)ceil_div(D, cd) * cd;
      const long long score = cost * 1024 - cw * 8 - chh;
      if (best < 0 || score < best) { best = score; bw = cw; bh = chh; bd = cd; }
    }
}

static int plan_wgrad(WgradParams& p, int N, int D, int H, int W, int Cin, int Cout, bool allow_halo) {
  p.N = N; p.D = D; p.H = H; p.W = W; p.Cin = Cin; p.Cout = Cout;
  choose_box_w(W, H, D, p.bw, p.bh, p.bd);
  p.tiles_w = ceil_div(W, p.bw);
  p.tiles_h = ceil_div(H, p.bh);
  p.tiles_d = ceil_div(D, p.bd);
  p.SWC = (Cin % 64 == 0) ? 64 : (Cin % 32 == 0 ? 32 : 16);
  p.n_cchunks = Cin / p.SWC;
  p.BN = (Cout % 256 == 0) ? 256 : (Cout % 192 == 0 ? 192 : (Cout % 128 == 0 ? 128 : (Cout % 64 == 0 ? 64 : 32)));
  p.n_cout_tiles = Cout / p.BN;
  // "dY-halo" mode for Cout <= 128 at one-plane tile boxes (decoders.2.conv2, encoders.0.conv2, encoders.1.*,
  // decoders.1.*: round 1 ran the Cout = 64 ones at 640-790 TFLOP/s, bound by re-loading the shifted operand 27 times
  // per K-step and by the 128 x 64 MMA's shared-memory read rate).  dW[tap] = sum_u X[u + s] dY[u + t] with
  // tap = s - t: the (d, w) part of the tap shifts X (9 slots per chunk instead of 27), the h part shifts dY — whose
  // 64-channel tile is loaded ONCE with an h-halo and read by the MMA as three N atoms one h-line apart (N = 192).
  // Needs an h-line to be bw consecutive, 1024-byte-aligned voxel rows.  Measured (us, incl. reduce): dec2.conv2
  // 293 -> 212, enc0.conv2 179 -> 143, enc1.conv1 59 -> 48, dec1.conv1 289 -> 257, dec1.conv2 112 -> 99, enc1.conv2
  // 86 -> 67.
  static const bool no_halo = getenv("B2_NO_WGRAD_HALO") != nullptr;
  static const int halo_max_c = getenv("B2_WGRAD_HALO_MAXC") ? atoi(getenv("B2_WGRAD_HALO_MAXC")) : 128;
  p.halo = (allow_halo && !no_halo && Cout % 32 == 0 && Cout <= halo_max_c && p.bd == 1 && p.bw % 8 == 0) ? 1 : 0;
  if (p.halo) {   // 64-channel N tiles (32 when Cout = 32), each read as three h-shifted atoms
    p.BN = (Cout % 64 == 0) ? 64 : 32;
    p.n_cout_tiles = Cout / p.BN;
  }
  static const bool plane_order = getenv("B2_WGRAD_PLANE_ORDER") != nullptr;
  p.d_fast = (p.halo && !plane_order) ? 1 : 0;
  p.total_slots = (p.halo ? 9 : 27) * p.n_cchunks;
  p.SPG = 128 / p.SWC;
  p.G = ceil_div(p.total_slots, p.SPG);
  // accumulators per CTA (one group per CTA measured slower: 237 vs 211 us); halo: 2 at BN = 64, 5 at BN = 32
  const int P = 512 / (p.halo ? 3 * p.BN : p.BN);
  p.n_gchunks = ceil_div(p.G, P);
  p.gpc = ceil_div(p.G, p.n_gchunks);
  p.n_gchunks = ceil_div(p.G, p.gpc);
  p.ksteps_total = (long long)N * p.tiles_d * p.tiles_h * p.tiles_w;
  const int columns = p.n_gchunks * p.n_cout_tiles;
  int splits = num_sms() / columns;
  if (splits < 1) splits = 1;
  if ((long long)splits > p.ksteps_total) splits = (int)p.ksteps_total;
  p.splits = splits;
  p.grid = columns * splits;
  p.streamk = 0;
  // more columns than half the SMs (decoders.0.conv1: 81): a uniform split cannot use the idle SMs, equal runs can
  static const bool no_streamk = getenv("B2_NO_WGRAD_STREAMK") != nullptr;
  if (!no_streamk && splits == 1 && columns < num_sms() && p.ksteps_total * columns >= 4LL * num_sms()) {
    p.streamk = 1;
    p.grid = num_sms();
    const long long K = p.ksteps_total, total = K * columns;
    int slices = 1;   // the most runs any column intersects (same arithmetic as wgrad_segment)
    for (long long col = 0; col < columns; ++col) {
      const long long first = ((col * K + 1) * p.grid - 1) / total, last = (((col + 1) * K) * p.grid - 1) / total;
      if ((int)(last - first + 1) > slices) slices = (int)(last - first + 1);
    }
    p.splits = slices;
  }
  p.slot_bytes = 128 * p.SWC * 2;
  p.a_bytes = 128 * 128 * 2;
  p.b_bytes = p.halo ? (p.bh + 2) * p.bw * p.BN * 2 : 128 * p.BN * 2;
  const int budget = 227 * 1024 - 1024 - 512;
  p.stages_a = (budget - 2 * p.b_bytes) / p.a_bytes;
  if (p.stages_a > 4) p.stages_a = 4;
  // a producer must never be two ring phases ahead of the consumer: give every stage a fixed owner
  p.n_prod = p.stages_a < kWgProducers ? p.stages_a : kWgProducers;
  p.stages_a = (p.stages_a / p.n_prod) * p.n_prod;
  if (p.stages_a < 2) return -1;
  // what is left deepens the fixed-operand ring (few groups per K-step = short steps: two stages do not cover the
  // load latency)
  p.stages_b = (budget - p.stages_a * p.a_bytes) / p.b_bytes;
  if (p.stages_b > 4) p.stages_b = 4;
  return 0;
}

}  // namespace b2

using namespace b2;

// Cin = 16 or a multiple of 32 (shifted slots of 16, 32 or 64 channels), Cout a multiple of 32
static bool wgrad_shape_ok(int Cin, int Cout) {
  return (Cin == 16 || (Cin % 32 == 0 && Cin >= 32)) && Cout % 32 == 0 && Cout >= 32;
}

extern "C" long long b2_conv3d_wgrad_workspace_bytes(int N, int D, int H, int W, int Cin, int Cout) {
  if (!wgrad_shape_ok(Cin, Cout) || N <= 0 || D <= 0 || H <= 0 || W <= 0) return -1;
  WgradParams p;
  const bool swap = wgrad_swap_roles(Cin, Cout);
  if (plan_wgrad(p, N, D, H, W, swap ? Cout : Cin, swap ? Cin : Cout, !swap) != 0) return -1;
  return (long long)p.splits * 27 * Cin * Cout * (long long)sizeof(float);
}

static int wgrad_partial_impl(const void* x, int ldx, int x_coff, const void* dy, int ldy, int y_coff, void* workspace,
                              long long workspace_bytes, int N, int D, int H, int W, int Cin, int Cout,
                              WgradParams& p, bool& swap, cudaStream_t stream) {
  B2_REQUIRE(x && dy && workspace, "b2_conv3d_wgrad: null pointer");
  B2_REQUIRE(N > 0 && D > 0 && H > 0 && W > 0, "b2_conv3d_wgrad: bad shape");
  B2_REQUIRE(wgrad_shape_ok(Cin, Cout), "b2_conv3d_wgrad: Cin=%d must be 16 or a multiple of 32, Cout=%d a multiple of 32",
             Cin, Cout);
  B2_REQUIRE(ldx % 8 == 0 && x_coff % 8 == 0 && ldy % 8 == 0 && y_coff % 8 == 0,
             "b2_conv3d_wgrad: channel strides/offsets must be multiples of 8");
  swap = wgrad_swap_roles(Cin, Cout);
  // kernel view: "shifted" operand (slots along M) and "fixed" operand (N); swapped roles shift dY by the flipped tap
  const void* sh_ptr = swap ? dy : x;
  const void* fx_ptr = swap ? x : dy;
  const int sh_c = swap ? Cout : Cin, fx_c = swap ? Cin : Cout;
  const int sh_ld = swap ? ldy : ldx, sh_off = swap ? y_coff : x_coff;
  const int fx_ld = swap ? ldx : ldy, fx_off = swap ? x_coff : y_coff;
  B2_REQUIRE(plan_wgrad(p, N, D, H, W, sh_c, fx_c, !swap) == 0, "b2_conv3d_wgrad: tile does not fit shared memory");
  const long long need = (long long)p.splits * 27 * Cin * Cout * (long long)sizeof(float);
  B2_REQUIRE(workspace_bytes >= need, "b2_conv3d_wgrad: workspace %lld < %lld bytes", workspace_bytes, need);
  p.ws = reinterpret_cast<float*>(workspace);

  CUtensorMap tx, ty;
  int rc = make_act_tmap(&tx, sh_ptr, N, D, H, W, sh_c, sh_ld, sh_off, p.SWC, p.bw, p.bh, p.bd);
  if (rc) return rc;
  rc = make_act_tmap(&ty, fx_ptr, N, D, H, W, fx_c, fx_ld, fx_off, p.BN < 64 ? p.BN : 64, p.bw,
                     p.halo ? p.bh + 2 : p.bh, p.bd);
  if (rc) return rc;

  const size_t smem_bytes = (size_t)p.stages_b * p.b_bytes + (size_t)p.stages_a * p.a_bytes + 1024 + 512;
  B2_CHECK_CUDA(cudaFuncSetAttribute(conv3d_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  dim3 grid((unsigned)p.grid);
  B2_LAUNCH(conv3d_wgrad_kernel, grid, kWgThreads, smem_bytes, stream, tx, ty, p);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

extern "C" int b2_conv3d_wgrad(const void* x, int ldx, int x_coff, const void* dy, int ldy, int y_coff, float* dw,
                               void* workspace, long long workspace_bytes, int N, int D, int H, int W, int Cin,
                               int Cout, cudaStream_t stream) {
  B2_REQUIRE(dw, "b2_conv3d_wgrad: null pointer");
  WgradParams p;
  bool swap = false;
  int rc = wgrad_partial_impl(x, ldx, x_coff, dy, ldy, y_coff, workspace, workspace_bytes, N, D, H, W, Cin, Cout, p,
                              swap, stream);
  if (rc) return rc;
  const long long total = 27LL * Cin * Cout;
  if (p.splits >= 32 && !swap) {
    // few elements, many splits (enc0.conv2 148, enc1.conv1 / dec2.conv2 74, enc1.conv2 37): split-parallel reduce
    B2_LAUNCH(wgrad_reduce_par_kernel<0>, (unsigned)((total + 31) / 32), 256, 0, stream, p.ws, dw, p.splits, Cin, Cout);
  } else if (swap) {
    B2_LAUNCH(wgrad_reduce_swapped_kernel, (unsigned)((total + 255) / 256), 256, 0, stream, p.ws, dw, p.splits, Cin, Cout);
  } else if ((Cout / 32) * (Cin / 8) >= num_sms()) {
    B2_LAUNCH(wgrad_reduce_kernel, dim3(Cout / 32, Cin / 8), 256, 0, stream, p.ws, dw, p.splits, Cin, Cout);
  } else {
    B2_LAUNCH(wgrad_reduce_simple_kernel, (unsigned)((total + 255) / 256), 256, 0, stream, p.ws, dw, p.splits, Cin, Cout);
  }
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

// The tensor-core half of b2_conv3d_wgrad only: the split partials stay in `workspace` (which must then be private to
// this layer until b2_wgrad_reduce_multi has run); *splits_out / *swapped_out describe their layout for the reduce.
extern "C" int b2_conv3d_wgrad_partial(const void* x, int ldx, int x_coff, const void* dy, int ldy, int y_coff,
                                       void* workspace, long long workspace_bytes, int N, int D, int H, int W, int Cin,
                                       int Cout, int* splits_out, int* swapped_out, cudaStream_t stream) {
  B2_REQUIRE(splits_out && swapped_out, "b2_conv3d_wgrad_partial: null pointer");
  WgradParams p;
  bool swap = false;
  int rc = wgrad_partial_impl(x, ldx, x_coff, dy, ldy, y_coff, workspace, workspace_bytes, N, D, H, W, Cin, Cout, p,
                              swap, stream);
  if (rc) return rc;
  *splits_out = p.splits;
  *swapped_out = swap ? 1 : 0;
  return B2_OK;
}

// One launch reduces the split partials of `count` layers (HOST arrays of `count` entries) into dW[co][ci][3][3][3].
extern "C" int b2_wgrad_reduce_multi(const float* const* ws, float* const* dw, const int* splits, const int* cin,
                                     const int* cout, const int* swapped, int count, cudaStream_t stream) {
  B2_REQUIRE(ws && dw && splits && cin && cout && swapped && count >= 0, "b2_wgrad_reduce_multi: null pointer");
  int done = 0;
  while (done < count) {
    WgReduceArgs a;
    int k = 0;
    long long blocks = 0;
    while (done + k < count && k < kMaxReduceLayers) {
      const int i = done + k;
      B2_REQUIRE(ws[i] && dw[i] && splits[i] > 0 && cin[i] % 8 == 0 && cout[i] % 32 == 0,
                 "b2_wgrad_reduce_multi: bad layer %d", i);
      a.ws[k] = ws[i]; a.dw[k] = dw[i];
      a.splits[k] = splits[i]; a.cin[k] = cin[i]; a.cout[k] = cout[i]; a.swapped[k] = swapped[i];
      a.mode[k] = (swapped[i] || splits[i] > 10) ? 1 : 0;
      a.first_block[k] = (int)blocks;
      const long long total = 27LL * cin[i] * cout[i];
      blocks += a.mode[k] == 0 ? (long long)(cout[i] / 32) * (cin[i] / 8) : (total + 31) / 32;
      B2_REQUIRE(blocks < (1LL << 31), "b2_wgrad_reduce_multi: too many blocks");
      ++k;
    }
    a.first_block[k] = (int)blocks;
    a.count = k;
    if (blocks > 0) {
      B2_LAUNCH(wgrad_reduce_multi_kernel, (unsigned)blocks, 256, 0, stream, a);
      B2_CHECK_CUDA(cudaGetLastError());
    }
    done += k;
  }
  return B2_OK;
}
