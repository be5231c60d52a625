// encoders.0.conv1: Cin = 1, K = 27 — a bandwidth-bound direct convolution (not tensor-core shaped).
//   fwd  : y[v, co] = relu( sum_tap x[v + off(tap)] * w[co][tap] )      x fp32 [N,D,H,W], y bf16 [N,D,H,W,Cout]
//   wgrad: dw[co][tap] = sum_v dy[v, co] * x[v + off(tap)]
// The input is a binary skeleton (~3 % ones): taps whose input voxel is 0 are skipped.
#include "common.h"
#include "ptx.cuh"

namespace b2 {


// One warp per 32 consecutive voxels, lane = voxel.  All 27 neighbour loads are issued before any arithmetic (the
// round-1 kernel walked the taps one dependent L1 load at a time and was latency-bound at 680 GB/s); a tap is skipped
// when no lane of the warp has a non-zero input there.  When stat_acc != NULL the kernel also accumulates, per
// channel, sum and sum of squares of the STORED (ReLU'd, bf16-rounded) outputs — the GroupNorm statistics — into
// the exact [COUT][4] accumulators of common.h (one atomic add per block and channel).  COUT = 16 (32-filter networks)
// sums one half-empty 32-column chunk: lanes 16..31 carry zeros and are not stored.
// bias (fp32 [COUT], may be NULL) is added to the accumulator before ReLU: a voxel whose 27 neighbours are all zero
// (every tap skipped) stores relu(bias) and contributes it to the statistics.
template <int COUT>
__global__ void __launch_bounds__(128)
conv_first_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w /*[COUT][27]*/,
                      __nv_bfloat16* __restrict__ y, int N, int D, int H, int W, int ldy, int y_coff, int relu,
                      long long* __restrict__ stat_acc, const float* __restrict__ bias) {
  pdl_prologue();
  __shared__ __align__(16) float ws[27][COUT];
  __shared__ float2 sred[4][COUT];
  __shared__ float bs[COUT];
  for (int i = threadIdx.x; i < 27 * COUT; i += blockDim.x) ws[i % 27][i / 27] = w[i];  // w[co*27+tap]
  if (bias != nullptr)
    for (int i = threadIdx.x; i < COUT; i += blockDim.x) bs[i] = bias[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long V = (long long)N * D * H * W;
  constexpr int kChunks = (COUT + 31) / 32;
  float st_s[kChunks], st_q[kChunks];   // lane L: channel 32*k + L, summed over this warp's voxels
#pragma unroll
  for (int k = 0; k < kChunks; ++k) { st_s[k] = 0.f; st_q[k] = 0.f; }
  for (long long v0 = ((long long)blockIdx.x * 4 + warp) * 32; v0 < V; v0 += (long long)gridDim.x * 128) {
    const long long v = v0 + lane;
    const bool active = v < V;
    const long long vv = active ? v : V - 1;
    const int wq = (int)(vv % W);
    long long r = vv / W;
    const int hq = (int)(r % H);
    r /= H;
    const int dq = (int)(r % D);
    const float* xc = x + vv;
    float xv[27];
#pragma unroll
    for (int tap = 0; tap < 27; ++tap) {
      const int dd = tap / 9 - 1, dh = (tap / 3) % 3 - 1, dw = tap % 3 - 1;
      const bool ok = active && (unsigned)(dq + dd) < (unsigned)D && (unsigned)(hq + dh) < (unsigned)H &&
                      (unsigned)(wq + dw) < (unsigned)W;
      xv[tap] = ok ? __ldg(xc + ((long long)dd * H + dh) * W + dw) : 0.f;
    }
    float acc[COUT];
#pragma unroll
    for (int c = 0; c < COUT; ++c) acc[c] = 0.f;
#pragma unroll
    for (int tap = 0; tap < 27; ++tap) {
      if (__any_sync(0xffffffffu, xv[tap] != 0.f)) {
        const float4* wr = reinterpret_cast<const float4*>(&ws[tap][0]);
#pragma unroll
        for (int c4 = 0; c4 < COUT / 4; ++c4) {
          const float4 q = wr[c4];
          acc[4 * c4 + 0] = fmaf(xv[tap], q.x, acc[4 * c4 + 0]);
          acc[4 * c4 + 1] = fmaf(xv[tap], q.y, acc[4 * c4 + 1]);
          acc[4 * c4 + 2] = fmaf(xv[tap], q.z, acc[4 * c4 + 2]);
          acc[4 * c4 + 3] = fmaf(xv[tap], q.w, acc[4 * c4 + 3]);
        }
      }
    }
    if (bias != nullptr) {
#pragma unroll
      for (int c = 0; c < COUT; ++c) acc[c] += bs[c];
    }
    if (relu) {
#pragma unroll
      for (int c = 0; c < COUT; ++c) acc[c] = relu_nan(acc[c]);
    }
    if (active) {
      uint4* dst = reinterpret_cast<uint4*>(y + v * ldy + y_coff);
#pragma unroll
      for (int j = 0; j < COUT / 8; ++j) {
        uint4 o;
        o.x = pack_bf16x2(acc[8 * j + 0], acc[8 * j + 1]);
        o.y = pack_bf16x2(acc[8 * j + 2], acc[8 * j + 3]);
        o.z = pack_bf16x2(acc[8 * j + 4], acc[8 * j + 5]);
        o.w = pack_bf16x2(acc[8 * j + 6], acc[8 * j + 7]);
        dst[j] = o;
      }
    }
    if (stat_acc != nullptr) {
#pragma unroll
      for (int k = 0; k < kChunks; ++k) {
        float xs[32], xq[32];
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const float f = (active && 32 * k + e < COUT) ? __bfloat162float(__float2bfloat16_rn(acc[32 * k + e])) : 0.f;
          xs[e] = f;
          xq[e] = f * f;
        }
        warp_column_sums(xs, lane);
        warp_column_sums(xq, lane);
        st_s[k] += xs[0];
        st_q[k] += xq[0];
      }
    }
  }
  if (stat_acc != nullptr) {
#pragma unroll
    for (int k = 0; k < kChunks; ++k)
      if (32 * k + lane < COUT) sred[warp][32 * k + lane] = make_float2(st_s[k], st_q[k]);
    __syncthreads();
    for (int c = threadIdx.x; c < COUT; c += blockDim.x) {
      const float2 a = sred[0][c], b = sred[1][c], cc = sred[2][c], d = sred[3][c];
      stat_atomic_add(stat_acc + 4 * c, (a.x + b.x) + (cc.x + d.x));
      stat_atomic_add(stat_acc + 4 * c + 2, (a.y + b.y) + (cc.y + d.y));
    }
  }
}

// dw[co][tap] = sum_u x[u] * dy[u - off(tap), co] over the NON-ZERO input voxels u (~3 % of a skeleton volume).
// Every block owns a contiguous range of input voxels: it first compacts the non-zero ones of a 2048-voxel
// sub-chunk into shared memory (ballot + prefix: ascending voxel order, deterministic).  Warp w then takes the
// voxels w, w+8, ... of that list; for one voxel a single 16-byte load instruction fetches 32/LPR different TAP rows
// at once (lane = (tap slot, channel octet), LPR = Cout/8 lanes per dy row), so the 27 taps cost ceil(27*LPR/32)
// load instructions instead of 27 (ncu, round 1: the one-row-per-instruction form executed 36 M warp instructions
// for 31 k voxels and sat at 25 % issue utilisation behind long-scoreboard stalls).  A lane owns its (tap, 8
// channels) sums; the 8 warps are combined through shared memory in warp order: no atomics, deterministic.
static constexpr int kFwChunk = 2048;

template <int COUT>
__global__ void __launch_bounds__(256)
conv_first_wgrad_kernel(const float* __restrict__ x, const __nv_bfloat16* __restrict__ dy, int lddy, int dy_coff,
                        float* __restrict__ partial /*[grid][27][COUT]*/, int N, int D, int H, int W,
                        long long per_block) {
  pdl_prologue();
  constexpr int LPR = COUT / 8;              // lanes per dy row
  constexpr int PPL = 32 / LPR;              // (voxel, tap) rows fetched by one load instruction
  constexpr int ROUNDS = (27 + PPL - 1) / PPL;
  __shared__ int s_u[kFwChunk];
  __shared__ uint32_t s_dhw[kFwChunk];
  __shared__ float s_x[kFwChunk];
  __shared__ int s_cnt[kFwChunk / 32 + 1];
  __shared__ float red[27 * COUT];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int slot = lane / LPR, cq = lane % LPR;
  const long long V = (long long)N * D * H * W;
  const long long r_begin = (long long)blockIdx.x * per_block;
  const long long r_end = (r_begin + per_block < V) ? r_begin + per_block : V;
  const __nv_bfloat16* dyc = dy + dy_coff + cq * 8;
  float acc[ROUNDS][8];
  int tdd[ROUNDS], tdh[ROUNDS], tdw[ROUNDS], toff[ROUNDS];
#pragma unroll
  for (int k = 0; k < ROUNDS; ++k) {
    const int tap = slot + PPL * k;
    tdd[k] = tap < 27 ? tap / 9 - 1 : 4096;   // 4096: never in bounds
    tdh[k] = (tap / 3) % 3 - 1;
    tdw[k] = tap % 3 - 1;
    toff[k] = tap < 27 ? (tdd[k] * H + tdh[k]) * W + tdw[k] : 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[k][e] = 0.f;
  }
  for (int i = threadIdx.x; i < 27 * COUT; i += blockDim.x) red[i] = 0.f;
  __syncthreads();
  for (long long c0 = r_begin; c0 < r_end; c0 += kFwChunk) {
    // ---- compaction of the non-zero voxels of [c0, c0 + kFwChunk) in ascending order
    float xv[kFwChunk / 256];
    unsigned bal[kFwChunk / 256];
#pragma unroll
    for (int k = 0; k < kFwChunk / 256; ++k) {
      const long long u = c0 + k * 256 + threadIdx.x;
      xv[k] = (u < r_end) ? __ldg(x + u) : 0.f;
      bal[k] = __ballot_sync(0xffffffffu, xv[k] != 0.f);
      if (lane == 0) s_cnt[k * 8 + warp] = __popc(bal[k]);
    }
    __syncthreads();
    if (warp == 0) {   // exclusive prefix over the 64 (k, warp) counts
      int a = s_cnt[lane], b = s_cnt[lane + 32];
      int ia = a, ib = b;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int ta = __shfl_up_sync(0xffffffffu, ia, o), tb = __shfl_up_sync(0xffffffffu, ib, o);
        if (lane >= o) { ia += ta; ib += tb; }
      }
      const int tot_a = __shfl_sync(0xffffffffu, ia, 31);
      s_cnt[lane] = ia - a;
      s_cnt[lane + 32] = tot_a + ib - b;
      if (lane == 31) s_cnt[64] = tot_a + ib;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kFwChunk / 256; ++k) {
      if (xv[k] != 0.f) {
        const int pos = s_cnt[k * 8 + warp] + __popc(bal[k] & ((1u << lane) - 1u));
        const long long u = c0 + k * 256 + threadIdx.x;
        const int wq = (int)(u % W);
        long long r = u / W;
        const int hq = (int)(r % H);
        r /= H;
        const int dq = (int)(r % D);
        s_u[pos] = (int)u;
        s_dhw[pos] = ((uint32_t)dq << 20) | ((uint32_t)hq << 10) | (uint32_t)wq;
        s_x[pos] = xv[k];
      }
    }
    __syncthreads();
    const int cnt = s_cnt[64];
    // ---- gather: two voxels x ROUNDS 16-byte loads in flight per lane
    for (int j0 = warp; j0 < cnt; j0 += 16) {
      uint4 g[2][ROUNDS];
      float xs[2];
#pragma unroll
      for (int jj = 0; jj < 2; ++jj) {
        const int j = j0 + 8 * jj;
        const bool live = j < cnt;
        const int js = live ? j : j0;
        const int u = s_u[js];
        const uint32_t c = s_dhw[js];
        const int dq = (int)(c >> 20), hq = (int)((c >> 10) & 1023u), wq = (int)(c & 1023u);
        xs[jj] = live ? s_x[js] : 0.f;
#pragma unroll
        for (int k = 0; k < ROUNDS; ++k) {
          // output voxel v with v + off(tap) = u
          const bool ok = live && (unsigned)(dq - tdd[k]) < (unsigned)D && (unsigned)(hq - tdh[k]) < (unsigned)H &&
                          (unsigned)(wq - tdw[k]) < (unsigned)W;
          g[jj][k] = make_uint4(0u, 0u, 0u, 0u);
          if (ok) g[jj][k] = __ldg(reinterpret_cast<const uint4*>(dyc + (long long)(u - toff[k]) * lddy));
        }
      }
#pragma unroll
      for (int jj = 0; jj < 2; ++jj)
#pragma unroll
        for (int k = 0; k < ROUNDS; ++k) {
          const uint32_t wd[4] = {g[jj][k].x, g[jj][k].y, g[jj][k].z, g[jj][k].w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            acc[k][2 * e] = fmaf(xs[jj], __uint_as_float(wd[e] << 16), acc[k][2 * e]);
            acc[k][2 * e + 1] = fmaf(xs[jj], __uint_as_float(wd[e] & 0xffff0000u), acc[k][2 * e + 1]);
          }
        }
    }
    __syncthreads();   // the list is rebuilt by the next sub-chunk
  }
  // deterministic block reduction: warps add their registers one after another (no float atomics)
  for (int w = 0; w < 8; ++w) {
    if (warp == w) {
#pragma unroll
      for (int k = 0; k < ROUNDS; ++k) {
        const int tap = slot + PPL * k;
        if (tap < 27) {
#pragma unroll
          for (int e = 0; e < 8; ++e) red[tap * COUT + cq * 8 + e] += acc[k][e];
        }
      }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < 27 * COUT; i += blockDim.x) partial[(size_t)blockIdx.x * 27 * COUT + i] = red[i];
}

// fixed-order sum of the per-block partials: block = 32 outputs x 8 row groups, fp64
__global__ void __launch_bounds__(256)
conv_first_wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, int nblocks, int Cout) {
  pdl_prologue();
  __shared__ double red[8][32];
  const int o = threadIdx.x & 31, rg = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + o;  // i = tap*Cout + co
  const int total = 27 * Cout;
  double acc = 0.0;
  if (i < total) {
    int r = rg;
    for (; r + 24 < nblocks; r += 32) {
      const float a0 = partial[(size_t)r * total + i], a1 = partial[(size_t)(r + 8) * total + i];
      const float a2 = partial[(size_t)(r + 16) * total + i], a3 = partial[(size_t)(r + 24) * total + i];
      acc += ((double)a0 + (double)a1) + ((double)a2 + (double)a3);
    }
    for (; r < nblocks; r += 8) acc += (double)partial[(size_t)r * total + i];
  }
  red[rg][o] = acc;
  __syncthreads();
  if (rg != 0 || i >= total) return;
#pragma unroll
  for (int k = 1; k < 8; ++k) acc += red[k][o];
  const int tap = i / Cout, co = i % Cout;
  dw[co * 27 + tap] = (float)acc;
}

static constexpr int kFirstWgradBlocks = 592;
static constexpr int kFirstFwdStatBlocks = 148 * 4;

}  // namespace b2

using namespace b2;

static int conv_first_fwd_impl(const float* x, const float* w, void* y, int ldy, int y_coff, int N, int D, int H,
                               int W, int Cout, int relu, long long* stat_acc, const float* bias,
                               cudaStream_t stream) {
  B2_REQUIRE(x && w && y, "b2_conv3d_first_fwd: null pointer");
  B2_REQUIRE(ldy % 8 == 0 && y_coff % 8 == 0, "b2_conv3d_first_fwd: ldy/y_coff must be multiples of 8");
  const long long V = (long long)N * D * H * W;
  long long blocks = (V + 127) / 128;
  const long long cap = stat_acc ? (long long)kFirstFwdStatBlocks : (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  __nv_bfloat16* yy = reinterpret_cast<__nv_bfloat16*>(y);
  switch (Cout) {
    case 16: B2_LAUNCH(conv_first_fwd_kernel<16>, (unsigned)blocks, 128, 0, stream, x, w, yy, N, D, H, W, ldy, y_coff, relu, stat_acc, bias); break;
    case 32: B2_LAUNCH(conv_first_fwd_kernel<32>, (unsigned)blocks, 128, 0, stream, x, w, yy, N, D, H, W, ldy, y_coff, relu, stat_acc, bias); break;
    case 64: B2_LAUNCH(conv_first_fwd_kernel<64>, (unsigned)blocks, 128, 0, stream, x, w, yy, N, D, H, W, ldy, y_coff, relu, stat_acc, bias); break;
    default:
      set_error("b2_conv3d_first_fwd: Cout=%d unsupported (16, 32 or 64)", Cout);
      return B2_ERR_UNSUPPORTED;
  }
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

extern "C" int b2_conv3d_first_fwd(const float* x, const float* w, void* y, int ldy, int y_coff, int N, int D, int H,
                                   int W, int Cout, int relu, cudaStream_t stream) {
  return conv_first_fwd_impl(x, w, y, ldy, y_coff, N, D, H, W, Cout, relu, nullptr, nullptr, stream);
}

// Same, with the GroupNorm statistics of the stored output fused in (batch 1): stat_acc int64 [Cout][4] exact
// accumulators (zero before the launch), consumed by b2_relu_gn_apply_acc.
extern "C" int b2_conv3d_first_fwd_stats(const float* x, const float* w, void* y, int ldy, int y_coff, int N, int D,
                                         int H, int W, int Cout, int relu, long long* stat_acc, cudaStream_t stream) {
  B2_REQUIRE(stat_acc, "b2_conv3d_first_fwd_stats: null pointer");
  B2_REQUIRE(N == 1, "b2_conv3d_first_fwd_stats: fused statistics need batch 1");
  return conv_first_fwd_impl(x, w, y, ldy, y_coff, N, D, H, W, Cout, relu, stat_acc, nullptr, stream);
}

// Same with a conv bias (fp32 [Cout]) added before ReLU; stat_acc may be NULL (no statistics) and needs batch 1.
extern "C" int b2_conv3d_first_fwd_bias(const float* x, const float* w, const float* bias, void* y, int ldy, int y_coff,
                                        int N, int D, int H, int W, int Cout, int relu, long long* stat_acc,
                                        cudaStream_t stream) {
  B2_REQUIRE(bias, "b2_conv3d_first_fwd_bias: null bias");
  B2_REQUIRE(!stat_acc || N == 1, "b2_conv3d_first_fwd_bias: fused statistics need batch 1");
  return conv_first_fwd_impl(x, w, y, ldy, y_coff, N, D, H, W, Cout, relu, stat_acc, bias, stream);
}

extern "C" long long b2_conv3d_first_wgrad_workspace_bytes(int Cout) {
  return (long long)kFirstWgradBlocks * 27 * Cout * (long long)sizeof(float);
}

extern "C" int b2_conv3d_first_wgrad(const float* x, const void* dy, int lddy, int dy_coff, float* dw, void* workspace,
                                     long long workspace_bytes, int N, int D, int H, int W, int Cout,
                                     cudaStream_t stream) {
  B2_REQUIRE(x && dy && dw && workspace, "b2_conv3d_first_wgrad: null pointer");
  B2_REQUIRE(Cout == 16 || Cout == 32 || Cout == 64, "b2_conv3d_first_wgrad: Cout=%d unsupported (16, 32 or 64)", Cout);
  B2_REQUIRE(workspace_bytes >= b2_conv3d_first_wgrad_workspace_bytes(Cout), "b2_conv3d_first_wgrad: workspace too small");
  B2_REQUIRE(D < 1024 && H < 1024 && W < 1024 && (long long)N * D * H * W < (1LL << 31),
             "b2_conv3d_first_wgrad: volume %dx%dx%dx%d too large", N, D, H, W);
  float* partial = reinterpret_cast<float*>(workspace);
  const long long V = (long long)N * D * H * W;
  long long per_block = (V + kFirstWgradBlocks - 1) / kFirstWgradBlocks;
  per_block = (per_block + 255) / 256 * 256;
  const int blocks = (int)((V + per_block - 1) / per_block);
  B2_REQUIRE(lddy % 8 == 0 && dy_coff % 8 == 0, "b2_conv3d_first_wgrad: lddy/dy_coff must be multiples of 8");
  auto* dyb = reinterpret_cast<const __nv_bfloat16*>(dy);
  if (Cout == 16)
    B2_LAUNCH(conv_first_wgrad_kernel<16>, blocks, 256, 0, stream, x, dyb, lddy, dy_coff, partial, N, D, H, W, per_block);
  else if (Cout == 32)
    B2_LAUNCH(conv_first_wgrad_kernel<32>, blocks, 256, 0, stream, x, dyb, lddy, dy_coff, partial, N, D, H, W, per_block);
  else
    B2_LAUNCH(conv_first_wgrad_kernel<64>, blocks, 256, 0, stream, x, dyb, lddy, dy_coff, partial, N, D, H, W, per_block);
  B2_CHECK_CUDA(cudaGetLastError());
  B2_LAUNCH(conv_first_wgrad_reduce_kernel, (27 * Cout + 31) / 32, 256, 0, stream, partial, dw, blocks, Cout);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}
