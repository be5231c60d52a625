// GroupNorm over post-ReLU activations ('crg' order: conv -> ReLU -> GroupNorm), NDHWC bf16, fp32 statistics.
//
// forward : stats pass  (sum x, sum x^2 per channel, per-block partials; the last block to finish reduces them in
//                        a fixed order -> per (n, group) mean, rstd; per (n, channel) scale = rstd*gamma,
//                        shift = beta - mean*scale; deterministic, no separate finalize launch)
//           apply pass  y = r*scale + shift  (optionally also writes the 2x2x2 max-pooled tensor in the same read)
// backward: stats pass  (sum dy, sum dy*xhat per channel), finalize (group sums, dgamma, dbeta, per-channel coefs),
//           apply pass  dr = relu'(r) * rstd*(dy*gamma - mean_g(dy*gamma) - xhat*mean_g(dy*gamma*xhat))
// All kernels are HBM-bound: one 16-byte (8-channel) vector per thread per voxel, coalesced along channels.
#include "common.h"
#include "vec.cuh"

namespace b2 {

static constexpr int kStatBlocks = 296;  // 2 x 148 SMs (upper bound; small tensors use fewer, >= 64 KB per block)
static constexpr int kStatThreads = 256;

// ------------------------------------------------------------------------------------------------- forward stats
// The block that finishes last (per sample, ticket from an integer atomic) reduces the per-block partials in a
// fixed order and writes mean/rstd and the per-channel scale/shift: deterministic, and no separate finalize launch.
__device__ __forceinline__ bool last_block_done(int* counter, int total) {
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(counter, 1) == total - 1) ? 1 : 0;
  __syncthreads();
  if (s_last) __threadfence();
  return s_last != 0;
}

// Last block only: per-channel totals over the per-block partials -> csum[C][2] (double, shared memory).
// L = 256/C lanes cooperate per channel (independent loads in flight), combined in a fixed order.
__device__ __forceinline__ void reduce_partials(const float* __restrict__ partial, int n, int nblk, int C,
                                                double* csum) {
  const int nthr = blockDim.x;
  const int L = (C >= nthr) ? 1 : (nthr / C > 32 ? 32 : nthr / C);   // lanes per channel: power of two <= 32
  const int sub = threadIdx.x % L;
  for (int c = threadIdx.x / L; c < C; c += nthr / L) {
    double a = 0.0, b = 0.0;
    const float* base = partial + ((size_t)n * nblk * C + c) * 2;
    int blk = sub;
    for (; blk + 7 * L < nblk; blk += 8 * L) {   // 8 independent loads in flight
      float2 pp[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) pp[k] = __ldcg(reinterpret_cast<const float2*>(base + (size_t)(blk + k * L) * C * 2));
#pragma unroll
      for (int k = 0; k < 8; ++k) { a += (double)pp[k].x; b += (double)pp[k].y; }
    }
    for (; blk + 3 * L < nblk; blk += 4 * L) {
      const float2 p0 = __ldcg(reinterpret_cast<const float2*>(base + (size_t)blk * C * 2));
      const float2 p1 = __ldcg(reinterpret_cast<const float2*>(base + (size_t)(blk + L) * C * 2));
      const float2 p2 = __ldcg(reinterpret_cast<const float2*>(base + (size_t)(blk + 2 * L) * C * 2));
      const float2 p3 = __ldcg(reinterpret_cast<const float2*>(base + (size_t)(blk + 3 * L) * C * 2));
      a += ((double)p0.x + (double)p1.x) + ((double)p2.x + (double)p3.x);
      b += ((double)p0.y + (double)p1.y) + ((double)p2.y + (double)p3.y);
    }
    for (; blk < nblk; blk += L) {
      const float2 p0 = __ldcg(reinterpret_cast<const float2*>(base + (size_t)blk * C * 2));
      a += (double)p0.x;
      b += (double)p0.y;
    }
    for (int o = L >> 1; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (sub == 0) { csum[2 * c] = a; csum[2 * c + 1] = b; }
  }
}

__global__ void __launch_bounds__(kStatThreads)
gn_stats_kernel(const __nv_bfloat16* __restrict__ r, long long V, int C, float* __restrict__ partial, int* counters,
                int G, float eps, const float* __restrict__ gamma, const float* __restrict__ beta,
                float* __restrict__ mean_rstd, float* __restrict__ scale_shift) {
  pdl_prologue();
  extern __shared__ float sh[];  // [vpi][C][2]
  const int C8 = C >> 3;
  const int vpi = kStatThreads / C8;
  const int oct = threadIdx.x % C8;
  const int vloc = threadIdx.x / C8;
  const int n = blockIdx.y;
  const int nblk = gridDim.x;
  const __nv_bfloat16* rn = r + (size_t)n * V * C + oct * 8;
  float s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { s[i] = 0.f; q[i] = 0.f; }
  {
    const long long stride = (long long)nblk * vpi;
    long long v = (long long)blockIdx.x * vpi + vloc;
    for (; v + 3 * stride < V; v += 4 * stride) {   // 4 independent 16-byte loads in flight per thread
      const uint4 u0 = ldg16(rn + v * C), u1 = ldg16(rn + (v + stride) * C);
      const uint4 u2 = ldg16(rn + (v + 2 * stride) * C), u3 = ldg16(rn + (v + 3 * stride) * C);
      const f8 x0 = unpack8(u0), x1 = unpack8(u1), x2 = unpack8(u2), x3 = unpack8(u3);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s[i] += (x0.v[i] + x1.v[i]) + (x2.v[i] + x3.v[i]);
        q[i] = fmaf(x0.v[i], x0.v[i], fmaf(x1.v[i], x1.v[i], fmaf(x2.v[i], x2.v[i], fmaf(x3.v[i], x3.v[i], q[i]))));
      }
    }
    for (; v < V; v += stride) {
      const f8 x = unpack8(ldg16(rn + v * C));
#pragma unroll
      for (int i = 0; i < 8; ++i) { s[i] += x.v[i]; q[i] = fmaf(x.v[i], x.v[i], q[i]); }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    sh[((size_t)vloc * C + oct * 8 + i) * 2 + 0] = s[i];
    sh[((size_t)vloc * C + oct * 8 + i) * 2 + 1] = q[i];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 0.f, b = 0.f;
    for (int j = 0; j < vpi; ++j) { a += sh[((size_t)j * C + c) * 2]; b += sh[((size_t)j * C + c) * 2 + 1]; }
    float* dst = partial + (((size_t)n * nblk + blockIdx.x) * C + c) * 2;
    dst[0] = a;
    dst[1] = b;
  }
  if (!last_block_done(&counters[n], nblk)) return;
  // ---- finalize sample n
  __syncthreads();
  double* csum = reinterpret_cast<double*>(sh);   // C*16 bytes <= the pass-1 scratch
  reduce_partials(partial, n, nblk, C, csum);
  __syncthreads();
  const int cpg = C / G;
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    double a = 0.0, b = 0.0;
    for (int k = 0; k < cpg; ++k) { a += csum[2 * (g * cpg + k)]; b += csum[2 * (g * cpg + k) + 1]; }
    const double m = (double)V * cpg;
    const double mean = a / m;
    double var = b / m - mean * mean;
    if (var < 0.0) var = 0.0;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    for (int k = 0; k < cpg; ++k) {
      const int c = g * cpg + k;
      const float sc = rstd * gamma[c];
      mean_rstd[((size_t)n * C + c) * 2 + 0] = (float)mean;
      mean_rstd[((size_t)n * C + c) * 2 + 1] = rstd;
      scale_shift[((size_t)n * C + c) * 2 + 0] = sc;
      scale_shift[((size_t)n * C + c) * 2 + 1] = beta[c] - (float)mean * sc;
    }
  }
  if (threadIdx.x == 0) counters[n] = 0;   // self-resetting ticket
}

// ---- statistics from the fixed-point accumulators (common.h) --------------------------------------------------------------
// The producers leave per-channel fixed-point sums in int64 [C][4]; one small block turns them into what the apply kernels
// read.  Reading C accumulators instead of ~148 x C fp32 partials makes this a ~3 us kernel (one L2 round trip, fp64
// only for the C conversions and the G group sums; no fp64 division or square root: 1/m comes from the host and rstd
// is rsqrtf + one Newton step on the well-conditioned variance).
// (Tried and measured slower, round 1: finalising in the prologue of EVERY block of the apply kernels — the dependent
// L2 round trips under a saturated memory system cost +13..35 us per launch.)
static constexpr int kMaxAccC = 512;

__device__ __forceinline__ float rstd_from_var(double var_eps) {
  const float v = (float)var_eps;
  float r = rsqrtf(v);
  return r * (1.5f - 0.5f * v * r * r);
}

__global__ void __launch_bounds__(kMaxAccC)
gn_finalize_acc_kernel(const long long* __restrict__ acc, int C, int G, double inv_m, float eps,
                       const float* __restrict__ gamma, const float* __restrict__ beta,
                       float* __restrict__ mean_rstd, float* __restrict__ scale_shift) {
  pdl_prologue();
  __shared__ double s_c[kMaxAccC][2];
  __shared__ float s_g[kMaxAccC][2];
  const int c = threadIdx.x;
  const int cpg = C / G;
  float gm = 0.f, bt = 0.f;
  if (c < C) {
    gm = gamma[c];
    bt = beta[c];
    s_c[c][0] = stat_read(acc + 4 * c);
    s_c[c][1] = stat_read(acc + 4 * c + 2);
  }
  __syncthreads();
  if (c < G) {
    double S = 0.0, Q = 0.0;
    for (int k = 0; k < cpg; ++k) { S += s_c[c * cpg + k][0]; Q += s_c[c * cpg + k][1]; }
    const double mean = S * inv_m;
    double var = Q * inv_m - mean * mean;
    if (var < 0.0) var = 0.0;
    s_g[c][0] = (float)mean;
    s_g[c][1] = rstd_from_var(var + (double)eps);
  }
  __syncthreads();
  if (c < C) {
    const float mean = s_g[c / cpg][0], rstd = s_g[c / cpg][1];
    const float sc = rstd * gm;
    mean_rstd[2 * c] = mean;
    mean_rstd[2 * c + 1] = rstd;
    scale_shift[2 * c] = sc;
    scale_shift[2 * c + 1] = bt - mean * sc;
  }
}

// backward: (sum dy, sum dy*r) per channel -> coef[c] = {a, b, c0, 0} (dr = a*dy + b*xhat + c0), dgamma, dbeta
__global__ void __launch_bounds__(kMaxAccC)
gn_bwd_finalize_acc_kernel(const long long* __restrict__ acc, int C, int G, double inv_m,
                           const float* __restrict__ gamma, const float* __restrict__ mean_rstd,
                           float* __restrict__ coef, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  pdl_prologue();
  __shared__ double s_c[kMaxAccC][2];
  __shared__ float s_g[kMaxAccC][2];
  const int c = threadIdx.x;
  const int cpg = C / G;
  float gm = 0.f, rstd = 0.f;
  if (c < C) {
    gm = gamma[c];
    const float mu = mean_rstd[2 * c];
    rstd = mean_rstd[2 * c + 1];
    const double sdy = stat_read(acc + 4 * c), sdyr = stat_read(acc + 4 * c + 2);
    const double sdyx = (double)rstd * (sdyr - (double)mu * sdy);   // sum dy*xhat
    s_c[c][0] = (double)gm * sdy;
    s_c[c][1] = (double)gm * sdyx;
    if (dgamma) dgamma[c] = (float)sdyx;
    if (dbeta) dbeta[c] = (float)sdy;
  }
  __syncthreads();
  if (c < G) {
    double S1 = 0.0, S2 = 0.0;
    for (int k = 0; k < cpg; ++k) { S1 += s_c[c * cpg + k][0]; S2 += s_c[c * cpg + k][1]; }
    s_g[c][0] = (float)(S2 * inv_m);
    s_g[c][1] = (float)(S1 * inv_m);
  }
  __syncthreads();
  if (c < C) {
    // dr = relu'(r) * (a*dy + b*xhat + c0), xhat = (r - mu)*rstd  ==  relu'(r) * (a*dy + kb*r + kc): the apply kernel
    // reads {a, kb, kc} as ONE 16-byte load per channel (it used to read mean/rstd as well and fold them itself)
    const float b = -rstd * s_g[c / cpg][0], c0 = -rstd * s_g[c / cpg][1];
    const float mu = mean_rstd[2 * c];
    float* o = coef + (size_t)c * 4;
    o[0] = rstd * gm;
    o[1] = b * rstd;
    o[2] = c0 - b * rstd * mu;
    o[3] = 0.f;
  }
}

// Blocks for the apply kernels (one channel octet of one voxel per thread and loop trip).  Every thread pays a fixed
// prologue (4-8 coefficient loads): a thread should own >= 4..8 voxels, but a small tensor must still cover one full
// resident wave (4 blocks/SM).  ncu, round 2: with one voxel per thread the 24x28x24 levels ran at 0.6-0.9 TB/s with the
// load-store unit throttled by the coefficient loads (lg_throttle 15 stall cycles per issue).
static inline int apply_blocks(long long items) {
  const long long wave = (long long)num_sms() * 4;
  const long long nb8 = (items + 2047) / 2048, nb2 = (items + 511) / 512;
  long long nb = nb8 >= wave ? nb8 : (nb2 < wave ? nb2 : wave);
  const long long cap = (long long)num_sms() * 16;
  if (nb > cap) nb = cap;
  if (nb < 1) nb = 1;
  return (int)nb;
}

// ------------------------------------------------------------------------------------------------- forward apply
// grid = (blocks, N).  A thread keeps one channel octet (256 % C8 == 0) and walks voxels with pointer increments only
// (no 64-bit divisions in the loop), two independent 16-byte loads in flight.
__global__ void __launch_bounds__(256)
gn_apply_kernel(const __nv_bfloat16* __restrict__ r, long long V, int C, const float* __restrict__ scale_shift,
                __nv_bfloat16* __restrict__ y, int ldy, int y_coff) {
  pdl_prologue();
  const int C8 = C >> 3;
  const int n = blockIdx.y;
  const int oct = threadIdx.x % C8;
  const int vpb = 256 / C8;                                   // voxels per block per sweep
  const long long vstride = (long long)gridDim.x * vpb;
  long long v = (long long)blockIdx.x * vpb + threadIdx.x / C8;
  float sc[8], sh[8];
  const float4* ss = reinterpret_cast<const float4*>(scale_shift + ((size_t)n * C + oct * 8) * 2);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float4 t = __ldg(ss + k);
    sc[2 * k] = t.x; sh[2 * k] = t.y; sc[2 * k + 1] = t.z; sh[2 * k + 1] = t.w;
  }
  const __nv_bfloat16* rp = r + ((size_t)n * V) * C + oct * 8;
  __nv_bfloat16* yp = y + ((size_t)n * V) * ldy + y_coff + oct * 8;
  for (; v + 3 * vstride < V; v += 4 * vstride) {   // 4 independent 16-byte loads in flight per thread
    uint4 u[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) u[j] = ldg16(rp + (v + j * vstride) * C);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const f8 x = unpack8(u[j]);
      f8 o;
#pragma unroll
      for (int k = 0; k < 8; ++k) o.v[k] = fmaf(x.v[k], sc[k], sh[k]);
      stg16(yp + (v + j * vstride) * ldy, pack8(o));
    }
  }
  for (; v + vstride < V; v += 2 * vstride) {
    const uint4 u0 = ldg16(rp + v * C), u1 = ldg16(rp + (v + vstride) * C);
    const f8 x0 = unpack8(u0), x1 = unpack8(u1);
    f8 o0, o1;
#pragma unroll
    for (int k = 0; k < 8; ++k) { o0.v[k] = fmaf(x0.v[k], sc[k], sh[k]); o1.v[k] = fmaf(x1.v[k], sc[k], sh[k]); }
    stg16(yp + v * ldy, pack8(o0));
    stg16(yp + (v + vstride) * ldy, pack8(o1));
  }
  for (; v < V; v += vstride) {
    const f8 x = unpack8(ldg16(rp + v * C));
    f8 o;
#pragma unroll
    for (int k = 0; k < 8; ++k) o.v[k] = fmaf(x.v[k], sc[k], sh[k]);
    stg16(yp + v * ldy, pack8(o));
  }
}

// apply + MaxPool3d(2,2,0): one thread per (2x2x2 cell, channel octet); also covers odd tails (no pooled output)
__global__ void __launch_bounds__(256)
gn_apply_pool_kernel(const __nv_bfloat16* __restrict__ r, int N, int D, int H, int W, int C,
                     const float* __restrict__ scale_shift, __nv_bfloat16* __restrict__ y, int ldy, int y_coff,
                     __nv_bfloat16* __restrict__ pooled /*[N][D/2][H/2][W/2][C]*/) {
  pdl_prologue();
  const int C8 = C >> 3;
  const int Dc = (D + 1) >> 1, Hc = (H + 1) >> 1, Wc = (W + 1) >> 1;
  const int Dp = D >> 1, Hp = H >> 1, Wp = W >> 1;
  const long long total = (long long)N * Dc * Hc * Wc * C8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int oct = (int)(i % C8);
    long long t = i / C8;
    const int cw = (int)(t % Wc); t /= Wc;
    const int ch = (int)(t % Hc); t /= Hc;
    const int cd = (int)(t % Dc);
    const int n = (int)(t / Dc);
    float sc[8], sh[8];
    const float4* ss = reinterpret_cast<const float4*>(scale_shift + ((size_t)n * C + oct * 8) * 2);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float4 q = __ldg(ss + k);
      sc[2 * k] = q.x; sh[2 * k] = q.y; sc[2 * k + 1] = q.z; sh[2 * k + 1] = q.w;
    }
    f8 mx;
#pragma unroll
    for (int k = 0; k < 8; ++k) mx.v[k] = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int d = 2 * cd + (j >> 2), h = 2 * ch + ((j >> 1) & 1), w = 2 * cw + (j & 1);
      if (d < D && h < H && w < W) {
        const long long v = (((long long)n * D + d) * H + h) * W + w;
        const f8 x = unpack8(ldg16(r + v * C + oct * 8));
        f8 o;
#pragma unroll
        for (int k = 0; k < 8; ++k) o.v[k] = fmaf(x.v[k], sc[k], sh[k]);
        const uint4 pk = pack8(o);
        stg16(y + v * ldy + y_coff + oct * 8, pk);
        const f8 ro = unpack8(pk);  // pool the bf16-rounded values (what the next layer reads)
#pragma unroll
        for (int k = 0; k < 8; ++k) mx.v[k] = fmaxf(mx.v[k], ro.v[k]);
      }
    }
    if (cd < Dp && ch < Hp && cw < Wp) {
      const long long pv = (((long long)n * Dp + cd) * Hp + ch) * Wp + cw;
      stg16(pooled + pv * C + oct * 8, pack8(mx));
    }
  }
}

// ------------------------------------------------------------------------------------------------- backward stats
// coef[n][c] = {a, b, c0, pad}: dr = a*dy + b*xhat + c0.  The last block per sample finalizes that sample; the last
// of those sums dgamma/dbeta over the samples (fixed order).
__global__ void __launch_bounds__(kStatThreads)
gn_bwd_stats_kernel(const __nv_bfloat16* __restrict__ dy, int lddy, int dy_coff, const __nv_bfloat16* __restrict__ r,
                    long long V, int C, const float* __restrict__ mean_rstd, float* __restrict__ partial,
                    int* counters, int N, int G, const float* __restrict__ gamma, float* __restrict__ coef,
                    float* __restrict__ dgb_n /*[N][C][2]*/, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  pdl_prologue();
  extern __shared__ float sh[];
  const int C8 = C >> 3;
  const int vpi = kStatThreads / C8;
  const int oct = threadIdx.x % C8;
  const int vloc = threadIdx.x / C8;
  const int n = blockIdx.y;
  const int nblk = gridDim.x;
  const __nv_bfloat16* rn = r + (size_t)n * V * C + oct * 8;
  const __nv_bfloat16* dyn = dy + (size_t)n * V * lddy + dy_coff + oct * 8;
  float mu[8], rs[8], s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    mu[i] = mean_rstd[((size_t)n * C + oct * 8 + i) * 2];
    rs[i] = mean_rstd[((size_t)n * C + oct * 8 + i) * 2 + 1];
    s[i] = 0.f;
    q[i] = 0.f;
  }
  {
    const long long stride = (long long)nblk * vpi;
    long long v = (long long)blockIdx.x * vpi + vloc;
    for (; v + stride < V; v += 2 * stride) {   // 4 independent 16-byte loads in flight per thread
      const uint4 ux0 = ldg16(rn + v * C), ug0 = ldg16(dyn + v * lddy);
      const uint4 ux1 = ldg16(rn + (v + stride) * C), ug1 = ldg16(dyn + (v + stride) * lddy);
      const f8 x0 = unpack8(ux0), g0 = unpack8(ug0), x1 = unpack8(ux1), g1 = unpack8(ug1);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s[i] += g0.v[i] + g1.v[i];
        q[i] = fmaf(g0.v[i], (x0.v[i] - mu[i]) * rs[i], fmaf(g1.v[i], (x1.v[i] - mu[i]) * rs[i], q[i]));
      }
    }
    for (; v < V; v += stride) {
      const f8 x = unpack8(ldg16(rn + v * C));
      const f8 g = unpack8(ldg16(dyn + v * lddy));
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s[i] += g.v[i];
        q[i] = fmaf(g.v[i], (x.v[i] - mu[i]) * rs[i], q[i]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    sh[((size_t)vloc * C + oct * 8 + i) * 2 + 0] = s[i];
    sh[((size_t)vloc * C + oct * 8 + i) * 2 + 1] = q[i];
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float a = 0.f, b = 0.f;
    for (int j = 0; j < vpi; ++j) { a += sh[((size_t)j * C + c) * 2]; b += sh[((size_t)j * C + c) * 2 + 1]; }
    float* dst = partial + (((size_t)n * nblk + blockIdx.x) * C + c) * 2;
    dst[0] = a;
    dst[1] = b;
  }
  if (!last_block_done(&counters[n], nblk)) return;
  // ---- finalize sample n
  __syncthreads();
  double* csum = reinterpret_cast<double*>(sh);   // [C][2] per-channel sums over blocks (C*16 bytes <= smem of pass 1)
  reduce_partials(partial, n, nblk, C, csum);
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    dgb_n[((size_t)n * C + c) * 2 + 0] = (float)csum[2 * c + 1];   // d gamma contribution of sample n
    dgb_n[((size_t)n * C + c) * 2 + 1] = (float)csum[2 * c];       // d beta
  }
  __syncthreads();
  const int cpg = C / G;
  for (int g = threadIdx.x; g < G; g += blockDim.x) {
    double S1 = 0.0, S2 = 0.0;
    for (int k = 0; k < cpg; ++k) {
      const double gm = (double)gamma[g * cpg + k];
      S1 += gm * csum[2 * (g * cpg + k)];
      S2 += gm * csum[2 * (g * cpg + k) + 1];
    }
    const double m = (double)V * cpg;
    for (int k = 0; k < cpg; ++k) {
      const int c = g * cpg + k;
      const float mu_f = mean_rstd[((size_t)n * C + c) * 2], rstd_f = mean_rstd[((size_t)n * C + c) * 2 + 1];
      const double rstd = (double)rstd_f;
      const float b = (float)(-rstd * S2 / m), c0 = (float)(-rstd * S1 / m);
      float* o = coef + ((size_t)n * C + c) * 4;   // {a, kb, kc}: see gn_bwd_finalize_acc_kernel
      o[0] = (float)(rstd * (double)gamma[c]);
      o[1] = b * rstd_f;
      o[2] = c0 - b * rstd_f * mu_f;
      o[3] = 0.f;
    }
  }
  if (threadIdx.x == 0) counters[n] = 0;
  if (!last_block_done(&counters[N], N)) return;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float dg = 0.f, db = 0.f;
    for (int k = 0; k < N; ++k) {
      const float2 v2 = __ldcg(reinterpret_cast<const float2*>(dgb_n + ((size_t)k * C + c) * 2));
      dg += v2.x;
      db += v2.y;
    }
    if (dgamma) dgamma[c] = dg;
    if (dbeta) dbeta[c] = db;
  }
  if (threadIdx.x == 0) counters[N] = 0;
}

// kBias (layers with a conv bias): the kernel also sums the STORED (bf16-rounded) dr per channel — the bias gradient.
// Each thread keeps fp32 running sums of its channel octet, the block combines them in thread order through shared
// memory and commits one fixed-point atomic per channel into dbias_acc int64 [C][2] (common.h): bit-identical run to run.
// Separate instantiations: neither the label test nor the sums touch the code of the other launches.
template <bool kRowLabels, bool kBias>
__global__ void __launch_bounds__(256)
gn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ dy, int lddy, int dy_coff, const __nv_bfloat16* __restrict__ r,
                    long long V, int C, const float* __restrict__ mean_rstd, const float* __restrict__ coef,
                    __nv_bfloat16* __restrict__ dr, const long long* __restrict__ row_labels,
                    long long* __restrict__ dbias_acc) {
  pdl_prologue();
  // row_labels != NULL (gradient produced by the head kernel): dy rows of voxels with label < 0 were never written
  // and count as zero — they are not read (no memset of dy, 97 % of its rows skipped)
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  const int C8 = C >> 3;
  const int n = blockIdx.y;
  const int oct = threadIdx.x % C8;
  const int vpb = 256 / C8;
  const long long vstride = (long long)gridDim.x * vpb;
  long long v = (long long)blockIdx.x * vpb + threadIdx.x / C8;
  // dr = relu'(r) * (ca*dy + cb*xhat + cc) with xhat = (r - mu)*rs  ==  relu'(r) * (ca*dy + kb*r + kc)
  float ca[8], kb[8], kc[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float4 cf = __ldg(reinterpret_cast<const float4*>(coef + ((size_t)n * C + oct * 8 + k) * 4));
    ca[k] = cf.x;
    kb[k] = cf.y;
    kc[k] = cf.z;
  }
  float sb[8];   // kBias: running sums of the stored dr of this thread's channel octet
#pragma unroll
  for (int k = 0; k < 8; ++k) sb[k] = 0.f;
  auto add_bias_sums = [&](const uint4& stored) {
    if constexpr (kBias) {
      const f8 q = unpack8(stored);
#pragma unroll
      for (int k = 0; k < 8; ++k) sb[k] += q.v[k];
    }
  };
  const __nv_bfloat16* rp = r + ((size_t)n * V) * C + oct * 8;
  const __nv_bfloat16* gp = dy + ((size_t)n * V) * lddy + dy_coff + oct * 8;
  __nv_bfloat16* op = dr + ((size_t)n * V) * C + oct * 8;
  for (; v + 3 * vstride < V; v += 4 * vstride) {   // 8 independent 16-byte loads in flight per thread
    bool lb[4];
    uint4 ux[4], ug[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) lb[j] = !kRowLabels || __ldg(row_labels + (size_t)n * V + v + j * vstride) >= 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      ux[j] = ldg16(rp + (v + j * vstride) * C);
      ug[j] = lb[j] ? ldg16(gp + (v + j * vstride) * lddy) : zero4;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const f8 x = unpack8(ux[j]), g = unpack8(ug[j]);
      f8 o;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const float d = fmaf(ca[k], g.v[k], fmaf(kb[k], x.v[k], kc[k]));
        o.v[k] = x.v[k] > 0.f ? d : 0.f;
      }
      const uint4 pk = pack8(o);
      add_bias_sums(pk);
      stg16(op + (v + j * vstride) * C, pk);
    }
  }
  for (; v + vstride < V; v += 2 * vstride) {
    const bool l0 = !kRowLabels || __ldg(row_labels + (size_t)n * V + v) >= 0;
    const bool l1 = !kRowLabels || __ldg(row_labels + (size_t)n * V + v + vstride) >= 0;
    const uint4 ux0 = ldg16(rp + v * C), ug0 = l0 ? ldg16(gp + v * lddy) : zero4;
    const uint4 ux1 = ldg16(rp + (v + vstride) * C), ug1 = l1 ? ldg16(gp + (v + vstride) * lddy) : zero4;
    const f8 x0 = unpack8(ux0), g0 = unpack8(ug0), x1 = unpack8(ux1), g1 = unpack8(ug1);
    f8 o0, o1;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float d0 = fmaf(ca[k], g0.v[k], fmaf(kb[k], x0.v[k], kc[k]));
      const float d1 = fmaf(ca[k], g1.v[k], fmaf(kb[k], x1.v[k], kc[k]));
      o0.v[k] = x0.v[k] > 0.f ? d0 : 0.f;
      o1.v[k] = x1.v[k] > 0.f ? d1 : 0.f;
    }
    const uint4 pk0 = pack8(o0), pk1 = pack8(o1);
    add_bias_sums(pk0);
    add_bias_sums(pk1);
    stg16(op + v * C, pk0);
    stg16(op + (v + vstride) * C, pk1);
  }
  for (; v < V; v += vstride) {
    const bool l0 = !kRowLabels || __ldg(row_labels + (size_t)n * V + v) >= 0;
    const f8 x = unpack8(ldg16(rp + v * C));
    const f8 g = unpack8(l0 ? ldg16(gp + v * lddy) : zero4);
    f8 o;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float d = fmaf(ca[k], g.v[k], fmaf(kb[k], x.v[k], kc[k]));
      o.v[k] = x.v[k] > 0.f ? d : 0.f;
    }
    const uint4 pk = pack8(o);
    add_bias_sums(pk);
    stg16(op + v * C, pk);
  }
  if constexpr (kBias) {
    __shared__ float s_sb[256][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) s_sb[threadIdx.x][k] = sb[k];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {   // threads j * C8 + c / 8 hold channel c, summed in order of j
      float a = 0.f;
      for (int j = 0; j < vpb; ++j) a += s_sb[j * C8 + (c >> 3)][c & 7];
      stat_atomic_add(dbias_acc + 2 * c, a);
    }
  }
}

// dbias_acc int64 [C][2] -> dbias fp32 [C]
__global__ void __launch_bounds__(kMaxAccC)
dbias_finalize_kernel(const long long* __restrict__ dbias_acc, int C, float* __restrict__ dbias) {
  pdl_prologue();
  const int c = threadIdx.x;
  if (c < C) dbias[c] = (float)stat_read(dbias_acc + 2 * c);
}

static inline int stat_blocks(long long V, int C) {
  // >= 16 KB of the tensor per block (round 1: 256 KB per block left the 12x14x12 and 24x28x24 levels with 3..31
  // blocks and 35 us of pure latency per launch), and at most ~16 k partial pairs for the finalising block to sum
  long long nb = (V * C * 2) / 16384;
  const long long by_partials = 16384 / C;
  if (nb > by_partials) nb = by_partials;
  if (nb > kStatBlocks) nb = kStatBlocks;
  if (nb < 1) nb = 1;
  return (int)nb;
}
static inline int ew_blocks(long long total) {
  long long nb = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 16;
  if (nb > cap) nb = cap;
  if (nb < 1) nb = 1;
  return (int)nb;
}

}  // namespace b2

using namespace b2;

extern "C" long long b2_relu_gn_bwd_workspace_bytes(int N, int C);
extern "C" long long b2_gn_workspace_bytes(int N, int C) {
  return (long long)N * kStatBlocks * C * 2 * (long long)sizeof(float);
}

static int check_gn_shape(const char* who, int N, long long V, int C, int G) {
  B2_REQUIRE(N > 0 && V > 0, "%s: bad shape", who);
  B2_REQUIRE(C % 8 == 0 && C >= 8 && C / 8 <= kStatThreads && kStatThreads % (C / 8) == 0,
             "%s: C=%d unsupported (C/8 must divide %d)", who, C, kStatThreads);
  B2_REQUIRE(G > 0 && C % G == 0 && C / G <= 64 && kStatThreads % G == 0 && (kStatThreads / G) <= 32 &&
                 ((kStatThreads / G) & (kStatThreads / G - 1)) == 0,
             "%s: groups=%d unsupported for C=%d", who, G, C);
  B2_REQUIRE(N <= 1024, "%s: batch %d too large", who, N);
  return B2_OK;
}

// r: bf16 [N][V][C] dense.  Outputs mean_rstd [N][C][2], scale_shift [N][C][2] (fp32).
extern "C" int b2_relu_gn_stats(const void* r, int N, long long V, int C, int G, float eps, const float* gamma,
                                const float* beta, float* mean_rstd, float* scale_shift, void* workspace,
                                long long workspace_bytes, int* counters, cudaStream_t stream) {
  B2_REQUIRE(r && gamma && beta && mean_rstd && scale_shift && workspace && counters,
             "b2_relu_gn_stats: null pointer");
  int rc = check_gn_shape("b2_relu_gn_stats", N, V, C, G);
  if (rc) return rc;
  B2_REQUIRE(workspace_bytes >= b2_gn_workspace_bytes(N, C), "b2_relu_gn_stats: workspace too small");
  const int nblk = stat_blocks(V, C);
  const int vpi = kStatThreads / (C / 8);
  const size_t sh = (size_t)vpi * C * 2 * sizeof(float);
  B2_LAUNCH(gn_stats_kernel, dim3(nblk, N), kStatThreads, sh, stream, reinterpret_cast<const __nv_bfloat16*>(r), V, C,
                                                               reinterpret_cast<float*>(workspace), counters, G, eps,
                                                               gamma, beta, mean_rstd, scale_shift);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

// GroupNorm statistics (batch 1) from the fixed-point accumulators a producer kernel filled (b2_conv3d_igemm_stats,
// b2_conv3d_first_fwd_stats): stat_acc int64 [C][4] -> mean_rstd fp32 [C][2], scale_shift fp32 [C][2].
extern "C" int b2_relu_gn_finalize_acc(const long long* stat_acc, long long V, int C, int G, float eps,
                                       const float* gamma, const float* beta, float* mean_rstd, float* scale_shift,
                                       cudaStream_t stream) {
  B2_REQUIRE(stat_acc && gamma && beta && mean_rstd && scale_shift, "b2_relu_gn_finalize_acc: null pointer");
  int rc = check_gn_shape("b2_relu_gn_finalize_acc", 1, V, C, G);
  if (rc) return rc;
  B2_REQUIRE(C <= kMaxAccC, "b2_relu_gn_finalize_acc: C=%d > %d", C, kMaxAccC);
  B2_LAUNCH_DEP(gn_finalize_acc_kernel, 1, (C + 31) / 32 * 32, 0, stream, stat_acc, C, G, 1.0 / ((double)V * (C / G)), eps,
            gamma, beta, mean_rstd, scale_shift);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

// y[(n,v)*ldy + y_coff + c] = r*scale + shift.  If pooled != NULL also writes MaxPool3d(2) of y (needs D,H,W).
extern "C" int b2_relu_gn_apply(const void* r, int N, int D, int H, int W, int C, const float* scale_shift, void* y,
                                int ldy, int y_coff, void* pooled, cudaStream_t stream) {
  B2_REQUIRE(r && scale_shift && y, "b2_relu_gn_apply: null pointer");
  B2_REQUIRE(C % 8 == 0 && ldy % 8 == 0 && y_coff % 8 == 0, "b2_relu_gn_apply: channel counts must be multiples of 8");
  const long long V = (long long)D * H * W;
  if (pooled) {
    const long long total = (long long)N * ((D + 1) / 2) * ((H + 1) / 2) * ((W + 1) / 2) * (C / 8);
    B2_LAUNCH_DEP(gn_apply_pool_kernel, ew_blocks(total), 256, 0, stream, reinterpret_cast<const __nv_bfloat16*>(r), N, D,
              H, W, C, scale_shift, reinterpret_cast<__nv_bfloat16*>(y), ldy, y_coff,
              reinterpret_cast<__nv_bfloat16*>(pooled));
  } else {
    B2_REQUIRE(256 % (C / 8) == 0, "b2_relu_gn_apply: C=%d unsupported", C);
    B2_LAUNCH_DEP(gn_apply_kernel, dim3(apply_blocks(V * (C / 8)), N), 256, 0, stream,
              reinterpret_cast<const __nv_bfloat16*>(r), V, C, scale_shift, reinterpret_cast<__nv_bfloat16*>(y), ldy,
              y_coff);
  }
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

// dr = relu'(r) * GroupNorm-backward(dy);  dgamma/dbeta fp32 [C] (overwritten; may be NULL)
extern "C" int b2_relu_gn_bwd(const void* dy, int lddy, int dy_coff, const void* r, int N, long long V, int C, int G,
                              const float* gamma, const float* mean_rstd, void* dr, float* dgamma, float* dbeta,
                              void* workspace, long long workspace_bytes, int* counters, cudaStream_t stream) {
  B2_REQUIRE(dy && r && gamma && mean_rstd && dr && workspace && counters, "b2_relu_gn_bwd: null pointer");
  int rc = check_gn_shape("b2_relu_gn_bwd", N, V, C, G);
  if (rc) return rc;
  B2_REQUIRE(lddy % 8 == 0 && dy_coff % 8 == 0, "b2_relu_gn_bwd: lddy/dy_coff must be multiples of 8");
  const long long need = b2_relu_gn_bwd_workspace_bytes(N, C);
  B2_REQUIRE(workspace_bytes >= need, "b2_relu_gn_bwd: workspace %lld < %lld", workspace_bytes, need);
  float* partial = reinterpret_cast<float*>(workspace);
  float* coef = partial + (size_t)N * kStatBlocks * C * 2;
  float* dgb_n = coef + (size_t)N * C * 4;
  const int nblk = stat_blocks(V, C);
  const int vpi = kStatThreads / (C / 8);
  const size_t sh = (size_t)vpi * C * 2 * sizeof(float);
  B2_LAUNCH(gn_bwd_stats_kernel, dim3(nblk, N), kStatThreads, sh, stream, 
      reinterpret_cast<const __nv_bfloat16*>(dy), lddy, dy_coff, reinterpret_cast<const __nv_bfloat16*>(r), V, C,
      mean_rstd, partial, counters, N, G, gamma, coef, dgb_n, dgamma, dbeta);
  B2_CHECK_CUDA(cudaGetLastError());
  B2_LAUNCH((gn_bwd_apply_kernel<false, false>), dim3(apply_blocks(V * (C / 8)), N), 256, 0, stream, 
      reinterpret_cast<const __nv_bfloat16*>(dy), lddy, dy_coff, reinterpret_cast<const __nv_bfloat16*>(r), V, C,
      mean_rstd, coef, reinterpret_cast<__nv_bfloat16*>(dr), static_cast<const long long*>(nullptr),
      static_cast<long long*>(nullptr));
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

extern "C" long long b2_relu_gn_bwd_workspace_bytes(int N, int C) {
  return b2_gn_workspace_bytes(N, C) + (long long)N * C * 6 * (long long)sizeof(float);
}

// GroupNorm backward (batch 1) when (sum dy, sum dy*r) arrive in the fixed-point accumulators a producer kernel filled
// (b2_conv3d_igemm_bstats, b2_maxpool3d_bwd_add_bstats, b2_upcat_bwd_separable_bstats, b2_head_ce_bstats): a one-block
// finalize (coefficients, dgamma, dbeta) + the apply pass; no statistics pass over (dy, r).  workspace >= C*16 bytes.
// dy_row_labels (int64 [V], may be NULL): dy comes from b2_head_ce_bstats with skip_dx_memset — only the rows of
// voxels with label >= 0 hold data, all others count as zero and are not read.
extern "C" int b2_relu_gn_bwd_acc(const long long* stat_acc, const void* dy, int lddy, int dy_coff, const void* r,
                                  long long V, int C, int G, const float* gamma, const float* mean_rstd, void* dr,
                                  float* dgamma, float* dbeta, void* workspace, long long workspace_bytes,
                                  const long long* dy_row_labels, cudaStream_t stream) {
  B2_REQUIRE(stat_acc && dy && r && gamma && mean_rstd && dr && workspace, "b2_relu_gn_bwd_acc: null pointer");
  int rc = check_gn_shape("b2_relu_gn_bwd_acc", 1, V, C, G);
  if (rc) return rc;
  B2_REQUIRE(C <= kMaxAccC, "b2_relu_gn_bwd_acc: C=%d > %d", C, kMaxAccC);
  B2_REQUIRE(lddy % 8 == 0 && dy_coff % 8 == 0, "b2_relu_gn_bwd_acc: lddy/dy_coff must be multiples of 8");
  B2_REQUIRE(workspace_bytes >= (long long)C * 4 * (long long)sizeof(float), "b2_relu_gn_bwd_acc: workspace too small");
  float* coef = reinterpret_cast<float*>(workspace);
  B2_LAUNCH_DEP(gn_bwd_finalize_acc_kernel, 1, (C + 31) / 32 * 32, 0, stream, stat_acc, C, G,
            1.0 / ((double)V * (C / G)), gamma, mean_rstd, coef, dgamma, dbeta);
  B2_CHECK_CUDA(cudaGetLastError());
  if (dy_row_labels != nullptr)
    B2_LAUNCH_DEP((gn_bwd_apply_kernel<true, false>), dim3(apply_blocks(V * (C / 8)), 1), 256, 0, stream,
              reinterpret_cast<const __nv_bfloat16*>(dy), lddy, dy_coff, reinterpret_cast<const __nv_bfloat16*>(r), V,
              C, mean_rstd, static_cast<const float*>(coef), reinterpret_cast<__nv_bfloat16*>(dr), dy_row_labels,
              static_cast<long long*>(nullptr));
  else
    B2_LAUNCH_DEP((gn_bwd_apply_kernel<false, false>), dim3(apply_blocks(V * (C / 8)), 1), 256, 0, stream,
              reinterpret_cast<const __nv_bfloat16*>(dy), lddy, dy_coff, reinterpret_cast<const __nv_bfloat16*>(r), V,
              C, mean_rstd, static_cast<const float*>(coef), reinterpret_cast<__nv_bfloat16*>(dr), dy_row_labels,
              static_cast<long long*>(nullptr));
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

// ---- layers with a conv bias: the same two GroupNorm-backward forms, also producing dbias = sum_v dr[v, c] --------------
// dbias_acc: int64 [C][2] fixed-point accumulators, zero before the call; dbias: fp32 [C] (overwritten).  The sums are
// fused into the apply pass (gn_bwd_apply_kernel<.., true>); one more one-block launch converts them to fp32.
static int launch_dbias_apply(const void* dy, int lddy, int dy_coff, const void* r, int N, long long V, int C,
                              const float* mean_rstd, const float* coef, void* dr, const long long* dy_row_labels,
                              long long* dbias_acc, float* dbias, cudaStream_t stream) {
  const dim3 grid(apply_blocks(V * (C / 8)), N);
  auto* dyb = reinterpret_cast<const __nv_bfloat16*>(dy);
  auto* rb = reinterpret_cast<const __nv_bfloat16*>(r);
  auto* drb = reinterpret_cast<__nv_bfloat16*>(dr);
  if (dy_row_labels != nullptr)
    B2_LAUNCH((gn_bwd_apply_kernel<true, true>), grid, 256, 0, stream, dyb, lddy, dy_coff, rb, V, C, mean_rstd, coef,
              drb, dy_row_labels, dbias_acc);
  else
    B2_LAUNCH((gn_bwd_apply_kernel<false, true>), grid, 256, 0, stream, dyb, lddy, dy_coff, rb, V, C, mean_rstd, coef,
              drb, dy_row_labels, dbias_acc);
  B2_CHECK_CUDA(cudaGetLastError());
  B2_LAUNCH(dbias_finalize_kernel, 1, (C + 31) / 32 * 32, 0, stream, static_cast<const long long*>(dbias_acc), C,
            dbias);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

extern "C" int b2_relu_gn_bwd_dbias(const void* dy, int lddy, int dy_coff, const void* r, int N, long long V, int C,
                                    int G, const float* gamma, const float* mean_rstd, void* dr, float* dgamma,
                                    float* dbeta, void* workspace, long long workspace_bytes, int* counters,
                                    long long* dbias_acc, float* dbias, cudaStream_t stream) {
  B2_REQUIRE(dy && r && gamma && mean_rstd && dr && workspace && counters && dbias_acc && dbias,
             "b2_relu_gn_bwd_dbias: null pointer");
  int rc = check_gn_shape("b2_relu_gn_bwd_dbias", N, V, C, G);
  if (rc) return rc;
  B2_REQUIRE(C <= kMaxAccC, "b2_relu_gn_bwd_dbias: C=%d > %d", C, kMaxAccC);
  B2_REQUIRE(lddy % 8 == 0 && dy_coff % 8 == 0, "b2_relu_gn_bwd_dbias: lddy/dy_coff must be multiples of 8");
  const long long need = b2_relu_gn_bwd_workspace_bytes(N, C);
  B2_REQUIRE(workspace_bytes >= need, "b2_relu_gn_bwd_dbias: workspace %lld < %lld", workspace_bytes, need);
  float* partial = reinterpret_cast<float*>(workspace);
  float* coef = partial + (size_t)N * kStatBlocks * C * 2;
  float* dgb_n = coef + (size_t)N * C * 4;
  const int nblk = stat_blocks(V, C);
  const int vpi = kStatThreads / (C / 8);
  const size_t sh = (size_t)vpi * C * 2 * sizeof(float);
  B2_LAUNCH(gn_bwd_stats_kernel, dim3(nblk, N), kStatThreads, sh, stream,
      reinterpret_cast<const __nv_bfloat16*>(dy), lddy, dy_coff, reinterpret_cast<const __nv_bfloat16*>(r), V, C,
      mean_rstd, partial, counters, N, G, gamma, coef, dgb_n, dgamma, dbeta);
  B2_CHECK_CUDA(cudaGetLastError());
  return launch_dbias_apply(dy, lddy, dy_coff, r, N, V, C, mean_rstd, coef, dr, nullptr, dbias_acc, dbias, stream);
}

extern "C" int b2_relu_gn_bwd_acc_dbias(const long long* stat_acc, const void* dy, int lddy, int dy_coff, const void* r,
                                        long long V, int C, int G, const float* gamma, const float* mean_rstd, void* dr,
                                        float* dgamma, float* dbeta, void* workspace, long long workspace_bytes,
                                        const long long* dy_row_labels, long long* dbias_acc, float* dbias,
                                        cudaStream_t stream) {
  B2_REQUIRE(stat_acc && dy && r && gamma && mean_rstd && dr && workspace && dbias_acc && dbias,
             "b2_relu_gn_bwd_acc_dbias: null pointer");
  int rc = check_gn_shape("b2_relu_gn_bwd_acc_dbias", 1, V, C, G);
  if (rc) return rc;
  B2_REQUIRE(C <= kMaxAccC, "b2_relu_gn_bwd_acc_dbias: C=%d > %d", C, kMaxAccC);
  B2_REQUIRE(lddy % 8 == 0 && dy_coff % 8 == 0, "b2_relu_gn_bwd_acc_dbias: lddy/dy_coff must be multiples of 8");
  B2_REQUIRE(workspace_bytes >= (long long)C * 4 * (long long)sizeof(float),
             "b2_relu_gn_bwd_acc_dbias: workspace too small");
  float* coef = reinterpret_cast<float*>(workspace);
  B2_LAUNCH_DEP(gn_bwd_finalize_acc_kernel, 1, (C + 31) / 32 * 32, 0, stream, stat_acc, C, G,
            1.0 / ((double)V * (C / G)), gamma, mean_rstd, coef, dgamma, dbeta);
  B2_CHECK_CUDA(cudaGetLastError());
  return launch_dbias_apply(dy, lddy, dy_coff, r, 1, V, C, mean_rstd, coef, dr, dy_row_labels, dbias_acc, dbias,
                            stream);
}
