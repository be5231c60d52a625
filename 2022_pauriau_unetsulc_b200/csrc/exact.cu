// Exact-label inference mode (north star: "inference labels bit-identical to the reference").
//
// The training / default inference path stores activations and weights in bf16: logits differ from the fp32 reference by
// ~2e-2 rel-L2 and ~3 % of the per-voxel arg-max labels flip on near-ties.  This mode keeps every activation in fp32 and
// runs each 3x3x3 convolution on the SAME tcgen05 implicit-GEMM kernel with split operands ("bf16x3"):
//     x = x_hi + x_lo (+ 2^-17 rel),  w = w_hi + w_lo     ->   x*w ~= x_hi*w_hi + x_lo*w_hi + x_hi*w_lo   (2^-16 rel)
// realised as ONE convolution over 3*Cin input channels, [x_hi | x_lo | x_hi] against [w_hi | w_hi | w_lo], with fp32
// accumulation in TMEM and an fp32 output.  The first layer (Cin = 1) is split the same way into 32 channels,
// [x_hi, x_hi, x_lo, 0...] against [w_hi, w_lo, w_hi, 0...], so any fp32 volume keeps its low half (for a binary
// volume x_lo = 0 and the extra products are exact zeros).  The element-wise operators in between (ReLU is fused in
// the conv epilogue; GroupNorm with fp64 statistics, MaxPool3d(2), trilinear upsample + concat, the 1x1x1 head +
// softmax at the skeleton points) are the plain fp32 kernels below.  ~3x the convolution work of the bf16 path;
// inference only.
#include "common.h"
#include <cuda_bf16.h>

namespace b2 {

static inline int ex_blocks(long long total, int per_block = 256) {
  long long nb = (total + per_block - 1) / per_block;
  const long long cap = (long long)num_sms() * 16;
  if (nb > cap) nb = cap;
  if (nb < 1) nb = 1;
  return (int)nb;
}

// out[v][0:C] = hi(x), out[v][C:2C] = lo(x) = bf16(x - hi), out[v][2C:3C] = hi(x)
__global__ void __launch_bounds__(256)
exact_split3_kernel(const float* __restrict__ x, long long V, int C, int ldx, int xoff, __nv_bfloat16* __restrict__ out) {
  pdl_prologue();
  const long long total = V * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long v = i / C;
    const int c = (int)(i % C);
    const float f = x[v * ldx + xoff + c];
    const __nv_bfloat16 hi = __float2bfloat16_rn(f);
    const __nv_bfloat16 lo = __float2bfloat16_rn(f - __bfloat162float(hi));
    __nv_bfloat16* o = out + v * 3 * C;
    o[c] = hi;
    o[C + c] = lo;
    o[2 * C + c] = hi;
  }
}

// network input: out[v][0] = out[v][1] = hi(x), out[v][2] = lo(x), channels 3..31 zero (pairs with
// [w_hi, w_lo, w_hi, 0...])
__global__ void __launch_bounds__(256)
exact_split_first_kernel(const float* __restrict__ x, long long V, __nv_bfloat16* __restrict__ out) {
  pdl_prologue();
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < V; v += (long long)gridDim.x * blockDim.x) {
    const float f = x[v];
    const __nv_bfloat16 h = __float2bfloat16_rn(f);
    const __nv_bfloat16 l = __float2bfloat16_rn(f - __bfloat162float(h));
    uint4* o = reinterpret_cast<uint4*>(out + v * 32);
    const uint32_t pair = (uint32_t)__bfloat16_as_ushort(h) | ((uint32_t)__bfloat16_as_ushort(h) << 16);
    o[0] = make_uint4(pair, (uint32_t)__bfloat16_as_ushort(l), 0u, 0u);
    o[1] = make_uint4(0u, 0u, 0u, 0u);
    o[2] = make_uint4(0u, 0u, 0u, 0u);
    o[3] = make_uint4(0u, 0u, 0u, 0u);
  }
}

// GroupNorm statistics in fp64, two deterministic stages: per-block per-channel partial sums, then a fixed-order finalize
static constexpr int kExStatBlocks = 296;
__global__ void __launch_bounds__(256)
exact_gn_partial_kernel(const float* __restrict__ r, long long V, int C, double* __restrict__ partial /*[blocks][C][2]*/) {
  pdl_prologue();
  extern __shared__ double ex_red[];   // [256 / C'] rows x C x 2, C' = min(C, 256)
  const int cpt = (C + 255) / 256;     // channels per thread when C > 256
  const int tc = C < 256 ? C : 256;    // threads along channels
  const int rows = 256 / tc;
  const int c0 = threadIdx.x % tc, row = threadIdx.x / tc;
  double s[2] = {0.0, 0.0}, q[2] = {0.0, 0.0};
  for (long long v = (long long)blockIdx.x * rows + row; v < V; v += (long long)gridDim.x * rows)
    for (int k = 0; k < cpt; ++k) {
      const int c = c0 + k * 256;
      if (c < C) {
        const double f = (double)r[v * C + c];
        s[k] += f;
        q[k] += f * f;
      }
    }
  for (int k = 0; k < cpt; ++k) {
    const int c = c0 + k * 256;
    if (c < C) {
      ex_red[((size_t)row * C + c) * 2] = s[k];
      ex_red[((size_t)row * C + c) * 2 + 1] = q[k];
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += 256) {
    double a = 0.0, b = 0.0;
    for (int j = 0; j < rows; ++j) { a += ex_red[((size_t)j * C + c) * 2]; b += ex_red[((size_t)j * C + c) * 2 + 1]; }
    partial[((size_t)blockIdx.x * C + c) * 2] = a;
    partial[((size_t)blockIdx.x * C + c) * 2 + 1] = b;
  }
}
__global__ void __launch_bounds__(512)
exact_gn_finalize_kernel(const double* __restrict__ partial, int blocks, long long V, int C, int G, double eps,
                         const float* __restrict__ gamma, const float* __restrict__ beta,
                         float* __restrict__ scale_shift /*[C][2]*/) {
  pdl_prologue();
  __shared__ double cs[512][2];
  const int c = threadIdx.x;
  if (c < C) {
    double a = 0.0, b = 0.0;
    for (int j = 0; j < blocks; ++j) { a += partial[((size_t)j * C + c) * 2]; b += partial[((size_t)j * C + c) * 2 + 1]; }
    cs[c][0] = a;
    cs[c][1] = b;
  }
  __syncthreads();
  if (c < C) {
    const int cpg = C / G, g0 = (c / cpg) * cpg;
    double a = 0.0, b = 0.0;
    for (int j = 0; j < cpg; ++j) { a += cs[g0 + j][0]; b += cs[g0 + j][1]; }
    const double m = (double)V * cpg;
    const double mean = a / m;
    double var = b / m - mean * mean;
    if (var < 0.0) var = 0.0;
    const double rstd = 1.0 / sqrt(var + eps);
    const double sc = rstd * (double)gamma[c];
    scale_shift[2 * c] = (float)sc;
    scale_shift[2 * c + 1] = (float)((double)beta[c] - mean * sc);
  }
}

// y[v][yoff + c] = r[v][c] * scale[c] + shift[c]   (fp32; one fused multiply-add of fp64-derived coefficients)
__global__ void __launch_bounds__(256)
exact_gn_apply_kernel(const float* __restrict__ r, long long V, int C, const float* __restrict__ scale_shift,
                      float* __restrict__ y, int ldy, int yoff) {
  pdl_prologue();
  const long long total = V * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long v = i / C;
    const int c = (int)(i % C);
    y[v * ldy + yoff + c] = fmaf(r[i], scale_shift[2 * c], scale_shift[2 * c + 1]);
  }
}

// MaxPool3d(2, 2, 0) on an fp32 NDHWC channel window; a NaN anywhere in a cell makes the cell NaN (as torch.max_pool3d)
__global__ void __launch_bounds__(256)
exact_maxpool_kernel(const float* __restrict__ x, int N, int D, int H, int W, int C, int ldx, int xoff,
                     float* __restrict__ y) {
  pdl_prologue();
  const int Dp = D >> 1, Hp = H >> 1, Wp = W >> 1;
  const long long total = (long long)N * Dp * Hp * Wp * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    long long t = i / C;
    const int pw = (int)(t % Wp); t /= Wp;
    const int ph = (int)(t % Hp); t /= Hp;
    const int pd = (int)(t % Dp);
    const int n = (int)(t / Dp);
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const long long v = (((long long)n * D + 2 * pd + (j >> 2)) * H + 2 * ph + ((j >> 1) & 1)) * W + 2 * pw + (j & 1);
      const float f = x[v * ldx + xoff + c];
      m = (f > m || f != f) ? f : m;
    }
    y[i] = m;
  }
}

__device__ __forceinline__ void ex_src_index(int dst, float scale, int in_size, int& i0, int& i1, float& l0, float& l1) {
  float src = scale * ((float)dst + 0.5f) - 0.5f;   // PyTorch area_pixel_compute_source_index, align_corners=False
  if (src < 0.f) src = 0.f;
  i0 = (int)src;
  if (i0 > in_size - 1) i0 = in_size - 1;
  i1 = i0 + ((i0 < in_size - 1) ? 1 : 0);
  l1 = src - (float)i0;
  l0 = 1.f - l1;
}

// trilinear upsample (align_corners=False), fp32, written into the channel window [yoff, yoff + C) of the concat buffer;
// same association order as ATen's upsample_trilinear3d kernel
__global__ void __launch_bounds__(256)
exact_upsample_kernel(const float* __restrict__ x, int N, int Di, int Hi, int Wi, int C, float* __restrict__ y, int ldy,
                      int yoff, int Do, int Ho, int Wo) {
  pdl_prologue();
  const float sd = (float)Di / (float)Do, sh = (float)Hi / (float)Ho, sw = (float)Wi / (float)Wo;
  const long long total = (long long)N * Do * Ho * Wo * C;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    long long t = i / C;
    const int w = (int)(t % Wo); t /= Wo;
    const int h = (int)(t % Ho); t /= Ho;
    const int d = (int)(t % Do);
    const int n = (int)(t / Do);
    int d0, d1, h0, h1, w0, w1;
    float ld0, ld1, lh0, lh1, lw0, lw1;
    ex_src_index(d, sd, Di, d0, d1, ld0, ld1);
    ex_src_index(h, sh, Hi, h0, h1, lh0, lh1);
    ex_src_index(w, sw, Wi, w0, w1, lw0, lw1);
    const float* xb = x + (size_t)n * Di * Hi * Wi * C + c;
#define EX_AT(dd, hh, ww) xb[(((size_t)(dd) * Hi + (hh)) * Wi + (ww)) * C]
    const float o = ld0 * (lh0 * (lw0 * EX_AT(d0, h0, w0) + lw1 * EX_AT(d0, h0, w1)) +
                           lh1 * (lw0 * EX_AT(d0, h1, w0) + lw1 * EX_AT(d0, h1, w1))) +
                    ld1 * (lh0 * (lw0 * EX_AT(d1, h0, w0) + lw1 * EX_AT(d1, h0, w1)) +
                           lh1 * (lw0 * EX_AT(d1, h1, w0) + lw1 * EX_AT(d1, h1, w1)));
#undef EX_AT
    const long long v = (((long long)n * Do + d) * Ho + h) * Wo + w;
    y[v * ldy + yoff + c] = o;
  }
}

// final 1x1x1 conv + Softmax(dim=1) + arg-max at gathered voxels, all fp32 (fp32 features in).  One warp per point.
__global__ void __launch_bounds__(256)
exact_head_gather_kernel(const float* __restrict__ x, const long long* __restrict__ index, long long n,
                         const float* __restrict__ W, const float* __restrict__ b, int Cin, int Cout, int softmax,
                         float* __restrict__ scores, int* __restrict__ preds) {
  pdl_prologue();
  extern __shared__ float ex_w[];   // [Cout][Cin + 1] + [Cout]
  float* sb = ex_w + (size_t)Cout * (Cin + 1);
  for (int e = threadIdx.x; e < Cout * Cin; e += blockDim.x) ex_w[(e / Cin) * (Cin + 1) + e % Cin] = W[e];
  for (int e = threadIdx.x; e < Cout; e += blockDim.x) sb[e] = b[e];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  for (long long p = (long long)blockIdx.x * wpb + warp; p < n; p += (long long)gridDim.x * wpb) {
    const float* xr = x + index[p] * Cin;
    // lane handles outputs o = lane, lane + 32; sequential fp32 accumulation over ci in index order (as a reference
    // 1x1x1 convolution would), features broadcast from L1
    float z[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int o = lane + 32 * k;
      if (o < Cout) {
        float acc = sb[o];
        const float* wr = ex_w + (size_t)o * (Cin + 1);
        for (int ci = 0; ci < Cin; ++ci) acc = fmaf(xr[ci], wr[ci], acc);
        z[k] = acc;
      }
    }
    float mx = fmaxf(z[0], z[1]);
    int am = z[1] > z[0] ? lane + 32 : lane;
    float mv = fmaxf(z[0], z[1]);
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, mv, s);
      const int oi = __shfl_xor_sync(0xffffffffu, am, s);
      if (ov > mv || (ov == mv && oi < am)) { mv = ov; am = oi; }   // ties -> lowest class index (torch.max)
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, s));
    }
    float e0 = 0.f, e1 = 0.f, sum = 0.f;
    if (softmax) {
      e0 = lane < Cout ? expf(z[0] - mx) : 0.f;
      e1 = lane + 32 < Cout ? expf(z[1] - mx) : 0.f;
      sum = e0 + e1;
#pragma unroll
      for (int s = 16; s >= 1; s >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, s);
    }
    if (lane < Cout) scores[p * Cout + lane] = softmax ? e0 / sum : z[0];
    if (lane + 32 < Cout) scores[p * Cout + lane + 32] = softmax ? e1 / sum : z[1];
    if (lane == 0) preds[p] = am;
  }
}

}  // namespace b2

using namespace b2;

extern "C" int b2_exact_split3(const float* x, long long V, int C, int ldx, int xoff, void* out, cudaStream_t stream) {
  B2_REQUIRE(x && out && V > 0 && C > 0 && xoff >= 0 && xoff + C <= ldx, "b2_exact_split3: bad arguments");
  B2_LAUNCH(exact_split3_kernel, ex_blocks(V * C), 256, 0, stream, x, V, C, ldx, xoff,
            reinterpret_cast<__nv_bfloat16*>(out));
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

extern "C" int b2_exact_split_first(const float* x, long long V, void* out, cudaStream_t stream) {
  B2_REQUIRE(x && out && V > 0, "b2_exact_split_first: bad arguments");
  B2_LAUNCH(exact_split_first_kernel, ex_blocks(V), 256, 0, stream, x, V, reinterpret_cast<__nv_bfloat16*>(out));
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

extern "C" long long b2_exact_gn_workspace_bytes(int C) { return (long long)kExStatBlocks * C * 2 * (long long)sizeof(double); }

// r fp32 dense [V][C] (post-ReLU conv output, one sample) -> scale_shift fp32 [C][2] of GroupNorm(G, C, eps) with affine
// (gamma, beta); statistics accumulated in fp64 in a fixed order (bit-identical run to run)
extern "C" int b2_exact_gn_stats(const float* r, long long V, int C, int G, float eps, const float* gamma,
                                 const float* beta, float* scale_shift, void* workspace, long long workspace_bytes,
                                 cudaStream_t stream) {
  B2_REQUIRE(r && gamma && beta && scale_shift && workspace, "b2_exact_gn_stats: null pointer");
  B2_REQUIRE(V > 0 && C > 0 && C <= 512 && G > 0 && C % G == 0, "b2_exact_gn_stats: bad shape C=%d G=%d", C, G);
  B2_REQUIRE(C <= 256 ? 256 % C == 0 : C % 256 == 0, "b2_exact_gn_stats: C=%d must divide or be a multiple of 256", C);
  B2_REQUIRE(workspace_bytes >= b2_exact_gn_workspace_bytes(C), "b2_exact_gn_stats: workspace too small");
  const int tc = C < 256 ? C : 256, rows = 256 / tc;
  long long nb = (V + rows - 1) / rows;
  const int blocks = (int)(nb < kExStatBlocks ? nb : kExStatBlocks);
  const size_t smem = (size_t)rows * C * 2 * sizeof(double);
  B2_CHECK_CUDA(cudaFuncSetAttribute(exact_gn_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  B2_LAUNCH(exact_gn_partial_kernel, blocks, 256, smem, stream, r, V, C, reinterpret_cast<double*>(workspace));
  B2_CHECK_CUDA(cudaGetLastError());
  B2_LAUNCH(exact_gn_finalize_kernel, 1, 512, 0, stream, static_cast<const double*>(workspace), blocks, V, C, G,
            (double)eps, gamma, beta, scale_shift);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

extern "C" int b2_exact_gn_apply(const float* r, long long V, int C, const float* scale_shift, float* y, int ldy,
                                 int yoff, cudaStream_t stream) {
  B2_REQUIRE(r && scale_shift && y && V > 0 && C > 0 && yoff >= 0 && yoff + C <= ldy, "b2_exact_gn_apply: bad arguments");
  B2_LAUNCH(exact_gn_apply_kernel, ex_blocks(V * C), 256, 0, stream, r, V, C, scale_shift, y, ldy, yoff);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

extern "C" int b2_exact_maxpool(const float* x, int N, int D, int H, int W, int C, int ldx, int xoff, float* y,
                                cudaStream_t stream) {
  B2_REQUIRE(x && y && N > 0 && D > 1 && H > 1 && W > 1 && C > 0 && xoff + C <= ldx, "b2_exact_maxpool: bad arguments");
  B2_LAUNCH(exact_maxpool_kernel, ex_blocks((long long)N * (D / 2) * (H / 2) * (W / 2) * C), 256, 0, stream, x, N, D, H,
            W, C, ldx, xoff, y);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

extern "C" int b2_exact_upsample(const float* x, int N, int Di, int Hi, int Wi, int C, float* y, int ldy, int yoff,
                                 int Do, int Ho, int Wo, cudaStream_t stream) {
  B2_REQUIRE(x && y && N > 0 && Di > 0 && Hi > 0 && Wi > 0 && C > 0 && yoff + C <= ldy, "b2_exact_upsample: bad arguments");
  B2_LAUNCH(exact_upsample_kernel, ex_blocks((long long)N * Do * Ho * Wo * C), 256, 0, stream, x, N, Di, Hi, Wi, C, y,
            ldy, yoff, Do, Ho, Wo);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}

extern "C" int b2_exact_head_gather(const float* x, const long long* index, long long n, const float* W,
                                    const float* b, int Cin, int Cout, int softmax, float* scores, int* preds,
                                    cudaStream_t stream) {
  if (n == 0) return B2_OK;
  B2_REQUIRE(x && index && W && b && scores && preds, "b2_exact_head_gather: null pointer");
  B2_REQUIRE(Cin > 0 && Cout > 0 && Cout <= 64, "b2_exact_head_gather: Cout=%d must be <= 64", Cout);
  const size_t smem = ((size_t)Cout * (Cin + 1) + Cout) * sizeof(float);
  B2_REQUIRE(smem <= 96 * 1024, "b2_exact_head_gather: head too large");
  B2_CHECK_CUDA(cudaFuncSetAttribute(exact_head_gather_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
  long long nb = (n + 7) / 8;
  if (nb > num_sms() * 4) nb = num_sms() * 4;
  B2_LAUNCH(exact_head_gather_kernel, (unsigned)nb, 256, smem, stream, x, index, n, W, b, Cin, Cout, softmax, scores,
            preds);
  B2_CHECK_CUDA(cudaGetLastError());
  return B2_OK;
}
