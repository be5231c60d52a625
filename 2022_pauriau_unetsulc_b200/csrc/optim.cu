// SGD with momentum (torch.optim.SGD semantics: v <- mu*v + g ; p <- p - lr*v ; dampening 0, no nesterov, wd 0)
// as one multi-tensor launch, plus the bf16 weight re-packs the tcgen05 conv kernels read:
//   fprop pack  Wf[tap][co][ci]      = W[co][ci][tap]
//   dgrad pack  Wd[tap][ci][co]      = W[co][ci][26 - tap]      (flipped taps, transposed channels)
#include "common.h"
#include "ptx.cuh"

namespace b2 {

static constexpr int kMaxTensors = 64;
static constexpr int kChunk = 4096;  // elements per block

struct SgdArgs {
  float* p[kMaxTensors];
  const float* g[kMaxTensors];
  float* v[kMaxTensors];
  long long n[kMaxTensors];
  int first_block[kMaxTensors + 1];
  int count;
  float lr, momentum, grad_scale;
};

__global__ void __launch_bounds__(256) sgd_multi_kernel(const SgdArgs a) {
  pdl_prologue();
  int t = 0;
  while (t + 1 < a.count && (int)blockIdx.x >= a.first_block[t + 1]) ++t;
  const long long base = (long long)(blockIdx.x - a.first_block[t]) * kChunk;
  float* __restrict__ p = a.p[t];
  const float* __restrict__ g = a.g[t];
  float* __restrict__ v = a.v[t];
  const long long n = a.n[t];
  const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(v)) & 15) == 0 &&
                   base + kChunk <= n;
  if (vec) {   // full, 16-byte aligned chunk: four float4 per thread, all loads issued before the first store
    float4 pv[4], gv[4], vv[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long j = base + (long long)(k * 256 + threadIdx.x) * 4;
      pv[k] = *reinterpret_cast<const float4*>(p + j);
      gv[k] = *reinterpret_cast<const float4*>(g + j);
      vv[k] = *reinterpret_cast<const float4*>(v + j);
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const long long j = base + (long long)(k * 256 + threadIdx.x) * 4;
      float4 nv, np;
      nv.x = a.momentum * vv[k].x + gv[k].x * a.grad_scale; np.x = pv[k].x - a.lr * nv.x;
      nv.y = a.momentum * vv[k].y + gv[k].y * a.grad_scale; np.y = pv[k].y - a.lr * nv.y;
      nv.z = a.momentum * vv[k].z + gv[k].z * a.grad_scale; np.z = pv[k].z - a.lr * nv.z;
      nv.w = a.momentum * vv[k].w + gv[k].w * a.grad_scale; np.w = pv[k].w - a.lr * nv.w;
      *reinterpret_cast<float4*>(v + j) = nv;
      *reinterpret_cast<float4*>(p + j) = np;
    }
    return;
  }
  for (int i = threadIdx.x; i < kChunk; i += 256) {
    const long long j = base + i;
    if (j < n) {
      const float vv = a.momentum * v[j] + g[j] * a.grad_scale;
      v[j] = vv;
      p[j] -= a.lr * vv;
    }
  }
}

// Multi-layer weight pack, one launch for every conv layer whose fp32 master changed.
// Block = (16 output channels x 64 input channels) of one layer: the fp32 master is read ONCE (16 contiguous runs of
// 64*27 floats), rounded to bf16 into shared memory, and written out twice: Wf[tap][co][ci0..] in 128-byte runs and
// Wd[26-tap][ci][co0..] in 32-byte runs.  (Round 1 used one 64x27 tile per block and per pack: 18 912 blocks, two
// reads of the master, 102 us.)
static constexpr int kMaxPackLayers = 16;
static constexpr int kPkCo = 16, kPkCi = 64;
struct PackArgs {
  const float* w[kMaxPackLayers];
  __nv_bfloat16* wf[kMaxPackLayers];
  __nv_bfloat16* wd[kMaxPackLayers];
  int cout[kMaxPackLayers], cin[kMaxPackLayers];
  int first_block[kMaxPackLayers + 1];
  int count;
};

// one (16 co x TW ci) tile; TW is a compile-time constant so that every index split is a multiply-shift
template <int TW>
__device__ __forceinline__ void pack_tile(const float* __restrict__ w, __nv_bfloat16* __restrict__ wf,
                                          __nv_bfloat16* __restrict__ wd, int Cout, int Cin, int co0, int ci0,
                                          __nv_bfloat16 (*tile)[kPkCi * 27 + 2]) {
  constexpr int RUN4 = TW * 27 / 4;   // float4 per co row
  for (int e = threadIdx.x; e < kPkCo * RUN4; e += 256) {
    const int j = e / RUN4, r4 = e - j * RUN4;
    const float4 v = __ldg(reinterpret_cast<const float4*>(w + ((size_t)(co0 + j) * Cin + ci0) * 27) + r4);
    __nv_bfloat162* d = reinterpret_cast<__nv_bfloat162*>(&tile[j][4 * r4]);   // r = ci*27 + tap
    d[0] = __floats2bfloat162_rn(v.x, v.y);
    d[1] = __floats2bfloat162_rn(v.z, v.w);
  }
  __syncthreads();
  if (wf != nullptr) {
    for (int e = threadIdx.x; e < 27 * kPkCo * (TW / 2); e += 256) {
      const int ci = (e % (TW / 2)) * 2, row = e / (TW / 2);
      const int j = row % kPkCo, tap = row / kPkCo;
      __nv_bfloat162 o;
      o.x = tile[j][ci * 27 + tap];
      o.y = tile[j][(ci + 1) * 27 + tap];
      *reinterpret_cast<__nv_bfloat162*>(wf + ((size_t)tap * Cout + co0 + j) * Cin + ci0 + ci) = o;
    }
  }
  if (wd != nullptr) {
    for (int e = threadIdx.x; e < 27 * TW * (kPkCo / 2); e += 256) {
      const int j = (e % (kPkCo / 2)) * 2, row = e / (kPkCo / 2);
      const int ci = row % TW, tap = row / TW;
      __nv_bfloat162 o;
      o.x = tile[j][ci * 27 + tap];
      o.y = tile[j + 1][ci * 27 + tap];
      *reinterpret_cast<__nv_bfloat162*>(wd + ((size_t)(26 - tap) * Cin + ci0 + ci) * Cout + co0 + j) = o;
    }
  }
}

__global__ void __launch_bounds__(256) pack_weights_multi_kernel(const PackArgs a) {
  pdl_prologue();
  extern __shared__ __align__(16) uint8_t pack_smem[];
  auto tile = reinterpret_cast<__nv_bfloat16(*)[kPkCi * 27 + 2]>(pack_smem);   // [kPkCo][..], odd word stride
  int l = 0;
  while (l + 1 < a.count && (int)blockIdx.x >= a.first_block[l + 1]) ++l;
  const int Cout = a.cout[l], Cin = a.cin[l];
  const int b = blockIdx.x - a.first_block[l];
  if (Cin % 64 == 0) {
    const int ci_tiles = Cin / 64;
    pack_tile<64>(a.w[l], a.wf[l], a.wd[l], Cout, Cin, (b / ci_tiles) * kPkCo, (b % ci_tiles) * 64, tile);
  } else if (Cin % 32 == 0) {
    const int ci_tiles = Cin / 32;
    pack_tile<32>(a.w[l], a.wf[l], a.wd[l], Cout, Cin, (b / ci_tiles) * kPkCo, (b % ci_tiles) * 32, tile);
  } else {   // Cin = 16 (encoders.0.conv2 of a 32-filter network) or 48 (its split operand in exact mode)
    const int ci_tiles = Cin / 16;
    pack_tile<16>(a.w[l], a.wf[l], a.wd[l], Cout, Cin, (b / ci_tiles) * kPkCo, (b % ci_tiles) * 16, tile);
  }
}

}  // namespace b2

using namespace b2;

// params/grads/moms: arrays of `count` device pointers (host arrays); numels: element counts.
extern "C" int b2_sgd_step(float* const* params, const float* const* grads, float* const* moms,
                           const long long* numels, int count, float lr, float momentum, float grad_scale,
                           cudaStream_t stream) {
  B2_REQUIRE(params && grads && moms && numels && count >= 0, "b2_sgd_step: null pointer");
  int done = 0;
  while (done < count) {
    SgdArgs a;
    int k = 0, blocks = 0;
    while (done + k < count && k < kMaxTensors) {
      const int idx = done + k;
      B2_REQUIRE(params[idx] && grads[idx] && moms[idx], "b2_sgd_step: null tensor %d", idx);
      a.p[k] = params[idx];
      a.g[k] = grads[idx];
      a.v[k] = moms[idx];
      a.n[k] = numels[idx];
      a.first_block[k] = blocks;
      blocks += (int)((numels[idx] + kChunk - 1) / kChunk);
      ++k;
    }
    a.first_block[k] = blocks;
    a.count = k;
    a.lr = lr;
    a.momentum = momentum;
    a.grad_scale = grad_scale;
    if (blocks > 0) {
      B2_LAUNCH(sgd_multi_kernel, blocks, 256, 0, stream, a);
      B2_CHECK_CUDA(cudaGetLastError());
    }
    done += k;
  }
  return B2_OK;
}

// count layers; w/wf/wd/cout/cin are HOST arrays.  w[i]: fp32 [Cout][Cin][3][3][3]; wf[i]/wd[i]: bf16 packs (may be NULL)
extern "C" int b2_pack_conv_weights_multi(const float* const* w, void* const* wf, void* const* wd, const int* cout,
                                          const int* cin, int count, cudaStream_t stream) {
  B2_REQUIRE(w && wf && wd && cout && cin && count >= 0, "b2_pack_conv_weights_multi: null pointer");
  int done = 0;
  while (done < count) {
    PackArgs a;
    int k = 0, blocks = 0;
    while (done + k < count && k < kMaxPackLayers) {
      const int i = done + k;
      B2_REQUIRE(w[i] && (wf[i] || wd[i]), "b2_pack_conv_weights_multi: null tensor %d", i);
      a.w[k] = w[i];
      a.wf[k] = reinterpret_cast<__nv_bfloat16*>(wf[i]);
      a.wd[k] = reinterpret_cast<__nv_bfloat16*>(wd[i]);
      a.cout[k] = cout[i];
      a.cin[k] = cin[i];
      a.first_block[k] = blocks;
      B2_REQUIRE(cout[i] % kPkCo == 0 && cin[i] % 16 == 0 && cin[i] > 0,
                 "b2_pack_conv_weights_multi: layer %d: Cout=%d and Cin=%d must be multiples of 16", i, cout[i], cin[i]);
      blocks += (cout[i] / kPkCo) * (cin[i] % 64 == 0 ? cin[i] / 64 : (cin[i] % 32 == 0 ? cin[i] / 32 : cin[i] / 16));
      ++k;
    }
    a.first_block[k] = blocks;
    a.count = k;
    if (blocks > 0) {
      const int sh = kPkCo * (kPkCi * 27 + 2) * 2;
      B2_CHECK_CUDA(cudaFuncSetAttribute(pack_weights_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, sh));
      B2_LAUNCH(pack_weights_multi_kernel, blocks, 256, sh, stream, a);
      B2_CHECK_CUDA(cudaGetLastError());
    }
    done += k;
  }
  return B2_OK;
}

// single layer convenience
extern "C" int b2_pack_conv_weights(const float* w, void* wf, void* wd, int Cout, int Cin, cudaStream_t stream) {
  B2_REQUIRE(w && (wf || wd), "b2_pack_conv_weights: null pointer");
  return b2_pack_conv_weights_multi(&w, &wf, &wd, &Cout, &Cin, 1, stream);
}
