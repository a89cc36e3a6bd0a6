// CUDA-core fp32 implementation of the emulator layers (cross-check path, PAYNE_PREC_SIMT_FP32)
// and the label-encode + first layer that every precision mode shares (K = D_in <= 8 is far too
// thin for the tensor cores).
//
//   encode  : Payne/train/NNmodels.py:164-168  (x as fp32) -> fp64 (x-xmin)/(xmax-xmin)-0.5 -> fp32
//   layers  : Payne/train/NNmodels.py:154-162  sigmoid(lin_k(h)), k=1..5; lin6 without activation
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "obs_star.cuh"

namespace payne {

// 1/(1+exp(-x)) with a correctly rounded reciprocal: the same value as the IEEE division, fewer instructions
__device__ __forceinline__ float sigmoidf_exact(float x) { return __frcp_rn(1.0f + expf(-x)); }
// LeakyReLU(0.01): torch's (NNmodels.py:101) and the numpy z*(z>0)+0.01*z*(z<0) of ystpred.py:41-45
__device__ __forceinline__ float leaky_relu(float x) { return x > 0.f ? x : 0.01f * x; }
constexpr int kActNone = 0, kActSigmoid = 1, kActLeaky = 2;
template <int ACT>
__device__ __forceinline__ float activate(float v) {
  if (ACT == kActSigmoid) return sigmoidf_exact(v);
  if (ACT == kActLeaky) return leaky_relu(v);
  return v;
}

struct EncodeParams {
  int D_in, H1;
  int col[8];        // column of each label in the input rows, -1 -> fixed
  double fixed[8];
  double xmin[8], xmax[8];
  double offset;
  int cast32;        // labels through fp32 first (predictspec.py:70); 0 for the fp64 YST1 path
  int act;           // kActSigmoid / kActLeaky for the first layer
  // per-star fixed values and layouts (payne_ctx_create_stars_opts), null without them: label i of point p is
  // parameter label_param(i) of star star[p] (param_of)
  const double* star_fixed;
  const int* star;   // [B] star of every row of this slab (null: star 0)
  int n_stars;
  const StarLayout* star_lay;
  // binaries (payne_ctx_set_binary): rows [half, 2 half) are the secondaries of points [0, half), whose theta rows
  // and stars are those of the primaries; null without a binary
  const PayneBinary* binary;
  int half;
};

// raw value of label i of row p
__device__ __forceinline__ double label_of(const EncodeParams& E, const double* x, long long ld, int p, int i) {
  const int which = label_param(i);
  const bool sec = E.binary && p >= E.half;
  if (sec) p -= E.half;
  const int k = (which >= 0 && (E.star_fixed || E.star_lay)) ? star_of(E.star, E.n_stars, p) : -1;
  const double v = param_of(E.star_lay, E.col[i], E.fixed[i], E.star_fixed, x + (long long)p * ld, k, which);
  return sec ? secondary_of(E.binary, x + (long long)p * ld, which, v) : v;
}

// h1[p, h] = sigmoid(W1[h, :] . enc(x_p) + b1[h]); optionally also the tf32 hi/lo split planes.
static __global__ void __launch_bounds__(256)
encode_layer1_kernel(const __grid_constant__ EncodeParams E, const double* __restrict__ x, long long ld,
                     const float* __restrict__ W1, const float* __restrict__ b1, float* __restrict__ out,
                     long long ldo, int B) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int H1 = E.H1;
  if (idx >= (long long)B * H1) return;
  const int p = (int)(idx / H1), h = (int)(idx % H1);
  float acc = 0.f;
  for (int i = 0; i < E.D_in; ++i) {
    const double raw = label_of(E, x, ld, p, i);
    const double x = E.cast32 ? (double)(float)raw : raw;            // predictspec.py:70
    const float enc = (float)((x - E.xmin[i]) / (E.xmax[i] - E.xmin[i]) - E.offset);
    acc = fmaf(enc, __ldg(W1 + h * E.D_in + i), acc);
  }
  const float v = acc + __ldg(b1 + h);
  out[(long long)p * ldo + h] = E.act == kActLeaky ? leaky_relu(v) : sigmoidf_exact(v);
}

// C[M,N] = act(A[M,K] . W[N,K]^T + bias[N]); all row-major; fp32 FMA accumulation.
template <int ACT>
__global__ void __launch_bounds__(256)
sgemm_bias_act_kernel(const float* __restrict__ A, long long lda, const float* __restrict__ W,
                      const float* __restrict__ bias, float* __restrict__ C, long long ldc,
                      int M, int N, int K, float bias_shift) {
  constexpr int BM = 128, BN = 128, BK = 16, PAD = 4;
  __shared__ float As[BK][BM + PAD];
  __shared__ float Ws[BK][BN + PAD];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += BK) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int e = tid + i * 256, r = e >> 4, kk = e & 15;
      const int gm = m0 + r, gn = n0 + r, gk = k0 + kk;
      As[kk][r] = (gm < M && gk < K) ? __ldg(A + (long long)gm * lda + gk) : 0.f;
      Ws[kk][r] = (gn < N && gk < K) ? __ldg(W + (long long)gn * K + gk) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[8], b[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = As[kk][ty * 8 + i];
#pragma unroll
      for (int j = 0; j < 8; ++j) b[j] = Ws[kk][tx * 8 + j];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int gm = m0 + ty * 8 + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int gn = n0 + tx * 8 + j;
      if (gn >= N) continue;
      float v = acc[i][j] + (__ldg(bias + gn) + bias_shift);
      v = activate<ACT>(v);
      C[(long long)gm * ldc + gn] = v;
    }
  }
}

}  // namespace payne
