// Translation unit of the general-grid fused tail (tail_general.cuh), the LSF-vector tail (tail_lsf.cuh) and
// the continuum-emulator multiply (continuum.cuh), the unit-test hook of the runtime-planned FFT (fft.cuh) and the
// dynamic shared-memory opt-in helper raise_max_dyn_smem;
// see launchers.h.
#include <map>
#include <mutex>
#include <utility>

#include "launchers.h"

namespace payne {

cudaError_t raise_max_dyn_smem(const void* func, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> mark;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  size_t& m = mark[std::make_pair(func, dev)];
  if (bytes <= m) return cudaSuccess;
  e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) m = bytes;
  return e;
}

#define PAYNE_GEN_SIZES(X) X(10) X(11) X(12) X(13) X(14) X(15)

bool probe_tail_general(int l2, size_t bytes, int* occ) {
  cudaError_t e1 = cudaErrorInvalidValue, e2 = cudaErrorInvalidValue;
  switch (l2 < 10 ? 10 : l2) {
#define X(L)                                                                                                      \
    case L:                                                                                                       \
      e1 = raise_max_dyn_smem((const void*)tail_general_kernel<L>, bytes);                                        \
      e2 = cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, tail_general_kernel<L>, kTailThreads, bytes);       \
      break;
    PAYNE_GEN_SIZES(X)
#undef X
    default: break;
  }
  if (e1 != cudaSuccess || e2 != cudaSuccess) { cudaGetLastError(); return false; }
  return true;
}

int launch_tail_general(int l2, int grid, size_t smem, cudaStream_t st, const TailParams& T, const TwConst& tc) {
  switch (l2 < 10 ? 10 : l2) {
#define X(L) case L: tail_general_kernel<L><<<grid, kTailThreads, smem, st>>>(T, tc); break;
    PAYNE_GEN_SIZES(X)
#undef X
    default: return PAYNE_E_UNSUPPORTED;
  }
  return cudaGetLastError() == cudaSuccess ? PAYNE_OK : PAYNE_E_CUDA;
}

template <bool TGT>
static bool probe_lsf(size_t bytes, int* occ) {
  if (raise_max_dyn_smem((const void*)tail_lsf_kernel<TGT>, bytes) != cudaSuccess ||
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, tail_lsf_kernel<TGT>, kTailThreads, bytes) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return true;
}

bool probe_tail_lsf(size_t bytes, int* occ) { return probe_lsf<false>(bytes, occ); }
bool probe_tail_lsf_targets(size_t bytes, int* occ) { return probe_lsf<true>(bytes, occ); }

int launch_tail_lsf(int grid, size_t smem, cudaStream_t st, const TailParams& T, const LsfParams& L) {
  tail_lsf_kernel<false><<<grid, kTailThreads, smem, st>>>(T, L);
  return cudaGetLastError() == cudaSuccess ? PAYNE_OK : PAYNE_E_CUDA;
}

int launch_tail_lsf_targets(int grid, size_t smem, cudaStream_t st, const TailParams& T, const LsfParams& L) {
  tail_lsf_kernel<true><<<grid, kTailThreads, smem, st>>>(T, L);
  return cudaGetLastError() == cudaSuccess ? PAYNE_OK : PAYNE_E_CUDA;
}

int launch_continuum(int grid, cudaStream_t st, const ContParams& C) {
  continuum_kernel<0><<<grid, 256, 0, st>>>(C);
  return cudaGetLastError() == cudaSuccess ? PAYNE_OK : PAYNE_E_CUDA;
}

// The runtime-planned convolution of fft.cuh on its own (payne_fft_test): one CTA packs x into the swizzled
// complex layout the tails use, runs forward -> filter -> inverse and unpacks the result in natural order.
struct TableH {
  const float* h;
  float invM;
  __device__ __forceinline__ float operator()(int k) const { return __ldg(h + k) * invM; }
};

__global__ void __launch_bounds__(kNT) fft_test_kernel(const float* __restrict__ x, int log2N,
                                                       const float* __restrict__ H, const float2* __restrict__ tw,
                                                       float* __restrict__ y) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* z = reinterpret_cast<float2*>(smem_raw);
  const int tid = threadIdx.x, log2M = log2N - 1, M = 1 << log2M;
  for (int m = tid; m < M; m += kNT) z[swz(m)] = make_float2(x[2 * m], x[2 * m + 1]);
  __syncthreads();
  const Twiddles twr{tw, log2N};
  FftPlan plan; plan.make(log2M);
  fft_forward(z, log2M, plan, twr, tid, kNT);
  filter_pairs(z, log2M, plan, twr, TableH{H, 1.0f / (float)M}, tid, kNT);
  fft_inverse(z, log2M, plan, twr, tid, kNT);
  for (int m = tid; m < M; m += kNT) {
    const float2 v = z[swz(m)];
    y[2 * m] = v.x; y[2 * m + 1] = v.y;
  }
}

int launch_fft_test(const float* x, int log2N, const float* H, const float2* tw, float* y) {
  const size_t smem = (size_t)4 << log2N;              // N/2 complex points of 8 bytes
  if (cudaFuncSetAttribute(fft_test_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
    return PAYNE_E_CUDA;
  fft_test_kernel<<<1, kNT, smem>>>(x, log2N, H, tw, y);
  return cudaGetLastError() == cudaSuccess ? PAYNE_OK : PAYNE_E_CUDA;
}

}  // namespace payne
