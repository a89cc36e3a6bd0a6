// Translation unit of the cluster-distributed fast tail (tail_cluster.cuh); see launchers.h.
#include "launchers.h"
#include "tail_cluster.cuh"

namespace payne {

#ifdef PAYNE_FAST_ONLY            // development builds compile one single-CTA size only; the cluster tail keeps 65536
#define PAYNE_CLUSTER_SIZES(X) X(16)
#else
#define PAYNE_CLUSTER_SIZES(X) X(15) X(16)
#endif

namespace {
template <class K>
cudaLaunchConfig_t cluster_config(K, int grid, size_t smem, cudaStream_t st, cudaLaunchAttribute* attr) {
  attr->id = cudaLaunchAttributeClusterDimension;
  attr->val.clusterDim.x = cl::kCluster;
  attr->val.clusterDim.y = 1;
  attr->val.clusterDim.z = 1;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)grid, 1, 1);
  cfg.blockDim = dim3(kNT, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cfg;
}
}  // namespace

int init_tail_cluster(const TwConst& tc) { return ct_set_twconst(tc) == cudaSuccess ? PAYNE_OK : PAYNE_E_CUDA; }

bool probe_tail_cluster(int l2, size_t bytes, int* ctas_per_sm, int* max_clusters) {
  cudaError_t e1 = cudaErrorInvalidValue, e2 = cudaErrorInvalidValue, e3 = cudaErrorInvalidValue;
  cudaLaunchAttribute attr;
  switch (l2) {
#define X(L)                                                                                                      \
    case L: {                                                                                                     \
      e1 = cudaFuncSetAttribute(tail_cluster_kernel<L, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes); \
      e2 = cudaOccupancyMaxActiveBlocksPerMultiprocessor(ctas_per_sm, tail_cluster_kernel<L, false>, kNT, bytes); \
      cudaLaunchConfig_t cfg = cluster_config(tail_cluster_kernel<L, false>, cl::kCluster, bytes, nullptr, &attr); \
      e3 = cudaOccupancyMaxActiveClusters(max_clusters, tail_cluster_kernel<L, false>, &cfg);                     \
      if (e1 == cudaSuccess && e2 == cudaSuccess && e3 == cudaSuccess) {   /* the multi-star instantiation alike */ \
        int o2 = 0, c2 = 0;                                                                                       \
        e1 = cudaFuncSetAttribute(tail_cluster_kernel<L, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes); \
        e2 = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o2, tail_cluster_kernel<L, true>, kNT, bytes);        \
        e3 = cudaOccupancyMaxActiveClusters(&c2, tail_cluster_kernel<L, true>, &cfg);                             \
        if (o2 < *ctas_per_sm) *ctas_per_sm = o2;                                                                 \
        if (c2 < *max_clusters) *max_clusters = c2;                                                               \
      }                                                                                                           \
      break;                                                                                                      \
    }
    PAYNE_CLUSTER_SIZES(X)
#undef X
    default: break;
  }
  if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) { cudaGetLastError(); return false; }
  return true;
}

int launch_tail_cluster(int l2, int n_clusters, size_t smem, cudaStream_t st, const TailParams& T, const FastGrid& F) {
  cudaLaunchAttribute attr;
  cudaError_t e = cudaErrorInvalidValue;
  switch (l2) {
#define X(L)                                                                                                        \
    case L: {                                                                                                       \
      cudaLaunchConfig_t cfg = cluster_config(tail_cluster_kernel<L, false>, n_clusters * cl::kCluster, smem, st, &attr); \
      e = T.n_stars > 1 ? cudaLaunchKernelEx(&cfg, tail_cluster_kernel<L, true>, T, F)                              \
                        : cudaLaunchKernelEx(&cfg, tail_cluster_kernel<L, false>, T, F);                            \
      break;                                                                                                        \
    }
    PAYNE_CLUSTER_SIZES(X)
#undef X
    default: return PAYNE_E_UNSUPPORTED;
  }
  return e == cudaSuccess ? PAYNE_OK : PAYNE_E_CUDA;
}

}  // namespace payne

#ifdef PAYNE_CLUSTER_PROF
extern "C" void payne_debug_cluster_prof(unsigned long long* out) {
  cudaDeviceSynchronize();
  cudaMemcpyFromSymbol(out, payne::cl::cl_prof, sizeof(unsigned long long) * 32);
  unsigned long long zero[32] = {0};
  cudaMemcpyToSymbol(payne::cl::cl_prof, zero, sizeof(zero));
}
#endif
