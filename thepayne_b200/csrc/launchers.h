// Plain-function front doors of the heavy kernel templates.  Each family of templates is instantiated
// in its own translation unit (gemm_tu.cu, tail_fast_tu.cu, tail_general_tu.cu) so that the library
// builds in parallel; payne_b200.cu holds the host logic and the small kernels and calls through here.
#pragma once
#include <cuda_runtime.h>

#include "mlp_simt.cuh"
#include "mlp_tc_types.h"
#include "tail_fast.cuh"
#include "tail_lsf.cuh"

namespace payne {

// cudaFuncAttributeMaxDynamicSharedMemorySize of `func` on the current device, raised to at least `bytes` and never
// lowered (tail_general_tu.cu).  The attribute belongs to the function on the device, not to a context: contexts that
// share one instantiation at different sizes (LSF, photometry and general tails) must not cap each other's launches.
// A high-water mark per (function, device) behind a mutex; only a successful call raises it.
cudaError_t raise_max_dyn_smem(const void* func, size_t bytes);

// ---- gemm_tu.cu: lin2..lin6 on tcgen05 (mlp_tc.cuh)
int tc_prepare_weights_x(TcWeights* w, const float* W_host, int N, int K, std::vector<void*>* owned);
int tc_alloc_acts_x(TcActs* a, long long rows, long long ld);
void tc_free_acts_x(TcActs* a);
// encode + lin1 + operand slicing (parity mode); grid_y = chunk nets (1 otherwise)
int launch_encode_x3(const EncodeParams& E, const double* x, long long ld, const float* W1, const float* b1,
                     TcActs* acts, int nb, int grid_y, long long plane_gstride, cudaStream_t st);
int tc_run_layers_x(const TcWeights* tcw, float* const* bias, const int* dims_in, const int* dims_out,
                    const float* h1, TcActs* actA, TcActs* actB, int nb, float* out, long long ldo,
                    float bias_shift, int prec, int sm_count, cudaStream_t st, long long* launches,
                    TcMapCache* caches, long long out_rows, TcStackCache* stack_cache = nullptr);
int tc_run_multinet_x(const TcWeights* tcw, float* const* bias, int H, int D_out, int groups, int chunk,
                      TcActs* actA, TcActs* actB, long long rows_per_group, int nb, float* out, long long ldo,
                      float bias_shift, int prec, int sm_count, cudaStream_t st, long long* launches,
                      long long out_rows);
// output layer of a leaky-ReLU stack from fp32 activations of any sign / magnitude (row-scaled slices)
int tc_run_scaled_layer_x(const TcWeights& w, const float* bias, const float* h, long long ldh, TcActs* acts,
                          float* rscale, int nb, float* out, long long ldo, float bias_shift, int sm_count,
                          cudaStream_t st, long long* launches);
// unit-test GEMM: slices dA [M, K] into the operand planes of `a`, then C = A . W^T + bias
int tc_gemm_test_x(const float* dA, int M, int N, int K, int precision, TcActs& a, const TcWeights& w,
                   const float* dbias, float* dC, int sm_count);

// ---- tail_fast_tu.cu / tail_fast_poly_tu.cu: fused tail on log-uniform grids (tail_fast.cuh)
// One form of tail_fast_kernel per kind of batch: points naming stars, targets (payne_ctx_set_targets), binaries
// (payne_ctx_set_binary) and continuum marginalisation (payne_ctx_set_cont_marg, for points or targets).  Each size
// has a form's instantiations in two translation units: without (tail_fast_tu.cu) and with (tail_fast_poly_tu.cu)
// continuum polynomial or model output in the final pass; Binary and Marg exist with them only.  tail_fast_tu.inl maps a
// form (and the second of its pair: several stars, or targets under Marg) to the kernel's point body, FastBody.
enum class FastForm { Point, Target, Binary, Marg };
// sets the dynamic shared-memory opt-in of every instantiation `form` may launch at 2^l2 samples on the current device
// and reports the smallest of their resident CTAs per SM; false when the kernel does not exist for l2 or a query fails
bool probe_tail_fast(int l2, FastForm form, size_t smem_bytes, int* ctas_per_sm);
// the instantiation follows from T: polynomial or model output (T.n_poly, T.model_out), several stars (Point,
// T.n_stars > 1) or targets (Marg, T.target)
int launch_tail_fast(int l2, FastForm form, int grid, size_t smem_bytes, cudaStream_t st, const TailParams& T, const FastGrid& F);
// the per-point setup of a slab of nb points (tail_setup_kernel<BODY>): one item per point, per (point, member) of a
// target (Target, or Marg with T.target) or per (point, component) of a binary
int launch_tail_setup(FastForm form, int nb, cudaStream_t st, const TailParams& T, const FastGrid& F);
// copies the first-pass constants into the translation units' __constant__ memory on the current device
// (call once per context, before the first launch)
int init_tail_fast(const TwConst& tc);
int init_tail_cluster(const TwConst& tc);

// ---- tail_cluster_tu.cu: the same tail with one transform spread over a cluster of four CTAs (tail_cluster.cuh;
// emulator grids above 16384 pixels).  max_clusters = co-resident clusters on the device.
bool probe_tail_cluster(int l2, size_t smem_bytes, int* ctas_per_sm, int* max_clusters);
int launch_tail_cluster(int l2, int n_clusters, size_t smem_bytes, cudaStream_t st, const TailParams& T, const FastGrid& F);

// ---- tail_general_tu.cu: any increasing grid (tail_general.cuh), LSF-vector broadening (tail_lsf.cuh)
bool probe_tail_general(int l2, size_t smem_bytes, int* ctas_per_sm);
int launch_tail_general(int l2, int grid, size_t smem_bytes, cudaStream_t st, const TailParams& T, const TwConst& tc);
bool probe_tail_lsf(size_t smem_bytes, int* ctas_per_sm);
int launch_tail_lsf(int grid, size_t smem_bytes, cudaStream_t st, const TailParams& T, const LsfParams& L);
// targets on a context with LSF vectors (payne_ctx_set_targets): the TGT instantiation of tail_lsf_kernel, same grid and
// dynamic shared memory as the star form (lsf_alloc)
bool probe_tail_lsf_targets(size_t smem_bytes, int* ctas_per_sm);
int launch_tail_lsf_targets(int grid, size_t smem_bytes, cudaStream_t st, const TailParams& T, const LsfParams& L);
int launch_continuum(int grid, cudaStream_t st, const ContParams& C);
// unit-test convolution: y = irfft(rfft(x) * H) of 2^log2N real samples (device buffers; H[0..N/2] without the
// 1/M; tw = the N/2-entry twiddle table of the tails), one CTA on the default stream
int launch_fft_test(const float* x, int log2N, const float* H, const float2* tw, float* y);

}  // namespace payne
