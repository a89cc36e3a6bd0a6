// Host-visible types of the tcgen05 GEMM path (mlp_tc.cuh) -- no device code, so that translation units
// which only hold these objects do not compile the GEMM kernels.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <vector>

namespace payne {

constexpr int kX3MaxK = 512;    // widest contraction the exact-accumulation split covers (see header)

struct TcWeights {
  void* plane[3] = {nullptr, nullptr, nullptr};   // T: fp32 hi, lo ; X3: bf16 q1, q2, q3
  void* xplane[3] = {nullptr, nullptr, nullptr};
  float* scale = nullptr;                          // X3: per-row power of two
  int N = 0, K = 0, Kp = 0;                        // Kp: row pitch in elements (16-byte multiple for TMA)
};
struct TcActs {
  void* plane[3] = {nullptr, nullptr, nullptr};    // sized for fp32; bf16 planes alias the storage
  long long rows = 0, ld = 0;
};

struct TcMaps {
  CUtensorMap a[3];
  CUtensorMap b[3];
  CUtensorMap c;       // EPI 0: fp32 output [M, N] (pitch ldc), boxes of 32 x 32, 128B swizzle
};

// Tensor maps of one layer, reusable while the buffers stay put: encoding seven descriptors through
// the driver costs several microseconds of host time per launch, which is what bounds the latency
// of small batches.  The maps cover `rows` (the allocated row count), not the batch: rows past the
// batch are computed on stale data and land in workspace rows nobody reads.
// The key holds every pointer the maps encode: a workspace that grows frees and reallocates all activation planes, and
// the allocator may hand one of them back at its old address while the others move.
struct TcMapCache {
  TcMaps maps;
  const void* ptr[7] = {};   // A planes 0-2, weight planes 0-2, output (unused planes of the mode: null)
  long long rows = 0, lda = 0, ldc = 0;
  int variant = -1;
};

// The hidden-layer stack as one launch (mlp_stack.cuh): maps of the two ping-pong activation buffers and of
// up to four layers' weight planes; arguments; and the cache of the encoded maps.
constexpr int kStackMaxLayers = 4;
struct TcStackMaps {
  CUtensorMap a[2][3];
  CUtensorMap b[kStackMaxLayers][3];
};
struct TcStackArgs {
  const float* bias[kStackMaxLayers];
  const float* wscale[kStackMaxLayers];   // per output column power-of-two scale of the weight slices
  void* plane[2][3];                      // bf16 planes of the two buffers; layer l reads (first + l) & 1, writes the other
  long long ld;                           // plane pitch in elements
  int M, H, layers, first;
};
struct TcStackCache {
  TcStackMaps maps;
  const void* ptr[6 + 3 * kStackMaxLayers] = {};   // every plane the maps encode (both buffers, every layer's weights)
  long long rows = 0, lda = 0;
  int H = 0, layers = 0;
  bool valid = false;
};

}  // namespace payne
