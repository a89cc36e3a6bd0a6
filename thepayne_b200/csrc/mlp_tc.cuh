// Emulator layers lin2..lin6 on the 5th-gen tensor cores (sm_100a): C = act(A . W^T + b).
//
//   reference: Payne/train/NNmodels.py:154-162  sigmoid(lin_k(h)) for k=2..5, lin6 linear.
//
// The reference runs fp32 Linear layers; the tensor cores have no fp32 MMA.  Three operand
// modes share one kernel:
//
//  X3 (parity mode)  "exact-accumulation" split.  Every operand is cut into three 8-bit
//      fixed-point slices stored as bf16: activations h in (0,1) as h = p1 + p2 + p3 with
//      p_i = k_i 2^-8i, |k_i| <= 256; weights row-wise as w = s_n (q1 + q2 + q3), s_n a power of
//      two >= max|w_n|, q_i = k_i 2^-(8i-1), |k_i| <= 128.  The dominant product sum
//      sum_k p1 q1 is then an integer multiple of 2^-15 below 2^24 for K <= 512 -- EXACTLY
//      representable in the fp32 TMEM accumulator, so the tensor core never rounds it -- and
//      the five cross terms p1q2, p2q1, p1q3, p2q2, p3q1 (<= 2^-8 of the result) go to a second
//      accumulator whose rounding is ~2^-32 of the result.  Six bf16 MMAs (K=16) cost the same
//      tensor time as three TF32 MMAs (K=8) but give a correctly rounded fp32 dot product
//      (3xTF32 measured here: coherent ~1e-6 bias from fp32 accumulator truncation over 96
//      MMA steps, which shows up as |dlnL| ~ 1e-2).
//  T3  3xTF32 error-compensated split (hi/lo), kept for comparison.
//  T1  1xTF32, fast mode (not a parity mode).
//
// Kernel anatomy (one CTA per SM, persistent over 128 x BN output tiles, 256 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor 128B-swizzled K-major boxes of the operand
//               planes into an NSTAGE ring, mbarrier complete_tx
//   warp 1      MMA issuer: one elected lane issues tcgen05.mma (M=128, N=BN) from shared-memory
//               descriptors; tcgen05.commit frees the ring slot / publishes the accumulator
//   warp 2      TMEM allocator (double-buffered accumulators)
//   warps 4-7   epilogue: tcgen05.ld 32 lanes x 32 columns -> scale, +bias (-> sigmoid -> split)
//               -> transposed through a padded smem patch -> 128-byte coalesced row stores
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <cmath>
#include <cstdlib>
#include <vector>

#include "../../include/payne_b200.h"
#include "mlp_simt.cuh"
#include "mlp_tc_types.h"

namespace payne {

enum { kModeT1 = 0, kModeT3 = 1, kModeX3 = 2 };

// ------------------------------------------------------------------ PTX wrappers
namespace ptx {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA store of a shared-memory box (128B-swizzled) into the output tensor; out-of-range rows /
// columns of the box are clipped by the tensor map.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }   // the 4 epilogue warps
template <int NTHREADS>
__device__ __forceinline__ void epi_bar_sync_n() { asm volatile("bar.sync 1, %0;" ::"n"(NTHREADS) : "memory"); }

__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void mma_bf16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accum) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
}  // namespace ptx

// K-major, 128-byte-swizzled operand tile: rows of 128 bytes, 8-row groups 1024 bytes apart.
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);          // start address
  d |= (uint64_t)1 << 16;                               // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                     // stride byte offset
  d |= (uint64_t)1 << 46;                               // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                               // SWIZZLE_128B
  return d;
}
// fp32 accumulate, A and B K-major, M=128; fmt: 2 = TF32 (kind::tf32), 1 = BF16 (kind::f16)
__host__ __device__ constexpr uint32_t umma_idesc(int N, uint32_t fmt) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// fixed-point slices of the exact-accumulation split -----------------------------------------
// activations (0 <= h < ~1): p1 = rint(h 2^8) 2^-8, p2 = rint(r1 2^16) 2^-16, p3 = rint(r2 2^24) 2^-24
// Rounding to a multiple of 2^-s is done by adding and subtracting 1.5 * 2^(23-s): in that binade one
// ulp is 2^-s, so the fp32 add itself rounds (to nearest, ties to even) exactly like rintf(h 2^s) 2^-s,
// without the three conversions per element that kept the epilogue on the slow XU pipe.
__device__ __forceinline__ float round_to_pow2_grid(float x, float magic) {
  return __fsub_rn(__fadd_rn(x, magic), magic);
}
__device__ __forceinline__ void x3_split_act(float h, __nv_bfloat16& p1, __nv_bfloat16& p2, __nv_bfloat16& p3) {
  const float a1 = round_to_pow2_grid(h, 49152.f);          // 1.5 * 2^15 : grid 2^-8
  const float r1 = h - a1;
  const float a2 = round_to_pow2_grid(r1, 192.f);           // 1.5 * 2^7  : grid 2^-16
  const float r2 = r1 - a2;
  const float a3 = round_to_pow2_grid(r2, 0.75f);           // 1.5 * 2^-1 : grid 2^-24
  p1 = __float2bfloat16_rn(a1); p2 = __float2bfloat16_rn(a2); p3 = __float2bfloat16_rn(a3);
}

// output-layer tile width; 64 (3-deep ring) was measured slower: MLP 0.274 vs 0.195 ms (A tile re-read twice as often)
#ifndef PAYNE_LIN6_BN
#define PAYNE_LIN6_BN 128
#endif
constexpr int kTcThreads = 256;
// Hidden layers (sigmoid + operand slicing epilogue, ~40 dependent instructions per element) get four
// groups of four epilogue warps: with one warp per scheduler the epilogue ran at IPC 0.16 and took more
// than half of the kernel; each group takes 16 of the tile's 64 columns.
template <int MODE, int EPI>
struct TcThreads {
  static constexpr int kEpiWarps = (EPI == 1 && MODE == kModeX3) ? 16 : 4;
  static constexpr int value = 128 + 32 * kEpiWarps;
};
constexpr int kBM = 128;
constexpr int kRowBytes = 128;   // one swizzle row: 32 tf32 or 64 bf16 along K

// Epilogue of one 32-row x 32-column block for the fp32 output layer: (main [+ corr]) * scale +
// bias, written as 16-byte chunks into a 128B-swizzled staging block and stored by TMA.
//   stage : this warp's 4 KB staging block (1024-byte aligned);  sb / ss : bias and scale of the
//   tile's columns in shared memory;  lane = row of the block.
template <bool X3>
__device__ __forceinline__ void epi_store_block(const CUtensorMap* cmap, float* stage, const float* sb,
                                                const float* ss, const uint32_t (&v)[32], const uint32_t (&c)[32],
                                                int colbase, int gcol0, int grow0, int lane, float rs = 1.f) {
  if (lane == 0) ptx::tma_store_wait_read();      // the previous store has finished reading the block
  __syncwarp();
  float4* st4 = reinterpret_cast<float4*>(stage) + lane * 8;
  const float4* b4 = reinterpret_cast<const float4*>(sb + colbase);
  const float4* s4 = reinterpret_cast<const float4*>(ss + colbase);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float4 bb = b4[k], sc = s4[k];
    float4 o;
    if (X3) {
      // rs and sc are powers of two: the products below are exact, the FMA rounds once
      o.x = fmaf((__uint_as_float(v[4 * k + 0]) + __uint_as_float(c[4 * k + 0])) * rs, sc.x, bb.x);
      o.y = fmaf((__uint_as_float(v[4 * k + 1]) + __uint_as_float(c[4 * k + 1])) * rs, sc.y, bb.y);
      o.z = fmaf((__uint_as_float(v[4 * k + 2]) + __uint_as_float(c[4 * k + 2])) * rs, sc.z, bb.z);
      o.w = fmaf((__uint_as_float(v[4 * k + 3]) + __uint_as_float(c[4 * k + 3])) * rs, sc.w, bb.w);
    } else {
      o.x = __uint_as_float(v[4 * k + 0]) + bb.x; o.y = __uint_as_float(v[4 * k + 1]) + bb.y;
      o.z = __uint_as_float(v[4 * k + 2]) + bb.z; o.w = __uint_as_float(v[4 * k + 3]) + bb.w;
    }
    st4[k ^ (lane & 7)] = o;                      // 128B swizzle: chunk index XOR (row mod 8)
  }
  ptx::fence_async_smem();
  __syncwarp();
  if (lane == 0) ptx::tma_store_2d(cmap, stage, gcol0, grow0);
}

template <int BN, int MODE>
struct TcCfg {
  static constexpr int kPlanes = MODE == kModeX3 ? 3 : (MODE == kModeT3 ? 2 : 1);
  static constexpr int kElemBytes = MODE == kModeX3 ? 2 : 4;
  static constexpr int kBK = kRowBytes / kElemBytes;              // K elements per stage
  static constexpr int kUmmaK = 32 / kElemBytes;                  // K per MMA
  static constexpr int kABytes = kBM * kRowBytes, kBBytes = BN * kRowBytes;
  static constexpr int kStageBytes = kPlanes * (kABytes + kBBytes);
  // epilogue staging (TMA-store blocks / transpose patches); the 64-wide parity tiles are the hidden
  // layers, whose epilogue stays in registers, so their ring gets the space: 3 stages instead of 2
  static constexpr int kPatchBytes = (MODE == kModeX3 && BN == 64) ? 0 : 4 * 32 * 33 * 4;
  static constexpr int kBudget = 232448 - kPatchBytes - 1024 - 256 - 2 * BN * 4;
  static constexpr int kStages = (kBudget / kStageBytes) > 6 ? 6 : (kBudget / kStageBytes);
  static constexpr int kSmem = kStages * kStageBytes + kPatchBytes + 1024 /*align*/ + 256 /*barriers*/ +
                               2 * BN * 4 /*bias, scale*/;
  static constexpr int kAccCols = MODE == kModeX3 ? 2 * BN : BN;  // columns per accumulator set
  static constexpr int kTmemCols = 2 * kAccCols;                  // double buffered
  static_assert(kTmemCols <= 512, "TMEM budget");
};


struct TcGemmArgs {
  const float* bias;
  const float* wscale;  // X3: per output column power-of-two scale
  const float* rscale;  // EPI 0, X3: per output ROW power-of-two scale of the A operand (null = 1): rows whose
                        // activations are not confined to [0,1) are sliced as h / rscale (x3_split_rows_kernel)
  void* out0;           // EPI 0: fp32 C ; EPI 1: plane 0 of the next layer's operand
  void* out1;
  void* out2;
  long long ldc;
  float bias_shift;     // EPI 0: added to the bias (-1 makes the layer emit line depth f - 1)
  int M, N, K;
  // Grouped launch (multi-chunk emulator, Payne/train/old/trainspec_multi.py:29-52): `groups` independent
  // GEMMs of the same shape share one persistent grid; the tile index carries the group.  Group g reads
  // activation rows [g a_grows, +M) of the planes, weight rows [g b_grows, +N) (bias / scale alike) and
  // writes columns [g b_grows, +N) of the fp32 output (EPI 0) or plane rows offset by g out_gstride
  // elements (EPI 1).  The last group may be narrower (n_last columns).  groups = 1: a plain GEMM.
  int groups, n_last;
  long long a_grows, b_grows, out_gstride;
};

template <int BN, int MODE, int EPI>
__global__ void __launch_bounds__(TcThreads<MODE, EPI>::value, 1)
tc_gemm_kernel(const __grid_constant__ TcMaps T, const __grid_constant__ TcGemmArgs G) {
  using Cfg = TcCfg<BN, MODE>;
  static_assert(Cfg::kPatchBytes > 0 || (EPI == 1 && MODE == kModeX3), "this epilogue needs its staging block");
  constexpr int NS = Cfg::kStages, NP = Cfg::kPlanes;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = (unsigned char*)(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
  unsigned char* stages = base;
  float* patch = (float*)(base + NS * Cfg::kStageBytes);
  uint64_t* bars = (uint64_t*)((unsigned char*)patch + Cfg::kPatchBytes);
  uint64_t* full = bars;                 // [NS]
  uint64_t* empty = bars + NS;           // [NS]
  uint64_t* tfull = bars + 2 * NS;       // [2]
  uint64_t* tempty = bars + 2 * NS + 2;  // [2]
  uint32_t* tmem_ptr = (uint32_t*)(bars + 2 * NS + 4);
  float* sbias = (float*)(bars + 32);    // 256 bytes reserved for barriers
  float* sscale = sbias + BN;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_m = (G.M + kBM - 1) / kBM, num_n = (G.N + BN - 1) / BN;
  const int tiles_per_group = num_m * num_n;
  const int num_tiles = tiles_per_group * G.groups;
  const int num_kb = (G.K + Cfg::kBK - 1) / Cfg::kBK;
  const int tile0 = (int)blockIdx.x;
  const int tstep = (int)gridDim.x;

  if (warp == 0 && lane == 0) {
    for (int p = 0; p < NP; ++p) { ptx::prefetch_tmap(&T.a[p]); ptx::prefetch_tmap(&T.b[p]); }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NS; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { ptx::mbar_init(&tfull[a], 1); ptx::mbar_init(&tempty[a], TcThreads<MODE, EPI>::kEpiWarps); }
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc(tmem_ptr, Cfg::kTmemCols);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // Programmatic dependent launch: everything above (barriers, TMEM, descriptor prefetch) touched no
  // global data, so it may run while the previous layer's grid drains; from here on the previous
  // grid must have completed.  The next layer is released right away -- it parks at this same point.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp == 0) {
    // ===================== TMA producer: stage = [A planes][B planes]
    if (lane == 0) {
      int s = 0; uint32_t ph = 0;
      for (int tile = tile0; tile < num_tiles; tile += tstep) {
        const int grp = tile / tiles_per_group, tig = tile - grp * tiles_per_group;
        const int m0 = (tig / num_n) * kBM, n0 = (tig % num_n) * BN;
        if (n0 >= (grp == G.groups - 1 ? G.n_last : G.N)) continue;       // narrower last group
        const int arow = (int)(grp * G.a_grows) + m0, brow = (int)(grp * G.b_grows) + n0;
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(&empty[s], ph ^ 1);
          unsigned char* st = stages + s * Cfg::kStageBytes;
          ptx::mbar_expect_tx(&full[s], Cfg::kStageBytes);
          const int k0 = kb * Cfg::kBK;
#pragma unroll
          for (int p = 0; p < NP; ++p) {
            ptx::tma_load_2d(&T.a[p], &full[s], st + p * Cfg::kABytes, k0, arow);
            ptx::tma_load_2d(&T.b[p], &full[s], st + NP * Cfg::kABytes + p * Cfg::kBBytes, k0, brow);
          }
          if (++s == NS) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc(BN, MODE == kModeX3 ? 1u : 2u);
      int s = 0; uint32_t ph = 0;
      int acc = 0; uint32_t aph = 0;
      for (int tile = tile0; tile < num_tiles; tile += tstep) {
        {
          const int grp = tile / tiles_per_group, tig = tile - grp * tiles_per_group;
          if ((tig % num_n) * BN >= (grp == G.groups - 1 ? G.n_last : G.N)) continue;
        }
        ptx::mbar_wait(&tempty[acc], aph ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_main = tmem_base + (uint32_t)(acc * Cfg::kAccCols);
        const uint32_t d_corr = d_main + BN;               // X3 only
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(&full[s], ph);
          ptx::tc_fence_after();
          const uint32_t st = ptx::smem_u32(stages + s * Cfg::kStageBytes);
          uint64_t da[3], db[3];
#pragma unroll
          for (int p = 0; p < NP; ++p) {
            da[p] = umma_desc_k_sw128(st + p * Cfg::kABytes);
            db[p] = umma_desc_k_sw128(st + NP * Cfg::kABytes + p * Cfg::kBBytes);
          }
#pragma unroll
          for (int ks = 0; ks < Cfg::kBK / Cfg::kUmmaK; ++ks) {
            const uint64_t ko = (uint64_t)((ks * 32) >> 4);   // 32 bytes of K per MMA
            const uint32_t first = (kb | ks) != 0;
            if constexpr (MODE == kModeX3) {
              ptx::mma_bf16(d_main, da[0] + ko, db[0] + ko, idesc, first);       // p1 q1 (exact)
              ptx::mma_bf16(d_corr, da[0] + ko, db[2] + ko, idesc, first);       // p1 q3
              ptx::mma_bf16(d_corr, da[1] + ko, db[1] + ko, idesc, 1);           // p2 q2
              ptx::mma_bf16(d_corr, da[2] + ko, db[0] + ko, idesc, 1);           // p3 q1
              ptx::mma_bf16(d_corr, da[0] + ko, db[1] + ko, idesc, 1);           // p1 q2
              ptx::mma_bf16(d_corr, da[1] + ko, db[0] + ko, idesc, 1);           // p2 q1
            } else if constexpr (MODE == kModeT3) {
              ptx::mma_tf32(d_main, da[1] + ko, db[0] + ko, idesc, first);       // lo hi
              ptx::mma_tf32(d_main, da[0] + ko, db[1] + ko, idesc, 1);           // hi lo
              ptx::mma_tf32(d_main, da[0] + ko, db[0] + ko, idesc, 1);           // hi hi
            } else {
              ptx::mma_tf32(d_main, da[0] + ko, db[0] + ko, idesc, first);
            }
          }
          ptx::mma_commit(&empty[s]);                  // frees the ring slot when the MMAs retire
          if (kb == num_kb - 1) ptx::mma_commit(&tfull[acc]);
          if (++s == NS) { s = 0; ph ^= 1; }
        }
        if (++acc == 2) { acc = 0; aph ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (warp w may only touch TMEM lanes 32*(w%4) .. +31)
    const int q = warp & 3;
    float* pt = patch + q * (EPI == 0 ? 1024 : 32 * 33);     // EPI 0: 4 KB swizzled staging block
    int acc = 0; uint32_t aph = 0;
    for (int tile = tile0; tile < num_tiles; tile += tstep) {
      const int grp = tile / tiles_per_group, tig = tile - grp * tiles_per_group;
      const int m0 = (tig / num_n) * kBM, n0 = (tig % num_n) * BN;
      const int Ng = grp == G.groups - 1 ? G.n_last : G.N;         // this group's output width
      if (n0 >= Ng) continue;
      const int gcol = (int)(grp * G.b_grows);                     // bias / scale / output-column offset
      const long long gout = grp * G.out_gstride;                  // EPI 1: plane offset of the group
      constexpr bool kRegEpi = (EPI == 1 && MODE == kModeX3);   // hidden layer, rows stay in registers
      if constexpr (EPI == 0 || kRegEpi) {
        // bias (+shift) and scale of this tile's columns -> shared memory, before the accumulator
        // is awaited so the loads are off the critical path
        constexpr int kEpiThreads = 32 * TcThreads<MODE, EPI>::kEpiWarps;
        ptx::epi_bar_sync_n<kEpiThreads>();        // previous tile's readers are done
        for (int cix = threadIdx.x - 128; cix < BN; cix += kEpiThreads) {
          const int gc = n0 + cix;
          sbias[cix] = (gc < Ng ? __ldg(G.bias + gcol + gc) : 0.f) + G.bias_shift;
          sscale[cix] = (MODE == kModeX3 && gc < Ng) ? __ldg(G.wscale + gcol + gc) : 1.f;
        }
        ptx::epi_bar_sync_n<kEpiThreads>();
      }
      ptx::mbar_wait(&tfull[acc], aph);
      ptx::tc_fence_after();
      const int row_base = m0 + q * 32;
      const uint32_t t_main = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * Cfg::kAccCols);
      if constexpr (EPI == 0) {
        const float rs = (MODE == kModeX3 && G.rscale && row_base + lane < G.M) ? __ldg(G.rscale + row_base + lane) : 1.f;
#pragma unroll 1
        for (int ch = 0; ch < BN / 32; ++ch) {
          const int col0 = n0 + ch * 32;
          if (col0 >= Ng) break;
          uint32_t v[32], c[32];
          ptx::tmem_ld32_nowait(t_main + (uint32_t)(ch * 32), v);
          if constexpr (MODE == kModeX3) ptx::tmem_ld32_nowait(t_main + (uint32_t)(BN + ch * 32), c);
          ptx::tmem_ld_wait();
          epi_store_block<MODE == kModeX3>(&T.c, pt, sbias, sscale, v, c, ch * 32, gcol + col0, row_base, lane, rs);
        }
      } else if constexpr (kRegEpi) {
        // Hidden layer: thread = row.  Its 32 accumulator columns never leave registers:
        // sigmoid, three fixed-point slices, and per plane four 16-byte stores of 8 bf16 (each
        // row's 64 bytes are contiguous, so the stores fill whole sectors without a transpose).
        const int grow = row_base + lane;
        const bool rowok = grow < G.M;
        constexpr int NG = TcThreads<MODE, EPI>::kEpiWarps / 4, CW = BN / NG;   // column groups, columns each
        static_assert(CW == 16, "hidden-layer epilogue: 16 columns per warp group");
        const int wgrp = (warp - 4) >> 2;
        const int cbase = wgrp * CW, col0 = n0 + cbase;
        if (col0 < Ng) {
          uint32_t v[CW], c[CW];
          ptx::tmem_ld16_nowait(t_main + (uint32_t)cbase, v);
          ptx::tmem_ld16_nowait(t_main + (uint32_t)(BN + cbase), c);
          ptx::tmem_ld_wait();
          const long long o = gout + (long long)grow * G.ldc + col0;
          const float4* b4 = reinterpret_cast<const float4*>(sbias + cbase);
          const float4* s4 = reinterpret_cast<const float4*>(sscale + cbase);
#pragma unroll
          for (int g8 = 0; g8 < CW / 8; ++g8) {
            __align__(16) __nv_bfloat16 q1[8], q2[8], q3[8];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const float4 bb = b4[2 * g8 + h], sc = s4[2 * g8 + h];
              const float bbv[4] = {bb.x, bb.y, bb.z, bb.w}, scv[4] = {sc.x, sc.y, sc.z, sc.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int j = 8 * g8 + 4 * h + e;
                const float val = sigmoidf_exact(fmaf(__uint_as_float(v[j]) + __uint_as_float(c[j]), scv[e], bbv[e]));
                x3_split_act(val, q1[4 * h + e], q2[4 * h + e], q3[4 * h + e]);
              }
            }
            if (rowok) {
              const int gc = col0 + 8 * g8;
              if (gc + 8 <= Ng) {
                *reinterpret_cast<uint4*>((__nv_bfloat16*)G.out0 + o + 8 * g8) = *reinterpret_cast<const uint4*>(q1);
                *reinterpret_cast<uint4*>((__nv_bfloat16*)G.out1 + o + 8 * g8) = *reinterpret_cast<const uint4*>(q2);
                *reinterpret_cast<uint4*>((__nv_bfloat16*)G.out2 + o + 8 * g8) = *reinterpret_cast<const uint4*>(q3);
              } else {
#pragma unroll
                for (int e = 0; e < 8; ++e)
                  if (gc + e < Ng) {
                    ((__nv_bfloat16*)G.out0)[o + 8 * g8 + e] = q1[e];
                    ((__nv_bfloat16*)G.out1)[o + 8 * g8 + e] = q2[e];
                    ((__nv_bfloat16*)G.out2)[o + 8 * g8 + e] = q3[e];
                  }
              }
            }
          }
        }
      } else {
#pragma unroll 1
      for (int ch = 0; ch < BN / 32; ++ch) {
        const int col0 = n0 + ch * 32;
        if (col0 >= Ng) break;
        uint32_t v[32];
        ptx::tmem_ld32_nowait(t_main + (uint32_t)(ch * 32), v);
        if constexpr (MODE == kModeX3) {
          uint32_t c[32];
          ptx::tmem_ld32_nowait(t_main + (uint32_t)(BN + ch * 32), c);
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) pt[lane * 33 + j] = __uint_as_float(v[j]) + __uint_as_float(c[j]);
        } else {
          ptx::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) pt[lane * 33 + j] = __uint_as_float(v[j]);
        }
        __syncwarp();
        const int lcol = col0 + lane;
        const bool colok = lcol < Ng;
        float bv = colok ? __ldg(G.bias + gcol + lcol) : 0.f;
        if (EPI == 0) bv += G.bias_shift;
        const float sc = (MODE == kModeX3 && colok) ? __ldg(G.wscale + gcol + lcol) : 1.f;
#pragma unroll 4
        for (int r = 0; r < 32; ++r) {
          const int grow = row_base + r;
          if (grow >= G.M) break;
          float val = fmaf(pt[r * 33 + lane], sc, bv);
          if (colok) {
            const long long o = (EPI == 0 ? (long long)gcol : gout) + (long long)grow * G.ldc + lcol;
            if (EPI == 0) {
              ((float*)G.out0)[o] = val;
            } else {
              val = sigmoidf_exact(val);
              if constexpr (MODE == kModeX3) {
                __nv_bfloat16 p1, p2, p3;
                x3_split_act(val, p1, p2, p3);
                ((__nv_bfloat16*)G.out0)[o] = p1; ((__nv_bfloat16*)G.out1)[o] = p2; ((__nv_bfloat16*)G.out2)[o] = p3;
              } else {
                const float hi = ptx::to_tf32(val);
                ((float*)G.out0)[o] = hi;
                ((float*)G.out1)[o] = ptx::to_tf32(val - hi);
              }
            }
          }
        }
        __syncwarp();
      }
      }
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tempty[acc]);
      if (++acc == 2) { acc = 0; aph ^= 1; }
    }
    if (EPI == 0 && lane == 0) ptx::tma_store_wait_all();
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

// fp32 -> operand planes of the next GEMM
static __global__ void tf32_split_kernel(const float* __restrict__ src, long long lds, float* __restrict__ hi,
                                  float* __restrict__ lo, long long ldd, long long rows, int cols) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const long long r = i / cols; const int c = (int)(i % cols);
  const float x = src[r * lds + c];
  const float h = ptx::to_tf32(x);
  hi[r * ldd + c] = h;
  lo[r * ldd + c] = ptx::to_tf32(x - h);
}
static __global__ void x3_split_kernel(const float* __restrict__ src, long long lds, __nv_bfloat16* __restrict__ p1,
                                __nv_bfloat16* __restrict__ p2, __nv_bfloat16* __restrict__ p3, long long ldd,
                                long long rows, int cols) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const long long r = i / cols; const int c = (int)(i % cols);
  __nv_bfloat16 a, b, d;
  x3_split_act(src[r * lds + c], a, b, d);
  p1[r * ldd + c] = a; p2[r * ldd + c] = b; p3[r * ldd + c] = d;
}

// Rows that are not confined to [0,1) (leaky-ReLU activations): one warp per row finds s = the power of two >= max|h|
// of the row, writes it to rscale and slices h / s (|h / s| <= 1, signed slices: the magic-number rounding of
// x3_split_act is sign-agnostic and bf16 holds the integers up to 256 exactly).  The leading product sum stays exact
// for K <= 512 (|p1 q1| <= 1, grid 2^-15).  Precision is 2^-24 of the ROW maximum rather than of each element, which
// for a dot product is what an fp32 GEMM's own rounding amounts to.
static __global__ void __launch_bounds__(256)
x3_split_rows_kernel(const float* __restrict__ src, long long lds, __nv_bfloat16* __restrict__ p1,
                     __nv_bfloat16* __restrict__ p2, __nv_bfloat16* __restrict__ p3, long long ldd,
                     float* __restrict__ rscale, int rows, int cols) {
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (r >= rows) return;
  const float* h = src + (long long)r * lds;
  float mx = 0.f;
  for (int c = lane; c < cols; c += 32) mx = fmaxf(mx, fabsf(h[c]));      // fmaxf drops NaN: those rows come out NaN anyway
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float s = 1.f;
  if (mx > 0.f && mx < 3.0e38f) {
    int e;
    const float m = frexpf(mx, &e);                  // mx = m 2^e, 0.5 <= m < 1
    s = ldexpf(1.f, (m == 0.5f) ? e - 1 : e);        // smallest power of two >= mx
  }
  if (lane == 0) rscale[r] = s;
  const float inv = 1.f / s;                          // exact
  for (int c = lane; c < cols; c += 32) {
    __nv_bfloat16 a, b, d;
    x3_split_act(h[c] * inv, a, b, d);
    const long long o = (long long)r * ldd + c;
    p1[o] = a; p2[o] = b; p3[o] = d;
  }
}

// Label encode + first layer + fixed-point slicing in one pass (parity mode): one warp per point.
// Lane i < D_in encodes label i once (fp64, NNmodels.py:164-168) and the warp shares the result;
// each lane then forms outputs h = lane, lane + 32, ... with the same fmaf order as
// encode_layer1_kernel and writes the three bf16 planes that lin2 reads.
static __global__ void __launch_bounds__(256)
encode_layer1_x3_kernel(const __grid_constant__ EncodeParams E, const double* __restrict__ x, long long ld,
                        const float* __restrict__ W1, const float* __restrict__ b1, __nv_bfloat16* __restrict__ p1,
                        __nv_bfloat16* __restrict__ p2, __nv_bfloat16* __restrict__ p3, long long ldp, int B,
                        long long plane_gstride) {
  const int lane = threadIdx.x & 31;
  const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  // multi-chunk emulator: blockIdx.y = chunk net; its first layer follows the previous one in W1 / b1 and
  // its operand planes start plane_gstride elements further on (gridDim.y = 1 otherwise)
  W1 += (long long)blockIdx.y * E.H1 * E.D_in;
  b1 += (long long)blockIdx.y * E.H1;
  p1 += blockIdx.y * plane_gstride; p2 += blockIdx.y * plane_gstride; p3 += blockIdx.y * plane_gstride;
  // lets the first tensor-core layer (launched with programmatic stream serialization) get resident and
  // run its prologue now; it still waits for this grid to finish before touching the planes
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (p >= B) return;
  float mine = 0.f;
  if (lane < E.D_in) {
    const double raw = label_of(E, x, ld, p, lane);
    const double xv = E.cast32 ? (double)(float)raw : raw;          // predictspec.py:70
    mine = (float)((xv - E.xmin[lane]) / (E.xmax[lane] - E.xmin[lane]) - E.offset);
  }
  float enc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) enc[i] = __shfl_sync(0xffffffffu, mine, i);
  // four outputs per trip so that their weight loads are in flight together (the kernel is a
  // chain of L2 latencies otherwise)
  for (int h0 = lane; h0 < E.H1; h0 += 128) {
    float w[4][8], bb[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int h = h0 + 32 * u;
      bb[u] = h < E.H1 ? __ldg(b1 + h) : 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) w[u][i] = (h < E.H1 && i < E.D_in) ? __ldg(W1 + h * E.D_in + i) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int h = h0 + 32 * u;
      if (h >= E.H1) break;
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (i < E.D_in) acc = fmaf(enc[i], w[u][i], acc);
      const float v = sigmoidf_exact(acc + bb[u]);
      __nv_bfloat16 a, b, c;
      x3_split_act(v, a, b, c);
      const long long o = (long long)p * ldp + h;
      p1[o] = a; p2[o] = b; p3[o] = c;
    }
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

// 2-D row-major [rows, K] (pitch ld elements) -> boxes of {128 bytes of K, box_rows}, 128B swizzle
// fp32 output [rows, cols] with pitch ld floats -> 32 x 32 boxes, 128B swizzle (TMA store)
inline int make_tmap_out(CUtensorMap* m, const void* ptr, long long rows, int cols, long long ld, int box_rows = 32) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return PAYNE_E_CUDA;
  if ((ld & 3) || ((uintptr_t)ptr & 15)) return PAYNE_E_INVALID;   // TMA: 16-byte base and pitch
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)ptr, gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? PAYNE_OK : PAYNE_E_CUDA;
}

inline int make_tmap(CUtensorMap* m, const void* ptr, long long rows, int K, long long ld, int box_rows,
                     int elem_bytes) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return PAYNE_E_CUDA;
  cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * elem_bytes};
  cuuint32_t box[2] = {(cuuint32_t)(kRowBytes / elem_bytes), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
                   (void*)ptr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? PAYNE_OK : PAYNE_E_CUDA;
}

// Host-side split of a weight matrix (done once per context).
inline int tc_prepare_weights(TcWeights* w, const float* W_host, int N, int K, std::vector<void*>* owned) {
  const int Kp = (K + 7) / 8 * 8;    // TMA needs 16-byte row pitches; the map's extent stays K (OOB = 0)
  w->N = N; w->K = K; w->Kp = Kp;
  const size_t n = (size_t)N * Kp;
  std::vector<float> hi(n), lo(n), sc(N);
  std::vector<uint16_t> q[3] = {std::vector<uint16_t>(n), std::vector<uint16_t>(n), std::vector<uint16_t>(n)};
  auto tf32 = [](float x) {   // cvt.rna.tf32: round to nearest, ties away, 10-bit mantissa
    uint32_t u; memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) == 0x7F800000u) return x;
    u += 0x1000u; u &= 0xFFFFE000u;
    float r; memcpy(&r, &u, 4); return r;
  };
  auto bf16bits = [](float x) { uint32_t u; memcpy(&u, &x, 4); return (uint16_t)(u >> 16); };   // exact by construction
  for (int r = 0; r < N; ++r) {
    float mx = 0.f;
    for (int k = 0; k < K; ++k) mx = std::max(mx, std::fabs(W_host[(size_t)r * K + k]));
    int e = 0;
    float s = 1.f;
    if (mx > 0.f && std::isfinite(mx)) { std::frexp(mx, &e); s = std::ldexp(1.f, e); }
    sc[r] = s;
    for (int k = 0; k < K; ++k) {
      const size_t i = (size_t)r * Kp + k;
      const float x = W_host[(size_t)r * K + k];
      hi[i] = tf32(x); lo[i] = tf32(x - hi[i]);
      const float u = x / s;                                            // exact (power of two)
      const float a1 = std::nearbyint(u * 128.f) / 128.f;
      const float r1 = u - a1;
      const float a2 = std::nearbyint(r1 * 32768.f) / 32768.f;
      const float r2 = r1 - a2;
      const float a3 = std::nearbyint(r2 * 8388608.f) / 8388608.f;
      q[0][i] = bf16bits(a1); q[1][i] = bf16bits(a2); q[2][i] = bf16bits(a3);
    }
  }
  auto up = [&](void** dst, const void* src, size_t bytes) {
    if (cudaMalloc(dst, bytes) != cudaSuccess) return PAYNE_E_NOMEM;
    owned->push_back(*dst);
    return cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice) == cudaSuccess ? PAYNE_OK : PAYNE_E_CUDA;
  };
  int rc = up(&w->plane[0], hi.data(), n * 4); if (rc) return rc;
  rc = up(&w->plane[1], lo.data(), n * 4); if (rc) return rc;
  for (int p = 0; p < 3; ++p) { rc = up(&w->xplane[p], q[p].data(), n * 2); if (rc) return rc; }
  rc = up((void**)&w->scale, sc.data(), (size_t)N * 4);
  return rc;
}

inline int tc_alloc_acts(TcActs* a, long long rows, long long ld) {
  a->rows = rows; a->ld = ld;
  for (int p = 0; p < 3; ++p)
    if (cudaMalloc(&a->plane[p], (size_t)rows * ld * 4) != cudaSuccess) return PAYNE_E_NOMEM;
  return PAYNE_OK;
}
inline void tc_free_acts(TcActs* a) {
  for (int p = 0; p < 3; ++p) { if (a->plane[p]) cudaFree(a->plane[p]); a->plane[p] = nullptr; }
  a->rows = 0;
}

// PAYNE_GEMM_PDL=0 switches programmatic dependent launch of the layer chain off.
inline bool tc_pdl_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("PAYNE_GEMM_PDL"); v = (e && e[0] == '0') ? 0 : 1; }
  return v != 0;
}

// Groups of a grouped launch (see TcGemmArgs).  n = output width of every group but the last.
struct TcGroups {
  int groups = 1, n = 0, n_last = 0;
  long long a_grows = 0, out_gstride = 0;
};

template <int BN, int MODE, int EPI>
inline int tc_launch(const TcActs& A, int K, const TcWeights& W, const float* bias, void* out0, void* out1,
                     void* out2, long long ldc, float bias_shift, int M, int sm_count, cudaStream_t st,
                     TcMapCache* cache = nullptr, long long map_rows = 0, const TcGroups* grp = nullptr,
                     int out_cols = 0, const float* rscale = nullptr) {
  using Cfg = TcCfg<BN, MODE>;
  static_assert(Cfg::kStages >= 2, "ring too shallow");
  constexpr int kVariant = BN * 100 + MODE * 10 + EPI;
  const bool grouped = grp && grp->groups > 1;
  // grouped: the maps span every group's rows of the planes (a_grows rows each)
  const long long mrows = grouped ? grp->groups * grp->a_grows : ((cache && map_rows >= M) ? map_rows : M);
  TcMaps local;
  TcMaps& T = cache ? cache->maps : local;
  const void* key[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, out0};
  for (int p = 0; p < Cfg::kPlanes; ++p) { key[p] = A.plane[p]; key[3 + p] = MODE == kModeX3 ? W.xplane[p] : W.plane[p]; }
  bool hit = cache && cache->variant == kVariant && cache->rows == mrows && cache->lda == A.ld && cache->ldc == ldc;
  for (int i = 0; i < 7 && hit; ++i) hit = cache->ptr[i] == key[i];
  if (!hit) {
    if (cache) cache->variant = -1;
    for (int p = 0; p < Cfg::kPlanes; ++p) {
      const void* wp = MODE == kModeX3 ? W.xplane[p] : W.plane[p];
      if (make_tmap(&T.a[p], A.plane[p], mrows, K, A.ld, kBM, Cfg::kElemBytes)) return PAYNE_E_CUDA;
      if (make_tmap(&T.b[p], wp, W.N, K, W.Kp, BN, Cfg::kElemBytes)) return PAYNE_E_CUDA;
    }
    for (int p = Cfg::kPlanes; p < 3; ++p) { T.a[p] = T.a[0]; T.b[p] = T.b[0]; }
    if (EPI == 0) {
      // out_cols: output width of a grouped launch (a launch of one group writes W.N columns)
      const long long orows = grouped ? ((cache && map_rows >= M) ? map_rows : M) : mrows;
      if (int rc = make_tmap_out(&T.c, out0, orows, (grouped && out_cols > 0) ? out_cols : W.N, ldc)) return rc;
    } else T.c = T.a[0];
    if (cache) {
      for (int i = 0; i < 7; ++i) cache->ptr[i] = key[i];
      cache->rows = mrows; cache->lda = A.ld; cache->ldc = ldc;
      cache->variant = kVariant;
    }
  }
  // the opt-in above 48 KB is a per-device attribute of the function: one flag per device ordinal
  static unsigned long long attr_set = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return PAYNE_E_CUDA;
  if (dev >= 64 || !((attr_set >> dev) & 1ull)) {
    if (cudaFuncSetAttribute(tc_gemm_kernel<BN, MODE, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             Cfg::kSmem) != cudaSuccess) return PAYNE_E_CUDA;
    if (dev < 64) attr_set |= 1ull << dev;
  }
  TcGemmArgs G{bias, W.scale, rscale, out0, out1, out2, ldc, bias_shift, M, W.N, K, 1, W.N, 0, 0, 0};
  if (grouped) {
    G.N = grp->n; G.groups = grp->groups; G.n_last = grp->n_last; G.a_grows = grp->a_grows; G.b_grows = grp->n;
    G.out_gstride = grp->out_gstride;
  }
  const int num_m = (M + kBM - 1) / kBM, num_n = (G.N + BN - 1) / BN;
  const int tiles = num_m * num_n * G.groups;
  const int grid = tiles < sm_count ? tiles : sm_count;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(TcThreads<MODE, EPI>::value); cfg.dynamicSmemBytes = Cfg::kSmem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = tc_pdl_enabled() ? 1 : 0;
  cfg.attrs = at; cfg.numAttrs = 1;
  if (cudaLaunchKernelEx(&cfg, tc_gemm_kernel<BN, MODE, EPI>, T, G) != cudaSuccess) return PAYNE_E_CUDA;
  return cudaGetLastError() == cudaSuccess ? PAYNE_OK : PAYNE_E_CUDA;
}

inline int tc_launch_hidden_stack(const TcWeights* tcw, float* const* bias, int layers, int H, TcActs* a0, TcActs* a1,
                                  int M, cudaStream_t st, TcStackCache* cache);      // mlp_stack.cuh

template <int MODE>
inline int tc_run_layers_mode(const TcWeights* tcw, float* const* bias, const int* dims_in, const int* dims_out,
                              const float* h1, TcActs* actA, TcActs* actB, int nb, float* out, long long ldo,
                              float bias_shift, int sm_count, cudaStream_t st, long long* launches,
                              TcMapCache* caches, long long out_rows, TcStackCache* stack_cache = nullptr) {
  const long long tot = (long long)nb * dims_out[0];
  const unsigned blocks = (unsigned)((tot + 255) / 256);
  if (h1 == nullptr)
    --*launches;      // the caller already wrote the sliced planes of layer 1 (encode_layer1_x3_kernel)
  else if (MODE == kModeX3)
    x3_split_kernel<<<blocks, 256, 0, st>>>(h1, dims_out[0], (__nv_bfloat16*)actA->plane[0],
                                            (__nv_bfloat16*)actA->plane[1], (__nv_bfloat16*)actA->plane[2],
                                            actA->ld, nb, dims_out[0]);
  else
    tf32_split_kernel<<<blocks, 256, 0, st>>>(h1, dims_out[0], (float*)actA->plane[0], (float*)actA->plane[1],
                                              actA->ld, nb, dims_out[0]);
  ++*launches;
  TcActs* cur = actA; TcActs* nxt = actB;
  int rc = PAYNE_OK;
  bool stacked = false;
  if constexpr (MODE == kModeX3) {
    // lin2 .. lin5 in one launch when they are all H -> H (mlp_stack.cuh); four layers end in actA again
    bool uniform = true;
    for (int k = 1; k < 5; ++k) uniform = uniform && dims_in[k] == dims_in[1] && dims_out[k] == dims_in[1];
    if (uniform && stack_cache && tc_launch_hidden_stack(tcw, bias, 4, dims_in[1], actA, actB, nb, st, stack_cache) == PAYNE_OK) {
      stacked = true;
      ++*launches;
    }
  }
  for (int k = 1; k < 5 && !rc && !stacked; ++k) {
    rc = tc_launch<64, MODE, 1>(*cur, dims_in[k], tcw[k], bias[k], nxt->plane[0], nxt->plane[1], nxt->plane[2],
                                nxt->ld, 0.f, nb, sm_count, st, caches ? caches + k : nullptr, cur->rows);
    ++*launches;
    TcActs* t = cur; cur = nxt; nxt = t;
  }
  if (rc) return rc;
  rc = tc_launch<PAYNE_LIN6_BN, MODE, 0>(*cur, dims_in[5], tcw[5], bias[5], out, nullptr, nullptr, ldo, bias_shift, nb,
                               sm_count, st, caches ? caches + 5 : nullptr, out_rows >= cur->rows ? cur->rows : 0);
  ++*launches;
  return rc;
}

// Multi-chunk emulator (Payne/train/old/trainspec_multi.py:29-52): G nets Net(D_in, H, P), sigmoid, 4 layers.
// lin1 was written by the caller as sliced planes [G][rows, H]; here lin2, lin3 (grouped hidden GEMMs) and
// lin4, whose G output blocks of P columns make up the contiguous flux row.  One launch per layer when
// every chunk but the last is a multiple of 32 pixels wide (TMA-store boxes are 32 columns; a partial
// box of chunk g would overwrite columns of chunk g+1), otherwise one launch per chunk for lin4.
template <int MODE>
inline int tc_run_multinet_mode(const TcWeights* tcw, float* const* bias, int H, int D_out, int groups, int chunk,
                                TcActs* actA, TcActs* actB, long long rows_per_group, int nb, float* out,
                                long long ldo, float bias_shift, int sm_count, cudaStream_t st, long long* launches,
                                long long out_rows) {
  TcGroups gh;
  gh.groups = groups; gh.n = H; gh.n_last = H; gh.a_grows = rows_per_group; gh.out_gstride = rows_per_group * actA->ld;
  TcActs* cur = actA; TcActs* nxt = actB;
  int rc = PAYNE_OK;
  for (int k = 1; k <= 2 && !rc; ++k) {
    rc = tc_launch<64, MODE, 1>(*cur, H, tcw[k], bias[k], nxt->plane[0], nxt->plane[1], nxt->plane[2], nxt->ld, 0.f,
                                nb, sm_count, st, nullptr, 0, &gh);
    ++*launches;
    TcActs* t = cur; cur = nxt; nxt = t;
  }
  if (rc) return rc;
  const int n_last = D_out - (groups - 1) * chunk;
  if (chunk % 32 == 0 || groups == 1) {
    TcGroups g4;
    g4.groups = groups; g4.n = chunk; g4.n_last = n_last; g4.a_grows = rows_per_group; g4.out_gstride = 0;
    rc = tc_launch<PAYNE_LIN6_BN, MODE, 0>(*cur, H, tcw[3], bias[3], out, nullptr, nullptr, ldo, bias_shift, nb, sm_count,
                                           st, nullptr, out_rows, &g4, D_out);
    ++*launches;
    return rc;
  }
  for (int g = 0; g < groups && !rc; ++g) {              // general chunk widths: one GEMM per chunk
    TcActs a = *cur;
    const long long off = (long long)g * rows_per_group * cur->ld;
    for (int p = 0; p < 3; ++p) a.plane[p] = (char*)cur->plane[p] + off * (MODE == kModeX3 ? 2 : 4);
    a.rows = rows_per_group;
    TcWeights w = tcw[3];
    const int ng = g == groups - 1 ? n_last : chunk;
    const long long woff = (long long)g * chunk * w.Kp;
    for (int p = 0; p < 3; ++p) {
      if (w.plane[p]) w.plane[p] = (char*)w.plane[p] + woff * 4;
      if (w.xplane[p]) w.xplane[p] = (char*)w.xplane[p] + woff * 2;
    }
    w.scale = tcw[3].scale + (long long)g * chunk;
    w.N = ng;
    // the output map of this chunk covers exactly its ng columns: TMA clips the partial box.  The base
    // must be 16-byte aligned: chunk widths that are not multiples of 4 go through the SIMT layers.
    rc = tc_launch<PAYNE_LIN6_BN, MODE, 0>(a, H, w, bias[3] + (long long)g * chunk, out + (long long)g * chunk, nullptr,
                                           nullptr, ldo, bias_shift, nb, sm_count, st, nullptr, out_rows);
    ++*launches;
  }
  return rc;
}

inline int tc_run_multinet(const TcWeights* tcw, float* const* bias, int H, int D_out, int groups, int chunk,
                           TcActs* actA, TcActs* actB, long long rows_per_group, int nb, float* out, long long ldo,
                           float bias_shift, int prec, int sm_count, cudaStream_t st, long long* launches,
                           long long out_rows) {
  if (prec == PAYNE_PREC_PARITY && H > kX3MaxK) return PAYNE_E_UNSUPPORTED;
  switch (prec) {
    case PAYNE_PREC_PARITY:
      return tc_run_multinet_mode<kModeX3>(tcw, bias, H, D_out, groups, chunk, actA, actB, rows_per_group, nb, out,
                                           ldo, bias_shift, sm_count, st, launches, out_rows);
    default:
      return PAYNE_E_UNSUPPORTED;
  }
}

// Output layer of a leaky-ReLU stack (SMLP / YST1) on the tensor cores: fp32 activations h [nb, K] (any sign and
// magnitude) -> row-scaled slices -> out = h . W^T + bias (+ bias_shift), exact-accumulation split.
inline int tc_run_scaled_layer(const TcWeights& w, const float* bias, const float* h, long long ldh, TcActs* acts,
                               float* rscale, int nb, float* out, long long ldo, float bias_shift, int sm_count,
                               cudaStream_t st, long long* launches) {
  if (!w.xplane[0] || w.K > kX3MaxK) return PAYNE_E_UNSUPPORTED;
  x3_split_rows_kernel<<<(unsigned)((nb + 7) / 8), 256, 0, st>>>(h, ldh, (__nv_bfloat16*)acts->plane[0],
                                                                 (__nv_bfloat16*)acts->plane[1],
                                                                 (__nv_bfloat16*)acts->plane[2], acts->ld, rscale, nb, w.K);
  ++*launches;
  const int rc = tc_launch<PAYNE_LIN6_BN, kModeX3, 0>(*acts, w.K, w, bias, out, nullptr, nullptr, ldo, bias_shift, nb, sm_count,
                                                      st, nullptr, 0, nullptr, 0, rscale);
  ++*launches;
  return rc;
}

// lin2..lin6 from the fp32 output of lin1 (h1, pitch = dims_out[0]).  bias_shift is added to the
// last layer's bias (the likelihood path asks for line depth f - 1 with bias_shift = -1).
inline int tc_run_layers(const TcWeights* tcw, float* const* bias, const int* dims_in, const int* dims_out,
                         const float* h1, TcActs* actA, TcActs* actB, int nb, float* out, long long ldo,
                         float bias_shift, int prec, int sm_count, cudaStream_t st, long long* launches,
                         TcMapCache* caches = nullptr, long long out_rows = 0, TcStackCache* stack_cache = nullptr) {
  for (int k = 1; k < 6; ++k)
    if (!tcw[k].plane[0]) return PAYNE_E_UNSUPPORTED;
  // exactness of the leading product sum (header): K * 2^8 * 2^7 <= 2^24 needs K <= 512
  if (prec == PAYNE_PREC_PARITY)
    for (int k = 1; k < 6; ++k)
      if (dims_in[k] > kX3MaxK) return PAYNE_E_UNSUPPORTED;
  switch (prec) {
    case PAYNE_PREC_PARITY:
      return tc_run_layers_mode<kModeX3>(tcw, bias, dims_in, dims_out, h1, actA, actB, nb, out, ldo, bias_shift,
                                         sm_count, st, launches, caches, out_rows, stack_cache);
    case PAYNE_PREC_3XTF32:
      return tc_run_layers_mode<kModeT3>(tcw, bias, dims_in, dims_out, h1, actA, actB, nb, out, ldo, bias_shift,
                                         sm_count, st, launches, caches, out_rows);
    case PAYNE_PREC_TF32:
      return tc_run_layers_mode<kModeT1>(tcw, bias, dims_in, dims_out, h1, actA, actB, nb, out, ldo, bias_shift,
                                         sm_count, st, launches, caches, out_rows);
    default:
      return PAYNE_E_UNSUPPORTED;
  }
}

}  // namespace payne
