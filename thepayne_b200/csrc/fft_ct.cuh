// Compile-time-planned variant of the in-shared-memory FFT convolution of fft.cuh (same
// algorithm, same storage swizzle, same digit-reversed filter stage) for the fast tail.
//
// What changes relative to fft.cuh:
//  * the radix plan is constexpr, so every shift/stride is an immediate and the digit reversal
//    of the filter stage unrolls to a few bit-field moves (no local-memory plan array);
//  * twiddles are hoisted: a thread's butterflies in one pass share j = tid mod S, so the R-1
//    factors W_L^{jq} are loaded ONCE per pass (a 22 KB, L1-resident subset of the table); in
//    the first pass of a large transform (S > blockDim) the i-th butterfly needs
//    W_L^{(tid + NT i) q} = W_L^{tid q} * exp(-2 pi i NT i q / L): base factor times a constant
//    that lives in the kernel-parameter (constant) bank.
#pragma once
#include "fft.cuh"

namespace payne {

constexpr int kNT = 256;   // threads per CTA in the tail kernels

template <int LOG2M>
struct CtPlan {
  // log2 radices of the strided passes; the contiguous radix-16 pass follows.
  static constexpr int rest0 = LOG2M - 4;
  __host__ __device__ static constexpr int pick(int rest) {
    return (rest == 5 || rest % 3 == 0) ? 3 : (rest >= 4 ? 4 : rest);
  }
  static constexpr int r0 = rest0 > 0 ? pick(rest0) : 0;
  static constexpr int rest1 = rest0 - r0;
  static constexpr int r1 = rest1 > 0 ? pick(rest1) : 0;
  static constexpr int rest2 = rest1 - r1;
  static constexpr int r2 = rest2 > 0 ? pick(rest2) : 0;
  static constexpr int rest3 = rest2 - r2;
  static constexpr int r3 = rest3 > 0 ? pick(rest3) : 0;
  static_assert(rest3 - r3 == 0, "plan needs more than four strided passes");
  static constexpr int n = (r0 > 0) + (r1 > 0) + (r2 > 0) + (r3 > 0);
  __host__ __device__ static constexpr int lr(int i) { return i == 0 ? r0 : i == 1 ? r1 : i == 2 ? r2 : r3; }
  __host__ __device__ static constexpr int log2L(int i) {   // sub-transform length entering pass i
    return i == 0 ? LOG2M : i == 1 ? LOG2M - r0 : i == 2 ? LOG2M - r0 - r1 : LOG2M - r0 - r1 - r2;
  }
  __host__ __device__ static constexpr int row_of(int klo) {
    int row = 0;
    int l = LOG2M - 4;
    if (r0 > 0) { l -= r0; row += (klo & ((1 << r0) - 1)) << l; klo >>= r0; }
    if (r1 > 0) { l -= r1; row += (klo & ((1 << r1) - 1)) << l; klo >>= r1; }
    if (r2 > 0) { l -= r2; row += (klo & ((1 << r2) - 1)) << l; klo >>= r2; }
    if (r3 > 0) { l -= r3; row += (klo & ((1 << r3) - 1)) << l; }
    return row;
  }
};

// First-pass constants exp(-2 pi i * ip * kNT * q / M) for transforms with M/R > kNT.
struct TwConst {
  float2 c[2][4][16];   // [log2M - 13][ip][q]
};

// Compact per-pass twiddle tables.  The factors W_L^{jq} a thread hoists for one strided pass are
// scattered over the main table (one useful 8 bytes per 128-byte line: 7 line fetches per thread,
// a >100 KB line footprint that the ~30 KB of L1 left beside the transform buffers cannot hold, so
// every pass started with L2-latency loads).  Here they are laid out [pass][j][q], q fastest: a
// thread reads R consecutive float2 (64 or 128 bytes), a warp 2-4 KB contiguous, and the whole
// set for one transform size is 25-42 KB.  Values are copies of main-table entries (bit-identical).
template <int LOG2M>
struct CtTwLayout {
  using P = CtPlan<LOG2M>;
  __host__ __device__ static constexpr int J(int p) {          // distinct j per pass held by a CTA
    const int S = 1 << (P::log2L(p) - P::lr(p));
    return S < kNT ? S : kNT;
  }
  __host__ __device__ static constexpr int off(int p) {        // float2 offset of pass p
    int o = 0;
    for (int i = 0; i < p; ++i) o += J(i) << P::lr(i);
    return o;
  }
  static constexpr int total = off(P::n);
};

struct TwTab {
  const float2* __restrict__ tab;   // exp(-2 pi i e / 2^log2n), e < 2^(log2n-1)
  int log2n;
  const float2* const* pass;        // pass[LOG2M] -> CtTwLayout<LOG2M> table (device pointers, in param space)
};

template <int LOG2L>
__device__ __forceinline__ float2 tw_load(const TwTab& tw, int x) {   // W_L^x, 0 <= x < L
  const int sh = tw.log2n - LOG2L;
  const int e = x << sh;
  const int half = 1 << (tw.log2n - 1);
#if defined(PAYNE_FFT_VARIANT) && PAYNE_FFT_VARIANT == 3     // microbenchmark: no table access
  float2 w = make_float2(__int_as_float(0x3f800000 | (e & 0xffff)), 0.5f);
#else
  float2 w = __ldg(tw.tab + (e & (half - 1)));
#endif
  if (e & half) { w.x = -w.x; w.y = -w.y; }
  return w;
}

template <int LOG2M, int PASS, bool INV>
__device__ __forceinline__ void ct_strided_pass(float2* z, const TwTab& tw, const TwConst& tc, int tid) {
  using P = CtPlan<LOG2M>;
  constexpr int LR = P::lr(PASS), R = 1 << LR, LOG2L = P::log2L(PASS), LOG2S = LOG2L - LR, S = 1 << LOG2S;
  constexpr int NBF = (1 << (LOG2M - LR));             // butterflies in the pass
  constexpr int NB = (NBF + kNT - 1) / kNT;            // per thread
  constexpr int SPAN = S > kNT ? S / kNT : 1;          // distinct j per thread
  static_assert(SPAN <= 4, "first pass too wide for the constant table");
  static_assert(SPAN == 1 || (PASS == 0 && LOG2M >= 13 && LOG2M <= 14), "constant table covers log2M 13..14");
  const int jb = tid & (S - 1);
  float2 wb[R];
#if defined(PAYNE_FFT_VARIANT) && PAYNE_FFT_VARIANT == 4     // microbenchmark: scattered main-table loads
#pragma unroll
  for (int q = 1; q < R; ++q) wb[q] = tw_load<LOG2L>(tw, jb * q);
#else
  {
    const float4* pt = reinterpret_cast<const float4*>(tw.pass[LOG2M] + CtTwLayout<LOG2M>::off(PASS) + (jb << LR));
#pragma unroll
    for (int q = 0; q < R; q += 2) {
      const float4 u = __ldg(pt + (q >> 1));
      wb[q] = make_float2(u.x, u.y);
      wb[q + 1] = make_float2(u.z, u.w);
    }
  }
#endif
#pragma unroll
  for (int i = 0; i < NB; ++i) {
    const int g = tid + kNT * i;
    if (NBF % kNT != 0 && g >= NBF) break;
    const int b = g >> LOG2S, j = g & (S - 1);
    const int base = (b << LOG2L) + j;
    float2 v[R];
    // stride >= 128 points: adding m*S never touches the bits the swizzle reads or flips
    const int sbase = swz(base);
#if defined(PAYNE_FFT_VARIANT) && PAYNE_FFT_VARIANT == 2     // microbenchmark: math only
#pragma unroll
    for (int m = 0; m < R; ++m) v[m] = make_float2(__int_as_float(sbase + m), __int_as_float(base - m));
#else
#pragma unroll
    for (int m = 0; m < R; ++m) v[m] = (LOG2S >= 7) ? z[sbase + (m << LOG2S)] : z[swz(base + (m << LOG2S))];
#endif
    constexpr int kSet = LOG2M >= 13 ? LOG2M - 13 : 0;
    const int ip = i % SPAN;
#if defined(PAYNE_FFT_VARIANT) && PAYNE_FFT_VARIANT == 1     // microbenchmark: memory traffic only
    if (false) {
#else
    if constexpr (!INV) {
#endif
      dftR<R, false>(v);
#pragma unroll
      for (int q = 1; q < R; ++q) {
        float2 w = wb[q];
        if (SPAN > 1 && ip != 0) w = cmul(w, tc.c[kSet][ip][q]);
        v[q] = cmul(v[q], w);
      }
    } else {
#pragma unroll
      for (int q = 1; q < R; ++q) {
        float2 w = wb[q];
        if (SPAN > 1 && ip != 0) w = cmul(w, tc.c[kSet][ip][q]);
        v[q] = cmulc(v[q], w);
      }
      dftR<R, true>(v);
    }
#if defined(PAYNE_FFT_VARIANT) && PAYNE_FFT_VARIANT == 2
    float2 acc = v[0];
#pragma unroll
    for (int m = 1; m < R; ++m) acc = acc + v[m];
    if (acc.x == 1.2345f) z[sbase] = acc;          // keeps the math alive, never true in practice
#else
#pragma unroll
    for (int m = 0; m < R; ++m) {
      if (LOG2S >= 7) z[sbase + (m << LOG2S)] = v[m];
      else z[swz(base + (m << LOG2S))] = v[m];
    }
#endif
  }
}

// The last strided pass works on blocks of 16*R points; thread tid + kNT*i of that pass owns
// block (tid>>4) + (kNT/16) i, i.e. warp w owns blocks {2w, 2w+1} + (kNT/16) i.  When the
// contiguous pass visits the 16-point groups in the SAME per-warp order, the two passes only need
// __syncwarp() between them (kWarpLocal): two block barriers fewer per transform.
template <int LOG2M>
struct CtLast {
  using P = CtPlan<LOG2M>;
  static constexpr int LRL = P::n > 0 ? P::lr(P::n - 1) : 0;          // log2 radix of the last strided pass
  static constexpr int NG = 1 << (LOG2M - 4);                          // 16-point groups
  static constexpr bool kWarpLocal = P::n > 0 && (NG % kNT == 0) && ((1 << (LOG2M - LRL)) % kNT == 0);
};

template <int LOG2M, bool INV>
__device__ __forceinline__ void ct_contiguous16(float2* z, int tid) {
  float4* z4 = reinterpret_cast<float4*>(z);
  using CL = CtLast<LOG2M>;
  constexpr int NG = CL::NG;
#pragma unroll
  for (int i = 0; i < (NG + kNT - 1) / kNT; ++i) {
    int g = tid + kNT * i;
    if (NG % kNT != 0 && g >= NG) break;
    if constexpr (CL::kWarpLocal) {
      constexpr int R = 1 << CL::LRL;                 // groups per block
      const int w = tid >> 5, idx = (tid & 31) + 32 * i;
      const int bl = idx >> CL::LRL, sub = idx & (R - 1);
      g = ((2 * w + (bl & 1) + (kNT / 16) * (bl >> 1)) << CL::LRL) + sub;
    }
    float4* p = z4 + 8 * g;
    const int x = g & 7;
    float2 v[16];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float4 u = p[c ^ x];
      v[2 * c] = make_float2(u.x, u.y);
      v[2 * c + 1] = make_float2(u.z, u.w);
    }
    dft16<INV>(v);
#pragma unroll
    for (int c = 0; c < 8; ++c) p[c ^ x] = make_float4(v[2 * c].x, v[2 * c].y, v[2 * c + 1].x, v[2 * c + 1].y);
  }
}

// passes 1.. of the forward transform and the contiguous pass (pass 0 done by the caller)
template <int LOG2M>
__device__ __forceinline__ void ct_fft_forward_rest(float2* z, const TwTab& tw, const TwConst& tc, int tid) {
  using P = CtPlan<LOG2M>;
  constexpr bool WL = CtLast<LOG2M>::kWarpLocal;
  if constexpr (P::n > 0) { if (WL && P::n == 1) __syncwarp(); else __syncthreads(); }
  if constexpr (P::n > 1) { ct_strided_pass<LOG2M, 1, false>(z, tw, tc, tid); if (WL && P::n == 2) __syncwarp(); else __syncthreads(); }
  if constexpr (P::n > 2) { ct_strided_pass<LOG2M, 2, false>(z, tw, tc, tid); if (WL && P::n == 3) __syncwarp(); else __syncthreads(); }
  if constexpr (P::n > 3) { ct_strided_pass<LOG2M, 3, false>(z, tw, tc, tid); if (WL && P::n == 4) __syncwarp(); else __syncthreads(); }
  ct_contiguous16<LOG2M, false>(z, tid);
  __syncthreads();
}
template <int LOG2M>
__device__ __forceinline__ void ct_fft_forward(float2* z, const TwTab& tw, const TwConst& tc, int tid) {
  using P = CtPlan<LOG2M>;
  if constexpr (P::n > 0) ct_strided_pass<LOG2M, 0, false>(z, tw, tc, tid);
  ct_fft_forward_rest<LOG2M>(z, tw, tc, tid);
}

// First forward pass with its inputs interpolated on the fly from a global row: complex element idx
// is the pair of real samples (2 idx, 2 idx + 1) of the regridded signal, sample k = np.interp at row
// position k * num / den (see tail_fast.cuh regrid_in, whose arithmetic this repeats).  Fusing the
// regrid into the pass saves one full write + read of the transform buffer and a block barrier, and
// lets the interpolation arithmetic run under the pass's shared-memory time.  The row must carry two
// finite pad floats behind its last used element; NaN samples read as 0 (nan_to_num in depth space) unless
// CLEAN says the row cannot hold any (finite labels, no continuum emulator: 6 of ~40 instructions per pair).
template <int LOG2M, bool CLEAN>
__device__ __forceinline__ void ct_pass0_regrid(float2* z, const TwTab& tw, const TwConst& tc, int tid,
                                                const float* __restrict__ row, int num, int den, float invden,
                                                float c) {
  using P = CtPlan<LOG2M>;
  static_assert(P::n > 0, "needs a strided pass");
  constexpr int LR = P::lr(0), R = 1 << LR, LOG2S = LOG2M - LR, S = 1 << LOG2S;
  constexpr int NBF = 1 << (LOG2M - LR);
  constexpr int NB = (NBF + kNT - 1) / kNT;
  constexpr int SPAN = S > kNT ? S / kNT : 1;
  static_assert(SPAN <= 4, "first pass too wide for the constant table");
  static_assert(SPAN == 1 || (LOG2M >= 13 && LOG2M <= 14), "constant table covers log2M 13..14");
  const int jb = tid & (S - 1);
  float2 wb[R];
  {
    const float4* pt = reinterpret_cast<const float4*>(tw.pass[LOG2M] + CtTwLayout<LOG2M>::off(0) + (jb << LR));
#pragma unroll
    for (int q = 0; q < R; q += 2) {
      const float4 u = __ldg(pt + (q >> 1));
      wb[q] = make_float2(u.x, u.y);
      wb[q + 1] = make_float2(u.z, u.w);
    }
  }
  // row position of complex element tid, and the steps for +kNT and +S elements
  const long long v0 = 2LL * tid * num;
  int j = (int)(v0 / den);
  int rem = (int)(v0 - (long long)j * den);
  const long long vi = 2LL * kNT * num, vm = 2LL * S * num;
  const int ij = (int)(vi / den), ir = (int)(vi - (long long)ij * den);
  const int mj = (int)(vm / den), mr = (int)(vm - (long long)mj * den);
#pragma unroll 1
  for (int i = 0; i < NB; ++i) {
    const int g = tid + kNT * i;
    if (NBF % kNT != 0 && g >= NBF) break;
    float2 v[R];
    {
      const float* src = row + j;
      int rr = rem;
#pragma unroll
      for (int m = 0; m < R; ++m) {
        float a0 = src[0], a1 = src[1], a2 = src[2];
        if (!CLEAN) {
          if (a0 != a0) a0 = 0.f;
          if (a1 != a1) a1 = 0.f;
          if (a2 != a2) a2 = 0.f;
        }
        const int rem1 = rr + num;
        const bool same = rem1 < den;              // second sample still between row[j] and row[j+1]
        const float lo = same ? a0 : a1, hi = same ? a1 : a2;
        const float d0 = (float)rr * invden, d1 = (float)(same ? rem1 : rem1 - den) * invden;
        v[m].x = fmaf(fmaf(d0 * (d0 - 1.f), c, d0), a1 - a0, a0);
        v[m].y = fmaf(fmaf(d1 * (d1 - 1.f), c, d1), hi - lo, lo);
        rr += mr;
        int adv = mj;
        if (rr >= den) { rr -= den; ++adv; }
        src += adv;
      }
    }
    rem += ir;
    j += ij;
    if (rem >= den) { rem -= den; ++j; }
    const int sbase = swz(g);
    constexpr int kSet = LOG2M >= 13 ? LOG2M - 13 : 0;
    const int ip = i % SPAN;
    dftR<R, false>(v);
#pragma unroll
    for (int q = 1; q < R; ++q) {
      float2 w = wb[q];
      if (SPAN > 1 && ip != 0) w = cmul(w, tc.c[kSet][ip][q]);
      v[q] = cmul(v[q], w);
    }
#pragma unroll
    for (int m = 0; m < R; ++m) {
      if (LOG2S >= 7) z[sbase + (m << LOG2S)] = v[m];
      else z[swz(g + (m << LOG2S))] = v[m];
    }
  }
}

// inverse transform = contiguous pass + strided passes n-1 .. 1 (`mid`), then strided pass 0 (`last`)
template <int LOG2M>
__device__ __forceinline__ void ct_fft_inverse_mid(float2* z, const TwTab& tw, const TwConst& tc, int tid) {
  using P = CtPlan<LOG2M>;
  constexpr bool WL = CtLast<LOG2M>::kWarpLocal;
  ct_contiguous16<LOG2M, true>(z, tid);
  if (WL) __syncwarp(); else __syncthreads();
  if constexpr (P::n > 3) { ct_strided_pass<LOG2M, 3, true>(z, tw, tc, tid); __syncthreads(); }
  if constexpr (P::n > 2) { ct_strided_pass<LOG2M, 2, true>(z, tw, tc, tid); __syncthreads(); }
  if constexpr (P::n > 1) { ct_strided_pass<LOG2M, 1, true>(z, tw, tc, tid); __syncthreads(); }
}
template <int LOG2M>
__device__ __forceinline__ void ct_fft_inverse_last(float2* z, const TwTab& tw, const TwConst& tc, int tid) {
  using P = CtPlan<LOG2M>;
  if constexpr (P::n > 0) { ct_strided_pass<LOG2M, 0, true>(z, tw, tc, tid); __syncthreads(); }
}
template <int LOG2M>
__device__ __forceinline__ void ct_fft_inverse(float2* z, const TwTab& tw, const TwConst& tc, int tid) {
  ct_fft_inverse_mid<LOG2M>(z, tw, tc, tid);
  ct_fft_inverse_last<LOG2M>(z, tw, tc, tid);
}

// The passes of a convolution that do not depend on the filter (the fused first pass, the other forward passes,
// all inverse passes) as ONE copy of code per size, called from the rotation and the instrumental stage alike.
// Inlined into both they made the point loop of the fused tail ~15 k instructions (240 KB), more than the
// instruction cache holds with three CTAs per SM in different phases, and the kernel spilled (324 bytes at the
// 80-register cap; 0 with the passes in functions of their own, each with its own register allocation):
// C2 tail 0.736 -> 0.699 ms, measured A/B on one box.
// The transform buffer is the base of the dynamic shared memory (re-declared inside so that the accesses stay
// LDS / STS); the first-pass constants come from a __constant__ copy (one per translation unit, set by
// ct_set_twconst at context creation) so that they stay constant-bank operands.
#ifndef PAYNE_SHARED_PASSES
#define PAYNE_SHARED_PASSES 1
#endif
#ifndef PAYNE_SHARE_PASS0
#define PAYNE_SHARE_PASS0 0
#endif
#ifndef PAYNE_SHARE_INV0
#define PAYNE_SHARE_INV0 0
#endif
static __constant__ TwConst g_twc;
static inline cudaError_t ct_set_twconst(const TwConst& h) { return cudaMemcpyToSymbol(g_twc, &h, sizeof(TwConst)); }

template <int LOG2M>
static __device__ __noinline__ void ct_fwd_mid_shared(const TwTab tw, int tid) {       // forward passes 1.. + contiguous
  extern __shared__ __align__(16) unsigned char ct_dyn_smem[];
  ct_fft_forward_rest<LOG2M>(reinterpret_cast<float2*>(ct_dyn_smem), tw, g_twc, tid);
}
template <int LOG2M>
static __device__ __noinline__ void ct_fwd_all_shared(const TwTab tw, int tid) {       // whole forward transform
  extern __shared__ __align__(16) unsigned char ct_dyn_smem[];
  ct_fft_forward<LOG2M>(reinterpret_cast<float2*>(ct_dyn_smem), tw, g_twc, tid);
}
template <int LOG2M>
static __device__ __noinline__ void ct_inv_mid_shared(const TwTab tw, int tid) {       // inverse contiguous + passes .. 1
  extern __shared__ __align__(16) unsigned char ct_dyn_smem[];
  ct_fft_inverse_mid<LOG2M>(reinterpret_cast<float2*>(ct_dyn_smem), tw, g_twc, tid);
}
template <int LOG2M>
static __device__ __noinline__ void ct_inv_all_shared(const TwTab tw, int tid) {       // whole inverse transform
  extern __shared__ __align__(16) unsigned char ct_dyn_smem[];
  ct_fft_inverse<LOG2M>(reinterpret_cast<float2*>(ct_dyn_smem), tw, g_twc, tid);
}
template <int LOG2M, bool CLEAN>
static __device__ __noinline__ void ct_pass0_regrid_shared(const TwTab tw, int tid, const float* row, int num, int den,
                                                           float invden, float c) {
  extern __shared__ __align__(16) unsigned char ct_dyn_smem[];
  ct_pass0_regrid<LOG2M, CLEAN>(reinterpret_cast<float2*>(ct_dyn_smem), tw, g_twc, tid, row, num, den, invden, c);
}

// Filter stage on digit-reversed storage; H(k), k in [0, M], includes the 1/M of the inverse.
// Work item w = tid + kNT i  ->  (klo = w >> 4, c = w & 15): c is fixed per thread, so the factor
// exp(-2 pi i c / 32) of the untangling twiddle W_N^k, k = klo + c M/16, is a per-thread constant.
// One pair (k, M-k) of the filter stage: z[pk] holds Z_k, z[pp] holds Z_{M-k}; W = exp(-2 pi i k / N).
template <class HF>
__device__ __forceinline__ void ct_filter_one(float2* z, int pk, int pp, float2 W, float hk, float hm) {
  const float2 Zk = z[pk], Zp = z[pp];
  const float A = 0.5f * (hk + hm), Bc = 0.5f * (hk - hm);
  const float2 E = make_float2(0.5f * (Zk.x + Zp.x), 0.5f * (Zk.y - Zp.y));
  const float2 O = make_float2(0.5f * (Zk.y + Zp.y), -0.5f * (Zk.x - Zp.x));
  const float2 WO = cmul(W, O), WcE = cmulc(E, W);
  const float2 E2 = make_float2(A * E.x + Bc * WO.x, A * E.y + Bc * WO.y);
  const float2 O2 = make_float2(Bc * WcE.x + A * O.x, Bc * WcE.y + A * O.y);
  z[pk] = make_float2(E2.x - O2.y, E2.y + O2.x);
  if (pp != pk) z[pp] = make_float2(E2.x + O2.y, O2.x - E2.y);
}

template <int LOG2M, class HF>
__device__ __forceinline__ void ct_filter_pairs(float2* z, const TwTab& tw, const HF& H, int tid) {
  using P = CtPlan<LOG2M>;
  constexpr int M = 1 << LOG2M, Mlo = M >> 4;
  const int c = tid & 15;
  const float2 wc = tw_load<5>(tw, c);                  // exp(-2 pi i c / 32)
  if constexpr (Mlo >= 2 * kNT / 16 * 1 && (Mlo % (2 * kNT / 16)) == 0) {
    // klo = kb + 16 i with kb = tid >> 4 < 16: the digit reversal is a bit permutation, so
    // row_of(klo) = row_of(kb) + row_of(16 i) and the second term (like the storage swizzle,
    // which only reads row bits that come from i) folds to a constant once the loop is unrolled.
    // The partner klo' = Mlo - klo = ((16 - kb) & 15) + 16 (Mlo/16 - 1 - i + (kb == 0)).
    constexpr int KB = kNT / 16, NI = Mlo / (2 * KB);
    static_assert(KB == 16, "item mapping assumes 256 threads");
    const int kb = tid >> 4;
    const int rk = P::row_of(kb), rq = P::row_of((KB - kb) & (KB - 1));
    const bool kb0 = (kb == 0);
    const int sh = tw.log2n - (LOG2M + 1);
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int klo = kb + KB * i;
      const int k = klo + (c << (LOG2M - 4));
      const float2 W = cmul(__ldg(tw.tab + (klo << sh)), wc);       // exp(-2 pi i k / N); klo < N/4
      const float hk = H(k), hm = H(M - k);
      const int row = rk + P::row_of(KB * i);
      int rowp, c_p;
      if (i == 0) {
        // kb == 0: the pair lives inside row 0 (k' = M - k <-> c' = 16 - c); c > 8 already done by c' < 8
        rowp = kb0 ? 0 : rq + P::row_of(KB * (Mlo / KB - 1));
        c_p = kb0 ? ((16 - c) & 15) : 15 - c;
        if (kb0 && c > 8) continue;
      } else {
        rowp = kb0 ? P::row_of(Mlo - KB * i) : rq + P::row_of(KB * (Mlo / KB - 1 - i));
        c_p = 15 - c;
      }
      ct_filter_one<HF>(z, swz((row << 4) + c), swz((rowp << 4) + c_p), W, hk, hm);
    }
    if (tid < 8) {                                       // klo = Mlo/2 pairs with itself: c <-> 15 - c
      constexpr int klo = Mlo / 2;
      const int k = klo + (c << (LOG2M - 4));
      const float2 W = cmul(__ldg(tw.tab + (klo << sh)), wc);
      constexpr int row = P::row_of(klo);
      ct_filter_one<HF>(z, swz((row << 4) + c), swz((row << 4) + 15 - c), W, H(k), H(M - k));
    }
  } else {
    constexpr int NITEMS = ((Mlo >> 1) + 1) << 4;
#pragma unroll 2
    for (int w = tid; w < NITEMS; w += kNT) {
      const int klo = w >> 4;
      int klo_p, c_p;
      if (klo == 0) {
        if (c > 8) continue;
        klo_p = 0; c_p = (16 - c) & 15;
      } else {
        klo_p = Mlo - klo; c_p = 15 - c;
        if (klo_p == klo && c > 7) continue;
      }
      const int k = klo + (c << (LOG2M - 4));
      const float2 W = cmul(tw_load<LOG2M + 1>(tw, klo), wc);   // exp(-2 pi i k / N)
      ct_filter_one<HF>(z, swz((P::row_of(klo) << 4) + c), swz((P::row_of(klo_p) << 4) + c_p), W, H(k), H(M - k));
    }
  }
  __syncthreads();
}

// Same for the odd-frequency half of a split transform (see ct_convolve_split): local index k'
// stands for frequency k = 2k'+1 of a transform of size M = 2 Mh, whose partner M-k = 2(Mh-1-k')+1
// is the bitwise complement of k' -- in digit-reversed storage: row' = Mlo-1-row, c' = 15-c.
// H(k), k in [0, M], includes 1/M.
template <int LOG2MH, class HF>
__device__ __forceinline__ void ct_filter_pairs_odd(float2* z, const TwTab& tw, const HF& H, int tid) {
  using P = CtPlan<LOG2MH>;
  constexpr int Mh = 1 << LOG2MH, Mlo = Mh >> 4, M = 2 * Mh;
  constexpr int NITEMS = (Mlo >> 1) << 4;
  const int c = tid & 15;
#pragma unroll 2
  for (int w = tid; w < NITEMS; w += kNT) {
    const int klo = w >> 4;
    const int row = P::row_of(klo);
    const int kp = klo + (c << (LOG2MH - 4));
    const int k = 2 * kp + 1;
    const int pk = swz((row << 4) + c);
    const int pp = swz(((Mlo - 1 - row) << 4) + (15 - c));
    const float2 Zk = z[pk], Zp = z[pp];
    const float2 W = tw_load<LOG2MH + 2>(tw, k);          // exp(-2 pi i k / N), N = 2M = 4 Mh
    const float hk = H(k), hm = H(M - k);
    const float A = 0.5f * (hk + hm), Bc = 0.5f * (hk - hm);
    const float2 E = make_float2(0.5f * (Zk.x + Zp.x), 0.5f * (Zk.y - Zp.y));
    const float2 O = make_float2(0.5f * (Zk.y + Zp.y), -0.5f * (Zk.x - Zp.x));
    const float2 WO = cmul(W, O), WcE = cmulc(E, W);
    const float2 E2 = make_float2(A * E.x + Bc * WO.x, A * E.y + Bc * WO.y);
    const float2 O2 = make_float2(Bc * WcE.x + A * O.x, Bc * WcE.y + A * O.y);
    z[pk] = make_float2(E2.x - O2.y, E2.y + O2.x);
    z[pp] = make_float2(E2.x + O2.y, O2.x - E2.y);
  }
  __syncthreads();
}

template <class HF>
struct EvenBins {      // H restricted to even frequencies: local k' -> H(2k')
  const HF& H;
  __device__ __forceinline__ float operator()(int k) const { return H(2 * k); }
};

// Convolution of a real signal of N = 4 Mh samples that does not fit one SM's shared memory:
// complex points [0, Mh) live in shared memory (swizzled), points [Mh, 2Mh) in a global scratch
// line `g` that stays in L2.  One radix-2 DIF step across the halves leaves the even frequencies
// in the first half and the odd ones in the second; the pairs (k, M-k) of the filter stage never
// mix the two classes, so each half is transformed, filtered and transformed back entirely in
// shared memory (the halves swap places once), and a radix-2 DIT step restores natural order.
template <int LOG2MH, class HF>
__device__ __forceinline__ void ct_convolve_split(float2* z, float2* g, const TwTab& tw, const TwConst& tc,
                                                  const HF& H, int tid) {
  constexpr int Mh = 1 << LOG2MH;
  for (int j = tid; j < Mh; j += kNT) {                  // cross DIF
    const float2 a = z[swz(j)], b = g[j];
    z[swz(j)] = a + b;
    g[j] = cmul(a - b, tw_load<LOG2MH + 1>(tw, j));      // W_M^j, M = 2 Mh
  }
  __syncthreads();
  ct_fft_forward<LOG2MH>(z, tw, tc, tid);
  ct_filter_pairs<LOG2MH>(z, tw, EvenBins<HF>{H}, tid);
  ct_fft_inverse<LOG2MH>(z, tw, tc, tid);
  for (int j = tid; j < Mh; j += kNT) {                  // swap halves
    const float2 a = z[swz(j)];
    z[swz(j)] = g[j];
    g[j] = a;
  }
  __syncthreads();
  ct_fft_forward<LOG2MH>(z, tw, tc, tid);
  ct_filter_pairs_odd<LOG2MH>(z, tw, H, tid);
  ct_fft_inverse<LOG2MH>(z, tw, tc, tid);
  for (int j = tid; j < Mh; j += kNT) {                  // cross DIT
    const float2 a = g[j];
    const float2 b = cmulc(z[swz(j)], tw_load<LOG2MH + 1>(tw, j));
    z[swz(j)] = a + b;
    g[j] = a - b;
  }
  __syncthreads();
}

// ct_convolve with the regrid of the input row fused into the first pass (see ct_pass0_regrid)
template <int LOG2M, class HF>
__device__ __forceinline__ void ct_convolve_regrid(float2* z, const TwTab& tw, const TwConst& tc, const HF& H, int tid,
                                                   const float* row, int num, int den, float invden, float c,
                                                   bool clean) {
#if PAYNE_SHARED_PASSES
  // z is the base of the dynamic shared memory (tail_fast.cuh) and tc the context's copy of g_twc
#if PAYNE_SHARE_PASS0
  if (clean) ct_pass0_regrid_shared<LOG2M, true>(tw, tid, row, num, den, invden, c);
  else ct_pass0_regrid_shared<LOG2M, false>(tw, tid, row, num, den, invden, c);
#else
  if (clean) ct_pass0_regrid<LOG2M, true>(z, tw, tc, tid, row, num, den, invden, c);
  else ct_pass0_regrid<LOG2M, false>(z, tw, tc, tid, row, num, den, invden, c);
#endif
  ct_fwd_mid_shared<LOG2M>(tw, tid);
  ct_filter_pairs<LOG2M>(z, tw, H, tid);
#if PAYNE_SHARE_INV0
  ct_inv_all_shared<LOG2M>(tw, tid);
#else
  ct_inv_mid_shared<LOG2M>(tw, tid);
  ct_fft_inverse_last<LOG2M>(z, tw, tc, tid);
#endif
#else
  if (clean) ct_pass0_regrid<LOG2M, true>(z, tw, tc, tid, row, num, den, invden, c);
  else ct_pass0_regrid<LOG2M, false>(z, tw, tc, tid, row, num, den, invden, c);
  ct_fft_forward_rest<LOG2M>(z, tw, tc, tid);
  ct_filter_pairs<LOG2M>(z, tw, H, tid);
  ct_fft_inverse<LOG2M>(z, tw, tc, tid);
#endif
}

template <int LOG2M, class HF>
__device__ __forceinline__ void ct_convolve(float2* z, const TwTab& tw, const TwConst& tc, const HF& H, int tid) {
  ct_fft_forward<LOG2M>(z, tw, tc, tid);
  ct_filter_pairs<LOG2M>(z, tw, H, tid);
  ct_fft_inverse<LOG2M>(z, tw, tc, tid);
}

// Host side: fill the CtTwLayout<LOG2M> table from a function w(x, log2L) = W_L^x.
template <int LOG2M, class WF>
inline void ct_build_pass_table(float2* out, WF&& w) {
  using P = CtPlan<LOG2M>;
  using Lay = CtTwLayout<LOG2M>;
  for (int p = 0; p < P::n; ++p) {
    const int lr = P::lr(p), R = 1 << lr, log2L = P::log2L(p), L = 1 << log2L;
    for (int j = 0; j < Lay::J(p); ++j)
      for (int q = 0; q < R; ++q) out[Lay::off(p) + (j << lr) + q] = w((int)(((long long)j * q) & (L - 1)), log2L);
  }
}
template <class WF>
inline int ct_pass_table(int log2m, float2* out, WF&& w) {     // returns the table length; out may be null
#define PAYNE_PT_CASE(L) case L: if (out) ct_build_pass_table<L>(out, w); return CtTwLayout<L>::total;
  switch (log2m) {
    PAYNE_PT_CASE(6) PAYNE_PT_CASE(7) PAYNE_PT_CASE(8) PAYNE_PT_CASE(9) PAYNE_PT_CASE(10) PAYNE_PT_CASE(11)
    PAYNE_PT_CASE(12) PAYNE_PT_CASE(13) PAYNE_PT_CASE(14)
    default: return 0;
  }
#undef PAYNE_PT_CASE
}

}  // namespace payne
