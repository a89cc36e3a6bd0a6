// Fast fused tail for emulators trained on a log-uniform wavelength grid (the grid every
// Payne trainer produces: Payne/utils/readc3k.py:441-451).  Same semantics as tail.cuh (which
// stays as the general-grid path); what differs is HOW the four np.interp regrids are done:
//
// On a log-uniform grid  w_i = w_0 q^i  every regrid of Payne/utils/smoothing.py:649-668 maps
// index k of one uniform-in-ln(lambda) grid to position  p = k * num / den  of another, an exact
// rational.  The bracketing index is floor(p) and the np.interp weight is
//     t = (e^{delta a} - 1) / (e^{a} - 1) = delta (1 + (delta - 1) a/2 + O(a^2)),
// delta = frac(p), a = the (tiny, ~3e-6) log-spacing of the source grid.  So the per-dataset
// tables and the per-point fp64 searches of the general path collapse into incremental integer
// arithmetic: each thread walks k -> k + 256 with (j, rem) += (inc_j, inc_rem).  The host
// verifies at context creation that these analytic weights reproduce the exact np.interp tables
// to < 2e-7 before this kernel is selected.
#pragma once
#include "fft_ct.cuh"
#include "tail.cuh"
#include "tail_general.cuh"

namespace payne {

struct FastGrid {
  // stage 1 forward (native -> 2^k grid) and back: p = k * num / den
  int f_num, f_den, f_incj, f_incr;   // num = n-1,  den = N1-1, inc = divmod(2*256*num, den) (pairs)
  int b_num, b_den, b_incj, b_incr;   // num = N1-1, den = n-1
  float f_invden, b_invden;
  float c_native;                     // dlnw / 2   (source spacing = native grid)
  float c_grid1;                      // du1 / 2    (source spacing = stage-1 grid)
  double dlnw, inv_dlnw;
  const double* obs_q;                // [n_obs] (ln lambda_j - ln w_0) / dlnw
  const double* obs_otm1;             // [n_obs] (flux - 1)/eflux : r = depth/eflux - otm1
  void* points;                       // [slab] FastPoint, written by tail_setup_kernel
  int win_floats;                     // shared-memory window for the rotation-kernel table (floats; 4 per table interval)
  float* scratch;                     // [grid, N1/2] second half of split transforms (N1 = 65536)
  TwConst twc;
  // (behind twc: the constant-bank offsets of the fields above are what the single-CTA kernel was tuned with)
  int obs_sorted;                     // single-star context: observed wavelengths are non-decreasing (cluster tail:
                                      // pixel ranges per CTA; a context of several stars decides per star, jcut[0])
  int cluster;                        // the cluster tail (tail_cluster.cuh) is in use: tail_setup fills FastSetup::jcut
  // dynamic point scheduling of tail_fast_kernel: CTA b starts with point b and takes further points from this
  // counter (reset to work_start = the tail's grid size by tail_setup_kernel); null = static round robin
  int* work_counter;
  int work_start;
};

struct FastSetup {
  int s_incj, s_incr, s_den, s_num;   // stage 2: num = nM-1, den = N2-1, inc for pairs (2*256*num)
  float s_invden;
  // cluster tail: first observed pixel at or beyond sample (r+1) N2/4 (the star's pixels sorted; jcut[0] = -1: not
  // sorted, every CTA scans the star's pixels)
  int jcut[3];
  double q0, scale;                   // final: p = (obs_q - q0) * scale
  ObsSlice obs;                       // the point's star
};

// Per-point setup, computed by tail_setup_kernel (one thread per point) ahead of the tail so that
// no CTA of the tail idles behind a single thread's fp64 logarithms.  Copied into shared memory as int4 (load_record).
struct alignas(16) FastPoint {
  PointSetup S;
  FastSetup FS;
};

template <class T>
__device__ __forceinline__ void divmod_init(int tid, int num, int den, int& j, int& rem) {
  const long long v = (long long)tid * num;
  j = (int)(v / den);
  rem = (int)(v - (long long)j * den);
}

__device__ __forceinline__ float interp_w(float delta, float c) {   // delta (1 + (delta-1) c)
  return fmaf(delta * (delta - 1.f), c, delta);
}

template <bool CLEAN>
__device__ __forceinline__ float ld_depth(const float* row, int j) {
  float v = row[j];
  if (!CLEAN && v != v) v = 0.f;        // nan_to_num(nan=1.0) (smoothing.py:138) in depth space
  return v;
}

// Where the N real samples of the current transform live.
struct ZSmem {                       // all in shared memory (N <= 32768)
  float* zf;
  __device__ __forceinline__ float ld(int k) const { return zf[zidx(k)]; }
  __device__ __forceinline__ void st2(int k, float2 v) const { *reinterpret_cast<float2*>(zf + zidx(k)) = v; }
};
struct ZSplit {                      // first half in shared memory, second half in an L2-resident scratch line
  float* zf;
  float* g;
  int half;
  __device__ __forceinline__ float ld(int k) const { return k < half ? zf[zidx(k)] : __ldcg(g + (k - half)); }
  __device__ __forceinline__ void st2(int k, float2 v) const {
    if (k < half) *reinterpret_cast<float2*>(zf + zidx(k)) = v;
    else *reinterpret_cast<float2*>(g + (k - half)) = v;
  }
};

// Regrid a line-depth row (global/L2) onto N uniform ln-lambda points in shared memory:
// out[k] = np.interp at native position j0 + k*num/den (num <= den).  Each thread makes PAIRS of
// adjacent outputs (three row loads for two outputs, one 8-byte smem store).  The very last
// output sits exactly on row[jlast] (weight 0), so row[jlast+1], row[jlast+2] are read but never
// contribute: rows carry two finite pad floats (ensure_workspace zero-fills them once).
// Two pairs per trip: six loads in flight per thread.
template <bool CLEAN, class ZV>
__device__ __forceinline__ void regrid_in(const float* row, const ZV& zv, int tid, int N, int num, int den,
                                          int j0, float invden, float c, int inc2j, int inc2r) {
  const long long v = 2LL * tid * num;
  int j = (int)(v / den);
  int rem = (int)(v - (long long)j * den);
  const float* src = row + j0 + j;
#pragma unroll 1
  for (int k = 2 * tid; k < N; k += 4 * kNT) {
    const int remA = rem;
    const float a0 = ld_depth<CLEAN>(src, 0), a1 = ld_depth<CLEAN>(src, 1), a2 = ld_depth<CLEAN>(src, 2);
    rem += inc2r;
    int adv = inc2j;
    if (rem >= den) { rem -= den; ++adv; }
    src += adv;
    const int remB = rem;
    const bool second = (k + 2 * kNT < N);         // false only for transforms below 1024 samples
    float b0 = 0.f, b1 = 0.f, b2 = 0.f;
    if (second) { b0 = ld_depth<CLEAN>(src, 0); b1 = ld_depth<CLEAN>(src, 1); b2 = ld_depth<CLEAN>(src, 2); }
    rem += inc2r;
    adv = inc2j;
    if (rem >= den) { rem -= den; ++adv; }
    src += adv;
    {
      const int rem1 = remA + num;
      const bool same = rem1 < den;                // second output still between row[j] and row[j+1]
      const float lo = same ? a0 : a1, hi = same ? a1 : a2;
      float2 o;
      o.x = fmaf(interp_w((float)remA * invden, c), a1 - a0, a0);
      o.y = fmaf(interp_w((float)(same ? rem1 : rem1 - den) * invden, c), hi - lo, lo);
      zv.st2(k, o);
    }
    if (second) {
      const int rem1 = remB + num;
      const bool same = rem1 < den;
      const float lo = same ? b0 : b1, hi = same ? b1 : b2;
      float2 o;
      o.x = fmaf(interp_w((float)remB * invden, c), b1 - b0, b0);
      o.y = fmaf(interp_w((float)(same ? rem1 : rem1 - den) * invden, c), hi - lo, lo);
      zv.st2(k + 2 * kNT, o);
    }
  }
}

// ---- per-stage building blocks, templated on the sample view -------------------------------
template <class ZV>
__device__ __forceinline__ void stage_regrid(const PointSetup& S, const float* row, const ZV& zv, int tid, int N,
                                             int num, int den, int j0, float invden, float c, int incj, int incr) {
  if (S.clean) regrid_in<true>(row, zv, tid, N, num, den, j0, invden, c, incj, incr);
  else regrid_in<false>(row, zv, tid, N, num, den, j0, invden, c, incj, incr);
}

// stage-1 output back onto the emulator grid (+ edge patch of predictspec.py:240-241); only
// pixels [ilo, ihi] are produced -- stage 2 reads nothing outside its mask
template <class ZV>
__device__ __forceinline__ void regrid_back(float* row, const ZV& zv, const FastGrid& F, int tid, int n, int N1,
                                            int ilo, int ihi) {
  // interior pixels [1, n-2] only: no edge tests and no clamp of k + 1 in the loop (pixel n-1 is the only one
  // that sits on the last grid point); the two end pixels are the patch of predictspec.py:240-241
  const int lo = max(ilo, 1), hi = min(ihi, n - 2);
  const long long v0 = (long long)(lo + tid) * F.b_num;
  int k = (int)(v0 / F.b_den);
  int rem = (int)(v0 - (long long)k * F.b_den);
  const int den = F.b_den, incj = F.b_incj, incr = F.b_incr;
  const float invden = F.b_invden, cg = F.c_grid1;
#pragma unroll 4
  for (int i = lo + tid; i <= hi; i += kNT) {
    const float dl = (float)rem * invden;
    const float g0 = zv.ld(k), g1 = zv.ld(k + 1);
    row[i] = fmaf(interp_w(dl, cg), g1 - g0, g0);
    k += incj; rem += incr;
    if (rem >= den) { rem -= den; ++k; }
  }
  if (tid == 0 && ilo == 0) {
    const long long v1 = F.b_num;                         // pixel 1
    const int k1 = (int)(v1 / den);
    const float d1 = (float)(int)(v1 - (long long)k1 * den) * invden;
    const float a = zv.ld(k1), b = zv.ld(k1 + 1);
    row[0] = fmaf(interp_w(d1, cg), b - a, a);
  }
  if (tid == 32 && ihi == n - 1) {
    const long long v1 = (long long)(n - 2) * F.b_num;    // pixel n-2
    const int k1 = (int)(v1 / den);
    const float d1 = (float)(int)(v1 - (long long)k1 * den) * invden;
    const float a = zv.ld(k1), b = zv.ld(k1 + 1);
    row[n - 1] = fmaf(interp_w(d1, cg), b - a, a);
  }
}

// The point's observed pixels [obs_lo, obs_hi).  STARS = false: a single-star context (launch-time specialisation),
// whose bounds are the kernel parameters' -- the per-point record is not consulted and the loops compile as they
// did before observation sets existed (measured: reading the bounds from the record cost 0.6 % of the C2 tail).
template <bool STARS>
__device__ __forceinline__ int obs_lo(const ObsSlice& o) { return STARS ? o.off : 0; }
template <bool STARS>
__device__ __forceinline__ int obs_hi(const TailParams& P, const ObsSlice& o) { return STARS ? o.off + o.n : P.n_obs; }

// Observed pixels with a continuum polynomial and / or model output (m = (1 + d) chebval(x), r = m / sigma -
// flux / sigma; fitutils.py:11-20, likelihood.py:95-97): four pixels per trip like the plain path, loads grouped
// (positions -> samples -> depth; then the per-pixel constants -> Clenshaw on four abscissae at once ->
// residuals).  It lives in its own instantiation of the kernel (POLY = true): the plain path sits at its 80-register
// cap and any code beside it changes its allocation (measured: +0.5 % with this loop behind a call).
// moff: column of the point's first pixel in its model row (a target's member m: the pixels of members 0 .. m-1).
template <bool STARS, class ZV>
__device__ __forceinline__ double final_pass_poly(const TailParams& P, const FastGrid& F, const PointSetup& S,
                                                  const FastSetup& FS, const ZV& zv, int tid, int p, int N2, int moff = 0) {
  const double nan = CUDART_NAN;
  const double pmax = (double)(N2 - 1);
  const float hdu = S.hdu;
  const double q0 = FS.q0, scale = FS.scale;
  const int off = obs_lo<STARS>(FS.obs), jend = obs_hi<STARS>(P, FS.obs);   // the point's star: pixels [off, jend)
  double* mrow = P.model_out ? P.model_out + (long long)p * P.ld_flux + moff : nullptr;
  double acc = 0.0;
  constexpr int U = 4;
#pragma unroll 1
  for (int j0 = off + tid; j0 < jend; j0 += U * kNT) {
    float d[U];
    unsigned okm = 0;
    {
      double q[U];
#pragma unroll
      for (int u = 0; u < U; ++u) q[u] = (j0 + u * kNT < jend) ? __ldcg(F.obs_q + j0 + u * kNT) : -1.0;
      float g0[U], g1[U], dl[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const double pp = (q[u] - q0) * scale;
        const bool ok = (pp >= 0.0 && pp <= pmax);         // smoothing.py:289 left/right = nan
        const int k = ok ? min((int)pp, N2 - 2) : 0;
        okm |= (unsigned)ok << u;
        dl[u] = (float)(pp - (double)k);
        g0[u] = zv.ld(k); g1[u] = zv.ld(k + 1);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) d[u] = fmaf(interp_w(dl[u], hdu), g1[u] - g0[u], g0[u]);
    }
    double is[U], ot[U], x[U], cv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const bool in = j0 + u * kNT < jend;
      is[u] = in ? __ldcg(P.obs_inv_s + j0 + u * kNT) : 0.0;
      ot[u] = in ? __ldcg(P.obs_ot + j0 + u * kNT) : 0.0;
      x[u] = (in && P.n_poly) ? __ldcg(P.obs_x + j0 + u * kNT) : 0.0;
    }
    if (P.n_poly) chebval_dev4(x, S.poly, P.n_poly, cv);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      double m = ((okm >> u) & 1u) ? 1.0 + (double)d[u] : nan;
      if (P.n_poly) m *= cv[u];
      if (j0 + u * kNT < jend) {
        if (mrow) mrow[j0 + u * kNT - off] = m;
        const double r = fma(m, is[u], -ot[u]);
        acc = fma(r, r, acc);
      }
    }
  }
  return acc;
}

// The residual pass of continuum marginalisation (marg_point) with an instrumental stage: final_pass_poly's thread
// mapping, order and residual arithmetic, with m = a_j read from the CTA's scratch (by the thread that wrote it in
// final_pass_bin<1>) and the star's own nk coefficients.  A separate function on purpose: a template switch inside
// final_pass_poly changed the spills of the 65536-sample target kernel.
__device__ __forceinline__ double final_pass_marg(const TailParams& P, const PointSetup& S, const FastSetup& FS, int tid,
                                                  int p, int moff, int nk) {
  const int off = FS.obs.off, jend = FS.obs.off + FS.obs.n;
  const double* scr = P.aj_scratch + (long long)blockIdx.x * P.aj_ld;
  double* mrow = P.model_out ? P.model_out + (long long)p * P.ld_flux + moff : nullptr;
  double acc = 0.0;
  constexpr int U = 4;
#pragma unroll 1
  for (int j0 = off + tid; j0 < jend; j0 += U * kNT) {
    double is[U], ot[U], x[U], cv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const bool in = j0 + u * kNT < jend;
      is[u] = in ? __ldcg(P.obs_inv_s + j0 + u * kNT) : 0.0;
      ot[u] = in ? __ldcg(P.obs_ot + j0 + u * kNT) : 0.0;
      x[u] = in ? __ldcg(P.obs_x + j0 + u * kNT) : 0.0;
    }
    chebval_dev4(x, S.poly, nk, cv);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (j0 + u * kNT < jend) {
        const double m = scr[j0 + u * kNT - off] * cv[u];
        if (mrow) mrow[j0 + u * kNT - off] = m;
        const double r = fma(m, is[u], -ot[u]);
        acc = fma(r, r, acc);
      }
    }
  }
  return acc;
}

// Binaries (payne_ctx_set_binary): the point's pixels with final_pass_poly's thread mapping and order.  BM = 1 (component
// 1, and the first pass of continuum marginalisation): a_1 = 1 + d (NaN outside the grid) into the CTA's scratch and
// comp row 0 (when given).  BM = 2 (component 2): a_2, a_1 read back from the scratch (by the thread that wrote it),
// m = (a_1 + k a_2) / (1 + k) with the blackbody flux ratio k, the continuum, chi2; a_2 into comp row 1 and m into the
// model row.  At k = 0 and a finite a_2, m is a_1 and the chi2 has
// the bits of final_pass_poly.
constexpr double kC2 = 1.438776877e8;   // second radiation constant hc / k_B, AA K

__device__ __forceinline__ double flux_ratio(double lam, double t1, double t2, double rr2) {
  return rr2 * expm1(kC2 / (lam * t1)) / expm1(kC2 / (lam * t2));
}

template <int BM, class ZV>
__device__ __forceinline__ double final_pass_bin(const TailParams& P, const FastGrid& F, const PointSetup& S,
                                                 const FastSetup& FS, const ZV& zv, int tid, int p, int N2) {
  const double nan = CUDART_NAN;
  const double pmax = (double)(N2 - 1);
  const float hdu = S.hdu;
  const double q0 = FS.q0, scale = FS.scale;
  const int off = FS.obs.off, jend = FS.obs.off + FS.obs.n;
  double* scr = P.aj_scratch + (long long)blockIdx.x * P.aj_ld;
  double* crow = P.comp_out ? P.comp_out + ((long long)p * 2 + (BM - 1)) * P.ld_flux : nullptr;
  double* mrow = (BM == 2 && P.model_out) ? P.model_out + (long long)p * P.ld_flux : nullptr;
  double t1 = 0.0, t2 = 0.0, rr2 = 0.0;
  if constexpr (BM == 2) {
    t1 = __ldg(P.bin_par + 3LL * p); t2 = __ldg(P.bin_par + 3LL * p + 1);
    const double rr = __ldg(P.bin_par + 3LL * p + 2);
    rr2 = rr * rr;
  }
  double acc = 0.0;
  constexpr int U = 4;
#pragma unroll 1
  for (int j0 = off + tid; j0 < jend; j0 += U * kNT) {
    float d[U];
    unsigned okm = 0;
    {
      double q[U];
#pragma unroll
      for (int u = 0; u < U; ++u) q[u] = (j0 + u * kNT < jend) ? __ldcg(F.obs_q + j0 + u * kNT) : -1.0;
      float g0[U], g1[U], dl[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const double pp = (q[u] - q0) * scale;
        const bool ok = (pp >= 0.0 && pp <= pmax);         // smoothing.py:289 left/right = nan
        const int k = ok ? min((int)pp, N2 - 2) : 0;
        okm |= (unsigned)ok << u;
        dl[u] = (float)(pp - (double)k);
        g0[u] = zv.ld(k); g1[u] = zv.ld(k + 1);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) d[u] = fmaf(interp_w(dl[u], hdu), g1[u] - g0[u], g0[u]);
    }
    if constexpr (BM == 1) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int j = j0 + u * kNT;
        if (j < jend) {
          const double a = ((okm >> u) & 1u) ? 1.0 + (double)d[u] : nan;
          scr[j - off] = a;
          if (crow) crow[j - off] = a;
        }
      }
    } else {
      double is[U], ot[U], x[U], cv[U], a1[U], lam[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int j = j0 + u * kNT;
        const bool in = j < jend;
        is[u] = in ? __ldcg(P.obs_inv_s + j) : 0.0;
        ot[u] = in ? __ldcg(P.obs_ot + j) : 0.0;
        x[u] = (in && P.n_poly) ? __ldcg(P.obs_x + j) : 0.0;
        a1[u] = in ? scr[j - off] : 0.0;
        lam[u] = in ? __ldcg(P.obs_w + j) : 1.0;
      }
      if (P.n_poly) chebval_dev4(x, S.poly, P.n_poly, cv);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int j = j0 + u * kNT;
        const double a2 = ((okm >> u) & 1u) ? 1.0 + (double)d[u] : nan;
        const double k = flux_ratio(lam[u], t1, t2, rr2);
        double m = (a1[u] + k * a2) / (1.0 + k);
        if (P.n_poly) m *= cv[u];
        if (j < jend) {
          if (crow) crow[j - off] = a2;
          if (mrow) mrow[j - off] = m;
          const double r = fma(m, is[u], -ot[u]);
          acc = fma(r, r, acc);
        }
      }
    }
  }
  return acc;
}

// The same without an instrumental stage (plain np.interp, predictspec.py:288-289), with the thread mapping and order of
// point_chi2's plain branch.
template <int BM>
__device__ __forceinline__ double plain_pass_bin(const TailParams& P, const PointSetup& S, const FastSetup& FS,
                                                 const float* row, int tid, int p) {
  const double nan = CUDART_NAN;
  const int n = P.n;
  const double wlo = __ldg(P.w) * S.D, whi = __ldg(P.w + n - 1) * S.D;
  const int off = FS.obs.off, jend = FS.obs.off + FS.obs.n;
  double* scr = P.aj_scratch + (long long)blockIdx.x * P.aj_ld;
  double* crow = P.comp_out ? P.comp_out + ((long long)p * 2 + (BM - 1)) * P.ld_flux : nullptr;
  double* mrow = (BM == 2 && P.model_out) ? P.model_out + (long long)p * P.ld_flux : nullptr;
  double t1 = 0.0, t2 = 0.0, rr2 = 0.0;
  if constexpr (BM == 2) {
    t1 = __ldg(P.bin_par + 3LL * p); t2 = __ldg(P.bin_par + 3LL * p + 1);
    const double rr = __ldg(P.bin_par + 3LL * p + 2);
    rr2 = rr * rr;
  }
  double acc = 0.0;
  for (int j = off + tid; j < jend; j += kNT) {
    const double x = __ldg(P.obs_w + j);
    double a;
    if (!(x >= wlo && x <= whi)) a = nan;
    else {
      const int g = (int)((__ldg(P.obs_lnw + j) - S.lnD - P.lnw0) * P.inv_dlnw);
      const int jj = locate(P.w, S.D, x, g, 0, n - 2);
      const double wa = __ldg(P.w + jj) * S.D, wb = __ldg(P.w + jj + 1) * S.D;
      const double va = (double)depth_of(row[jj], true, false);
      const double vb = (double)depth_of(row[jj + 1], true, false);
      a = 1.0 + np_interp_pair(x, wa, wb, va, vb);
    }
    if constexpr (BM == 1) {
      scr[j - off] = a;
      if (crow) crow[j - off] = a;
    } else {
      const double k = flux_ratio(x, t1, t2, rr2);
      double m = (scr[j - off] + k * a) / (1.0 + k);
      if (P.n_poly) m *= chebval_dev(__ldg(P.obs_x + j), S.poly, P.n_poly);
      if (crow) crow[j - off] = a;
      if (mrow) mrow[j - off] = m;
      const double r = m * __ldg(P.obs_inv_s + j) - __ldg(P.obs_ot + j);
      acc += r * r;
    }
  }
  return acc;
}

// No instrumental profile: plain np.interp (predictspec.py:288-289), continuum, residuals.  MARG: the residual pass of
// continuum marginalisation (marg_point), m = a_j from the CTA's scratch and nk coefficients, with this loop's own
// arithmetic, thread mapping and order.
template <bool STARS, bool MARG = false>
__device__ __forceinline__ double plain_pass(const TailParams& P, const PointSetup& S, const FastSetup& FS,
                                             const float* row, int tid, int p, int moff, int nk = 0) {
  const double nan = CUDART_NAN;
  const bool is_depth = true;   // this kernel is only launched on line-depth rows (f - 1)
  const int npoly = MARG ? nk : P.n_poly;
  const double* scr = MARG ? P.aj_scratch + (long long)blockIdx.x * P.aj_ld : nullptr;
  double acc = 0.0;
  const int n = P.n;
  const double wlo = __ldg(P.w) * S.D, whi = __ldg(P.w + n - 1) * S.D;
  const int off = obs_lo<STARS>(FS.obs), jend = obs_hi<STARS>(P, FS.obs);
  for (int j = off + tid; j < jend; j += kNT) {
    const double x = __ldg(P.obs_w + j);
    double m;
    if constexpr (MARG) m = scr[j - off];
    else if (!(x >= wlo && x <= whi)) m = nan;
    else {
      const int g = (int)((__ldg(P.obs_lnw + j) - S.lnD - P.lnw0) * P.inv_dlnw);
      const int jj = locate(P.w, S.D, x, g, 0, n - 2);
      const double wa = __ldg(P.w + jj) * S.D, wb = __ldg(P.w + jj + 1) * S.D;
      const double a = (double)depth_of(row[jj], is_depth, false);
      const double b = (double)depth_of(row[jj + 1], is_depth, false);
      m = 1.0 + np_interp_pair(x, wa, wb, a, b);
    }
    if (npoly) m *= chebval_dev(__ldg(P.obs_x + j), S.poly, npoly);
    if (P.model_out) P.model_out[(long long)p * P.ld_flux + moff + (j - off)] = m;
    const double r = m * __ldg(P.obs_inv_s + j) - __ldg(P.obs_ot + j);
    acc += r * r;
  }
  return acc;
}

// observed pixels, continuum, residuals; returns this thread's partial chi2
template <bool POLY, bool STARS, class ZV>
__device__ __forceinline__ double final_pass(const TailParams& P, const FastGrid& F, const PointSetup& S,
                                             const FastSetup& FS, const ZV& zv, int tid, int p, int N2, int moff = 0) {
  const double nan = CUDART_NAN;
  const double pmax = (double)(N2 - 1);
  const float hdu = S.hdu;
  const double q0 = FS.q0, scale = FS.scale;
  double acc = 0.0;
  if (!POLY) {
    // four pixels per trip: the twelve per-pixel constants are requested together, then the eight
    // shared-memory samples, then the arithmetic (the phase is latency-bound at 24 warps per SM)
    constexpr int U = 4;
    const int jend = obs_hi<STARS>(P, FS.obs);                // the point's star: pixels [obs_lo, jend)
#pragma unroll 1
    for (int j0 = obs_lo<STARS>(FS.obs) + tid; j0 < jend; j0 += U * kNT) {
      double q[U], is[U], ot[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int j = j0 + u * kNT;
        const bool in = j < jend;
        q[u] = in ? __ldcg(F.obs_q + j) : -1.0;          // -1 -> outside the grid -> contributes through `in` only
        is[u] = in ? __ldcg(P.obs_inv_s + j) : 0.0;
        ot[u] = in ? __ldcg(F.obs_otm1 + j) : 0.0;
      }
      float g0[U], g1[U], dl[U];
      bool ok[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const double pp = (q[u] - q0) * scale;
        ok[u] = (pp >= 0.0 && pp <= pmax);               // smoothing.py:289 left/right = nan
        const int k = ok[u] ? min((int)pp, N2 - 2) : 0;
        dl[u] = (float)(pp - (double)k);
        g0[u] = zv.ld(k); g1[u] = zv.ld(k + 1);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float d = fmaf(interp_w(dl[u], hdu), g1[u] - g0[u], g0[u]);
        double r = fma((double)d, is[u], -ot[u]);
        if (!ok[u]) r = nan;
        if (j0 + u * kNT < jend) acc = fma(r, r, acc);
      }
    }
  } else {
    acc = final_pass_poly<STARS>(P, F, S, FS, zv, tid, p, N2, moff);
  }
  return acc;
}

// Drop the L2 lines lying wholly inside row[0, n) without write-back.  Not inlined on purpose: the tail kernel
// sits at its 80-register cap, and these few instructions inlined at the end of the point loop changed the
// allocation of the whole kernel (+1.5 % time).
static __device__ __noinline__ void discard_lines(const float* row, int n, int tid) {
  const unsigned long long a0 = (unsigned long long)row, a1 = a0 + 4ull * (unsigned long long)n;
  const unsigned long long last = a1 & ~127ull;
  for (unsigned long long a = ((a0 + 127ull) & ~127ull) + 128ull * (unsigned)tid; a < last; a += 128ull * kNT)
    asm volatile("discard.global.L2 [%0], 128;" ::"l"(a));
}

// Stage 2 and the final pass of one point against its star (S, FS) on the row that stage 1 left; returns this
// thread's partial chi2.  z / zs / zp / gline: the kernel's transform buffer and its views.
// BM: 0 a point of one star; 1 / 2 component 1 / 2 of a binary (final_pass_bin, plain_pass_bin).
template <int LOG2N1, bool POLY, bool STARS, int BM = 0>
__device__ __forceinline__ double point_chi2(const TailParams& P, const FastGrid& F, const PointSetup& S,
                                             const FastSetup& FS, float2* z, const ZSmem& zs, const ZSplit& zp,
                                             float* gline, const TwTab& tw, const float* row, int tid, int p, int moff) {
  constexpr bool kSplit = LOG2N1 >= 16;
  constexpr int LOG2MH = kSplit ? LOG2N1 - 2 : 8;
  const double nan = CUDART_NAN;
  double acc = 0.0;
  if (S.use_inst) {
    // ---------------- stage 2: mask, regrid, Gaussian broadening
    const int log2N2 = S.log2N2, N2 = 1 << log2N2;
    const int i0 = S.i0;
    GaussH H{S.taper_a, 2.0f / (float)N2};
    bool split2 = false;
    if constexpr (kSplit) split2 = (log2N2 == LOG2N1);
    if (split2) {
      if constexpr (kSplit) {
        stage_regrid(S, row, zp, tid, N2, FS.s_num, FS.s_den, i0, FS.s_invden, F.c_native, FS.s_incj, FS.s_incr);
        __syncthreads();
        ct_convolve_split<LOG2MH>(z, reinterpret_cast<float2*>(gline), tw, F.twc, H, tid);
        if constexpr (BM == 0) acc = final_pass<POLY, STARS>(P, F, S, FS, zp, tid, p, N2, moff);
        else acc = final_pass_bin<BM>(P, F, S, FS, zp, tid, p, N2);
      }
    } else {
      constexpr int LA = LOG2N1 > 15 ? 15 : LOG2N1;       // largest all-in-smem transform
      if (!(log2N2 == LA || (LA >= 10 && log2N2 == LA - 1))) {
        // small masks: separate regrid, runtime-planned transform
        stage_regrid(S, row, zs, tid, N2, FS.s_num, FS.s_den, i0, FS.s_invden, F.c_native, FS.s_incj, FS.s_incr);
        __syncthreads();
        const Twiddles twr{tw.tab, tw.log2n};
        FftPlan plan; plan.make(log2N2 - 1);
        fft_forward(z, log2N2 - 1, plan, twr, tid, kNT);
        filter_pairs(z, log2N2 - 1, plan, twr, H, tid, kNT);
        fft_inverse(z, log2N2 - 1, plan, twr, tid, kNT);
      } else if (log2N2 == LA) {
        ct_convolve_regrid<LA - 1>(z, tw, F.twc, H, tid, row + i0, FS.s_num, FS.s_den, FS.s_invden, F.c_native, S.clean != 0);
      } else {
        ct_convolve_regrid<(LA >= 10 ? LA - 2 : 8)>(z, tw, F.twc, H, tid, row + i0, FS.s_num, FS.s_den,
                                                     FS.s_invden, F.c_native, S.clean != 0);
      }
      if constexpr (BM == 0) acc = final_pass<POLY, STARS>(P, F, S, FS, zs, tid, p, N2, moff);
      else acc = final_pass_bin<BM>(P, F, S, FS, zs, tid, p, N2);
    }
  } else if constexpr (BM != 0) {
    acc = plain_pass_bin<BM>(P, S, FS, row, tid, p);
  } else {
    acc = plain_pass<STARS>(P, S, FS, row, tid, p, moff);
  }
  return acc;
}

// ---- continuum marginalisation (payne_ctx_set_cont_marg) ------------------------------------------------------------
// Column pair (a, b), a >= b, of entry e of the lower triangle of [B | y]^T [B | y] without y.y (K + 1 columns: the
// star's K Chebyshev columns b_jk = a_j T_k(x_j) / s_j, then y_j = o_j / s_j): G below column K, h = row K.
__device__ __forceinline__ void marg_entry(int e, int& a, int& b) {
  a = 0;
  while (e > a) { e -= a + 1; ++a; }
  b = e;
}

// NaN coefficients and Cholesky factor of star k's K coefficients at columns cofs / lofs of row p
__device__ __forceinline__ void marg_nan_out(const TailParams& P, int p, int K, int cofs, int lofs, int tid) {
  const double nan = CUDART_NAN;
  for (int i = tid; P.coef_out && i < K; i += kNT) P.coef_out[(long long)p * P.ld_coef + cofs + i] = nan;
  for (int i = tid; P.chol_out && i < K * (K + 1) / 2; i += kNT) P.chol_out[(long long)p * P.ld_chol + lofs + i] = nan;
}

// One point against star k with its continuum integrated out.  Returns this thread's partial Q (the chi2 at c-hat, with
// final_pass_poly's or plain_pass's thread mapping and order, so the warp and CTA reduction of the caller gives Q the bits
// of -2 lnL of a context that samples the coefficients); thread 0 gets M = -sum ln L_kk + C_k in `M`.
//  1. stage 2 and the final pass of a binary's component 1 (point_chi2 BM = 1): a_j into the CTA's scratch;
//  2. G and h in fp64 over chunks of pixels staged in the (dead) transform buffer: thread (e, r) sums entry e over
//     pixels r, r + R, ... of every chunk in four accumulators, then thread e adds its R partials in order -- a fixed
//     pixel-to-thread mapping and order that depends on K and the transform size only;
//  3. warp 0: Cholesky G = L L^T, L z = h, L^T c = z; c-hat into S.poly (NaN with a pivot at or below 1e-10 of its diagonal entry: status bit 3
//     when G is finite);
//  4. the residual pass at c-hat on the scratch.
template <int LOG2N1>
__device__ __forceinline__ double marg_point(const TailParams& P, const FastGrid& F, PointSetup& S, const FastSetup& FS,
                                             float2* z, const ZSmem& zs, const ZSplit& zp, float* gline, const TwTab& tw,
                                             const float* row, int tid, int p, int moff, int k, int cofs, int lofs,
                                             double& M) {
  constexpr int kBufD = (LOG2N1 >= 16 ? (1 << LOG2N1) / 2 : (1 << LOG2N1)) / 2;   // doubles of the transform buffer
  constexpr int kG = PAYNE_MAX_POLY + 1;                                           // row stride of G / L
  const double nan = CUDART_NAN;
  point_chi2<LOG2N1, true, true, 1>(P, F, S, FS, z, zs, zp, gline, tw, row, tid, p, 0);
  __syncthreads();                                        // a_j in the scratch; the transform buffer is free
  const int K = __ldg(P.marg_k + k);
  const int off = FS.obs.off, n = FS.obs.n;
  const double* scr = P.aj_scratch + (long long)blockIdx.x * P.aj_ld;
  double* sm = reinterpret_cast<double*>(z);
  const int nc = K + 1, nent = nc * (nc + 1) / 2 - 1;
  const int R = kNT / nent;
  const int C = (kBufD - kNT) / nc;                       // pixels per chunk; the last kNT doubles take the partials
  const bool act = tid < nent * R;
  int ea = 0, eb = 0;
  if (act) marg_entry(tid / R, ea, eb);
  const int r = act ? tid % R : 0;
  double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
  for (int c0 = 0; c0 < n; c0 += C) {
    const int cn = min(C, n - c0);
    for (int i = tid; i < cn; i += kNT) {
      const int j = off + c0 + i;
      const double as = scr[c0 + i] * __ldg(P.obs_inv_s + j);
      const double x = __ldg(P.obs_x + j);
      double t0 = 1.0, t1 = x;
      sm[i] = as;
      for (int q = 1; q < K; ++q) {
        sm[q * C + i] = as * t1;
        const double t2 = 2.0 * x * t1 - t0;
        t0 = t1; t1 = t2;
      }
      sm[K * C + i] = __ldg(P.obs_ot + j);
    }
    __syncthreads();
    if (act) {
      const double* ba = sm + ea * C;
      const double* bb = sm + eb * C;
      int i = r;
      for (; i + 3 * R < cn; i += 4 * R) {
        s0 = fma(ba[i], bb[i], s0);
        s1 = fma(ba[i + R], bb[i + R], s1);
        s2 = fma(ba[i + 2 * R], bb[i + 2 * R], s2);
        s3 = fma(ba[i + 3 * R], bb[i + 3 * R], s3);
      }
      for (; i < cn; i += R) s0 = fma(ba[i], bb[i], s0);
    }
    __syncthreads();
  }
  double* part = sm + (kBufD - kNT);
  if (act) part[tid] = ((s0 + s1) + s2) + s3;
  __syncthreads();
  double g = 0.0;
  if (tid < nent) {
    for (int q = 0; q < R; ++q) g += part[tid * R + q];
    marg_entry(tid, ea, eb);
  }
  __syncthreads();                                        // G overlaps the partials of the smallest buffers
  double* G = sm;                                         // G[a * kG + b], a >= b; h_b = G[K * kG + b]
  if (tid < nent) G[ea * kG + eb] = g;
  __syncthreads();
  if (tid < 32) {
    const unsigned full = 0xffffffffu;
    const int lane = tid;
    bool fin = true;
    for (int e = lane; e < nent; e += 32) {
      int a, b;
      marg_entry(e, a, b);
      fin = fin && isfinite(G[a * kG + b]);
    }
    fin = __all_sync(full, fin);
    bool ok = true;
    double* L = G;                                        // in place, column by column
    for (int jc = 0; jc < K; ++jc) {
      double v = 0.0, g0 = 0.0;
      if (lane >= jc && lane < K) {
        v = g0 = G[lane * kG + jc];
        for (int q = 0; q < jc; ++q) v = fma(-L[lane * kG + q], L[jc * kG + q], v);
      }
      // a rank-deficient G leaves pivots of rounding size and either sign: fail at or below 1e-10 of the diagonal entry
      const double d = __shfl_sync(full, v, jc), gd = __shfl_sync(full, g0, jc);
      ok = ok && d > 1e-10 * gd;
      const double ljj = sqrt(d);
      if (lane > jc && lane < K) L[lane * kG + jc] = v / ljj;
      if (lane == jc) L[jc * kG + jc] = ljj;
      __syncwarp();
    }
    double v = lane < K ? G[K * kG + lane] : 0.0;         // L z = h
    for (int i = 0; i < K; ++i) {
      const double zi = __shfl_sync(full, v, i) / L[i * kG + i];
      if (lane == i) v = zi;
      else if (lane > i && lane < K) v = fma(-L[lane * kG + i], zi, v);
    }
    for (int i = K - 1; i >= 0; --i) {                    // L^T c = z
      const double ci = __shfl_sync(full, v, i) / L[i * kG + i];
      if (lane == i) v = ci;
      else if (lane < i) v = fma(-L[i * kG + lane], ci, v);
    }
    if (!ok) v = nan;
    if (lane < K) {
      S.poly[lane] = v;
      if (P.coef_out) P.coef_out[(long long)p * P.ld_coef + cofs + lane] = v;
    }
    if (P.chol_out)
      for (int e = lane; e < K * (K + 1) / 2; e += 32) {
        int a, b;
        marg_entry(e, a, b);
        P.chol_out[(long long)p * P.ld_chol + lofs + e] = ok ? L[a * kG + b] : nan;
      }
    if (lane == 0) {
      double lsum = 0.0;
      for (int i = 0; i < K; ++i) lsum += log(L[i * kG + i]);
      M = ok ? __ldg(P.marg_c + k) - lsum : nan;
      if (!ok && fin) atomicOr(P.status, 8);
    }
  }
  __syncthreads();                                        // c-hat in S.poly
  if (S.use_inst) return final_pass_marg(P, S, FS, tid, p, moff, K);
  return plain_pass<true, true>(P, S, FS, row, tid, p, moff, K);
}

// The point body a tail_fast_kernel runs per point, its form (tail_fast_tu.inl maps the host's FastForm to it):
//  OneStar      a single-star context, whose pixel bounds are the kernel parameters' (obs_lo / obs_hi);
//  Stars        a context of several stars: the point's star;
//  Target       every point names a target (TailParams::target): stage 1 runs once on the row, then stage 2 and the final
//               pass once per member against that member's record, and lnL is the members' chi2 summed in member order;
//  Binary       every point is a binary (TailParams::binary): component 1's record and row, stage 1, stage 2 and a final
//               pass that keeps a_1; then component 2's, whose final pass combines the two (final_pass_bin);
//  MargStars /  continuum marginalisation (TailParams::marg_k) of a point or of every member of a target, through
//  MargTargets  marg_point: lnL = -0.5 (Q + chi2_sed) + M (members: Q and M each summed in member order).
// Binary and Marg* have the polynomial / model-output final pass only (POLY).
enum class FastBody { OneStar, Stars, Target, Binary, MargStars, MargTargets };

__host__ __device__ constexpr bool body_target(FastBody b) { return b == FastBody::Target || b == FastBody::MargTargets; }
__host__ __device__ constexpr bool body_marg(FastBody b) { return b == FastBody::MargStars || b == FastBody::MargTargets; }

// What a point body needs of its kernel: the transform buffer and its views, the rotation-table window, the reduction
// slots
struct FastCta {
  float2* z;
  ZSmem zs;
  ZSplit zp;
  float* gline;
  TwTab tw;
  float* win;
  int win_have;                                           // table intervals already in the window
  double* red;
  int tid;
};

// Stage 1 (rotational broadening on the full emulator grid): writes back the row's pixels [blo, bhi] (those stage 2
// reads) and ends with a barrier.
template <int LOG2N1>
__device__ __forceinline__ void rot_stage(const TailParams& P, const FastGrid& F, const PointSetup& S, FastCta& c,
                                          float* row, int blo, int bhi) {
  constexpr int N1 = 1 << LOG2N1;
  constexpr bool kSplit = LOG2N1 >= 16;
  constexpr int LOG2MH = kSplit ? LOG2N1 - 2 : 8;          // complex points per half (split only)
  const int n = P.n, tid = c.tid;
  // (the barrier after the regrid below publishes the window)
  const RotHT<2> H = rot_window(P, S, N1, c.win, F.win_floats, c.win_have, tid);
  if constexpr (!kSplit) {
    // regrid fused into the first FFT pass (measured against the separate regrid: tail -5 %)
    ct_convolve_regrid<LOG2N1 - 1>(c.z, c.tw, F.twc, H, tid, row, F.f_num, F.f_den, F.f_invden, F.c_native, S.clean != 0);
    regrid_back(row, c.zs, F, tid, n, N1, blo, bhi);
  } else {
    stage_regrid(S, row, c.zp, tid, N1, F.f_num, F.f_den, 0, F.f_invden, F.c_native, F.f_incj, F.f_incr);
    __syncthreads();
    ct_convolve_split<LOG2MH>(c.z, reinterpret_cast<float2*>(c.gline), c.tw, F.twc, H, tid);
    regrid_back(row, c.zp, F, tid, n, N1, blo, bhi);
  }
  __syncthreads();
}

// A point against its star (OneStar, Stars, MargStars; not a bad one): stage 1, then point_chi2 or marg_point, and lnL.
template <int LOG2N1, bool POLY, FastBody BODY>
__device__ __forceinline__ void star_point(const TailParams& P, const FastGrid& F, PointSetup& S, const FastSetup& FS,
                                           FastCta& c, float* row, int p) {
  constexpr bool STARS = BODY != FastBody::OneStar;
  const int tid = c.tid;
  if (POLY && !body_marg(BODY) && S.do_rot) {
    rot_stage<LOG2N1>(P, F, S, c, row, S.use_inst ? max(S.i0 - 1, 0) : 0, S.use_inst ? min(S.i1 + 1, P.n - 1) : P.n - 1);
  } else if (S.do_rot) {
    // The plain kernels (the sampler's hot path) and MargStars keep their own copy of stage 1 and of its window
    // staging: calling rot_stage cost the 4096- and 8192-sample plain kernels 92 to 124 bytes of spills and the
    // MargStars kernels of those sizes 72 / 84 and 92 / 104 bytes of spill stores / loads, and rot_window alone
    // changed the code of every plain kernel.
    constexpr int N1 = 1 << LOG2N1;
    constexpr bool kSplit = LOG2N1 >= 16;
    constexpr int LOG2MH = kSplit ? LOG2N1 - 2 : 8;
    const int n = P.n;
    // the table entries this point can touch: [0, vsini_scale * N1/2 + 3]; staged in shared memory when they fit (the
    // barrier after the regrid below publishes them)
    const double xt_max = S.vsini_scale * (double)(N1 >> 1);
    float4* win4 = reinterpret_cast<float4*>(c.win);
    const int nwin = (int)fmin(fmin(xt_max + 2.0, (double)(F.win_floats >> 2)), (double)P.ntab);
    for (int i = c.win_have + tid; i < nwin; i += kNT) win4[i] = __ldg(P.sbtab + i);
    c.win_have = max(c.win_have, nwin);
    const RotHT<2> H{P.sbtab, win4, nwin, S.vsini_scale, P.sb_h, 1.0f / (float)(N1 >> 1), P.ntab, RotHT<2>::fix40(S.vsini_scale)};
    // pixels stage 2 will read: its mask [i0, i1] (one more on each side keeps the edge patch exact)
    const int blo = S.use_inst ? max(S.i0 - 1, 0) : 0;
    const int bhi = S.use_inst ? min(S.i1 + 1, n - 1) : n - 1;
    if constexpr (!kSplit) {
      ct_convolve_regrid<LOG2N1 - 1>(c.z, c.tw, F.twc, H, tid, row, F.f_num, F.f_den, F.f_invden, F.c_native, S.clean != 0);
      regrid_back(row, c.zs, F, tid, n, N1, blo, bhi);
    } else {
      stage_regrid(S, row, c.zp, tid, N1, F.f_num, F.f_den, 0, F.f_invden, F.c_native, F.f_incj, F.f_incr);
      __syncthreads();
      ct_convolve_split<LOG2MH>(c.z, reinterpret_cast<float2*>(c.gline), c.tw, F.twc, H, tid);
      regrid_back(row, c.zp, F, tid, n, N1, blo, bhi);
    }
    __syncthreads();
  }
  if constexpr (body_marg(BODY)) {
    double M = 0.0;
    double c2 = cta_sum(marg_point<LOG2N1>(P, F, S, FS, c.z, c.zs, c.zp, c.gline, c.tw, row, tid, p, 0,
                                           star_of(P.star, P.n_stars, p), 0, 0, M), c.red, tid);
    if (tid == 0) {
      if (P.chi2_out) P.chi2_out[(long long)p * P.ld_chi2] = c2;
      if (P.chi2_sed) c2 += P.chi2_sed[p];
      if (P.lnl) store_lnl(P, p, -0.5 * c2 + M);
    }
  } else {
    // (the CTA reduction of cta_sum written out, the warps' sum taken only where lnL is stored: cta_sum here changed
    // the code of the plain kernels and the stack and spills of the 2048-sample polynomial one)
    double acc = point_chi2<LOG2N1, POLY, STARS>(P, F, S, FS, c.z, c.zs, c.zp, c.gline, c.tw, row, tid, p, 0);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((tid & 31) == 0) c.red[tid >> 5] = acc;
    __syncthreads();
    if (tid == 0 && P.lnl) {
      double c2 = 0.0;
#pragma unroll
      for (int wdx = 0; wdx < kNT / 32; ++wdx) c2 += c.red[wdx];
      if (P.chi2_sed) c2 += P.chi2_sed[p];
      store_lnl(P, p, -0.5 * c2);
    }
  }
}

// A point naming a target (Target, MargTargets) of K > 0 members, whose records rec[0, K) the kernel loaded from rec[0]
// on: stage 1 once on the row's pixels tu = the union of the members' windows, then every member against its own
// record; the row is read-only from there on.
template <int LOG2N1, bool POLY, FastBody BODY>
__device__ __forceinline__ void target_point(const TailParams& P, const FastGrid& F, FastPoint& SP, FastCta& c,
                                             float* row, int p, const FastPoint* rec, int K, int2 tu) {
  PointSetup& S = SP.S;
  const FastSetup& FS = SP.FS;
  const int tid = c.tid;
  // the labels and Vrot of every member are the first member's (payne_ctx_set_targets), so its do_rot, vsini_scale
  // and clean hold for the row; skipped when every member is bad
  if (S.do_rot && tu.x <= tu.y) rot_stage<LOG2N1>(P, F, S, c, row, tu.x, tu.y);
  // Member m's model pixels follow those of members 0 .. m-1 (the members' observations lie back to back in the set's
  // arrays).
  const int off0 = FS.obs.off;
  double tot = 0.0;                                       // thread 0: chi2 of members 0 .. m, summed in that order
  double mtot = 0.0;                                      // Marg, thread 0: M of members 0 .. m, likewise
  int cofs = 0, lofs = 0;                                 // Marg: the member's first coefficient / Cholesky column
  for (int m = 0; m < K; ++m) {
    if (m > 0) {
      __syncthreads();                                    // member m-1's record, transform buffer and red[] are free
      load_record(SP, rec + m, tid);
      __syncthreads();
    }
    const bool bad = S.bad != 0;
    const int moff = FS.obs.off - off0;
    double acc = 0.0;
    double M = 0.0;                                       // Marg: the member's M (thread 0)
    int km = 0;                                           // Marg: the member's coefficients
    if constexpr (body_marg(BODY)) {
      const int k = __ldg(P.tfirst + __ldg(P.target + p)) + m;
      km = __ldg(P.marg_k + k);
      if (!bad) acc = marg_point<LOG2N1>(P, F, S, FS, c.z, c.zs, c.zp, c.gline, c.tw, row, tid, p, moff, k, cofs, lofs, M);
      else {
        model_nan(P, p, moff, FS.obs.n, tid);
        marg_nan_out(P, p, km, cofs, lofs, tid);
      }
    } else {
      if (!bad) acc = point_chi2<LOG2N1, POLY, true>(P, F, S, FS, c.z, c.zs, c.zp, c.gline, c.tw, row, tid, p, moff);
      else model_nan(P, p, moff, FS.obs.n, tid);
    }
    double c2 = cta_sum(acc, c.red, tid);
    if (tid == 0) {
      if (bad) c2 = CUDART_NAN;
      if (P.chi2_out) P.chi2_out[(long long)p * P.ld_chi2 + m] = c2;
      tot = m == 0 ? c2 : tot + c2;
      if constexpr (body_marg(BODY)) mtot = m == 0 ? M : mtot + M;
    }
    if constexpr (body_marg(BODY)) { cofs += km; lofs += km * (km + 1) / 2; }
  }
  if (tid == 0 && P.lnl) {
    if (P.chi2_sed) tot += P.chi2_sed[p];
    if constexpr (body_marg(BODY)) store_lnl(P, p, -0.5 * tot + mtot);
    else store_lnl(P, p, -0.5 * tot);
  }
}

// A binary: component c's record c * B + p (component 0's loaded by the kernel) on its row c * B + p, stage 1, stage 2
// and final_pass_bin<c + 1>.  A bad component makes a_c, the model and lnL NaN.
template <int LOG2N1>
__device__ __forceinline__ void binary_point(const TailParams& P, const FastGrid& F, FastPoint& SP, FastCta& c,
                                             float* row, int p, const FastPoint* points) {
  PointSetup& S = SP.S;
  const FastSetup& FS = SP.FS;
  const int tid = c.tid;
  double acc = 0.0;
  bool bad = false;
  for (int cc = 0; cc < 2; ++cc) {
    float* rowc = row + (long long)cc * P.B * P.ldf;
    if (cc == 1) {
      __syncthreads();                                    // component 1's record and transform buffer are free
      load_record(SP, points + P.B + p, tid);
      __syncthreads();
    }
    if (S.bad) {
      bad = true;
      // (a_c, the component row and the model row in one loop: model_nan in its place changed the spills of the
      // 16384- and 65536-sample binary kernels)
      double* scr = P.aj_scratch + (long long)blockIdx.x * P.aj_ld;
      for (int j = tid; j < FS.obs.n; j += kNT) {
        if (cc == 0) scr[j] = CUDART_NAN;
        if (P.comp_out) P.comp_out[((long long)p * 2 + cc) * P.ld_flux + j] = CUDART_NAN;
        if (cc == 1 && P.model_out) P.model_out[(long long)p * P.ld_flux + j] = CUDART_NAN;
      }
      continue;
    }
    if (S.do_rot) {
      const int blo = S.use_inst ? max(S.i0 - 1, 0) : 0;
      const int bhi = S.use_inst ? min(S.i1 + 1, P.n - 1) : P.n - 1;
      rot_stage<LOG2N1>(P, F, S, c, rowc, blo, bhi);
    }
    if (cc == 0) point_chi2<LOG2N1, true, true, 1>(P, F, S, FS, c.z, c.zs, c.zp, c.gline, c.tw, rowc, tid, p, 0);
    else acc = point_chi2<LOG2N1, true, true, 2>(P, F, S, FS, c.z, c.zs, c.zp, c.gline, c.tw, rowc, tid, p, 0);
  }
  const double c2 = cta_sum(acc, c.red, tid);
  if (tid == 0 && P.lnl) store_lnl(P, p, bad ? CUDART_NAN : -0.5 * c2);
}

// LOG2N1 <= 15: the whole transform sits in shared memory (3 CTAs/SM up to 2^14).
// LOG2N1 == 16: split transform, half in shared memory (128 KB), half in the scratch line.
// POLY: continuum polynomial and / or model output in the final pass (the host picks the instantiation).
// BODY: what a point is (FastBody).
// (3 CTAs/SM, 80 registers with a few spills, measured at C2 0.76 ms against 0.84 ms with 2 CTAs/SM and no spills)
template <int LOG2N1, bool POLY, FastBody BODY>
__global__ void __launch_bounds__(kNT, LOG2N1 <= 14 ? 3 : 1)
tail_fast_kernel(const __grid_constant__ TailParams P, const __grid_constant__ FastGrid F) {
  static_assert(POLY || !(BODY == FastBody::Binary || body_marg(BODY)), "Binary and Marg* have the POLY final pass only");
  constexpr bool STARS = BODY != FastBody::OneStar;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* zf = reinterpret_cast<float*>(smem_raw);
  __shared__ FastPoint SP;
  __shared__ double red[kNT / 32];
  const int tid = threadIdx.x;
  constexpr int N1 = 1 << LOG2N1;
  constexpr bool kSplit = LOG2N1 >= 16;
  float* gline = kSplit ? F.scratch + (size_t)blockIdx.x * (N1 / 2) : nullptr;
  // (the rotation-table window lies behind the transform buffer)
  FastCta c{reinterpret_cast<float2*>(smem_raw), ZSmem{zf}, ZSplit{zf, gline, N1 / 2}, gline,
            TwTab{P.tw, P.log2tw, P.twpass}, zf + (kSplit ? N1 / 2 : N1), 0, red, tid};
  const FastPoint* points = reinterpret_cast<const FastPoint*>(F.points);

  // (lives in red[0], which is dead between the end of one point and the reduction of the next: 16 more bytes of
  // static shared memory would come out of every point's rotation-table window)
  int& s_next = *reinterpret_cast<int*>(&red[0]);
  int pn;
  for (int p = blockIdx.x; p < P.B; p = pn) {
    float* row = P.flux + (long long)p * P.ldf;
    // the next point is claimed now (its latency hides under this point) and read after the barrier below; thread 0
    // writes s_next again only behind this iteration's last barrier
    if (tid == 0) s_next = F.work_counter ? atomicAdd(F.work_counter, 1) : p + (int)gridDim.x;
    const FastPoint* rec = points + p;
    int K = 1;                                            // members (targets; 0: no such target)
    if constexpr (body_target(BODY)) {
      const int t = __ldg(P.target + p);
      K = (t >= 0 && t < P.n_targets) ? __ldg(P.tfirst + t + 1) - __ldg(P.tfirst + t) : 0;
      rec = points + (long long)p * P.kmax;
      if (tid >= 32 && tid < 64) {
        // warp 1: the pixels that the members' stage 2 and final passes read, the union of their windows (in red[1],
        // dead like red[0] until the first member's reduction)
        int lo = P.n, hi = -1;
        for (int m = tid - 32; m < K; m += 32) {
          const PointSetup& Sm = rec[m].S;
          if (Sm.bad) continue;
          lo = min(lo, Sm.use_inst ? max(Sm.i0 - 1, 0) : 0);
          hi = max(hi, Sm.use_inst ? min(Sm.i1 + 1, P.n - 1) : P.n - 1);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
          hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if (tid == 32) *reinterpret_cast<int2*>(&red[1]) = make_int2(lo, hi);
      }
    }
    load_record(SP, rec, tid);
    __syncthreads();
    pn = s_next;
    int2 tu = make_int2(0, -1);
    if constexpr (body_target(BODY)) {
      tu = *reinterpret_cast<const int2*>(&red[1]);
      __syncthreads();                                    // red[1] is read everywhere before a member's reduction
    }
    if constexpr (BODY == FastBody::Binary) {
      binary_point<LOG2N1>(P, F, SP, c, row, p, points);
    } else {
      if (body_target(BODY) ? K == 0 : SP.S.bad) {        // NaN lnL and model row; the row is not read
        // (the model row's NaN fill written out: model_nan here changed the code of the plain kernels)
        if (P.model_out)
          for (int j = tid; j < obs_hi<STARS>(P, SP.FS.obs) - obs_lo<STARS>(SP.FS.obs); j += kNT)
            P.model_out[(long long)p * P.ld_flux + j] = CUDART_NAN;
        if constexpr (BODY == FastBody::MargStars) {
          const int k = star_of(P.star, P.n_stars, p);
          if (k >= 0) marg_nan_out(P, p, __ldg(P.marg_k + k), 0, 0, tid);
          if (tid == 0 && P.chi2_out) P.chi2_out[(long long)p * P.ld_chi2] = CUDART_NAN;
        }
        if (tid == 0 && P.lnl) store_lnl(P, p, CUDART_NAN);
        __syncthreads();
        continue;
      }
      if constexpr (body_target(BODY)) target_point<LOG2N1, POLY, BODY>(P, F, SP, c, row, p, rec, K, tu);
      else star_point<LOG2N1, POLY, BODY>(P, F, SP.S, SP.FS, c, row, p);
    }
    // The row is scratch and fully consumed: L2 is told to drop its lines instead of writing them back
    // (discard.global.L2).  Without this every row crosses HBM three times (the emulator's write is evicted --
    // the slab is larger than L2 --, the tail reads it, and the in-place rewrite after the rotation stage is
    // evicted again): measured DRAM traffic of the tail 456 MB = 2.0x the algorithmic bytes, 254 MB = 1.09x
    // with the discard, for +1.4 % of kernel time.  Only lines that lie wholly inside this row are dropped.
    if (P.discard_rows) {
      discard_lines(row, P.n, tid);
      if constexpr (BODY == FastBody::Binary) discard_lines(row + (long long)P.B * P.ldf, P.n, tid);
    }
    __syncthreads();
  }
  if (tid == 0) gather_exit(P, gridDim.x);
}

// stage-2 and final regrid ratios of a point with an instrumental stage
__device__ __forceinline__ void stage2_setup(const FastGrid& F, const PointSetup& S, FastSetup& FS) {
  const int nM = S.i1 - S.i0 + 1, N2 = 1 << S.log2N2;
  FS.s_num = nM - 1; FS.s_den = N2 - 1;
  const long long inc = 2LL * kNT * (nM - 1);
  FS.s_incj = (int)(inc / (N2 - 1));
  FS.s_incr = (int)(inc - (long long)FS.s_incj * (N2 - 1));
  FS.s_invden = 1.0f / (float)(N2 - 1);
  FS.scale = (double)(N2 - 1) / (double)(nM - 1);
  FS.q0 = (double)S.i0 + S.lnD * F.inv_dlnw;
}

// One thread per setup item (the serial prologue of the tail, done for the whole slab at once): mask limits, transform
// sizes, Doppler factor, taper constant and the stage-2 / final regrid ratios of FastPoint record `item`.  The item of
// tail_fast_kernel<BODY>'s point p:
//  - a point of one star (OneStar, Stars, MargStars; launched as Stars): item p;
//  - a target's member m (Target, MargTargets; launched as Target): item p * kmax + m.  The items of members a target
//    does not have are not written; a point whose target lies outside [0, n_targets) gets a bad record at p * kmax;
//  - a binary's component c (Binary): item c * B + p, the secondary's labels, Vrad and Vrot through P.binary, and from
//    component 0's thread the point's Teff_1, Teff_2 and Rratio.
template <FastBody BODY>
__global__ void __launch_bounds__(64)
tail_setup_kernel(const __grid_constant__ TailParams P, const __grid_constant__ FastGrid F) {
  constexpr bool TGT = body_target(BODY), BIN = BODY == FastBody::Binary;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)P.B * (TGT ? P.kmax : BIN ? 2 : 1)) return;
  if (i == 0 && F.work_counter) *F.work_counter = F.work_start;
  int p, k, c = 0;                                        // point, star, component
  if constexpr (TGT) {
    p = (int)(i / P.kmax);
    const int m = (int)(i - (long long)p * P.kmax);
    const int t = P.target[p];
    k = -1;
    if (t >= 0 && t < P.n_targets) {
      const int f = P.tfirst[t];
      if (m >= P.tfirst[t + 1] - f) return;
      k = f + m;
    } else if (m > 0) {
      return;
    }
  } else {
    if constexpr (BIN) c = (int)(i / P.B);
    p = (int)(i - (long long)c * P.B);
    k = star_of(P.star, P.n_stars, p);
  }
  const double* th = P.theta + (long long)p * P.ld;
  PointSetup S{};
  FastSetup FS{};
  tail_setup_star(P, th, k, S, FS.obs, c ? P.binary : nullptr);
  if (!S.bad && S.use_inst) {
    stage2_setup(F, S, FS);
    // (F.cluster is set for batches of points naming stars only)
    if (F.cluster && P.stars[k].sorted) {
      // tail_cluster.cuh: CTA r of the cluster serves the observed pixels whose position falls into quarter r
      for (int r = 0; r < 3; ++r) {
        const double thr = (double)((long long)(r + 1) << (S.log2N2 - 2));
        int a = FS.obs.off, b = FS.obs.off + FS.obs.n;   // first j of the star with (obs_q[j] - q0) * scale >= thr
        while (a < b) {
          const int mid = (a + b) >> 1;
          if ((__ldg(F.obs_q + mid) - FS.q0) * FS.scale >= thr) b = mid; else a = mid + 1;
        }
        FS.jcut[r] = a;
      }
    } else if (F.cluster) {
      FS.jcut[0] = -1;
    }
  }
  FastPoint* out = reinterpret_cast<FastPoint*>(F.points) + i;
  out->S = S;
  out->FS = FS;
  if (BIN && c == 0) {
    const double t1 = get_par(P, th, PAYNE_P_TEFF, k);
    const PayneBinary& b = *P.binary;
    P.bin_par[3LL * p] = t1;
    P.bin_par[3LL * p + 1] = secondary_of(&b, th, PAYNE_P_TEFF, t1);
    P.bin_par[3LL * p + 2] = b.rratio_col >= 0 ? th[b.rratio_col] : b.rratio_fixed;
  }
}

}  // namespace payne
