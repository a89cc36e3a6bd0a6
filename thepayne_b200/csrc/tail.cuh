// Fused tail of the likelihood: emulator flux row -> rotational broadening -> Doppler shift ->
// instrumental broadening -> resample onto the observed pixels -> Chebyshev continuum -> chi2.
// One CTA owns one live point at a time; the only HBM/L2 traffic per point is the fp32 flux
// row (read once, rewritten in place after the rotational stage) plus per-dataset tables.
//
// Reference semantics reproduced step by step (paths relative to the reference checkout):
//   Payne/predict/predictspec.py:228-289   getspec: vsini -> edge patch -> Doppler -> inst_R / interp
//   Payne/utils/smoothing.py:132-143       mask_wave (+-20 sigma, strict), nan_to_num(nan=1)
//   Payne/utils/smoothing.py:649-668       resample_wave: 2^k uniform ln-lambda regrid by np.interp
//   Payne/utils/smoothing.py:293-314,610-629  rotational kernel in Fourier space, np.interp back
//   Payne/utils/smoothing.py:252-291,588-608  Gaussian taper, np.interp onto outwave (NaN outside)
//   Payne/fitting/fitutils.py:11-20        polycalc (chebval on the normalised observed grid)
//   Payne/fitting/likelihood.py:95-97,117  chi2 and lnL
//
// Numerics: wavelength / index arithmetic in fp64, flux arithmetic in fp32 on the line depth
// d = f - 1 (both transfer functions have unit DC gain, so the FFTs only see the ~0.1-amplitude
// depth signal), residuals and the chi2 sum in fp64.
#pragma once
#include <math_constants.h>
#include "fft.cuh"
#include "obs_star.cuh"
#include "../../include/payne_b200.h"

namespace payne {

constexpr double kCkms = 2.998e5;               // smoothing.py:16
constexpr double kSpeedOfLight = 299792.458;    // predictspec.py:12
constexpr double kFwhmFit = 2.355;              // genmod.py:83
constexpr int kTailThreads = 256;

struct TailParams {
  // emulator grid
  int n;
  const double* w;        // [n]
  const double* inv_dw;   // [n-1] 1/(w[j+1]-w[j])
  double lnw0, inv_dlnw;  // index guess: (ln x - lnw0) * inv_dlnw
  double sigma_in;        // ckms / ANN.resolution  (smoothing.py:113)
  // stage 1 (rotation): per-dataset regrid tables, np.interp semantics baked in on the host
  int log2N1;
  const int2* fwd1;       // [N1]  {j, bits(t)}: g_k = f[j] + t (f[j+1]-f[j])
  const int2* back1;      // [n]   {k, bits(t)}: f_i = g[k] + t (g[k+1]-g[k])
  double sb_scale;        // 2 pi / (N1 dv1 h): table coordinate of bin k is |vsini| k sb_scale
  double sb_h;            // table spacing in u
  const float4* sbtab;    // [ntab] cubic through sb((i-1)h) .. sb((i+2)h) as Horner coefficients in f = u/h - i
  int ntab;
  // twiddles exp(-2 pi i e / Ntw), e < Ntw/2
  const float2* tw;
  int log2tw;
  const float2* twpass[16]; // [log2 M] compact per-pass twiddle tables of the compile-time plans (fft_ct.cuh)
  int max_log2N;          // largest FFT the shared-memory carve-out holds
  // observation: the stars' arrays back to back (obs_star.cuh); n_obs / obs_min / obs_max are star 0's
  int n_obs;
  const double* obs_w;      // [n_obs] wavelength
  const double* obs_lnw;    // [n_obs] ln wavelength
  const double* obs_ot;     // [n_obs] flux / eflux
  const double* obs_inv_s;  // [n_obs] 1 / eflux
  const double* obs_x;      // [n_obs] Chebyshev abscissa (fitutils.py:13-14)
  double obs_min, obs_max;
  // parameter layout
  int col[PAYNE_NPAR];
  double fixed[PAYNE_NPAR];
  int n_poly;
  int poly_col[PAYNE_MAX_POLY];
  int n_labels;                 // emulator inputs: a row whose labels are all finite cannot hold NaN
  int label_col[8];
  double label_fixed[8];
  // batch
  const double* theta;
  long long ld;
  float* flux;              // [B, ldf] emulator output; scratch, overwritten
  long long ldf;
  int flux_is_depth;        // rows hold f - 1 (tensor-core path) instead of f
  const double* chi2_sed;   // [B] or null
  double* lnl;              // [B] or null
  double* model_out;        // [B, ld_flux] or null: row p holds the first n_obs of p's star
  int* status;              // device flag: bit0 = a point needed a larger FFT than the carve-out
  int B;
  double inst_scale;        // Inst_R -> sigma-resolution: 2.355 (genmod.py:83, FWHM given) or 1 (getspec callers)
  int discard_rows;         // fast tail: drop a consumed row's lines from L2 without write-back (discard.global.L2)
  int rows_may_nan;         // rows can hold NaN although the labels are finite (continuum emulator attached)
  // Multi-GPU all-gather of lnL fused into the tail (payne_lnlike_batch_gather; fast and cluster tails): the thread
  // that writes a point's lnL also stores it into every peer's gathered buffer through the NVLink peer mappings, and
  // the last CTA to leave the kernel raises this rank's flag on every rank behind a system-scope fence.  g_world = 0: off.
  // (at the END of the struct: the fields above keep the constant-bank offsets the kernels were tuned with)
  int g_world, g_rank;
  double* g_dst[16];                 // rank r's buffer of this step at this rank's slice, slab offset included
  unsigned long long* g_flag[16];    // rank r's flag word of this rank
  unsigned long long g_raise;        // 0: this launch does not finish the step (a slab before the last one)
  int* g_done;                       // CTA counter (zero between launches)
  // Observation set (payne_ctx_create_stars): star of every point of this slab (null: star 0) and the per-star
  // records.  A point whose star lies outside [0, n_stars) gets lnL NaN, no model row, and status bit 2.
  const int* star;
  const ObsStar* stars;
  int n_stars;
  long long ld_flux;                 // model_out row stride
  // Per-star fixed values (payne_ctx_create_stars_opts): [n_stars, PAYNE_NPAR], read where col < 0 in place of
  // `fixed` / `label_fixed`; null when the context was created without them.
  const double* star_fixed;
  const StarLayout* star_lay;        // [n_stars] per-star layouts (obs_star.cuh), null without them
  // Targets (payne_ctx_set_targets; fast tail only): point p names target[p], whose members are the stars
  // [tfirst[t], tfirst[t + 1]); member m's per-point record is FastPoint p * kmax + m.  A target outside
  // [0, n_targets) gets lnL NaN, no model row and status bit 2.  Null target: the points name stars.
  const int* target;
  const int* tfirst;                 // [n_targets + 1]
  int n_targets, kmax;               // kmax: the largest member count
  double* chi2_out;                  // [B, ld_chi2] chi2 of every member, or null
  long long ld_chi2;
  // Binaries (payne_ctx_set_binary; fast tail only): point p's component c has emulator row c * B + p and FastPoint
  // record c * B + p.  Null binary: no binary.
  const PayneBinary* binary;         // device copy
  double* bin_par;                   // [B, 3] Teff_1, Teff_2, Rratio of every point (tail_setup_kernel)
  double* aj_scratch;                // [grid, aj_ld] a_1 (binaries) or a_j (marginalisation) of the CTA's current point
  long long aj_ld;
  double* comp_out;                  // [B, 2, ld_flux] a_1 and a_2, or null
  // Continuum marginalisation (payne_ctx_set_cont_marg; fast tail only): star k's K = marg_k[k] coefficients are
  // integrated out, C = marg_c[k] = sum_k (ln 2 pi / 2 - ln w_k).  aj_scratch / aj_ld hold a_j of the CTA's current point,
  // chi2_out / ld_chi2 every point's (or member's) Q.  Null marg_k: off.
  const int* marg_k;
  const double* marg_c;
  double* coef_out;                  // [B, ld_coef] c-hat (a target's members back to back), or null
  long long ld_coef;
  double* chol_out;                  // [B, ld_chol] L, packed lower triangles K (K + 1) / 2 each, or null
  long long ld_chol;
};

// lnL of point p: local result and, with the fused gather on, the copy in every peer's buffer
__device__ __forceinline__ void store_lnl(const TailParams& P, int p, double v) {
  P.lnl[p] = v;
  for (int r = 0; r < P.g_world; ++r)
    if (r != P.g_rank) P.g_dst[r][p] = v;
}
// every CTA, once, behind its last point (thread 0): the CTA's peer stores are fenced; the last CTA raises the flags
__device__ __forceinline__ void gather_exit(const TailParams& P, unsigned nctas) {
  if (P.g_world == 0) return;
  __threadfence_system();
  if (P.g_raise && atomicAdd(P.g_done, 1) == (int)nctas - 1) {
    *P.g_done = 0;
    __threadfence_system();
    for (int r = 0; r < P.g_world; ++r) *reinterpret_cast<volatile unsigned long long*>(P.g_flag[r]) = P.g_raise;
  }
}

// The CTA's sum of every thread's acc, complete in thread 0 (0 elsewhere): warp shuffles, then the warps' partials in
// warp order, so the bits do not depend on scheduling.  red: kTailThreads / 32 doubles of shared memory, written before
// the barrier this ends with.
__device__ __forceinline__ double cta_sum(double acc, double* red, int tid) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((tid & 31) == 0) red[tid >> 5] = acc;
  __syncthreads();
  double c2 = 0.0;
  if (tid == 0) {
#pragma unroll
    for (int w = 0; w < kTailThreads / 32; ++w) c2 += red[w];
  }
  return c2;
}

// NaN into the n model pixels of a bad point (or member) from column moff of row p; nothing without model output
__device__ __forceinline__ void model_nan(const TailParams& P, int p, int moff, int n, int tid) {
  if (P.model_out)
    for (int j = tid; j < n; j += kTailThreads) P.model_out[(long long)p * P.ld_flux + moff + j] = CUDART_NAN;
}

// A per-point record into shared memory, as int4 by threads 0 .. sizeof(T) / 16 - 1; the caller's barrier publishes it
template <class T>
__device__ __forceinline__ void load_record(T& dst, const T* src, int tid) {
  static_assert(sizeof(T) % 16 == 0, "records are copied as int4");
  if (tid < (int)(sizeof(T) / 16)) reinterpret_cast<int4*>(&dst)[tid] = __ldg(reinterpret_cast<const int4*>(src) + tid);
}

struct PointSetup {
  double vsini_scale;   // |vsini| * sb_scale
  double D;             // Doppler factor
  double u0, inv_du;    // resampled grid of stage 2 (observed frame)
  double rho;           // rest-frame grid ratio per kTailThreads steps
  double du, rM;
  double lnD, u0t;      // u0t = ln w[i0] in the rest frame
  double poly[PAYNE_MAX_POLY];
  float taper_a;        // exp(-a k^2)
  float hdu;
  int do_rot, use_inst, bad, i0, i1, log2N2, clean;
};

// The point's star: observed pixels [off, off + n) of the concatenated arrays (0 pixels for an invalid star).
struct ObsSlice {
  int off, n;
};

// parameter `which` of point th of star k
__device__ __forceinline__ double get_par(const TailParams& P, const double* th, int which, int k) {
  return param_of(P.star_lay, P.col[which], P.fixed[which], P.star_fixed, th, k, which);
}

// float index of real sample k: 2*swz(k>>1) + (k&1) == k ^ (((k>>5)&7)<<2)
__device__ __forceinline__ int zidx(int k) { return k ^ (((k >> 5) & 7) << 2); }

// np.interp between (wa, a) and (wb, b), wa <= x <= wb, as numpy's compiled_interp has it: an exact hit returns its
// value (also beside a NaN neighbour, e.g. where a continuum emulator's NaN ends meet the grid), else
// slope * (x - wa) + a, with its fallbacks for NaN / inf neighbours
__device__ __forceinline__ double np_interp_pair(double x, double wa, double wb, double a, double b) {
  if (x == wa) return a;
  if (x == wb) return b;
  const double slope = (b - a) / (wb - wa);
  double r = slope * (x - wa) + a;
  if (r != r) {
    r = slope * (x - wb) + b;
    if (r != r && a == b) r = a;
  }
  return r;
}

// largest j in [lo, hi] with w[j]*D <= x, assuming w[lo]*D <= x; starts from a guess.
__device__ __forceinline__ int locate(const double* __restrict__ w, double D, double x, int guess,
                                      int lo, int hi) {
  int j = min(max(guess, lo), hi);
  int steps = 0;
  while (j > lo && x < __ldg(w + j) * D && steps < 4) { --j; ++steps; }
  while (j < hi && x >= __ldg(w + j + 1) * D && steps < 8) { ++j; ++steps; }
  if (steps >= 4) {  // far-off guess (irregular grid): bisection
    int a = lo, b = hi;
    if (x < __ldg(w + a) * D) return a;
    while (b > a) {
      int mid = (a + b + 1) >> 1;
      if (__ldg(w + mid) * D <= x) a = mid; else b = mid - 1;
    }
    j = a;
  }
  return j;
}

// Rotational transfer function sb(u) (smoothing.py:612-619): 4-point Lagrange interpolation of a table with
// spacing h, stored per interval as the monomial coefficients of that cubic (one 16-byte load and three
// FMAs per value instead of four loads and the weight polynomials).
// WINDOW 0: global table only; 1: every interval the point can touch sits in the shared-memory copy `win`;
// 2: the first nwin intervals do, the rest come from the global table.
template <int WINDOW>
struct RotHT {
  const float4* __restrict__ tab;   // global table
  const float4* win;                // copy of its first nwin intervals in shared memory
  int nwin;
  double scale;     // table coordinate per bin
  double h;
  float invM;
  int ntab;
  // Table position of bin k in 24.40 fixed point (k < 2^15, scale < 2^8): one wide integer multiply, a shift
  // and an int->float conversion instead of four double-precision conversions per value; the position is
  // good to 2^-28 of a table interval.
  unsigned long long s40;
  __device__ static unsigned long long fix40(double scale) {
    return scale < 256.0 ? (unsigned long long)__double2ll_rn(scale * 1099511627776.0) : ~0ull;
  }
  __device__ __forceinline__ float operator()(int k) const {
    if (WINDOW != 1 && s40 == ~0ull) return direct(scale * (double)k * h) * invM;     // absurdly broad kernel: closed form
    const unsigned long long pos = (unsigned long long)(unsigned)k * s40;
    const int i = (int)(pos >> 40);
    if (WINDOW != 1 && i >= ntab) return direct(scale * (double)k * h) * invM;
    const float f = (float)(unsigned)(pos >> 8) * 2.3283064365386963e-10f;   // low 32 of the 40 fraction bits
    float4 c;
    if (WINDOW == 1) c = win[i];
    else if (WINDOW == 2) c = i < nwin ? win[i] : __ldg(tab + i);
    else c = __ldg(tab + i);
    return fmaf(f, fmaf(f, fmaf(f, c.w, c.z), c.y), c.x) * invM;
  }
  static __device__ __noinline__ float direct(double u) {  // beyond the table: fp64 closed form
    if (u == 0.0) return 1.f;
    double s, c;
    sincos(u, &s, &c);
    return (float)(j1(u) / u - 3.0 * c / (2.0 * u * u) + 3.0 * s / (2.0 * u * u * u));
  }
};
using RotH = RotHT<0>;

// Stage 1's transfer function at N1 samples, with the rotation table's first intervals staged in the CTA's shared-memory
// window `win` (win_floats floats, 4 per interval).  The point can touch the entries [0, vsini_scale * N1/2 + 3]; a point
// whose range is longer keeps its first win_floats/4 intervals there and reads the rest from the global table.  The
// window holds the first intervals of the one table, so the win_have intervals an earlier point of the CTA staged stay
// valid.  The caller's next barrier publishes the new entries.
__device__ __forceinline__ RotHT<2> rot_window(const TailParams& P, const PointSetup& S, int N1, float* win, int win_floats,
                                               int& win_have, int tid) {
  const double xt_max = S.vsini_scale * (double)(N1 >> 1);
  float4* win4 = reinterpret_cast<float4*>(win);
  const int nwin = (int)fmin(fmin(xt_max + 2.0, (double)(win_floats >> 2)), (double)P.ntab);
  for (int i = win_have + tid; i < nwin; i += kTailThreads) win4[i] = __ldg(P.sbtab + i);
  win_have = max(win_have, nwin);
  return RotHT<2>{P.sbtab, win4, nwin, S.vsini_scale, P.sb_h, 1.0f / (float)(N1 >> 1), P.ntab, RotHT<2>::fix40(S.vsini_scale)};
}

// Gaussian taper exp(-2 pi^2 sigma^2 ss^2) (smoothing.py:598-600), ss = k / (N dv).
struct GaussH {
  float a, invM;
  __device__ __forceinline__ float operator()(int k) const {
    const float kf = (float)k;
    return expf(-a * kf * kf) * invM;
  }
};

__device__ __forceinline__ double chebval_dev(double x, const double* c, int nc) {
  // numpy.polynomial.chebyshev.chebval (Clenshaw), same operation order
  if (nc == 1) return c[0];
  if (nc == 2) return c[0] + c[1] * x;
  const double x2 = 2.0 * x;
  double c0 = c[nc - 2], c1 = c[nc - 1];
  for (int i = 3; i <= nc; ++i) {
    const double tmp = c0;
    c0 = c[nc - i] - c1;
    c1 = tmp + c1 * x2;
  }
  return c0 + c1 * x;
}

// The same for four abscissae at once (identical operations per abscissa, coefficient loads shared, four
// independent dependency chains instead of one).
__device__ __forceinline__ void chebval_dev4(const double (&x)[4], const double* c, int nc, double (&out)[4]) {
  if (nc == 1) {
#pragma unroll
    for (int u = 0; u < 4; ++u) out[u] = c[0];
    return;
  }
  if (nc == 2) {
    const double a = c[0], b = c[1];
#pragma unroll
    for (int u = 0; u < 4; ++u) out[u] = a + b * x[u];
    return;
  }
  double c0[4], c1[4];
  {
    const double a = c[nc - 2], b = c[nc - 1];
#pragma unroll
    for (int u = 0; u < 4; ++u) { c0[u] = a; c1[u] = b; }
  }
  for (int i = 3; i <= nc; ++i) {
    const double ci = c[nc - i];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const double tmp = c0[u];
      c0[u] = ci - c1[u];
      c1[u] = tmp + c1[u] * (2.0 * x[u]);
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) out[u] = c0[u] + c1[u] * x[u];
}

__device__ __forceinline__ float depth_of(float v, bool is_depth, bool fill_nan) {
  if (fill_nan && v != v) return 0.f;   // nan_to_num(nan=1.0) (smoothing.py:138) in depth space
  return is_depth ? v : v - 1.f;
}

// Point setup of theta row th against star k (k < 0: no such star).  sec: the binary whose secondary this record
// describes (its labels, Vrad and Vrot; secondary_of), null for the primary or a single star.
static __device__ __forceinline__ void tail_setup_star(const TailParams& P, const double* th, int k, PointSetup& S,
                                                       ObsSlice& obs, const PayneBinary* sec = nullptr) {
  if (k < 0) {                                    // no observation to compare with: NaN, nothing written
    S.bad = 1; S.use_inst = 0; S.do_rot = 0;
    obs.off = 0; obs.n = 0;
    atomicOr(P.status, 4);
    return;
  }
  const ObsStar& st = P.stars[k];
  obs.off = st.off; obs.n = st.n_obs;
  const double vrot = secondary_of(sec, th, PAYNE_P_VROT, get_par(P, th, PAYNE_P_VROT, k));
  const double vrad = secondary_of(sec, th, PAYNE_P_VRAD, get_par(P, th, PAYNE_P_VRAD, k));
  const double instR = get_par(P, th, PAYNE_P_INSTR, k);
  S.bad = 0;
  S.clean = P.rows_may_nan ? 0 : 1;
  for (int i = 0; i < P.n_labels; ++i) {
    const int which = label_param(i);
    const double v = secondary_of(sec, th, which,
                                  param_of(P.star_lay, P.label_col[i], P.label_fixed[i], P.star_fixed, th, which >= 0 ? k : -1, which));
    if (!isfinite(v)) S.clean = 0;
  }
  S.do_rot = (vrot != 0.0);                       // predictspec.py:231 (NaN != 0 is true)
  if (vrot != vrot) S.bad = 1;                    // NaN kernel -> NaN spectrum
  S.vsini_scale = fabs(vrot) * P.sb_scale;        // sigma = sqrt(vsini^2 - 0) (smoothing.py:297)
  S.D = (vrad != 0.0) ? 1.0 + (vrad / kSpeedOfLight) : 1.0;   // predictspec.py:245-249
  if (!(S.D > 0.0)) S.bad = 1;
  S.lnD = log(S.D);
  // A star with fewer coefficients than the launch's n_poly (per-star layouts: the largest) gets zeros after its own.
  // Clenshaw's recurrence passes through trailing zero coefficients exactly at a finite abscissa ((a, 0) -> (c, a)),
  // so the final passes keep one constant-bank n_poly and every star gets the bits of its own continuum order.
  for (int i = poly_of(P.star_lay, P.n_poly, P.poly_col, th, k, S.poly); i < P.n_poly; ++i) S.poly[i] = 0.0;
  const double Rs = P.inst_scale * instR;         // genmod.py:83 (inst_scale = 2.355) or predictspec.py:255-263 (1)
  S.use_inst = (Rs > 0.0);                        // predictspec.py:257 (false for NaN)
  S.log2N2 = 0; S.i0 = 0; S.i1 = P.n - 1;
  if (!S.use_inst || S.bad) return;
  // mask_wave (smoothing.py:631-647): wlim * (1 + 20/width * [-1, 1]), strict inequalities
  const double lo = st.obs_min * (1.0 + 20.0 / Rs * -1.0);
  const double hi = st.obs_max * (1.0 + 20.0 / Rs * 1.0);
  const int n = P.n;
  // first index with w*D > lo
  int g0 = (int)ceil((log(lo) - S.lnD - P.lnw0) * P.inv_dlnw);
  int i0;
  if (!(__ldg(P.w + n - 1) * S.D > lo)) i0 = n;
  else if (__ldg(P.w) * S.D > lo) i0 = 0;
  else i0 = locate(P.w, S.D, lo, g0, 0, n - 2) + 1;   // locate: last with w*D <= lo
  // last index with w*D < hi
  int i1;
  if (!(__ldg(P.w) * S.D < hi)) i1 = -1;
  else if (__ldg(P.w + n - 1) * S.D < hi) i1 = n - 1;
  else {
    int g1 = (int)floor((log(hi) - S.lnD - P.lnw0) * P.inv_dlnw);
    i1 = locate(P.w, S.D, hi, g1, 0, n - 2);          // last with w*D <= hi
    if (__ldg(P.w + i1) * S.D == hi) --i1;              // strict
  }
  const int nM = i1 - i0 + 1;
  if (nM < 17) { S.bad = 1; return; }
  int l2 = 32 - __clz(nM - 1);                     // ceil(log2(nM))
  if (l2 > P.max_log2N) { S.bad = 2; atomicOr(P.status, 1); return; }
  S.i0 = i0; S.i1 = i1; S.log2N2 = l2;
  const int N2 = 1 << l2;
  const double u0 = log(__ldg(P.w + i0) * S.D), u1 = log(__ldg(P.w + i1) * S.D);
  S.du = (u1 - u0) / (double)(N2 - 1);             // np.linspace step
  S.u0 = u0;
  S.u0t = log(__ldg(P.w + i0));
  S.inv_du = 1.0 / S.du;
  S.hdu = (float)(0.5 * S.du);
  S.rM = (double)(nM - 1) / (double)(N2 - 1);
  S.rho = exp(S.du * (double)kTailThreads);
  const double sig_out = kCkms / Rs;               // smoothing.py:106
  const double s2 = sig_out * sig_out - P.sigma_in * P.sigma_in;   // smoothing.py:271
  if (!(s2 >= 0.0)) { S.bad = 1; return; }         // sqrt(<0) = NaN everywhere
  const double dv = kCkms * S.du;                  // smoothing.py:282
  const double nd = (double)N2 * dv;
  S.taper_a = (float)(2.0 * CUDART_PI * CUDART_PI * s2 / (nd * nd));
}

static __device__ void tail_setup(const TailParams& P, const double* th, int p, PointSetup& S, ObsSlice& obs) {
  tail_setup_star(P, th, star_of(P.star, P.n_stars, p), S, obs);
}

}  // namespace payne
