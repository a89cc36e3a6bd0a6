// Tail for an LSF vector: PayneSpecPredict.getspec with a non-float ``inst_R`` (the dispersion in AA at
// every observed pixel) -- Payne/predict/predictspec.py:265-286 -> smoothspec(smoothtype='lsf')
// Payne/utils/smoothing.py:126-150 -> smooth_lsf_fft :482-586 -> smooth_fft :588-608.
//
// The rotational stage, the edge patch and the Doppler factor are those of tail_general.cuh.  The
// instrumental stage differs from the scalar-R one in every step, and all of it depends on the point
// (the dispersion is interpolated at the Doppler-shifted emulator wavelengths):
//   disparr = np.interp(modwave, outwave, lsf)                          predictspec.py:270-272
//   mask    = modwave within [outwave.min() - 2000, outwave.max() + 2000]   smoothing.py:126-133, 640-646
//   dw = np.gradient(wave); cdf = np.cumsum(dw / sigma); cdf /= cdf.max()   :525-527
//   x_per_sigma = np.nanmedian(np.gradient(cdf) / (dw / sigma)); nx = 2**ceil(log2(2 / x_per_sigma))  :548-565
//   lam = np.interp(linspace(0, 1, nx), cdf, wave); newspec = np.interp(lam, wave, spec)  :568-573
//   spec_conv = irfft(rfft(newspec) * exp(-2 pi^2 x_per_sigma^2 k^2))                     :581, 596-607
//   outspec = np.interp(outwave, lam, spec_conv)          (edges clamp, no NaN)           :584
// One CTA per point; the cumulative sum is a block scan, the median an exact radix selection
// (continuum.cuh), the three np.interp are bisections with numpy's slope formula, and the convolution is
// the runtime-planned in-shared-memory FFT of fft.cuh on the line depth (nx = 2 .. 16, below its smallest plan: a
// direct circular convolution, lsf_small_conv; nx = 1 is NaN).  Wavelength arithmetic is fp64.
#pragma once
#include "continuum.cuh"
#include "tail.cuh"

namespace payne {

struct LsfParams {
  const double* lsf;      // dispersion (AA) at the observed pixels, the stars' vectors back to back like obs_w
  double* cdf;            // [grid, n]  scratch
  double* aux;            // [grid, n]  scratch: dw/sigma, then gradient(cdf)/(dw/sigma)
  double* lam;            // [grid, 2^log2nx_max] scratch
  int log2nx_max;         // largest transform the shared-memory carve-out and the twiddle table hold
};

// last j in [0, n-1] with xs(j) <= x, given xs(0) <= x
template <class XF>
__device__ __forceinline__ int last_le(const XF& xs, int n, double x) {
  int a = 0, b = n - 1;
  while (b > a) {
    const int mid = (a + b + 1) >> 1;
    if (xs(mid) <= x) a = mid; else b = mid - 1;
  }
  return a;
}

// np.interp(x, xp, fp) with the default clamped edges (numpy's compiled_interp: slope * (x - xp[j]) + fp[j])
template <class XF, class FF>
__device__ __forceinline__ double np_interp(double x, const XF& xp, const FF& fp, int n, int* jout = nullptr) {
  if (jout) *jout = 0;
  if (x != x) return x;
  if (x > xp(n - 1)) { if (jout) *jout = n - 1; return fp(n - 1); }
  if (x < xp(0)) return fp(0);
  const int j = last_le(xp, n, x);
  if (jout) *jout = j;
  if (j == n - 1) return fp(j);
  const double x0 = xp(j);
  if (x0 == x) return fp(j);
  const double f0 = fp(j), f1 = fp(j + 1), x1 = xp(j + 1);
  const double slope = (f1 - f0) / (x1 - x0);
  double r = slope * (x - x0) + f0;
  if (r != r) {
    r = slope * (x - x1) + f1;
    if (r != r && f0 == f1) r = f0;
  }
  return r;
}

// irfft(rfft(x) * exp(-2 pi^2 xps^2 k^2)) of the nx < 32 samples zf[zidx(0 .. nx)], below the smallest plan of the
// runtime FFT: the same transfer function as a direct circular convolution in fp64 with its impulse response
// h[m] = (T_0 + 2 sum_{0<k<nx/2} T_k cos(2 pi k m / nx) + T_{nx/2} cos(pi m)) / nx (the Nyquist term real, as irfft
// takes it).  h goes to hbuf[0, nx); all threads call it, and the result is in zf when it returns.
__device__ __forceinline__ void lsf_small_conv(float* zf, int nx, double xps, double* hbuf, int tid) {
  const double a = 2.0 * CUDART_PI * CUDART_PI * xps * xps;
  if (tid < nx) {
    double h = 0.0;
    for (int k = 0; k <= nx / 2; ++k) {
      const double t = exp(-a * (double)k * (double)k);
      h += ((k == 0 || 2 * k == nx) ? 1.0 : 2.0) * t * cospi((double)((2 * k * tid) % (2 * nx)) / (double)nx);
    }
    hbuf[tid] = h / (double)nx;
  }
  __syncthreads();
  double y = 0.0;
  if (tid < nx)
    for (int j = 0; j < nx; ++j) y += (double)zf[zidx(j)] * hbuf[(tid - j) & (nx - 1)];
  __syncthreads();
  if (tid < nx) zf[zidx(tid)] = (float)y;
  __syncthreads();
}

// Emulator pixels [i0, i1] inside the LSF mask of star st at Doppler factor D (thread 0; i1 < i0: none).
__device__ __forceinline__ int2 lsf_mask(const TailParams& P, const ObsStar& st, double D) {
  const int n = P.n;
  const double lo = st.obs_min + 20.0 * 100.0 * -1.0, hi = st.obs_max + 20.0 * 100.0 * 1.0;   // smoothing.py:128, 643
  const double* w = P.w;
  auto ws = [w, D](int i) { return __ldg(w + i) * D; };
  int i0 = n, i1 = -1;
  if (ws(n - 1) > lo) i0 = ws(0) > lo ? 0 : last_le(ws, n, lo) + 1;        // first with w D > lo
  if (ws(0) < hi) {
    i1 = last_le(ws, n, hi);                                               // last with w D <= hi
    if (ws(i1) == hi) --i1;                                                // strict
  }
  return make_int2(i0, i1);
}

// TGT false: point p names a star (TailParams::star).
// TGT true: point p names a target (TailParams::target), whose members are the stars [tfirst[t], tfirst[t + 1]).  The
// members share the labels and Vrot (payne_ctx_set_targets), so stage 1 runs once on the row, before the first member
// that is good after its setup and mask; from there on the row is read-only, and each member in order gets its own
// Doppler factor, mask, LSF stage, pixels, continuum and chi2 in the CTA's scratch.  Member m's model pixels follow those
// of members 0 .. m-1, chi2_out[p, m] is its chi2 (NaN when the member is bad by itself), and lnL is
// -0.5 ((((chi2_0 + chi2_1) + ...) + chi2_{K-1}) + chi2_sed).
// (The star form keeps its own inline copy of the stages: sharing the target form's lambdas changed its registers and
// stack frame.)
template <bool TGT>
__global__ void __launch_bounds__(kTailThreads, 1)
tail_lsf_kernel(const __grid_constant__ TailParams P, const __grid_constant__ LsfParams L) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* z = reinterpret_cast<float2*>(smem_raw);
  float* zf = reinterpret_cast<float*>(smem_raw);
  __shared__ PointSetup S;
  __shared__ double red[kTailThreads / 32];
  __shared__ double part[kTailThreads];
  __shared__ int hist[256];
  __shared__ unsigned long long sh_prefix;
  __shared__ int sh_rank, sh_count, sh_i0, sh_i1;
  __shared__ ObsSlice so;               // the point's star (a target: the current member): observed pixels [off, off + n)
  const int tid = threadIdx.x;
  const Twiddles twr{P.tw, P.log2tw};
  const double nan = CUDART_NAN;
  const int n = P.n;
  double* cdf = L.cdf + (size_t)blockIdx.x * n;
  double* aux = L.aux + (size_t)blockIdx.x * n;
  double* lam = L.lam + ((size_t)blockIdx.x << L.log2nx_max);

  if constexpr (!TGT) {
    for (int p = blockIdx.x; p < P.B; p += gridDim.x) {
      const double* th = P.theta + (long long)p * P.ld;
      float* row = P.flux + (long long)p * P.ldf;
      if (tid == 0) {
        tail_setup(P, th, p, S, so);             // Inst_R is absent in this mode: Doppler, rotation and polynomial only
        const double D = S.D;
        int i0 = n, i1 = -1;
        if (!S.bad) {
          const ObsStar& st = P.stars[star_of(P.star, P.n_stars, p)];
          const double lo = st.obs_min + 20.0 * 100.0 * -1.0, hi = st.obs_max + 20.0 * 100.0 * 1.0;   // smoothing.py:128, 643
          const double* w = P.w;
          auto ws = [w, D](int i) { return __ldg(w + i) * D; };
          if (ws(n - 1) > lo) i0 = ws(0) > lo ? 0 : last_le(ws, n, lo) + 1;        // first with w D > lo
          if (ws(0) < hi) {
            i1 = last_le(ws, n, hi);                                               // last with w D <= hi
            if (ws(i1) == hi) --i1;                                                // strict
          }
        }
        sh_i0 = i0; sh_i1 = i1;
      }
      __syncthreads();
      const int i0 = sh_i0, i1 = sh_i1, nM = i1 - i0 + 1;
      const int off = so.off, no = so.n;
      if (S.bad || nM < 17) {
        model_nan(P, p, 0, no, tid);
        if (tid == 0 && P.lnl) P.lnl[p] = nan;
        __syncthreads();
        continue;
      }
      bool is_depth = P.flux_is_depth != 0;
      const double D = S.D;

      // ---------------- stage 1: rotational broadening (as tail_general.cuh)
      if (S.do_rot) {
        const int N1 = 1 << P.log2N1, log2M = P.log2N1 - 1;
        for (int k = tid; k < N1; k += kTailThreads) {
          const int2 e = __ldg(P.fwd1 + k);
          const float t = __int_as_float(e.y);
          const float a = depth_of(row[e.x], is_depth, true), b = depth_of(row[e.x + 1], is_depth, true);
          zf[zidx(k)] = a + t * (b - a);
        }
        __syncthreads();
        RotH H{P.sbtab, nullptr, 0, S.vsini_scale, P.sb_h, 1.0f / (float)(1 << log2M), P.ntab, RotH::fix40(S.vsini_scale)};
        FftPlan plan; plan.make(log2M);
        fft_forward(z, log2M, plan, twr, tid, kTailThreads);
        filter_pairs(z, log2M, plan, twr, H, tid, kTailThreads);
        fft_inverse(z, log2M, plan, twr, tid, kTailThreads);
        for (int i = tid; i < n; i += kTailThreads) {
          if (i == 0 || i == n - 1) continue;
          const int2 e = __ldg(P.back1 + i);
          const float t = __int_as_float(e.y);
          const float g0 = zf[zidx(e.x)], g1 = zf[zidx(e.x + 1)];
          const float v = g0 + t * (g1 - g0);
          row[i] = v;
          if (i == 1) row[0] = v;
          if (i == n - 2) row[n - 1] = v;
        }
        is_depth = true;
        __syncthreads();
      }

      // ---------------- dw / sigma on the masked, shifted emulator grid
      const double* w = P.w + i0;
      const double* ow = P.obs_w + off;
      const double* lsf = L.lsf + off;
      auto wave = [w, D](int i) { return __ldg(w + i) * D; };
      auto owf = [ow](int j) { return __ldg(ow + j); };
      auto lsff = [lsf](int j) { return __ldg(lsf + j); };
      for (int i = tid; i < nM; i += kTailThreads) {
        const double disp = np_interp(wave(i), owf, lsff, no);
        const double dw = i == 0 ? wave(1) - wave(0)
                                 : (i == nM - 1 ? wave(nM - 1) - wave(nM - 2) : (wave(i + 1) - wave(i - 1)) / 2.0);
        aux[i] = dw / disp;
      }
      __syncthreads();
      // ---------------- cdf = cumsum / max: every thread sums a contiguous chunk, offsets by a serial pass
      const int chunk = (nM + kTailThreads - 1) / kTailThreads;
      const int c0 = min(tid * chunk, nM), c1 = min(c0 + chunk, nM);
      {
        double s = 0.0;
        for (int i = c0; i < c1; ++i) s += aux[i];
        part[tid] = s;
      }
      __syncthreads();
      if (tid == 0) {
        double run = 0.0;
        for (int t = 0; t < kTailThreads; ++t) { const double v = part[t]; part[t] = run; run += v; }
      }
      __syncthreads();
      {
        double s = part[tid];
        for (int i = c0; i < c1; ++i) { s += aux[i]; cdf[i] = s; }
      }
      __syncthreads();
      const double total = cdf[nM - 1];
      __syncthreads();
      for (int i = tid; i < nM; i += kTailThreads) cdf[i] = cdf[i] / total;
      __syncthreads();
      // ---------------- x_per_sigma = nanmedian(gradient(cdf) / (dw / sigma))
      for (int i = tid; i < nM; i += kTailThreads) {
        const double g = i == 0 ? cdf[1] - cdf[0]
                                : (i == nM - 1 ? cdf[nM - 1] - cdf[nM - 2] : (cdf[i + 1] - cdf[i - 1]) / 2.0);
        aux[i] = g / aux[i];
      }
      __syncthreads();
      const double* auxc = aux;
      const double xps = nanmedian_dev([auxc](int j) { return auxc[j]; }, nM, hist, &sh_prefix, &sh_rank, &sh_count);
      const double Nf = 2.0 / xps;                                    // pix_per_sigma = 2
      const int log2nx = (Nf == Nf && Nf > 0.0 && Nf < 1e9) ? (int)ceil(log2(Nf)) : -1;
      if (log2nx < 1 || log2nx > L.log2nx_max) {               // nx = 1: the reference's irfft raises (DESIGN §5)
        if (tid == 0) { if (log2nx > L.log2nx_max) atomicOr(P.status, 1); if (P.lnl) P.lnl[p] = nan; }
        model_nan(P, p, 0, no, tid);
        __syncthreads();
        continue;
      }
      const int nx = 1 << log2nx;
      // ---------------- even grid in the cdf coordinate, spectrum on it
      {
        const double step = 1.0 / (double)(nx - 1);                   // np.linspace(0, 1, nx)
        const double* cdfc = cdf;
        auto cdff = [cdfc](int j) { return cdfc[j]; };
        const float* rowm = row + i0;
        auto specf = [rowm, is_depth](int j) { return (double)depth_of(rowm[j], is_depth, true); };
        for (int k = tid; k < nx; k += kTailThreads) {
          const double x = k == nx - 1 ? 1.0 : (double)k * step;
          const double lk = np_interp(x, cdff, wave, nM);
          lam[k] = lk;
          zf[zidx(k)] = (float)np_interp(lk, wave, specf, nM);
        }
      }
      __syncthreads();
      if (log2nx < 5) {
        lsf_small_conv(zf, nx, xps, part, tid);
      } else {
        const int log2M = log2nx - 1;
        const float a = (float)(2.0 * CUDART_PI * CUDART_PI * xps * xps);   // ss = rfftfreq(nx, 1/nx) = k
        GaussH H{a, 1.0f / (float)(1 << log2M)};
        FftPlan plan; plan.make(log2M);
        fft_forward(z, log2M, plan, twr, tid, kTailThreads);
        filter_pairs(z, log2M, plan, twr, H, tid, kTailThreads);
        fft_inverse(z, log2M, plan, twr, tid, kTailThreads);
      }
      // ---------------- onto the observed pixels (edges clamp), continuum polynomial, chi2
      double acc = 0.0;
      {
        const double* lamc = lam;
        auto lamf = [lamc](int k) { return lamc[k]; };
        const float* zc = zf;
        auto convf = [zc](int k) { return (double)zc[zidx(k)]; };
        for (int j = off + tid; j < off + no; j += kTailThreads) {
          double m = 1.0 + np_interp(__ldg(P.obs_w + j), lamf, convf, nx);
          if (P.n_poly) m *= chebval_dev(__ldg(P.obs_x + j), S.poly, P.n_poly);
          if (P.model_out) P.model_out[(long long)p * P.ld_flux + j - off] = m;
          const double r = m * __ldg(P.obs_inv_s + j) - __ldg(P.obs_ot + j);
          acc += r * r;
        }
      }
      double c2 = cta_sum(acc, red, tid);
      if (tid == 0 && P.lnl) {
        if (P.chi2_sed) c2 += P.chi2_sed[p];
        P.lnl[p] = -0.5 * c2;
      }
      __syncthreads();
    }
  } else {
    // ---------------- stage 1: rotational broadening of the row in place (as tail_general.cuh)
    auto rotate = [&](float* row, bool is_depth) {
      const int N1 = 1 << P.log2N1, log2M = P.log2N1 - 1;
      for (int k = tid; k < N1; k += kTailThreads) {
        const int2 e = __ldg(P.fwd1 + k);
        const float t = __int_as_float(e.y);
        const float a = depth_of(row[e.x], is_depth, true), b = depth_of(row[e.x + 1], is_depth, true);
        zf[zidx(k)] = a + t * (b - a);
      }
      __syncthreads();
      RotH H{P.sbtab, nullptr, 0, S.vsini_scale, P.sb_h, 1.0f / (float)(1 << log2M), P.ntab, RotH::fix40(S.vsini_scale)};
      FftPlan plan; plan.make(log2M);
      fft_forward(z, log2M, plan, twr, tid, kTailThreads);
      filter_pairs(z, log2M, plan, twr, H, tid, kTailThreads);
      fft_inverse(z, log2M, plan, twr, tid, kTailThreads);
      for (int i = tid; i < n; i += kTailThreads) {
        if (i == 0 || i == n - 1) continue;
        const int2 e = __ldg(P.back1 + i);
        const float t = __int_as_float(e.y);
        const float g0 = zf[zidx(e.x)], g1 = zf[zidx(e.x + 1)];
        const float v = g0 + t * (g1 - g0);
        row[i] = v;
        if (i == 1) row[0] = v;
        if (i == n - 2) row[n - 1] = v;
      }
      __syncthreads();
    };

    // ---------------- everything after stage 1, against the star of S / so and the mask [i0, i0 + nM): this thread's
    // share of chi2 in acc; false when the transform size is out of range (status bit 0 above log2nx_max).  The model
    // pixels go to mrow[0, so.n).
    auto lsf_star = [&](const float* row, bool is_depth, int i0, int nM, double* mrow, double& acc) -> bool {
      const double D = S.D;
      const int off = so.off, no = so.n;
      // ---------------- dw / sigma on the masked, shifted emulator grid
      const double* w = P.w + i0;
      const double* ow = P.obs_w + off;
      const double* lsf = L.lsf + off;
      auto wave = [w, D](int i) { return __ldg(w + i) * D; };
      auto owf = [ow](int j) { return __ldg(ow + j); };
      auto lsff = [lsf](int j) { return __ldg(lsf + j); };
      for (int i = tid; i < nM; i += kTailThreads) {
        const double disp = np_interp(wave(i), owf, lsff, no);
        const double dw = i == 0 ? wave(1) - wave(0)
                                 : (i == nM - 1 ? wave(nM - 1) - wave(nM - 2) : (wave(i + 1) - wave(i - 1)) / 2.0);
        aux[i] = dw / disp;
      }
      __syncthreads();
      // ---------------- cdf = cumsum / max: every thread sums a contiguous chunk, offsets by a serial pass
      const int chunk = (nM + kTailThreads - 1) / kTailThreads;
      const int c0 = min(tid * chunk, nM), c1 = min(c0 + chunk, nM);
      {
        double s = 0.0;
        for (int i = c0; i < c1; ++i) s += aux[i];
        part[tid] = s;
      }
      __syncthreads();
      if (tid == 0) {
        double run = 0.0;
        for (int t = 0; t < kTailThreads; ++t) { const double v = part[t]; part[t] = run; run += v; }
      }
      __syncthreads();
      {
        double s = part[tid];
        for (int i = c0; i < c1; ++i) { s += aux[i]; cdf[i] = s; }
      }
      __syncthreads();
      const double total = cdf[nM - 1];
      __syncthreads();
      for (int i = tid; i < nM; i += kTailThreads) cdf[i] = cdf[i] / total;
      __syncthreads();
      // ---------------- x_per_sigma = nanmedian(gradient(cdf) / (dw / sigma))
      for (int i = tid; i < nM; i += kTailThreads) {
        const double g = i == 0 ? cdf[1] - cdf[0]
                                : (i == nM - 1 ? cdf[nM - 1] - cdf[nM - 2] : (cdf[i + 1] - cdf[i - 1]) / 2.0);
        aux[i] = g / aux[i];
      }
      __syncthreads();
      const double* auxc = aux;
      const double xps = nanmedian_dev([auxc](int j) { return auxc[j]; }, nM, hist, &sh_prefix, &sh_rank, &sh_count);
      const double Nf = 2.0 / xps;                                    // pix_per_sigma = 2
      const int log2nx = (Nf == Nf && Nf > 0.0 && Nf < 1e9) ? (int)ceil(log2(Nf)) : -1;
      if (log2nx < 1 || log2nx > L.log2nx_max) {               // nx = 1: the reference's irfft raises (DESIGN §5)
        if (tid == 0 && log2nx > L.log2nx_max) atomicOr(P.status, 1);
        if (mrow)
          for (int j = tid; j < no; j += kTailThreads) mrow[j] = nan;
        return false;
      }
      const int nx = 1 << log2nx;
      // ---------------- even grid in the cdf coordinate, spectrum on it
      {
        const double step = 1.0 / (double)(nx - 1);                   // np.linspace(0, 1, nx)
        const double* cdfc = cdf;
        auto cdff = [cdfc](int j) { return cdfc[j]; };
        const float* rowm = row + i0;
        auto specf = [rowm, is_depth](int j) { return (double)depth_of(rowm[j], is_depth, true); };
        for (int k = tid; k < nx; k += kTailThreads) {
          const double x = k == nx - 1 ? 1.0 : (double)k * step;
          const double lk = np_interp(x, cdff, wave, nM);
          lam[k] = lk;
          zf[zidx(k)] = (float)np_interp(lk, wave, specf, nM);
        }
      }
      __syncthreads();
      if (log2nx < 5) {
        lsf_small_conv(zf, nx, xps, part, tid);
      } else {
        const int log2M = log2nx - 1;
        const float a = (float)(2.0 * CUDART_PI * CUDART_PI * xps * xps);   // ss = rfftfreq(nx, 1/nx) = k
        GaussH H{a, 1.0f / (float)(1 << log2M)};
        FftPlan plan; plan.make(log2M);
        fft_forward(z, log2M, plan, twr, tid, kTailThreads);
        filter_pairs(z, log2M, plan, twr, H, tid, kTailThreads);
        fft_inverse(z, log2M, plan, twr, tid, kTailThreads);
      }
      // ---------------- onto the observed pixels (edges clamp), continuum polynomial, chi2
      {
        const double* lamc = lam;
        auto lamf = [lamc](int k) { return lamc[k]; };
        const float* zc = zf;
        auto convf = [zc](int k) { return (double)zc[zidx(k)]; };
        for (int j = off + tid; j < off + no; j += kTailThreads) {
          double m = 1.0 + np_interp(__ldg(P.obs_w + j), lamf, convf, nx);
          if (P.n_poly) m *= chebval_dev(__ldg(P.obs_x + j), S.poly, P.n_poly);
          if (mrow) mrow[j - off] = m;
          const double r = m * __ldg(P.obs_inv_s + j) - __ldg(P.obs_ot + j);
          acc += r * r;
        }
      }
      return true;
    };

    for (int p = blockIdx.x; p < P.B; p += gridDim.x) {
      const double* th = P.theta + (long long)p * P.ld;
      float* row = P.flux + (long long)p * P.ldf;
      double* mrow = P.model_out ? P.model_out + (long long)p * P.ld_flux : nullptr;
      const int t = __ldg(P.target + p);
      const bool valid = t >= 0 && t < P.n_targets;
      const int k0 = valid ? __ldg(P.tfirst + t) : -1;
      const int K = valid ? __ldg(P.tfirst + t + 1) - k0 : 1;
      int off0 = 0;
      bool is_depth = P.flux_is_depth != 0, rotated = false;
      double tot = 0.0;                                  // thread 0: chi2 of members 0 .. m, summed in that order
      for (int m = 0; m < K; ++m) {
        if (tid == 0) {
          tail_setup_star(P, th, valid ? k0 + m : -1, S, so);   // an invalid target: status bit 2, no pixels
          int2 r = make_int2(n, -1);
          if (!S.bad) r = lsf_mask(P, P.stars[k0 + m], S.D);
          sh_i0 = r.x; sh_i1 = r.y;
        }
        __syncthreads();
        if (m == 0) off0 = so.off;
        const int i0 = sh_i0, nM = sh_i1 - i0 + 1;
        double* mrow_m = mrow ? mrow + (so.off - off0) : nullptr;
        double acc = 0.0;
        bool ok = !(S.bad || nM < 17);
        if (ok) {
          if (S.do_rot && !rotated) {
            rotate(row, is_depth);
            rotated = is_depth = true;
          }
          ok = lsf_star(row, is_depth, i0, nM, mrow_m, acc);
        } else if (mrow_m) {
          for (int j = tid; j < so.n; j += kTailThreads) mrow_m[j] = nan;
        }
        double c2 = cta_sum(acc, red, tid);              // (its barrier also frees S, so and the scratch)
        if (tid == 0) {
          if (!ok) c2 = nan;
          if (valid && P.chi2_out) P.chi2_out[(long long)p * P.ld_chi2 + m] = c2;
          tot = m == 0 ? c2 : tot + c2;
        }
      }
      if (tid == 0 && P.lnl) {
        if (P.chi2_sed) tot += P.chi2_sed[p];
        P.lnl[p] = -0.5 * tot;
      }
      __syncthreads();
    }
  }
}

}  // namespace payne
