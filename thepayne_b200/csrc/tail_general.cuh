// General-grid fused tail: any strictly increasing emulator wavelength grid.  Same chain as
// tail_fast.cuh; the regrids use exact np.interp tables (stage 1) and fp64 searches on w[]
// (stage 2, fallback) instead of the analytic weights of the log-uniform fast path.
#pragma once
#include "fft_ct.cuh"
#include "tail.cuh"

namespace payne {

// FFT convolution of 2^log2N real samples held in shared memory: compile-time-planned transform for
// the sizes this instantiation is built around, runtime-planned otherwise.
template <int LOG2N1, class HF>
__device__ __forceinline__ void convolve_any(float2* z, int log2N, const TwTab& tw, const TwConst& tc, const HF& H,
                                             int tid) {
  constexpr int LA = LOG2N1 > 15 ? 15 : LOG2N1;       // largest all-in-smem transform
  if (log2N == LA) {
    ct_convolve<LA - 1>(z, tw, tc, H, tid);
  } else if (LA >= 10 && log2N == LA - 1) {
    ct_convolve<(LA >= 10 ? LA - 2 : 8)>(z, tw, tc, H, tid);
  } else {
    const Twiddles twr{tw.tab, tw.log2n};
    FftPlan plan; plan.make(log2N - 1);
    fft_forward(z, log2N - 1, plan, twr, tid, kNT);
    filter_pairs(z, log2N - 1, plan, twr, H, tid, kNT);
    fft_inverse(z, log2N - 1, plan, twr, tid, kNT);
  }
}

template <int LOG2N1>
__global__ void __launch_bounds__(kTailThreads, LOG2N1 <= 14 ? 3 : 1)
tail_general_kernel(const __grid_constant__ TailParams P, const __grid_constant__ TwConst TC) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* z = reinterpret_cast<float2*>(smem_raw);
  float* zf = reinterpret_cast<float*>(smem_raw);
  __shared__ PointSetup S;
  __shared__ ObsSlice SL;
  __shared__ double red[kTailThreads / 32];
  const int tid = threadIdx.x;
  const TwTab tw{P.tw, P.log2tw, P.twpass};
  const double nan = CUDART_NAN;

  for (int p = blockIdx.x; p < P.B; p += gridDim.x) {
    const double* th = P.theta + (long long)p * P.ld;
    float* row = P.flux + (long long)p * P.ldf;
    if (tid == 0) tail_setup(P, th, p, S, SL);
    __syncthreads();
    if (S.bad) {
      model_nan(P, p, 0, SL.n, tid);
      if (tid == 0 && P.lnl) P.lnl[p] = nan;
      __syncthreads();
      continue;
    }
    bool is_depth = P.flux_is_depth != 0;

    // ---------------- stage 1: rotational broadening on the full emulator grid
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
      convolve_any<LOG2N1>(z, P.log2N1, tw, TC, H, tid);
      // back onto the emulator grid + the edge patch of predictspec.py:240-241
      const int n = P.n;
      for (int i = tid; i < n; i += kTailThreads) {
        if (i == 0 || i == n - 1) continue;
        const int2 e = __ldg(P.back1 + i);
        const float t = __int_as_float(e.y);
        const float g0 = zf[zidx(e.x)], g1 = zf[zidx(e.x + 1)];
        const float v = g0 + t * (g1 - g0);      // t = NaN marks "outside" (smoothing.py:313-314)
        row[i] = v;
        if (i == 1) row[0] = v;
        if (i == n - 2) row[n - 1] = v;
      }
      is_depth = true;
      __syncthreads();
    }

    double acc = 0.0;
    if (S.use_inst) {
      // ---------------- stage 2: mask, regrid, Gaussian broadening
      const int N2 = 1 << S.log2N2, log2M = S.log2N2 - 1;
      const int i0 = S.i0, i1 = S.i1;
      double xt = exp(S.u0t + S.du * (double)tid);   // rest-frame grid point
      for (int k = tid; k < N2; k += kTailThreads, xt *= S.rho) {
        int j = locate(P.w, 1.0, xt, i0 + (int)((double)k * S.rM), i0, i1 - 1);
        double t = (xt - __ldg(P.w + j)) * __ldg(P.inv_dw + j);
        t = fmin(fmax(t, 0.0), 1.0);
        const float a = depth_of(row[j], is_depth, true), b = depth_of(row[j + 1], is_depth, true);
        zf[zidx(k)] = a + (float)t * (b - a);
      }
      __syncthreads();
      GaussH H{S.taper_a, 1.0f / (float)(1 << log2M)};
      convolve_any<LOG2N1>(z, S.log2N2, tw, TC, H, tid);
      // ---------------- onto the observed pixels, continuum, chi2
      const double pmax = (double)(N2 - 1);
      const int off = SL.off, jend = off + SL.n;            // the point's star
      for (int j = off + tid; j < jend; j += kTailThreads) {
        const double pp = (__ldg(P.obs_lnw + j) - S.u0) * S.inv_du;
        double m;
        if (!(pp >= 0.0 && pp <= pmax)) m = nan;            // smoothing.py:289 left/right = nan
        else {
          const int k = min((int)pp, N2 - 2);
          const float dl = (float)(pp - (double)k);
          const float t = dl * (1.f + (dl - 1.f) * S.hdu);   // (e^{dl du}-1)/(e^{du}-1) to O(du^2)
          const float g0 = zf[zidx(k)], g1 = zf[zidx(k + 1)];
          m = 1.0 + (double)(g0 + t * (g1 - g0));
        }
        if (P.n_poly) m *= chebval_dev(__ldg(P.obs_x + j), S.poly, P.n_poly);
        if (P.model_out) P.model_out[(long long)p * P.ld_flux + (j - off)] = m;
        const double r = m * (double)__ldg(P.obs_inv_s + j) - __ldg(P.obs_ot + j);
        acc += r * r;
      }
    } else {
      // ---------------- no instrumental profile: plain np.interp (predictspec.py:288-289)
      const int n = P.n;
      const double wlo = __ldg(P.w) * S.D, whi = __ldg(P.w + n - 1) * S.D;
      const int off = SL.off, jend = off + SL.n;
      for (int j = off + tid; j < jend; j += kTailThreads) {
        const double x = __ldg(P.obs_w + j);
        double m;
        if (!(x >= wlo && x <= whi)) m = nan;
        else {
          const int g = (int)((__ldg(P.obs_lnw + j) - S.lnD - P.lnw0) * P.inv_dlnw);
          const int jj = locate(P.w, S.D, x, g, 0, n - 2);
          const double wa = __ldg(P.w + jj) * S.D, wb = __ldg(P.w + jj + 1) * S.D;
          const double a = (double)depth_of(row[jj], is_depth, false);
          const double b = (double)depth_of(row[jj + 1], is_depth, false);
          m = 1.0 + np_interp_pair(x, wa, wb, a, b);
        }
        if (P.n_poly) m *= chebval_dev(__ldg(P.obs_x + j), S.poly, P.n_poly);
        if (P.model_out) P.model_out[(long long)p * P.ld_flux + (j - off)] = m;
        const double r = m * (double)__ldg(P.obs_inv_s + j) - __ldg(P.obs_ot + j);
        acc += r * r;
      }
    }
    // ---------------- block reduction -> one lnL per live point (likelihood.py:117)
    double c2 = cta_sum(acc, red, tid);
    if (tid == 0 && P.lnl) {
      if (P.chi2_sed) c2 += P.chi2_sed[p];
      P.lnl[p] = -0.5 * c2;
    }
    __syncthreads();
  }
}

}  // namespace payne
