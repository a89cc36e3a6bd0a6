// Photometric SED emulator + SED chi2 for a batch of live points (fp64, like the reference's
// numpy path: fp32 weights up-cast against fp64 activations).
//
//   Payne/predict/photANN.py:118-131    fastANN.encode / eval: (x-xmin)/(xmax-xmin) (no -0.5),
//                                       a1 = s(W1 x + b1), a2 = s(W2 a1 + b2), y = W3 a2 + b3
//   Payne/predict/predictsed.py:75-103  sed(): Av < 5 -> BC = ANN(x); else high-Av extension
//   Payne/predict/highred.py:19-25      BC0 - (a1 + b1 Av (a2 + b2 Rv + c2 Rv^2))
//   Payne/fitting/genmod.py:110-187     genphot (logR, Dist) / genphot_scaled (logA); Rv = 3.1
//   Payne/fitting/likelihood.py:109-112 SED chi2
//
// A CTA evaluates kPhotTile points against every band so each weight is loaded once per tile.
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include "../../include/payne_b200.h"
#include "obs_star.cuh"

namespace payne {

constexpr int kPhotTile = 8;
constexpr int kPhotThreads = 128;

struct PhotParams {
  int nb, H;
  const float *w1, *b1, *w2t, *b2, *w3, *b3;   // w2t[b][h_in][h_out] (transposed on the host)
  double xmin[6], xmax[6];
  const double* hiav;        // [nb,5]
  const double *obs_mag, *obs_err;   // [n_stars, nb]
  int col[PAYNE_NPAR];
  double fixed[PAYNE_NPAR];
  int photscale;
  const double* theta;
  long long ld;
  double* chi2_sed;          // [B] or null
  double* mags_out;          // [B, nb] or null
  int B;
  // observation set (obs_star.cuh): star of every point of this slab (null: star 0); a point whose star lies outside
  // [0, n_stars) gets chi2 NaN, no magnitudes row, and status bit 2
  const int* star;
  const ObsStar* stars;
  int n_stars;
  int* status;
  // Per-star options (payne_ctx_create_stars_opts), null without them:
  const double* star_fixed;  // [n_stars, PAYNE_NPAR] star k's values where col < 0
  // [n_stars, nb] slot of net band b among star k's magnitudes (its PayneObs order), -1 if it has none in that band.
  // With it, a point's terms are stored per slot and summed in slot order at the end, so that its chi2 has the order
  // a single-star context of that star's bands gives; mags_out row p gets its magnitudes in slots [0, nb_k).
  const int* band_slot;
  const StarLayout* star_lay;   // [n_stars] per-star layouts (columns, photscale), null without them; a star without
                                // photometry has no slots (band_slot row all -1)
};

__device__ __forceinline__ double phot_par(const PhotParams& P, const double* th, int which, int k) {
  return param_of(P.star_lay, P.col[which], P.fixed[which], P.star_fixed, th, k, which);
}
__device__ __forceinline__ double sigmoid_d(double a) { return 1.0 / (1.0 + exp(-a)); }

// SLOTS: P.band_slot is set (the kernel without it is the one of contexts without band lists)
template <bool SLOTS>
__global__ void __launch_bounds__(kPhotThreads)
phot_kernel(const __grid_constant__ PhotParams P) {
  extern __shared__ double sm[];
  const int H = P.H;
  double* a1 = sm;                       // [tile][H]
  double* a2 = sm + kPhotTile * H;       // [tile][H]
  double* term = a2 + kPhotTile * H;     // [tile][nb] per-slot chi2 terms (band_slot only)
  __shared__ double zin[kPhotTile][6];
  __shared__ double aux[kPhotTile][4];   // logt, av, rv(for hiav), scale term
  __shared__ double chi[kPhotTile];
  __shared__ int moff[kPhotTile];        // the point's star: first of its magnitudes (-1: no such star)
  __shared__ int kst[kPhotTile];         // the point's star (band_slot only)
  __shared__ int slot[kPhotTile];        // band b's slot among the point's magnitudes, -1: none (band_slot only)
  const int tid = threadIdx.x;
  const int p0 = blockIdx.x * kPhotTile;
  const double log10_tsun = log10(5770.0);

  if (tid < kPhotTile) {
    const int p = p0 + tid;
    chi[tid] = 0.0;
    if (p < P.B) {
      const int k = star_of(P.star, P.n_stars, p);
      moff[tid] = k < 0 ? -1 : P.stars[k].phot_off;
      kst[tid] = k;
      if (k < 0) { chi[tid] = CUDART_NAN; atomicOr(P.status, 4); }
      const double* th = P.theta + (long long)p * P.ld;
      const double teff = phot_par(P, th, PAYNE_P_TEFF, k);
      const double logt = log10(teff);
      double av = phot_par(P, th, PAYNE_P_AV, k);
      const double rv = 3.1;                                   // likelihood.py:103-106 never frees Rv
      const bool hi = !(av < 5.0);                             // predictsed.py:86
      double x[6] = {pow(10.0, logt), phot_par(P, th, PAYNE_P_LOGG, k), phot_par(P, th, PAYNE_P_FEH, k),
                     phot_par(P, th, PAYNE_P_AFE, k), hi ? 0.0 : av, hi ? 3.1 : rv};
      for (int i = 0; i < 6; ++i) zin[tid][i] = (x[i] - P.xmin[i]) / (P.xmax[i] - P.xmin[i]);
      aux[tid][0] = logt; aux[tid][1] = av; aux[tid][2] = hi ? 1.0 : 0.0;
      double base;
      if ((P.star_lay && k >= 0) ? P.star_lay[k].photscale : P.photscale) {
        base = 5.0 * phot_par(P, th, PAYNE_P_LOGA, k) - 10.0 * (logt - log10_tsun) - 0.26;   // predictsed.py:96
      } else {
        const double logl = 2.0 * phot_par(P, th, PAYNE_P_LOGR, k) + 4.0 * (logt - log10_tsun);   // genmod.py:128
        const double mu = 5.0 * log10(phot_par(P, th, PAYNE_P_DIST, k)) - 5.0;
        base = -2.5 * logl + 4.74 + mu;                          // predictsed.py:93-94 (BC subtracted below)
      }
      aux[tid][3] = base;
    }
  }
  __syncthreads();

  for (int b = 0; b < P.nb; ++b) {
    if (SLOTS) {
      // a band no point of the tile has is skipped (CTA-uniform: every thread reads the same slots)
      if (tid < kPhotTile) slot[tid] = (p0 + tid < P.B && kst[tid] >= 0) ? P.band_slot[kst[tid] * P.nb + b] : -1;
      __syncthreads();
      bool any = false;
#pragma unroll
      for (int q = 0; q < kPhotTile; ++q) any |= slot[q] >= 0;
      __syncthreads();                   // every thread has its answer before a skipped band's successor rewrites slot
      if (!any) continue;
    }
    const float* w1 = P.w1 + (long long)b * H * 6;
    const float* w2t = P.w2t + (long long)b * H * H;
    for (int h = tid; h < H; h += kPhotThreads) {
      double w[6];
      for (int i = 0; i < 6; ++i) w[i] = (double)__ldg(w1 + h * 6 + i);
      const double bb = (double)__ldg(P.b1 + b * H + h);
      for (int q = 0; q < kPhotTile; ++q) {
        double s = 0.0;
        for (int i = 0; i < 6; ++i) s += w[i] * zin[q][i];
        a1[q * H + h] = sigmoid_d(s + bb);
      }
    }
    __syncthreads();
    for (int h = tid; h < H; h += kPhotThreads) {
      double acc[kPhotTile];
#pragma unroll
      for (int q = 0; q < kPhotTile; ++q) acc[q] = 0.0;
      for (int hi = 0; hi < H; ++hi) {
        const double wv = (double)__ldg(w2t + (long long)hi * H + h);
#pragma unroll
        for (int q = 0; q < kPhotTile; ++q) acc[q] += wv * a1[q * H + hi];
      }
      const double bb = (double)__ldg(P.b2 + b * H + h);
#pragma unroll
      for (int q = 0; q < kPhotTile; ++q) a2[q * H + h] = sigmoid_d(acc[q] + bb);
    }
    __syncthreads();
    // output layer: one warp per point (round-robin)
    const int warp = tid >> 5, lane = tid & 31;
    for (int q = warp; q < kPhotTile; q += kPhotThreads / 32) {
      double s = 0.0;
      for (int h = lane; h < H; h += 32) s += (double)__ldg(P.w3 + b * H + h) * a2[q * H + h];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      const int p = p0 + q;
      if (lane == 0 && p < P.B && moff[q] >= 0 && (!SLOTS || slot[q] >= 0)) {
        double BC = s + (double)__ldg(P.b3 + b);
        if (aux[q][2] != 0.0) {                                  // highred.py:19-25
          const double* c = P.hiav + b * 5;
          const double av = aux[q][1], rv = 3.1;
          BC = BC - (c[0] + c[1] * av * (c[2] + c[3] * rv + c[4] * (rv * rv)));
        }
        const double m = aux[q][3] - BC;
        if (SLOTS) {
          const int sl = slot[q];
          if (P.mags_out) P.mags_out[(long long)p * P.nb + sl] = m;
          const double d = m - P.obs_mag[moff[q] + sl], e = P.obs_err[moff[q] + sl];
          term[q * P.nb + sl] = (d * d) / (e * e);
        } else {
          if (P.mags_out) P.mags_out[(long long)p * P.nb + b] = m;
          const double d = m - P.obs_mag[moff[q] + b], e = P.obs_err[moff[q] + b];
          chi[q] += (d * d) / (e * e);
        }
      }
    }
    __syncthreads();
  }
  if (SLOTS && tid < kPhotTile && p0 + tid < P.B && moff[tid] >= 0) {
    // the point's terms in its own band order (likelihood.py:109-112 enumerates obs_phot)
    const int nbk = P.stars[kst[tid]].nb;
    for (int sl = 0; sl < nbk; ++sl) chi[tid] += term[tid * P.nb + sl];
  }
  if (tid < kPhotTile && p0 + tid < P.B && P.chi2_sed) P.chi2_sed[p0 + tid] = chi[tid];
}

// lnL when there is no spectrum: -0.5 * chi2_sed
__global__ void lnl_from_sed_kernel(const double* __restrict__ chi2_sed, double* __restrict__ lnl, int B) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) lnl[i] = -0.5 * chi2_sed[i];
}

}  // namespace payne
