// Per-star record of a context's observation set (payne_ctx_create_stars).  A context holds the observations of
// S stars back to back in one set of device arrays; every point of a batch names its star, and every consumer of
// the observation resolves that star's record once per point and then reads its slice [off, off + n_obs).
// A single-star context is the case S = 1 (record 0 covers the whole arrays).
#pragma once
#include "../../include/payne_b200.h"

namespace payne {

struct ObsStar {
  int off, n_obs;              // first observed pixel in the concatenated arrays, number of pixels
  double obs_min, obs_max;     // wavelength range (mask limits of the instrumental stage)
  int sorted;                  // wavelengths finite and non-decreasing (cluster tail: pixel ranges per CTA)
  int phot_off;                // first of this star's nb magnitudes / errors
  int nb;                      // number of this star's magnitudes (the photometry net's nb unless given a band list)
};

// PAYNE_P_* parameter behind emulator label i (Teff, log(g), [Fe/H], [a/Fe], Vmic), -1 for a label beyond those
__host__ __device__ constexpr int label_param(int i) {
  return i == 0 ? PAYNE_P_TEFF : i == 1 ? PAYNE_P_LOGG : i == 2 ? PAYNE_P_FEH : i == 3 ? PAYNE_P_AFE
       : i == 4 ? PAYNE_P_VMIC : -1;
}

// Value of a parameter the layout does not sample (col < 0): star k's own value when the context was created with
// per-star fixed values (star_fixed [n_stars, PAYNE_NPAR]), the layout's otherwise.  k < 0 (no such star): the
// layout's; every consumer turns such a point into NaN anyway.
__device__ __forceinline__ double fixed_of(const double* star_fixed, const double* fixed, int k, int which) {
  return (star_fixed && k >= 0) ? star_fixed[(long long)k * PAYNE_NPAR + which] : fixed[which];
}

// star index of batch point p (null array: star 0), or -1 when outside [0, n_stars)
__device__ __forceinline__ int star_of(const int* star, int n_stars, int p) {
  const int k = star ? star[p] : 0;
  return (k >= 0 && k < n_stars) ? k : -1;
}

}  // namespace payne
