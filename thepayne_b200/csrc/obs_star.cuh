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

// Per-star parameter layout (PayneStarOpts.layout): where star k's parameters sit in its own theta row.  The records
// [n_stars] are uploaded only when some star of the set gives a layout (a star without one gets the context layout's
// record); without them the pointer is null and every consumer reads its own copy of the context layout.
struct StarLayout {
  int col[PAYNE_NPAR];            // column in theta, -1: not sampled (star_fixed)
  int n_poly;                     // pc_k coefficients (0 without a continuum polynomial)
  int poly_col[PAYNE_MAX_POLY];
  int photscale;                  // photscale_bool
};

// Parameter `which` of theta row th of star k: the column of star k's layout when the context has per-star layouts,
// ctx_col (the consumer's copy of the context layout) otherwise.  Where that column is -1: star k's own value when the
// context has per-star fixed values (star_fixed [n_stars, PAYNE_NPAR]), ctx_fixed otherwise.  k < 0 (no such star --
// every consumer turns such a point into NaN anyway -- or a label beyond PAYNE_P_*): the context's column and value.
__device__ __forceinline__ double param_of(const StarLayout* star_lay, int ctx_col, double ctx_fixed,
                                           const double* star_fixed, const double* th, int k, int which) {
  const int c = (star_lay && k >= 0) ? star_lay[k].col[which] : ctx_col;
  if (c >= 0) return th[c];
  return (star_fixed && k >= 0) ? star_fixed[(long long)k * PAYNE_NPAR + which] : ctx_fixed;
}

// Parameter `which` of a binary's secondary (payne_ctx_set_binary) in theta row th: its own column, else its own fixed
// value when that is not NaN, else `prim`, the primary's value (param_of).  bin null (no binary): prim.
__device__ __forceinline__ double secondary_of(const PayneBinary* bin, const double* th, int which, double prim) {
  if (!bin || which < 0) return prim;
  const int c = bin->col[which];
  if (c >= 0) return th[c];
  const double f = bin->fixed[which];
  return f == f ? f : prim;
}

// Continuum coefficients of theta row th of star k into poly[]; returns their number.
__device__ __forceinline__ int poly_of(const StarLayout* star_lay, int ctx_n_poly, const int* ctx_poly_col,
                                       const double* th, int k, double* poly) {
  const bool own = star_lay && k >= 0;
  const int n = own ? star_lay[k].n_poly : ctx_n_poly;
  for (int i = 0; i < n; ++i) poly[i] = th[own ? star_lay[k].poly_col[i] : ctx_poly_col[i]];
  return n;
}

// star index of batch point p (null array: star 0), or -1 when outside [0, n_stars)
__device__ __forceinline__ int star_of(const int* star, int n_stars, int p) {
  const int k = star ? star[p] : 0;
  return (k >= 0 && k < n_stars) ? k : -1;
}

}  // namespace payne
