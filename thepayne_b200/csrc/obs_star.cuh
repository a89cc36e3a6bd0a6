// Per-star record of a context's observation set (payne_ctx_create_stars).  A context holds the observations of
// S stars back to back in one set of device arrays; every point of a batch names its star, and every consumer of
// the observation resolves that star's record once per point and then reads its slice [off, off + n_obs).
// A single-star context is the case S = 1 (record 0 covers the whole arrays).
#pragma once

namespace payne {

struct ObsStar {
  int off, n_obs;              // first observed pixel in the concatenated arrays, number of pixels
  double obs_min, obs_max;     // wavelength range (mask limits of the instrumental stage)
  int sorted;                  // wavelengths finite and non-decreasing (cluster tail: pixel ranges per CTA)
  int phot_off;                // first of this star's nb magnitudes / errors
};

// star index of batch point p (null array: star 0), or -1 when outside [0, n_stars)
__device__ __forceinline__ int star_of(const int* star, int n_stars, int p) {
  const int k = star ? star[p] : 0;
  return (k >= 0 && k < n_stars) ? k : -1;
}

}  // namespace payne
