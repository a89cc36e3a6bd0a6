/*
 * payne_b200.h -- C ABI of the B200-native batched likelihood path of The Payne.
 *
 * The reference (pacargile/ThePayne) is pure Python and has no FFI layer; the boundary it
 * exposes for this path is a set of Python method signatures.  Each entry point below
 * names the reference interface it replaces (paths relative to the reference checkout):
 *
 *   payne_ctx_create        likelihood.__init__            Payne/fitting/likelihood.py:7-40
 *                           GenMod._initspecnn/_initphotnn Payne/fitting/genmod.py:15-43
 *                           ANN.__init__ / readNN          Payne/predict/predictspec.py:31-59,
 *                                                          Payne/train/NNmodels.py:44-89
 *                           fastANN.__init__               Payne/predict/photANN.py:97-116
 *   payne_lnlike_batch      likelihood.lnlikefn + lnlike   Payne/fitting/likelihood.py:42-117
 *   payne_lnlike_batch_host same, host buffers in/out (what dynesty hands over)
 *   payne_model_batch       GenMod.genspec / genphot(_scaled)  Payne/fitting/genmod.py:58-187
 *                           PayneSpecPredict.getspec       Payne/predict/predictspec.py:136-294
 *                           FastPayneSEDPredict.sed        Payne/predict/predictsed.py:75-103
 *   payne_ann_eval          ANN.eval / LinNet.forward      Payne/predict/predictspec.py:61-74,
 *                                                          Payne/train/NNmodels.py:154-168
 *   payne_ctx_attach_continuum  PayneSpecPredict(Cnnpath=...) / predictcont + the continuum multiply of getspec
 *                                                          Payne/predict/predictspec.py:96-102,122-134,208-226
 *   payne_ctx_set_lsf       getspec(inst_R=<vector>)       Payne/predict/predictspec.py:265-286 ->
 *                           smoothspec(smoothtype='lsf')   Payne/utils/smoothing.py:126-150,482-586
 *   payne_ctx_create_stars, payne_*_stars   one context for the observations of many stars that share the
 *                           emulators and the parameter layout (likelihood.__init__ per star; a survey fits
 *                           thousands of stars with one emulator): every point of a batch names its star.
 *   payne_ctx_create_stars_opts  the same with each star's own fixed parameter values (fitstar.py:193-198 per star),
 *                           photometric bands (likelihood.py:109-112 over the star's obs_phot), LSF vector and
 *                           parameter layout (fitstar.py:50-65, 202-207 per star).
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a
 * negative PAYNE_E_* code and never throws; payne_last_error() gives the message of the
 * last failure on the calling thread.  "dev" pointers are CUDA device pointers on the
 * context's device, owned by the caller; the context owns only its copies of the network
 * weights, the observation and its workspaces.  Calls are stream-ordered on `stream`
 * (a cudaStream_t passed as void*, NULL = legacy default stream) and do not synchronise,
 * except the *_host entry which returns with the results in host memory.  One context
 * per device; distinct contexts may be used from distinct threads concurrently.
 *
 * NaN semantics follow the reference: NaN is returned (never an error) for observed
 * pixels outside the emulator's coverage (smoothing.py:289), for a requested resolution
 * finer than the emulator's (smoothing.py:271) and for NaN inputs.
 */
#ifndef PAYNE_B200_H
#define PAYNE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PAYNE_ABI_VERSION 8

enum {
  PAYNE_OK = 0,
  PAYNE_E_INVALID = -1,   /* bad argument / unsupported shape */
  PAYNE_E_CUDA = -2,      /* CUDA runtime / driver error */
  PAYNE_E_NOMEM = -3,
  PAYNE_E_UNSUPPORTED = -4
};

/* Named parameters of the sampler vector, in the order of fitstar.fitpars
 * (Payne/fitting/fitstar.py:50-65).  pc_k continuum coefficients are listed separately. */
enum {
  PAYNE_P_TEFF = 0, PAYNE_P_LOGG, PAYNE_P_FEH, PAYNE_P_AFE, PAYNE_P_VRAD, PAYNE_P_VROT,
  PAYNE_P_VMIC, PAYNE_P_INSTR, PAYNE_P_LOGR, PAYNE_P_DIST, PAYNE_P_LOGA, PAYNE_P_AV,
  PAYNE_P_RV, PAYNE_NPAR
};
#define PAYNE_MAX_POLY 16

/* MLP arithmetic.  PARITY reproduces the reference's fp32 Linear layers on the tensor cores
 * with an exact-accumulation split (three 8-bit fixed-point bf16 slices per operand, six bf16
 * MMAs per product, fp32 accumulate in TMEM; see csrc/mlp_tc.cuh).  3XTF32 is the classic
 * error-compensated TF32 split (kept for comparison: its accumulator truncation bias costs
 * ~1e-2 in lnL).  TF32 trades accuracy for speed and does NOT meet the 1e-5 / 1e-3 parity bar
 * (reported separately).  SIMT_FP32 is a plain CUDA-core fp32 FMA implementation kept as an
 * on-device cross-check.  BF16 is reserved. */
enum {
  PAYNE_PREC_PARITY = 0,
  PAYNE_PREC_TF32 = 1,
  PAYNE_PREC_BF16 = 2,
  PAYNE_PREC_SIMT_FP32 = 3,
  PAYNE_PREC_3XTF32 = 4
};

/* Spectrum emulator; HOST pointers, copied at create.  W[k] is layer k's weight, row-major
 * [out,in] fp32; b[k] its bias.  Layer widths follow from n_layers:
 *   6 (or 0): LinNet  D_in-H1-H1-H2-H2-H3-D_out, sigmoid          (NNmodels.py:140-168)
 *   4       : SMLP    D_in-H1-H2-H3-D_out,      leaky ReLU 0.01   (NNmodels.py:92-115)
 *   3       : YST1    D_in-H1-H2-D_out,         leaky ReLU 0.01   (predict/ystpred.py:18-58)
 *   4 + SIGMOID + n_groups >= 1 : multi-chunk emulator, n_groups nets Net(D_in,H1,P) of four sigmoid-sigmoid-
 *             sigmoid-linear layers each covering group_size consecutive pixels (Payne/train/old/
 *             trainspec_multi.py:29-52); W[0] = [n_groups,H1,D_in], W[1], W[2] = [n_groups,H1,H1], W[3] =
 *             [D_out,H1] (the chunks' output layers one after another), biases alike; H2 = H3 = H1;
 *             encode_offset 0 (trainspec_multi.py:56-67).
 * The leaky-ReLU stacks keep their (narrow) hidden layers on the CUDA-core fp32 kernels; in PARITY mode their wide
 * output layer -- nearly all of their flops -- runs on the tensor cores with row-scaled operand slices (activations
 * divided by the power of two above the row maximum; contraction width <= 512), SIMT_FP32 keeps everything on CUDA cores. */
enum { PAYNE_ACT_SIGMOID = 0, PAYNE_ACT_LEAKY_RELU = 1 };
typedef struct {
  int32_t D_in, H1, H2, H3, D_out;
  const float* W[6];
  const float* b[6];
  const double* xmin;        /* [D_in] */
  const double* xmax;        /* [D_in] */
  const double* wavelength;  /* [D_out], strictly increasing */
  double resolution;         /* sigma-R of the emulator grid (predictspec.py:49) */
  double encode_offset;      /* 0.5 for every reference net (NNmodels.py:166, ystpred.py:49) */
  int32_t n_layers;          /* 0 = 6 */
  int32_t activation;        /* PAYNE_ACT_* ; must be LEAKY_RELU for 3/4 layers, SIGMOID for 6 */
  int32_t label_fp32_cast;   /* 1: labels pass through fp32 first (ANN.eval, predictspec.py:70); 0: fp64 (ystpred.py:47-50) */
  int32_t n_groups;          /* multi-chunk emulator: number of chunk nets (0 or 1 = one monolithic net) */
  int32_t group_size;        /* pixels per chunk net; the last one may be narrower (trainspec_multi.py:242-243) */
  int32_t reserved_;
} PayneSpecNet;

/* Photometry emulator: stacked per-band Net(6,H,1) (photANN.py:97-106); HOST pointers. */
typedef struct {
  int32_t nb, H;
  const float *w1, *b1;      /* [nb,H,6], [nb,H]  */
  const float *w2, *b2;      /* [nb,H,H], [nb,H]  */
  const float *w3, *b3;      /* [nb,H],   [nb]    */
  const double *xmin, *xmax; /* [6] */
  const double *hiav;        /* [nb,5] a1,b1,a2,b2,c2 (highred.py:10-25), NaN if absent */
} PaynePhotNet;

/* Observation (fitargs of likelihood.py:84-112); HOST pointers, copied at create. */
typedef struct {
  int32_t n_obs;
  const double *wave, *flux, *eflux;   /* [n_obs]; wave increasing */
  int32_t nb;
  const double *phot_mag, *phot_err;   /* [nb] */
} PayneObs;

/* How a row of theta maps onto named parameters (likelihood.py:42-72). */
typedef struct {
  int32_t ndim;
  int32_t col[PAYNE_NPAR];        /* column in theta, or -1 if not sampled */
  double  fixed[PAYNE_NPAR];      /* value used when col<0; NaN = absent (likelihood.py:51-55) */
  int32_t n_poly;                 /* number of pc_k coefficients (0 = no continuum polynomial) */
  int32_t poly_col[PAYNE_MAX_POLY];
  int32_t spec_bool, phot_bool, modpoly_bool, photscale_bool;  /* runbools, fitstar.py:202-207 */
  int32_t precision;              /* PAYNE_PREC_* */
} PayneLayout;

typedef struct PayneCtx PayneCtx;

int payne_abi_version(void);
const char* payne_last_error(void);

/* spec / phot may be NULL when the corresponding runbool is 0. device = CUDA ordinal.
 * Same as payne_ctx_create_stars(spec, phot, obs, 1, layout, device, out). */
int payne_ctx_create(const PayneSpecNet* spec, const PaynePhotNet* phot, const PayneObs* obs,
                     const PayneLayout* layout, int device, PayneCtx** out);

/* Observation set: obs is an array of n_stars PayneObs, HOST pointers, copied.  Every star must have the same nb
 * (= phot->nb when phot_bool; payne_ctx_create_stars_opts lifts this with band lists).  Star k keeps its own n_obs, wavelength range, sort order and Chebyshev
 * normalisation (polycalc on its own wave, fitutils.py:13-14).  The emulators, the parameter layout and every table
 * built from the emulator grid are shared.  A single-star context is the case n_stars = 1.
 * On a context of several stars, payne_ctx_set_lsf (the LSF vector is per observed pixel) and payne_gather_create
 * (the fused all-gather has no star argument) return PAYNE_E_UNSUPPORTED; payne_ctx_attach_continuum works. */
int payne_ctx_create_stars(const PayneSpecNet* spec, const PaynePhotNet* phot, const PayneObs* obs,
                           int32_t n_stars, const PayneLayout* layout, int device, PayneCtx** out);

/* What may differ between the stars of an observation set besides the observation itself; HOST pointers, copied. */
typedef struct {
  const double*  fixed;  /* [PAYNE_NPAR] or NULL (= layout->fixed): this star's values of the parameters the layout
                            does not sample (col < 0); NaN = absent, as in PayneLayout */
  const int32_t* band;   /* [PayneObs.nb] or NULL: photometry-net band of each of this star's magnitudes, in PayneObs
                            order, distinct, in [0, phot->nb); NULL = net order (then PayneObs.nb == phot->nb) */
  const double*  lsf;    /* [PayneObs.n_obs] or NULL: dispersion (AA) at every observed pixel, as payne_ctx_set_lsf */
  const PayneLayout* layout;  /* or NULL (= the context layout): this star's own parameter layout (ABI 8) */
} PayneStarOpts;

/* payne_ctx_create_stars with per-star options: opts is an array of n_stars PayneStarOpts or NULL
 * (payne_ctx_create_stars = this with opts NULL; a star whose fields are all NULL is a star of that call).
 *   fixed: star k's row replaces the layout's fixed values everywhere they are read (emulator labels, Vrad, Vrot,
 *          Inst_R, the photometry parameters).
 *   band:  PayneObs.nb may differ between stars.  A star's SED chi2 is summed over its own bands in its PayneObs
 *          order; payne_model_batch_stars writes row p's magnitudes in that order into columns [0, nb_k) of the
 *          [B, phot->nb] output and leaves the other columns unwritten.  Out of range, duplicated or too many
 *          entries: PAYNE_E_INVALID.
 *   lsf:   given for every star or for none (a mix is PAYNE_E_UNSUPPORTED: the LSF tail and the scalar-R tails are
 *          different kernels); every vector is checked as payne_ctx_set_lsf checks one, and while the vectors are set
 *          Inst_R is ignored.  The vectors are fixed at creation: payne_ctx_set_lsf still refuses several stars.
 *   layout: the star's own ndim, col[], fixed[], n_poly, poly_col[], photscale_bool and phot_bool: its free parameters,
 *          their order in its theta row, its continuum order and its photometry may differ from the other stars'.
 *          fixed[] is the star's fixed values (giving `fixed` too is PAYNE_E_INVALID).  phot_bool 0: the star has no
 *          magnitudes (PayneObs.nb must be 0) and its SED chi2 is 0.  PAYNE_E_INVALID: a col or poly_col outside
 *          [0, ndim) or used twice (col -1 = not sampled), n_poly above PAYNE_MAX_POLY, spec_bool or precision other
 *          than the context layout's, nothing to fit, photometry in a context whose layout has phot_bool 0.
 *          PAYNE_E_UNSUPPORTED: stars with and without a continuum polynomial (modpoly_bool with n_poly >= 1) in one
 *          set -- the polynomial and the plain final pass round differently, so such a star would not get the bits of
 *          its single-star context; n_poly >= 1 may differ.  Every star's polynomial is evaluated to the set's largest
 *          order, its own coefficients followed by zeros (exact at finite abscissae): PAYNE_E_UNSUPPORTED as well for a
 *          star below that order whose Chebyshev abscissae are not finite (n_obs = 1 or all its wavelengths equal).  A star without a layout has the context layout.  In the
 *          batch entries ld must be at least the largest ndim (context layout's and the stars'); row p reads columns
 *          [0, ndim) of its star only. */
int payne_ctx_create_stars_opts(const PayneSpecNet* spec, const PaynePhotNet* phot, const PayneObs* obs,
                                const PayneStarOpts* opts, int32_t n_stars, const PayneLayout* layout, int device,
                                PayneCtx** out);
void payne_ctx_destroy(PayneCtx* ctx);

/* theta_dev: [B, ld] fp64 row-major on the device, ld >= ndim (with per-star layouts: the largest).  lnl_dev: [B] fp64.
 * star_dev: [B] int32 on the device, the star of every row of theta; NULL = star 0 for every row, which a context of
 * several stars refuses (PAYNE_E_INVALID).  A row whose star lies outside [0, n_stars) cannot be checked without a
 * synchronise: it gets lnL NaN, no model row and sets status bit 2; the other rows are not affected.
 * payne_lnlike_batch = payne_lnlike_batch_stars with star_dev = NULL. */
int payne_lnlike_batch(PayneCtx* ctx, const double* theta_dev, int64_t B, int64_t ld,
                       double* lnl_dev, void* stream);
int payne_lnlike_batch_stars(PayneCtx* ctx, const double* theta_dev, const int32_t* star_dev, int64_t B, int64_t ld,
                             double* lnl_dev, void* stream);

/* Same with HOST buffers: copies theta (and star) in, runs, copies lnL out, synchronises.  A star index outside
 * [0, n_stars) returns PAYNE_E_INVALID before anything is launched or written. */
int payne_lnlike_batch_host(PayneCtx* ctx, const double* theta_host, int64_t B, int64_t ld,
                            double* lnl_host);
int payne_lnlike_batch_stars_host(PayneCtx* ctx, const double* theta_host, const int32_t* star_host, int64_t B,
                                  int64_t ld, double* lnl_host);

/* Model spectrum on the observed grid and magnitudes; either output may be NULL.
 * flux_dev: [B, n_obs] fp64, mags_dev: [B, nb] fp64, lnl_dev: [B] fp64 or NULL.
 * _stars: flux_dev: [B, ld_flux], ld_flux >= the largest n_obs; row p gets the first n_obs[star[p]] entries, the
 * rest are not written.  payne_model_batch = payne_model_batch_stars with star_dev = NULL, ld_flux = n_obs. */
int payne_model_batch(PayneCtx* ctx, const double* theta_dev, int64_t B, int64_t ld,
                      double* flux_dev, double* mags_dev, double* lnl_dev, void* stream);
int payne_model_batch_stars(PayneCtx* ctx, const double* theta_dev, const int32_t* star_dev, int64_t B, int64_t ld,
                            double* flux_dev, int64_t ld_flux, double* mags_dev, double* lnl_dev, void* stream);

/* Targets: stars observed in several spectra (echelle orders, spectrograph arms, epochs).  A target is a run of
 * consecutive stars of the observation set, its members, that describe one physical star: target t holds the stars
 * [first[t], first[t+1]).  first[n_targets + 1] (HOST, copied) must start at 0, increase strictly and end at n_stars;
 * NULL removes the targets.  A point of the _targets entries names a target, and is evaluated as
 *   the emulator row (and the continuum emulator) once, from the first member's labels;
 *   rotational broadening once;
 *   for every member m in order: Doppler shift, mask, instrumental broadening, resampling on m's pixels, m's continuum
 *     polynomial, chi2_m -- each chi2_m has the bits of -2 lnL of a single-star context of star m without photometry;
 *   the SED chi2 once, from the first member's magnitudes;
 *   lnL = -0.5 * ((((chi2_0 + chi2_1) + ...) + chi2_{K-1}) + chi2_sed).
 * Members may differ in Vrad, Inst_R (column or fixed value) or LSF vector, pixels and continuum order.  With LSF vectors
 * (PayneStarOpts.lsf) the instrumental stage of every member is its own vector's; the emulator grid need not be uniform
 * in ln wavelength then.  At set time PAYNE_E_INVALID: members that resolve Teff, log(g), [Fe/H], [a/Fe], Vmic or Vrot
 * to different columns or fixed values; magnitudes on a member other than the first; with LSF vectors, a member whose
 * Inst_R is a theta column (nothing reads it beside the vector).  PAYNE_E_UNSUPPORTED: without LSF vectors, a context
 * without the fast tail (emulator grid not uniform in ln wavelength); a context with the fused gather.  A one-star
 * context may switch its LSF vector on or off afterwards (payne_ctx_set_lsf); the _targets entries then check these
 * rules again.  The entries without _targets keep naming stars.  A target outside [0, n_targets): PAYNE_E_INVALID from
 * the _host entry before anything is launched; on the device lnL NaN, no model row or chi2, status bit 2.  A member that
 * is bad by itself (e.g. Inst_R above the emulator's resolution, a mask of fewer than 17 emulator pixels, or an LSF
 * transform above 32768 samples: status bit 0) makes lnL NaN; the other members' model rows and chi2 keep their values.
 * ld >= the largest ndim.  Without LSF vectors, per-(point, member) records bound a slab to
 * min(max_batch, 65536 / the largest member count) points. */
int payne_ctx_set_targets(PayneCtx* ctx, const int32_t* first, int32_t n_targets);
int payne_lnlike_batch_targets(PayneCtx* ctx, const double* theta_dev, const int32_t* target_dev, int64_t B, int64_t ld,
                               double* lnl_dev, void* stream);
int payne_lnlike_batch_targets_host(PayneCtx* ctx, const double* theta_host, const int32_t* target_host, int64_t B,
                                    int64_t ld, double* lnl_host);
/* flux_dev [B, ld_flux]: row p holds the members' model spectra back to back in member order (ld_flux >= the largest
 * target's pixel count); chi2_dev [B, ld_chi2]: chi2_dev[p, m] = chi2_m (ld_chi2 >= the largest member count); mags_dev
 * [B, nb]: the first member's magnitudes.  Any output may be NULL. */
int payne_model_batch_targets(PayneCtx* ctx, const double* theta_dev, const int32_t* target_dev, int64_t B, int64_t ld,
                              double* flux_dev, int64_t ld_flux, double* chi2_dev, int64_t ld_chi2, double* mags_dev,
                              double* lnl_dev, void* stream);

/* Double-lined binaries: one observed spectrum modelled as the flux-weighted sum of two stars.  Component 1 (the
 * primary) has the parameters of the layout, as everywhere else.  Component 2 (the secondary) resolves each of Teff,
 * log(g), [Fe/H], [a/Fe], Vmic, Vrad and Vrot to col[P] (a theta column) if col[P] >= 0, else to fixed[P] if that is
 * not NaN, else to the primary's value.  Inst_R and the continuum polynomial are shared.  Rratio = R_sec / R_pri is
 * theta column rratio_col, or rratio_fixed when rratio_col < 0.  Per observed pixel j (wavelength lambda_j):
 *   a_c[j]  component c's model before the continuum (1 + line depth after rotation, Doppler shift, instrumental
 *           stage or plain interpolation, resampling; NaN where the single-star model is NaN);
 *   k_j     = Rratio^2 * expm1(c2 / (lambda_j Teff_1)) / expm1(c2 / (lambda_j Teff_2)), c2 = 1.438776877e8 AA K
 *           (both stars radiate as blackbodies of radius R);
 *   m_j     = (a_1[j] + k_j a_2[j]) / (1 + k_j), times the continuum polynomial when the layout has one;
 * chi2 and lnL as for one star.  With Rratio = 0 and a finite a_2, m and lnL have the bits of the primary alone
 * through payne_model_batch_stars.  A component that is bad by itself makes lnL and the model NaN. */
typedef struct {
  int32_t col[PAYNE_NPAR];   /* secondary's theta column, -1: not sampled */
  double  fixed[PAYNE_NPAR]; /* secondary's fixed value where col < 0; NaN: the primary's value */
  int32_t rratio_col;        /* Rratio's theta column, -1: rratio_fixed */
  double  rratio_fixed;
} PayneBinary;

/* Sets the binary description (HOST pointer, copied); NULL removes it.  PAYNE_E_INVALID: a column or non-NaN fixed
 * value on a parameter other than the seven above, a column outside [0, ndim), Rratio neither sampled nor fixed to a
 * finite value.  PAYNE_E_UNSUPPORTED, here and again in every _binary entry: photometry (phot_bool), LSF vectors, an
 * attached continuum emulator, targets, per-star layouts (PayneStarOpts.layout), the fused gather, and contexts without
 * the fast tail (emulator grid not uniform in ln wavelength).  Per-star fixed values apply to the shared parameters.
 * The entries without _binary are unchanged by it.  Every point runs both components' emulator rows in one pass of the
 * emulator, so a slab holds max_batch / 2 points. */
int payne_ctx_set_binary(PayneCtx* ctx, const PayneBinary* binary);
/* star_dev: [B] int32 or NULL (star 0), as in the _stars entries (a star outside [0, n_stars): lnL NaN, status bit 2;
 * the _host entry returns PAYNE_E_INVALID before launching). */
int payne_lnlike_batch_binary(PayneCtx* ctx, const double* theta_dev, const int32_t* star_dev, int64_t B, int64_t ld,
                              double* lnl_dev, void* stream);
int payne_lnlike_batch_binary_host(PayneCtx* ctx, const double* theta_host, const int32_t* star_host, int64_t B,
                                   int64_t ld, double* lnl_host);
/* flux_dev [B, ld_flux]: m; comp_dev [B, 2, ld_flux]: a_1 and a_2 (ld_flux >= the largest n_obs); lnl_dev [B].  Any
 * output may be NULL; row p gets the first n_obs of its star, the rest is not written. */
int payne_model_batch_binary(PayneCtx* ctx, const double* theta_dev, const int32_t* star_dev, int64_t B, int64_t ld,
                             double* flux_dev, int64_t ld_flux, double* comp_dev, double* lnl_dev, void* stream);

/* Continuum marginalisation: the Chebyshev continuum of a star's model, m_j = a_j * sum_k c_k T_k(x_j), is linear in
 * its K coefficients, so chi2 is an exact quadratic in c and the coefficients can be integrated out per point instead
 * of being sampled (K fewer dimensions for the sampler per spectrum).  Per star with the setting, over its pixels j:
 *   a_j     the model before the continuum (1 + depth after rotation, Doppler shift, instrumental stage or plain
 *           interpolation, resampling; NaN where the sampled model is NaN); x_j its Chebyshev abscissa;
 *   b_jk    = a_j T_k(x_j) / sigma_j,  y_j = flux_j / sigma_j;
 *   G       = sum_j b_j b_j^T = L L^T (Cholesky),  h = sum_j b_j y_j,  c-hat = G^-1 h, all in fp64;
 *   Q       = chi2 at c-hat, with the bits of -2 lnL of a context that samples pc_0 .. pc_{K-1} (no photometry) at
 *           theta with c-hat appended;
 *   M       = -sum_k ln L_kk + sum_k (ln(2 pi) / 2 - ln(hi_k - lo_k));
 *   lnL     = -0.5 (Q + chi2_sed) + M, the log of the integral of exp(-chi2(c) / 2) prod_k dc_k / (hi_k - lo_k) over R^K
 *           (equal to the box integral when the box holds the coefficients' conditional posterior; not truncated).
 * A target (payne_ctx_set_targets) of n members: lnL = -0.5 ((((Q_0 + Q_1) + ...) + Q_{n-1}) + chi2_sed) +
 * ((M_0 + M_1) + ...) + M_{n-1}.  Any NaN a_j makes lnL NaN.  A finite G with a pivot at or below 1e-10 of its
 * diagonal entry (fewer usable pixels than K, all a_j zero) makes lnL, c-hat, Q and the model NaN and sets status bit 3.
 * While the setting is on, every likelihood and model entry (plain, _stars, _targets, their _host twins) returns this
 * lnL and the model at c-hat. */
typedef struct {
  int32_t n_coef;                /* K in [1, PAYNE_MAX_POLY]; 0: the star has no setting */
  double lo[PAYNE_MAX_POLY];     /* the coefficients' box: its widths enter M */
  double hi[PAYNE_MAX_POLY];
} PayneContMarg;

/* per_star [n_stars] (HOST, copied); NULL removes the setting.  PAYNE_E_INVALID: a star with the setting whose layout
 * also samples pc_k (modpoly_bool with n_poly > 0), n_coef outside [0, PAYNE_MAX_POLY] or 0 for every star, a
 * non-finite box or lo >= hi.  PAYNE_E_UNSUPPORTED: some stars with the setting and others without, LSF vectors, a
 * binary, an attached continuum emulator, a grid without the fast tail, the fused gather.  Every entry checks these
 * rules again (the context may change in between).  Transforms of 65536 samples run on the single-CTA kernel. */
int payne_ctx_set_cont_marg(PayneCtx* ctx, const PayneContMarg* per_star);
/* Per point p (all outputs device pointers, any may be NULL): coef_dev[p, :K] c-hat, chol_dev[p, :K(K+1)/2] L as packed
 * lower triangle (row by row: L00, L10, L11, L20, ...), chi2_dev[p] Q, lnl_dev[p] lnL.  ld_coef >= the largest K,
 * ld_chol >= the largest K(K+1)/2.  star_dev as in the _stars entries. */
int payne_cont_batch_stars(PayneCtx* ctx, const double* theta_dev, const int32_t* star_dev, int64_t B, int64_t ld,
                           double* coef_dev, int64_t ld_coef, double* chol_dev, int64_t ld_chol,
                           double* chi2_dev, double* lnl_dev, void* stream);
/* The same for targets: the members' c-hat and L lie back to back in member order (ld_coef >= the largest sum of the
 * members' K, ld_chol likewise), chi2_dev[p, m] = Q_m (ld_chi2 >= the largest member count). */
int payne_cont_batch_targets(PayneCtx* ctx, const double* theta_dev, const int32_t* target_dev, int64_t B, int64_t ld,
                             double* coef_dev, int64_t ld_coef, double* chol_dev, int64_t ld_chol,
                             double* chi2_dev, int64_t ld_chi2, double* lnl_dev, void* stream);

/* Continuum emulator (HOST pointers, copied): any PayneSpecNet the spectrum emulator could be; its
 * `wavelength` is the continuum's own grid.  From then on every model spectrum is multiplied, right after
 * the emulator and before any broadening, by np.interp(modwave, contwave, c / nanmedian(c), left=nan,
 * right=nan) with c = F_nu -> F_lambda of the continuum net's output (predictspec.py:208-226).  Attaching
 * again replaces the previous one.  Not reachable from the likelihood (it never passes Cnnpath). */
int payne_ctx_attach_continuum(PayneCtx* ctx, const PayneSpecNet* cont);

/* LSF vector: lsf_host[n_obs] = dispersion (sigma, in AA) at every observed pixel.  While set, the
 * instrumental stage is smooth_lsf_fft (smoothing.py:482-586) instead of the scalar-R Gaussian and the
 * Inst_R parameter is ignored; observed pixels outside the emulator's coverage take the edge value (the
 * reference's np.interp clamps there) instead of NaN.  NULL switches back.  Emulator grids up to 32768
 * pixels; a point whose cdf grid would need more than 32768 samples returns NaN and sets status bit 0.
 * Targets (payne_ctx_set_targets) run with LSF vectors too, see there. */
int payne_ctx_set_lsf(PayneCtx* ctx, const double* lsf_host, int64_t n);

/* Emulator forward pass only.  x_dev: [B, D_in] fp64 labels; y_dev: [B, ldy] fp32, ldy>=D_out.
 * Tensor-core precisions write y with TMA stores: y_dev 16-byte aligned, ldy a multiple of 4. */
int payne_ann_eval(PayneCtx* ctx, const double* x_dev, int64_t B, float* y_dev, int64_t ldy,
                   void* stream);

/* Multi-GPU: all-gather of lnL over peer memory (one process per GPU on one node; replaces the ncclAllGather behind
 * every step of the sharded likelihood, thepayne_b200/dist.py).  Every rank holds three rotating buffers of
 * world * slots doubles.  payne_gather_create allocates them and writes PAYNE_GATHER_HANDLE_BYTES of CUDA IPC handles to
 * handles_out; the ranks exchange those bytes (any transport: the Python side uses torch.distributed's all_gather_object)
 * and pass the concatenation, in rank order, to payne_gather_connect, which maps the peers' buffers (NVLink P2P).
 * payne_lnlike_batch_gather = payne_lnlike_batch of this rank's B = slots points with the all-gather fused into the tail
 * kernel: the thread that writes a point's lnL also stores it into every rank's buffer (plain stores through the peer
 * mappings), and the last CTA of the kernel raises this rank's flag on every rank behind a system-scope fence (tails
 * without the hook -- general grid, LSF, photometry only -- are followed by one small push kernel doing the same);
 * stream-ordered, no host synchronisation, every rank must call it the same number of times.
 * PAYNE_GATHER_FUSED=0 (environment): always the separate push kernel.
 * *gathered_prev receives the device pointer of the complete gathered vector [world * slots] of the PREVIOUS call (NULL on
 * the first): it is valid for work enqueued on `stream` after this call and must be consumed before the next call.
 * payne_gather_flush enqueues the wait for the last step and returns its vector.  A peer that never arrives sets
 * status bit 1 after ~10 s instead of hanging the device. */
#define PAYNE_GATHER_HANDLE_BYTES 128
int payne_gather_create(PayneCtx* ctx, int world, int rank, int64_t slots, void* handles_out);
int payne_gather_connect(PayneCtx* ctx, const void* all_handles);
int payne_lnlike_batch_gather(PayneCtx* ctx, const double* theta_dev, int64_t B, int64_t ld, void* stream,
                              double** gathered_prev);
int payne_gather_flush(PayneCtx* ctx, void* stream, double** gathered_last);

/* Introspection for benches/tests: key is one of "n_ann","n_obs" (the largest star's),"n_stars","n_obs_total"
 * (observed pixels of all stars),"n_targets","binary" (1 while a PayneBinary is set),"nfft1","launches",
 * "grid_loguniform","fast_tail","max_batch","sm_count","tail_grid","precision","continuum","lsf","legacy_tc"
 * (a leaky-ReLU stack whose output layer runs on the tensor cores),"status"
 * (bit0: a point needed a larger transform than the shared-memory carve-out; bit1: a peer of the gather never arrived;
 * bit2: a point named a star outside [0, n_stars), or a target outside [0, n_targets); bit3: continuum marginalisation
 * met a finite Gram matrix with a pivot at or below 1e-10 of its diagonal entry), "cont_marg" (1 while payne_ctx_set_cont_marg is on).
 * Returns the value or -1. */
int64_t payne_ctx_query(PayneCtx* ctx, const char* key);
/* Runtime switches: "precision" (PAYNE_PREC_*), "max_batch" (workspace slab, points), "timing" (0/1,
 * see payne_ctx_last_ms), "fast_tail" (0 forces the general-grid tail), "gemm_stack" (0: one launch per hidden layer instead of
 * one cluster launch for lin2..lin5; bit-identical), "tail_cluster" (transforms above
 * 16384 samples spread over a cluster of four CTAs: default 1 for 65536-sample transforms, 0 for 32768).
 * Environment, read once: PAYNE_TAIL_CLUSTER=0 (never use the cluster tail) / 1 (also for 32768-sample transforms), PAYNE_ROT_WINDOW=0 (no shared-memory slice of the rotation-kernel table),
 * PAYNE_GEMM_PDL=0 (no programmatic dependent launch along the layer chain), PAYNE_GEMM_STACK=0 (see "gemm_stack"). */
int payne_ctx_set(PayneCtx* ctx, const char* key, int64_t value);

/* Kernel unit-test hook: C[M,N] = A[M,K] . W[N,K]^T + bias[N] through the tensor-core GEMM of
 * the given PAYNE_PREC_* mode, HOST buffers in and out (A must lie in [0,1) for PARITY, like
 * the sigmoid activations it is built for).  Synchronous. */
int payne_gemm_test(const float* A_host, const float* W_host, const float* bias_host, int M, int N, int K,
                    int precision, int device, float* C_host);

/* Kernel unit-test hook: y = irfft(rfft(x) * H) through the runtime-planned shared-memory FFT convolution of
 * the fused tails (csrc/fft.cuh), one CTA.  x, y: N = 2^log2N real samples, log2N in [5, 15]; H: the N/2 + 1
 * real transfer-function values at frequencies 0 .. N/2 (the hook applies the 1/(N/2) of the inverse).
 * HOST buffers in and out.  Synchronous. */
int payne_fft_test(const float* x_host, int log2N, const float* H_host, int device, float* y_host);

/* Per-kernel device time of the most recent payne_lnlike_batch call on this context,
 * measured with CUDA events on the launching stream when timing is enabled
 * (payne_ctx_set(ctx,"timing",1)).  which: 0 = emulator GEMM stages, 1 = fused tail,
 * 2 = photometry.  Returns milliseconds, or a negative value if unavailable. */
double payne_ctx_last_ms(PayneCtx* ctx, int which);

#ifdef __cplusplus
}
#endif
#endif /* PAYNE_B200_H */
