// C-ABI implementation: context creation (weights + per-dataset tables to HBM) and the
// stream-ordered launch sequence  encode+lin1 -> lin2..lin6 -> photometry -> fused tail.
// See include/payne_b200.h for the contract and the reference interfaces each entry replaces.
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <limits>
#include <string>
#include <utility>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/payne_b200.h"
#include "launchers.h"
#include "phot.cuh"
#include "continuum.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CU_TRY(expr)                                                                     \
  do {                                                                                   \
    cudaError_t e__ = (expr);                                                            \
    if (e__ != cudaSuccess)                                                              \
      return fail(PAYNE_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));   \
  } while (0)

template <class T>
int upload(T** dst, const T* src, size_t n) {
  *dst = nullptr;
  if (n == 0) return PAYNE_OK;
  CU_TRY(cudaMalloc((void**)dst, n * sizeof(T)));
  CU_TRY(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
  return PAYNE_OK;
}

inline int ceil_log2(long long v) {
  int l = 0;
  while ((1LL << l) < v) ++l;
  return l;
}

// np.linspace(a, b, n)
std::vector<double> linspace(double a, double b, int n) {
  std::vector<double> y(n);
  const double step = (b - a) / (double)(n - 1);
  for (int i = 0; i < n; ++i) y[i] = (double)i * step + a;
  y[n - 1] = b;
  return y;
}

// np.interp index/weight of x in the increasing grid xp (value = fp[j] + t (fp[j+1]-fp[j])).
// outside: clamp (left=fp[0], right=fp[-1]) or NaN weight when nan_outside.
void interp_entry(const std::vector<double>& xp, double x, bool nan_outside, int* j, float* t) {
  const int n = (int)xp.size();
  if (x < xp[0] || x > xp[n - 1]) {
    if (nan_outside) { *j = 0; *t = std::numeric_limits<float>::quiet_NaN(); return; }
    if (x < xp[0]) { *j = 0; *t = 0.f; } else { *j = n - 2; *t = 1.f; }
    return;
  }
  if (x == xp[n - 1]) { *j = n - 2; *t = 1.f; return; }
  int k = (int)(std::upper_bound(xp.begin(), xp.end(), x) - xp.begin()) - 1;   // xp[k] <= x < xp[k+1]
  k = std::min(std::max(k, 0), n - 2);
  *j = k;
  *t = (float)((x - xp[k]) / (xp[k + 1] - xp[k]));
}

// exp(i a) rounded to floats with the modulus as close to 1 as the float grid allows: among the
// neighbouring floats of cos a and sin a pick the pair minimising | |W|^2 - 1 |.  Plain rounding
// leaves a table whose mean |W|^2 - 1 is a few 1e-9 negative; every element meets ~6 twiddles
// per transform pair, so that becomes a coherent -1.4e-8 amplitude loss per convolution.
float2 unit_round(double a) {
  const double c = std::cos(a), s = std::sin(a);
  const float cf = (float)c, sf = (float)s;
  const float cc[3] = {cf, std::nextafter(cf, INFINITY), std::nextafter(cf, -INFINITY)};
  const float ss[3] = {sf, std::nextafter(sf, INFINITY), std::nextafter(sf, -INFINITY)};
  const double uc = std::fabs((double)std::nextafter(std::fabs(cf), INFINITY) - std::fabs((double)cf));
  const double us = std::fabs((double)std::nextafter(std::fabs(sf), INFINITY) - std::fabs((double)sf));
  float bc = cf, bs = sf;
  double best = std::fabs((double)cf * cf + (double)sf * sf - 1.0);
  for (float x : cc)
    for (float y : ss) {
      if (std::fabs((double)x - c) > uc || std::fabs((double)y - s) > us) continue;
      const double e = std::fabs((double)x * x + (double)y * y - 1.0);
      if (e < best) { best = e; bc = x; bs = y; }
    }
  return make_float2(bc, bs);
}

// sb(u) of smoothing.py:612-619 without the small-u cancellation
double rot_sb(double u) {
  u = std::fabs(u);
  if (u < 0.5) {
    // J1(u)/u = sum (-1)^m (u/2)^(2m) / (2 m! (m+1)!),  (3/(2u^2))(sin u/u - cos u) = 1.5 sum (-1)^(m+1) 2m u^(2m-2)/(2m+1)!
    double a = 0.0, q = u * u, term1 = 0.5, term2 = 0.5;
    // term1_m = (-1)^m (q/4)^m / (2 m!(m+1)!), term2_m = 1.5 (-1)^m (2m+2) q^m / (2m+3)!
    for (int m = 0; m < 12; ++m) {
      a += term1 + term2;
      term1 *= -(q / 4.0) / ((double)(m + 1) * (double)(m + 2));
      term2 *= -q * (double)(2 * m + 4) / ((double)(2 * m + 2) * (double)(2 * m + 4) * (double)(2 * m + 5));
    }
    return a;
  }
  return j1(u) / u - 3.0 * std::cos(u) / (2.0 * u * u) + 3.0 * std::sin(u) / (2.0 * u * u * u);
}

}  // namespace

struct PayneCtx {
  int device = 0, sm_count = 0;
  cudaStream_t stream = nullptr;   // used by the *_host entry
  int n_layers = 6;
  bool legacy = false;             // leaky-ReLU stack (SMLP / YST1): hidden layers on the CUDA-core fp32 kernels
  bool legacy_tc = false;          // ... and the wide output layer on the tensor cores (row-scaled slices, parity mode)
  float* rscale = nullptr;         // [slab] per-row scale of that layer's operand (workspace)
  // multi-chunk emulator (trainspec_multi.py:29-52): n_groups sigmoid nets of 4 layers, `chunk` pixels each
  bool multinet = false;
  int n_groups = 1, chunk = 0;
  long long rows_per_group = 0;    // rows of one group's block in the activation planes (workspace)
  payne::TcMapCache mapc[6];       // tensor maps per layer, valid while the workspace stays put
  payne::TcStackCache stackc;      // ... and of the hidden-layer stack (one launch for lin2..lin5)
  bool use_stack = true;           // PAYNE_GEMM_STACK=0 / payne_ctx_set("gemm_stack", 0): one launch per hidden layer
  cudaStream_t side = nullptr;     // per-point tail setup runs here, beside the emulator GEMMs
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaEvent_t ev_done = nullptr;   // end of the last call that used the workspace
  cudaStream_t last_stream = nullptr;
  bool has_last = false;
  PayneLayout lay{};
  // spectrum emulator
  bool has_spec = false;
  int D_in = 0, H[4] = {0, 0, 0, 0}, D_out = 0;   // H[0]=H1 (lin1,lin2 out), H[1]=H2, H[2]=H3
  int dims_in[6], dims_out[6];
  float* W[6] = {nullptr};
  float* b[6] = {nullptr};
  payne::TcWeights tcw[6];
  payne::EncodeParams enc{};
  payne::TailParams tail{};
  payne::FastGrid fast{};
  size_t tail_smem = 0;
  size_t fast_smem = 0;      // tail_smem + rotation-table window (fast kernels)
  int tail_grid = 0;
  int fast_grid[4] = {0, 0, 0, 0};   // CTAs of the fast tail of every payne::FastForm (form_grid), 0 until probed
  int grid_loguniform = 0;
  int use_fast = 0;        // analytic-regrid tail selected (log-uniform emulator grid)
  int allow_fast = 1;
  // cluster-distributed fast tail (tail_cluster.cuh) for transforms above 16384 samples
  int grid_cap = 0;        // > 0: at most this many CTAs (clusters) in the persistent tail grids (tests: forces the
                           // dynamic point scheduling to hand several points to every CTA of a small batch)
  int use_cluster = 0, allow_cluster = 1;
  size_t cluster_smem = 0;
  int cluster_win_floats = 0, cluster_n = 0, cluster_occ = 0;
  // continuum emulator (predictspec.py:96-102, 208-226): a second emulator context (weights, operand
  // planes, its own output rows) and the per-dataset tables of the multiply
  PayneCtx* cont = nullptr;
  payne::ContParams contp{};
  // LSF vector (predictspec.py:265-286): replaces the scalar-R stage of the tail
  bool lsf_on = false;
  payne::LsfParams lsf{};
  size_t lsf_smem = 0;
  int lsf_grid = 0;
  // observation set: n_stars observations back to back in the tail's and photometry's arrays (obs_star.cuh)
  int n_stars = 1, n_obs_max = 0;
  long long n_obs_total = 0;
  std::vector<payne::ObsStar> stars;    // host copy of the records
  payne::ObsStar* stars_dev = nullptr;
  double* star_fixed_dev = nullptr;     // [n_stars, PAYNE_NPAR] per-star fixed values (payne_ctx_create_stars_opts), or null
  payne::StarLayout* star_lay_dev = nullptr;   // [n_stars] per-star layouts (PayneStarOpts.layout), or null
  int ndim_max = 0;                     // the largest ndim of the context layout and the stars' layouts
  std::vector<double> star_fixed_h;     // host copies of star_fixed_dev / star_lay_dev (empty without them)
  std::vector<payne::StarLayout> star_lay_h;
  // targets (payne_ctx_set_targets): runs of consecutive stars that describe one physical star
  int n_targets = 0, tgt_kmax = 0;
  bool tgt_lsf_probed = false;          // the LSF target kernel's shared-memory opt-in is set
  std::string tgt_instr_col;            // the first member with an Inst_R column (refused beside LSF vectors), or empty
  long long tgt_nobs_max = 0;           // the largest sum of the members' n_obs (model row of a target)
  int* tfirst_dev = nullptr;            // [n_targets + 1]
  std::vector<int> tfirst_h;            // its host copy
  // per-mode buffers (resize_buffer; *_n: elements allocated)
  payne::FastPoint* tgt_points = nullptr;   // [rows * tgt_kmax] per-(point, member) records of a slab (fast tail only)
  int* tgt_star = nullptr;              // [rows] first member's star of every point of a slab
  double* bin_par = nullptr;            // [rows, 3] Teff_1, Teff_2, Rratio of the points of a slab (binaries)
  double* aj_scratch = nullptr;         // [grid, n_obs_max] a_j of every CTA's current point (binaries or continuum
                                        // marginalisation, which never go together; grid: that form's)
  long long tgt_points_n = 0, tgt_star_n = 0, bin_par_n = 0, aj_scratch_n = 0;
  // binaries (payne_ctx_set_binary): the secondary's description
  bool has_binary = false;
  PayneBinary* binary_dev = nullptr;
  // continuum marginalisation (payne_ctx_set_cont_marg): every star's K and C
  bool has_marg = false;
  std::vector<int> marg_k_h;            // [n_stars] K of every star
  int* marg_k_dev = nullptr;
  double* marg_c_dev = nullptr;         // [n_stars] sum_k (ln(2 pi) / 2 - ln w_k)
  // photometry
  bool has_phot = false;
  payne::PhotParams phot{};
  size_t phot_smem = 0;
  // workspace
  long long slab = 8192, slab_alloc = 0, ldf = 0;
  float *flux = nullptr, *hA = nullptr, *hB = nullptr;
  payne::TcActs actA, actB;
  double* chi2_sed = nullptr;
  int* status = nullptr;
  // all-gather of lnL over peer memory (payne_gather_*): three rotating buffers [world * slots] on every rank, each
  // rank's push kernel stores its slice into every rank's copy and then raises its flag there
  int g_world = 0, g_rank = 0;
  long long g_slots = 0, g_seq = 0;            // g_seq: steps submitted so far
  double* g_buf = nullptr;                      // local [3][world * slots]
  unsigned long long* g_flag = nullptr;         // local [world]: last step whose slice of rank r has landed here (+1)
  double* g_peer_buf[16] = {nullptr};           // every rank's g_buf as mapped into this process (own = local)
  unsigned long long* g_peer_flag[16] = {nullptr};
  bool g_opened[16] = {false};
  int* g_done = nullptr;                        // CTA counter of the fused tail's exit
  bool g_fuse = true;                           // PAYNE_GATHER_FUSED=0: always the separate push kernel
  bool g_active = false, g_fused = false;       // set around run_batch by payne_lnlike_batch_gather
  unsigned long long g_wait_for = 0, g_raise_to = 0;
  size_t g_bufoff = 0;
  // host staging
  long long stage_cap = 0, stage_ld = 0;
  double *theta_pin = nullptr, *lnl_pin = nullptr, *theta_stage = nullptr, *lnl_stage = nullptr;
  double* lnl_map = nullptr;       // device view of lnl_pin (zero-copy result: the tail writes lnL straight to the host)
  long long star_cap = 0;
  int *star_pin = nullptr, *star_stage = nullptr;   // star indices of the *_stars_host entry
  // device allocations to free
  std::vector<void*> owned;
  // timing
  bool timing = false;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  double ms_acc[3] = {0, 0, 0};
  bool ms_valid = false;
  std::vector<std::array<cudaEvent_t, 4>> pending;
  long long launches = 0;
};

namespace {

// Entry points select the context's device and put the caller's device back on return.
struct DeviceGuard {
  int prev = -1;
  bool changed = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) changed = (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() { if (changed) cudaSetDevice(prev); }
};

// The workspace (flux slab, activation planes, per-point records) is shared by every entry point, and
// entry points may be given different streams: a call on another stream than the previous one first
// waits for the previous call's work.
int order_after_previous(PayneCtx* c, cudaStream_t st) {
  if (c->has_last && c->last_stream != st) CU_TRY(cudaStreamWaitEvent(st, c->ev_done, 0));
  return PAYNE_OK;
}
int mark_done(PayneCtx* c, cudaStream_t st) {
  CU_TRY(cudaEventRecord(c->ev_done, st));
  c->last_stream = st; c->has_last = true;
  return PAYNE_OK;
}

template <class T>
int upload_owned(PayneCtx* c, T** dst, const T* src, size_t n) {
  int rc = upload(dst, src, n);
  if (rc == PAYNE_OK && *dst) c->owned.push_back((void*)*dst);
  return rc;
}

// One star's observation (fitargs of likelihood.py:84-112) appended to the context's concatenated arrays, and its
// record: pixel offset and count, wavelength range, sort order.  The Chebyshev abscissa is normalised on the
// star's own grid (polycalc, fitutils.py:13-14).
struct ObsArrays {
  std::vector<double> w, lnw, ot, inv_s, x;   // wavelength, ln wavelength, flux / eflux, 1 / eflux, Chebyshev abscissa
  std::vector<double> q, otm1;                // fast tail: grid position (ln w - ln w_0) / dlnw, (flux - 1) / eflux
};
int append_star_obs(const PayneObs* obs, double lnw0, double inv_dlnw, ObsArrays& A, payne::ObsStar* rec) {
  const int no = obs->n_obs;
  if (no < 1) return fail(PAYNE_E_INVALID, "n_obs must be >= 1");
  if (!obs->wave || !obs->flux || !obs->eflux) return fail(PAYNE_E_INVALID, "null observation array");
  const double* ow = obs->wave;
  const double omin = *std::min_element(ow, ow + no);
  const double omax = *std::max_element(ow, ow + no);
  rec->off = (int)A.w.size(); rec->n_obs = no; rec->obs_min = omin; rec->obs_max = omax; rec->sorted = 1;
  for (int j = 0; j < no; ++j) {
    const double lnw = std::log(ow[j]);
    A.w.push_back(ow[j]);
    A.lnw.push_back(lnw);
    A.ot.push_back(obs->flux[j] / obs->eflux[j]);
    A.inv_s.push_back(1.0 / obs->eflux[j]);
    const double x = ow[j] - omin;                     // fitutils.py:13-14
    A.x.push_back(2.0 * (x / (omax - omin)) - 1.0);
    A.q.push_back((lnw - lnw0) * inv_dlnw);
    A.otm1.push_back((obs->flux[j] - 1.0) / obs->eflux[j]);
    if (!std::isfinite(ow[j]) || (j > 0 && ow[j] < ow[j - 1])) rec->sorted = 0;
  }
  return PAYNE_OK;
}

// Per-dataset tables of the fused tail: emulator grid, stage-1 regrid tables, rotation-kernel table,
// twiddles, observation arrays, analytic regrid constants, kernel occupancy.
int build_tail(PayneCtx* c, const PayneSpecNet* s, const PayneObs* obs) {
  using namespace payne;
  EncodeParams& E = c->enc;
  // ---- emulator grid
  const int n = s->D_out;
  std::vector<double> w(s->wavelength, s->wavelength + n), inv_dw(n - 1);
  for (int i = 0; i + 1 < n; ++i) {
    if (!(w[i + 1] > w[i])) return fail(PAYNE_E_INVALID, "wavelength grid must be strictly increasing");
    inv_dw[i] = 1.0 / (w[i + 1] - w[i]);
  }
  TailParams& T = c->tail;
  T.n = n;
  double *dw, *dinv;
  int rc = upload_owned(c, &dw, w.data(), n); if (rc) return rc;
  rc = upload_owned(c, &dinv, inv_dw.data(), n - 1); if (rc) return rc;
  T.w = dw; T.inv_dw = dinv;
  T.lnw0 = std::log(w[0]);
  T.inv_dlnw = (double)(n - 1) / (std::log(w[n - 1]) - std::log(w[0]));
  T.sigma_in = kCkms / s->resolution;
  {
    const char* e = getenv("PAYNE_DISCARD_ROWS");            // "0": leave the consumed rows to L2's write-back
    T.discard_rows = !(e && e[0] == '0');
  }
  T.inst_scale = kFwhmFit;
  // log-uniform check (informational; enables the analytic regrid fast path later)
  double maxdev = 0.0;
  for (int i = 0; i < n; ++i)
    maxdev = std::max(maxdev, std::fabs((std::log(w[i]) - T.lnw0) * T.inv_dlnw - (double)i));
  c->grid_loguniform = maxdev < 1e-7;

  // ---- stage 1 (rotation) regrid: smoothing.py:649-668, 306-314
  const int l2 = ceil_log2(n);
  const int N1 = 1 << l2;
  T.log2N1 = l2;
  std::vector<double> x1 = linspace(std::log(w[0]), std::log(w[n - 1]), N1);
  for (auto& v : x1) v = std::exp(v);
  std::vector<int2> fwd(N1), back(n);
  for (int k = 0; k < N1; ++k) {
    int j; float t;
    interp_entry(w, x1[k], false, &j, &t);
    fwd[k] = make_int2(j, 0);
    std::memcpy(&fwd[k].y, &t, 4);
  }
  for (int i = 0; i < n; ++i) {
    int k; float t;
    interp_entry(x1, w[i], true, &k, &t);
    back[i] = make_int2(k, 0);
    std::memcpy(&back[i].y, &t, 4);
  }
  std::vector<double> dl(N1 - 1);
  for (int k = 0; k + 1 < N1; ++k) dl[k] = std::log(x1[k + 1]) - std::log(x1[k]);
  std::nth_element(dl.begin(), dl.begin() + (N1 - 1) / 2, dl.end());
  const double dv1 = kCkms * dl[(N1 - 1) / 2];          // odd count -> the middle element
  int2 *dfwd, *dback;
  rc = upload_owned(c, &dfwd, fwd.data(), N1); if (rc) return rc;
  rc = upload_owned(c, &dback, back.data(), n); if (rc) return rc;
  T.fwd1 = dfwd; T.back1 = dback;
  // rotational transfer function table
  const double h = 1.0 / 32.0;
  const double vmax = 600.0;
  long long ntab = (long long)std::ceil(3.14159265358979323846 * vmax / dv1 / h) + 8;
  ntab = std::min<long long>(ntab, 1LL << 21);
  // interval i: the cubic through sb((i-1)h), sb(ih), sb((i+1)h), sb((i+2)h) in f = u/h - i, as c0 + f(c1 + f(c2 + f c3))
  std::vector<float4> sbt(ntab);
  {
    double tm = rot_sb(-h), t0 = rot_sb(0.0), t1 = rot_sb(h);
    for (long long i = 0; i < ntab; ++i) {
      const double t2 = rot_sb((double)(i + 2) * h);
      sbt[i] = make_float4((float)t0, (float)(-tm / 3.0 - t0 / 2.0 + t1 - t2 / 6.0), (float)(tm / 2.0 - t0 + t1 / 2.0),
                           (float)(-tm / 6.0 + t0 / 2.0 - t1 / 2.0 + t2 / 6.0));
      tm = t0; t0 = t1; t1 = t2;
    }
  }
  float4* dsb;
  rc = upload_owned(c, &dsb, sbt.data(), sbt.size()); if (rc) return rc;
  T.sbtab = dsb; T.ntab = (int)ntab; T.sb_h = h;
  T.sb_scale = 2.0 * 3.14159265358979323846 / ((double)N1 * dv1) / h;
  // twiddles
  std::vector<float2> tw(N1 / 2);
  for (int e = 0; e < N1 / 2; ++e) {
    tw[e] = unit_round(-2.0 * 3.14159265358979323846 * (double)e / (double)N1);
  }
  float2* dtw;
  rc = upload_owned(c, &dtw, tw.data(), tw.size()); if (rc) return rc;
  T.tw = dtw; T.log2tw = l2; T.max_log2N = l2;
  // compact per-pass copies for the compile-time-planned transforms (fft_ct.cuh, CtTwLayout)
  {
    auto wfun = [&](int x, int log2L) {
      const int e = x << (l2 - log2L);
      if (e < N1 / 2) return tw[e];
      const float2 t = tw[e - N1 / 2];
      return make_float2(-t.x, -t.y);
    };
    for (int m = 0; m < 16; ++m) T.twpass[m] = nullptr;
    for (int m = 6; m <= std::min(14, l2 - 1); ++m) {
      const int len = payne::ct_pass_table(m, (float2*)nullptr, wfun);
      if (len <= 0) continue;
      std::vector<float2> pt(len);
      payne::ct_pass_table(m, pt.data(), wfun);
      float2* dpt;
      rc = upload_owned(c, &dpt, pt.data(), pt.size()); if (rc) return rc;
      T.twpass[m] = dpt;
    }
  }
  // one 8-byte slot per complex point; from 65536 samples on only half of them sit in shared
  // memory (split transform, fast tail only)
  c->tail_smem = l2 >= 16 ? (size_t)2 * N1 : (size_t)4 * N1;
  if (l2 > 16) return fail(PAYNE_E_UNSUPPORTED, "emulator grids above 65536 pixels are not supported");

  // ---- observation: every star's arrays back to back, one record per star
  {
    FastGrid& F = c->fast;
    const double dlnw = (std::log(w[n - 1]) - std::log(w[0])) / (double)(n - 1);
    F.dlnw = dlnw; F.inv_dlnw = 1.0 / dlnw;
  }
  ObsArrays A;
  for (int k = 0; k < c->n_stars; ++k) {
    rc = append_star_obs(&obs[k], T.lnw0, c->fast.inv_dlnw, A, &c->stars[k]);
    if (rc) return rc;
    c->n_obs_max = std::max(c->n_obs_max, obs[k].n_obs);
  }
  const size_t no = A.w.size();
  if (no > (size_t)std::numeric_limits<int>::max()) return fail(PAYNE_E_INVALID, "more than 2^31 - 1 observed pixels in all");
  c->n_obs_total = (long long)no;
  double *d1, *d2, *d3, *d4, *d5;
  rc = upload_owned(c, &d1, A.w.data(), no); if (rc) return rc;
  rc = upload_owned(c, &d2, A.lnw.data(), no); if (rc) return rc;
  rc = upload_owned(c, &d3, A.ot.data(), no); if (rc) return rc;
  rc = upload_owned(c, &d4, A.inv_s.data(), no); if (rc) return rc;
  rc = upload_owned(c, &d5, A.x.data(), no); if (rc) return rc;
  T.n_obs = obs[0].n_obs; T.obs_w = d1; T.obs_lnw = d2; T.obs_ot = d3; T.obs_inv_s = d4; T.obs_x = d5;
  T.obs_min = c->stars[0].obs_min; T.obs_max = c->stars[0].obs_max;
  for (int i = 0; i < PAYNE_NPAR; ++i) { T.col[i] = c->lay.col[i]; T.fixed[i] = c->lay.fixed[i]; }
  T.n_poly = c->lay.modpoly_bool ? c->lay.n_poly : 0;
  for (int i = 0; i < PAYNE_MAX_POLY; ++i) T.poly_col[i] = c->lay.poly_col[i];
  T.n_labels = s->D_in;
  for (int i = 0; i < 8; ++i) { T.label_col[i] = E.col[i]; T.label_fixed[i] = E.fixed[i]; }
  c->ldf = ((long long)n + 2 + 3) / 4 * 4;   // two finite pad floats per row (read, never used: tail_fast.cuh regrid_in)

  // ---- analytic regrid constants for the fast tail, verified against the exact tables
  {
    FastGrid& F = c->fast;
    const double dlnw = F.dlnw;
    F.f_num = n - 1; F.f_den = N1 - 1;
    F.f_incj = (int)((2LL * kNT * F.f_num) / F.f_den);       // forward regrid walks in pairs
    F.f_incr = (int)((2LL * kNT * F.f_num) % F.f_den);
    F.b_num = N1 - 1; F.b_den = n - 1;
    F.b_incj = (int)(((long long)kNT * F.b_num) / F.b_den);
    F.b_incr = (int)(((long long)kNT * F.b_num) % F.b_den);
    F.f_invden = 1.0f / (float)F.f_den; F.b_invden = 1.0f / (float)F.b_den;
    F.c_native = (float)(0.5 * dlnw);
    F.c_grid1 = (float)(0.5 * dlnw * (double)(n - 1) / (double)(N1 - 1));
    double worst = maxdev;
    for (int k = 0; k < N1; ++k) {
      const long long v = (long long)k * F.f_num;
      int j = (int)(v / F.f_den); double dl = (double)(v % F.f_den) / (double)F.f_den;
      if (j >= n - 1) { j = n - 2; dl = 1.0; }
      const double ta = dl * (1.0 + (dl - 1.0) * (double)F.c_native);
      float te; std::memcpy(&te, &fwd[k].y, 4);
      worst = std::max(worst, std::fabs(((double)j + ta) - ((double)fwd[k].x + (double)te)));
    }
    for (int i = 1; i + 1 < n; ++i) {
      const long long v = (long long)i * F.b_num;
      int k = (int)(v / F.b_den); double dl = (double)(v % F.b_den) / (double)F.b_den;
      if (k >= N1 - 1) { k = N1 - 2; dl = 1.0; }
      const double ta = dl * (1.0 + (dl - 1.0) * (double)F.c_grid1);
      float te; std::memcpy(&te, &back[i].y, 4);
      worst = std::max(worst, std::fabs(((double)k + ta) - ((double)back[i].x + (double)te)));
    }
    c->use_fast = (worst < 2e-7) && l2 >= 10 && l2 <= 16;
    double *dq, *dot;
    rc = upload_owned(c, &dq, A.q.data(), no); if (rc) return rc;
    rc = upload_owned(c, &dot, A.otm1.data(), no); if (rc) return rc;
    F.obs_q = dq; F.obs_otm1 = dot;
    F.obs_sorted = c->stars[0].sorted;
    for (int set = 0; set < 2; ++set)
      for (int ip = 0; ip < 4; ++ip)
        for (int q = 0; q < 16; ++q) {
          const double M = (double)(1 << (13 + set));
          F.twc.c[set][ip][q] = unit_round(-2.0 * 3.14159265358979323846 * (double)ip * (double)kNT * (double)q / M);
        }
  }
  if (c->use_fast) {
    if (payne::init_tail_fast(c->fast.twc) || payne::init_tail_cluster(c->fast.twc))
      return fail(PAYNE_E_CUDA, "tail constants");
    // Shared memory left over next to the transform buffer holds the slice of the rotation-kernel
    // table a point actually uses (its lookups are scattered across lanes; from shared memory each
    // costs one wavefront instead of one per touched line).  Take the largest slice that does not
    // cost a resident CTA.
    int occf = 0;
    auto probe = [&](size_t bytes, int* occ) { return payne::probe_tail_fast(l2, payne::FastForm::Point, bytes, occ); };
    int occ0 = 0;
    const bool ok0 = probe(c->tail_smem, &occ0);
    size_t win = 0;
    const char* wenv = getenv("PAYNE_ROT_WINDOW");            // "0": keep the table in L1/L2 only
    if (ok0 && occ0 >= 1 && !(wenv && wenv[0] == '0')) {
      for (size_t cand : {(size_t)32768, (size_t)16384, (size_t)12288, (size_t)11008, (size_t)10880, (size_t)10752, (size_t)10496, (size_t)10240, (size_t)9216, (size_t)8448, (size_t)8192, (size_t)6144,
                          (size_t)4096, (size_t)2048}) {
        int o = 0;
        if (probe(c->tail_smem + cand, &o) && o == occ0) { win = cand; break; }
      }
    }
    c->fast_smem = c->tail_smem + win;
    c->fast.win_floats = (int)(win / 4);
    probe(c->fast_smem, &occf);
    c->fast_grid[(int)payne::FastForm::Point] = occf * c->sm_count;
    {
      const char* denv = getenv("PAYNE_TAIL_DYNAMIC");       // "0": static round robin of points over the CTAs
      if (!(denv && denv[0] == '0')) {
        int* wc = nullptr;
        CU_TRY(cudaMalloc((void**)&wc, sizeof(int)));
        CU_TRY(cudaMemset(wc, 0, sizeof(int)));
        c->owned.push_back(wc);
        c->fast.work_counter = wc;
      }
    }
    if (c->use_fast && l2 >= 16) {
      float* sc = nullptr;
      CU_TRY(cudaMalloc((void**)&sc, (size_t)c->fast_grid[(int)payne::FastForm::Point] * (N1 / 2) * sizeof(float)));
      c->owned.push_back(sc);
      c->fast.scratch = sc;
    }
    // Transforms above 16384 samples: one transform spread over a cluster of four CTAs (an eighth of the packed
    // signal each, three CTAs per SM) instead of one CTA per SM holding all (32768) or half (65536) of it.
    const char* cenv = getenv("PAYNE_TAIL_CLUSTER");         // "0": keep the single-CTA kernels
    if (l2 >= 15 && !(cenv && cenv[0] == '0')) {
      const size_t base = (size_t)N1;                         // N1/8 complex points of 8 bytes per CTA
      int occ0 = 0, ncl0 = 0;
      if (payne::probe_tail_cluster(l2, base, &occ0, &ncl0) && occ0 >= 1 && ncl0 >= 1) {
        size_t win = 0;
        const char* wenv = getenv("PAYNE_ROT_WINDOW");
        if (!(wenv && wenv[0] == '0'))
          for (size_t cand : {(size_t)32768, (size_t)16384, (size_t)12288, (size_t)11008, (size_t)10880, (size_t)10752, (size_t)10496,
                              (size_t)10240, (size_t)9216, (size_t)8448, (size_t)8192, (size_t)6144, (size_t)4096, (size_t)2048}) {
            int o = 0, ncl = 0;
            if (payne::probe_tail_cluster(l2, base + cand, &o, &ncl) && o == occ0 && ncl == ncl0) { win = cand; break; }
          }
        int occ = 0, ncl = 0;
        if (payne::probe_tail_cluster(l2, base + win, &occ, &ncl) && ncl >= 1) {
          c->use_cluster = 1;
          // default: 65536-sample transforms only.  Measured on B200 (4096 points): N1 = 65536 (C4) tail 8.0 ms
          // single-CTA split kernel vs 5.3 ms cluster; N1 = 32768 2.26 ms single CTA (whole transform in 128 KB)
          // vs 3.13 ms cluster -- there the twelve cluster barriers per point outweigh the occupancy.
          c->allow_cluster = (l2 >= 16) || (cenv && cenv[0] == '1');
          c->cluster_smem = base + win;
          c->cluster_win_floats = (int)(win / 4);
          c->cluster_n = ncl;
          c->cluster_occ = occ;
        }
      }
    }
    c->fast.cluster = c->use_cluster;
  }
  if (l2 <= 15) {
    int occ = 0;
    if (!payne::probe_tail_general(l2, c->tail_smem, &occ) || occ < 1)
      return fail(PAYNE_E_UNSUPPORTED, "tail kernel does not fit on an SM");
    c->tail_grid = occ * c->sm_count;
  } else if (!c->use_fast) {
    return fail(PAYNE_E_UNSUPPORTED,
                "a 65536-point transform needs the log-uniform fast tail (emulator grid is not log-uniform)");
  }
  return PAYNE_OK;
}

int build_spec(PayneCtx* c, const PayneSpecNet* s, const PayneObs* obs, bool emulator_only = false) {
  using namespace payne;
  c->D_in = s->D_in; c->H[0] = s->H1; c->H[1] = s->H2; c->H[2] = s->H3; c->D_out = s->D_out;
  if (s->D_in < 1 || s->D_in > 8) return fail(PAYNE_E_INVALID, "D_in must be in [1,8]");
  if (s->D_out < 32) return fail(PAYNE_E_INVALID, "D_out must be >= 32");
  const int nl = s->n_layers == 0 ? 6 : s->n_layers;
  if (nl != 6 && nl != 4 && nl != 3) return fail(PAYNE_E_INVALID, "n_layers must be 6 (LinNet), 4 (SMLP / multi-chunk) or 3 (YST1)");
  c->multinet = (nl == 4 && s->activation == PAYNE_ACT_SIGMOID && s->n_groups >= 1);
  if (!c->multinet && (nl == 6) != (s->activation == PAYNE_ACT_SIGMOID))
    return fail(PAYNE_E_UNSUPPORTED, "supported emulators: 6 sigmoid layers, 4 sigmoid layers in chunks, or 3/4 leaky-ReLU layers");
  c->n_layers = nl;
  c->legacy = (nl != 6) && !c->multinet;
  if (c->multinet) {
    c->n_groups = s->n_groups; c->chunk = s->group_size;
    if (c->chunk < 32 || (long long)(c->n_groups - 1) * c->chunk >= s->D_out || (long long)c->n_groups * c->chunk < s->D_out)
      return fail(PAYNE_E_INVALID, "multi-chunk emulator: n_groups chunks of group_size pixels must tile D_out (last one may be narrower)");
    if (s->H2 != s->H1 || s->H3 != s->H1) return fail(PAYNE_E_INVALID, "multi-chunk emulator: H2 and H3 must equal H1");
    if (c->n_groups > 64) return fail(PAYNE_E_UNSUPPORTED, "at most 64 chunk nets");
  }
  int din[6] = {s->D_in, s->H1, s->H1, s->H2, s->H2, s->H3};
  int dout[6] = {s->H1, s->H1, s->H2, s->H2, s->H3, s->D_out};
  if (nl == 4) {                                   // NNmodels.py:99-107
    const int a[4] = {s->D_in, s->H1, s->H2, s->H3}, b[4] = {s->H1, s->H2, s->H3, s->D_out};
    for (int k = 0; k < 4; ++k) { din[k] = a[k]; dout[k] = b[k]; }
  } else if (nl == 3) {                            // ystpred.py:25-30
    const int a[3] = {s->D_in, s->H1, s->H2}, b[3] = {s->H1, s->H2, s->D_out};
    for (int k = 0; k < 3; ++k) { din[k] = a[k]; dout[k] = b[k]; }
  }
  if (c->multinet) {
    // stacked over the chunks: [G*H, D_in], [G*H, H], [G*H, H], [D_out, H]
    const int G = c->n_groups, H = s->H1;
    const int a[4] = {s->D_in, H, H, H}, b[4] = {G * H, G * H, G * H, s->D_out};
    for (int k = 0; k < 4; ++k) { din[k] = a[k]; dout[k] = b[k]; }
  }
  for (int k = 0; k < nl; ++k) {
    c->dims_in[k] = din[k]; c->dims_out[k] = dout[k];
    int rc = upload_owned(c, &c->W[k], s->W[k], (size_t)din[k] * dout[k]);
    if (rc) return rc;
    rc = upload_owned(c, &c->b[k], s->b[k], (size_t)dout[k]);
    if (rc) return rc;
  }
  EncodeParams& E = c->enc;
  E.D_in = s->D_in; E.H1 = s->H1; E.offset = s->encode_offset;
  E.cast32 = (nl == 6 || c->multinet) ? 1 : (s->label_fp32_cast != 0);
  E.act = c->legacy ? kActLeaky : kActSigmoid;
  const int label_par[5] = {PAYNE_P_TEFF, PAYNE_P_LOGG, PAYNE_P_FEH, PAYNE_P_AFE, PAYNE_P_VMIC};
  for (int i = 0; i < 8; ++i) {
    E.col[i] = -1; E.fixed[i] = std::numeric_limits<double>::quiet_NaN(); E.xmin[i] = 0; E.xmax[i] = 1;
  }
  for (int i = 0; i < s->D_in; ++i) {
    E.xmin[i] = s->xmin[i]; E.xmax[i] = s->xmax[i];
    if (i < 5) { E.col[i] = c->lay.col[label_par[i]]; E.fixed[i] = c->lay.fixed[label_par[i]]; }
  }

  int rc = PAYNE_OK;
  if (!emulator_only) {
    rc = build_tail(c, s, obs);
    if (rc) return rc;
  }
  // Parity mode's "the tensor core never rounds the leading product sum" holds for contractions up to
  // 512 wide (mlp_tc.cuh header); wider hidden layers must use the CUDA-core fp32 mode.
  if (!c->legacy && c->lay.precision == PAYNE_PREC_PARITY)
    for (int k = 1; k < (c->multinet ? 4 : 6); ++k)
      if (din[k] > payne::kX3MaxK)
        return fail(PAYNE_E_UNSUPPORTED, "parity precision supports hidden widths up to 512 (layer " + std::to_string(k + 1) +
                    " contracts over " + std::to_string(din[k]) + "); use precision 'simt'");
  if (c->multinet) {
    // chunk widths that are not multiples of 4 cannot be TMA-stored (16-byte bases): CUDA-core layers
    if (c->chunk % 4 != 0 && c->lay.precision != PAYNE_PREC_SIMT_FP32)
      return fail(PAYNE_E_UNSUPPORTED, "multi-chunk emulator: group_size must be a multiple of 4 for the tensor-core modes (use precision 'simt')");
    if (c->lay.precision != PAYNE_PREC_SIMT_FP32 && c->lay.precision != PAYNE_PREC_PARITY)
      return fail(PAYNE_E_UNSUPPORTED, "multi-chunk emulator: precision must be 'parity' or 'simt'");
    const int G = c->n_groups, H = s->H1;
    for (int k = 1; k <= 2; ++k) {
      rc = payne::tc_prepare_weights_x(&c->tcw[k], s->W[k], G * H, H, &c->owned);
      if (rc) return fail(rc, "tc_prepare_weights failed");
    }
    // output layers padded to G * chunk rows so that every group's weight block has the same height
    std::vector<float> w4((size_t)G * c->chunk * H, 0.f);
    std::memcpy(w4.data(), s->W[3], (size_t)s->D_out * H * sizeof(float));
    rc = payne::tc_prepare_weights_x(&c->tcw[3], w4.data(), G * c->chunk, H, &c->owned);
    if (rc) return fail(rc, "tc_prepare_weights failed");
    return PAYNE_OK;
  }
  // leaky-ReLU stacks: the output layer (nearly all of their flops) takes row-scaled slices, K <= 512
  if (c->legacy && din[nl - 1] <= payne::kX3MaxK && din[nl - 1] >= 8) {
    rc = payne::tc_prepare_weights_x(&c->tcw[nl - 1], s->W[nl - 1], dout[nl - 1], din[nl - 1], &c->owned);
    if (rc) return fail(rc, "tc_prepare_weights failed");
    c->legacy_tc = true;
  }
  // tensor-core operand copies of the weights (sigmoid LinNet only)
  for (int k = 1; k < 6 && !c->legacy; ++k) {
    rc = payne::tc_prepare_weights_x(&c->tcw[k], s->W[k], dout[k], din[k], &c->owned);
    if (rc) return fail(rc, "tc_prepare_weights failed: " + std::string(cudaGetErrorString(cudaGetLastError())));
  }
  return PAYNE_OK;
}

int build_phot(PayneCtx* c, const PaynePhotNet* p, const PayneObs* obs, const PayneStarOpts* opts) {
  using namespace payne;
  const int nb = p->nb, H = p->H;
  // band list of every star: net band of each of its magnitudes; none given = the net's order
  // a star whose own layout has no photometry (phot_bool 0, PayneObs.nb 0) has no slots
  auto no_phot = [&](int k) { return opts && opts[k].layout && !opts[k].layout->phot_bool; };
  bool any_band = false;
  for (int k = 0; k < c->n_stars; ++k) any_band |= opts && (opts[k].band || no_phot(k));
  std::vector<int> band_slot(any_band ? (size_t)c->n_stars * nb : 0, -1);
  for (int k = 0; k < c->n_stars; ++k) {
    if (no_phot(k)) continue;
    const int32_t* band = opts ? opts[k].band : nullptr;
    if (!band) {
      if (p->nb != obs[k].nb)
        return fail(PAYNE_E_INVALID, "photometry net and observation of star " + std::to_string(k) + " disagree on nb");
      for (int b = 0; b < nb && any_band; ++b) band_slot[(size_t)k * nb + b] = b;
      continue;
    }
    if (obs[k].nb < 0 || obs[k].nb > nb)
      return fail(PAYNE_E_INVALID, "star " + std::to_string(k) + ": " + std::to_string(obs[k].nb) +
                  " magnitudes but the photometry net has " + std::to_string(nb) + " bands");
    for (int i = 0; i < obs[k].nb; ++i) {
      if (band[i] < 0 || band[i] >= nb)
        return fail(PAYNE_E_INVALID, "star " + std::to_string(k) + ": band " + std::to_string(band[i]) + " outside [0, " +
                    std::to_string(nb) + ")");
      int& sl = band_slot[(size_t)k * nb + band[i]];
      if (sl >= 0) return fail(PAYNE_E_INVALID, "star " + std::to_string(k) + ": band " + std::to_string(band[i]) + " given twice");
      sl = i;
    }
  }
  PhotParams& P = c->phot;
  P.nb = nb; P.H = H;
  std::vector<float> w2t((size_t)nb * H * H);
  for (int b = 0; b < nb; ++b)
    for (int ho = 0; ho < H; ++ho)
      for (int hi = 0; hi < H; ++hi)
        w2t[((size_t)b * H + hi) * H + ho] = p->w2[((size_t)b * H + ho) * H + hi];
  float *d1, *d2, *d3, *d4, *d5, *d6;
  int rc;
  rc = upload_owned(c, &d1, p->w1, (size_t)nb * H * 6); if (rc) return rc;
  rc = upload_owned(c, &d2, p->b1, (size_t)nb * H); if (rc) return rc;
  rc = upload_owned(c, &d3, w2t.data(), w2t.size()); if (rc) return rc;
  rc = upload_owned(c, &d4, p->b2, (size_t)nb * H); if (rc) return rc;
  rc = upload_owned(c, &d5, p->w3, (size_t)nb * H); if (rc) return rc;
  rc = upload_owned(c, &d6, p->b3, (size_t)nb); if (rc) return rc;
  P.w1 = d1; P.b1 = d2; P.w2t = d3; P.b2 = d4; P.w3 = d5; P.b3 = d6;
  for (int i = 0; i < 6; ++i) { P.xmin[i] = p->xmin[i]; P.xmax[i] = p->xmax[i]; }
  // every star's magnitudes and errors back to back, in its own order (without band lists star k is at k * nb)
  std::vector<double> mag, err;
  for (int k = 0; k < c->n_stars; ++k) {
    const int nbk = obs[k].nb;
    if (nbk > 0 && (!obs[k].phot_mag || !obs[k].phot_err)) return fail(PAYNE_E_INVALID, "null photometry array");
    c->stars[k].phot_off = (int)mag.size();
    c->stars[k].nb = nbk;
    mag.insert(mag.end(), obs[k].phot_mag, obs[k].phot_mag + nbk);
    err.insert(err.end(), obs[k].phot_err, obs[k].phot_err + nbk);
  }
  double *h1, *h2, *h3;
  rc = upload_owned(c, &h1, p->hiav, (size_t)nb * 5); if (rc) return rc;
  rc = upload_owned(c, &h2, mag.data(), mag.size()); if (rc) return rc;
  rc = upload_owned(c, &h3, err.data(), err.size()); if (rc) return rc;
  P.hiav = h1; P.obs_mag = h2; P.obs_err = h3;
  for (int i = 0; i < PAYNE_NPAR; ++i) { P.col[i] = c->lay.col[i]; P.fixed[i] = c->lay.fixed[i]; }
  P.photscale = c->lay.photscale_bool;
  c->phot_smem = (size_t)2 * kPhotTile * H * sizeof(double);
  if (any_band) {
    int* ds = nullptr;
    rc = upload_owned(c, &ds, band_slot.data(), band_slot.size()); if (rc) return rc;
    P.band_slot = ds;
    c->phot_smem += (size_t)kPhotTile * nb * sizeof(double);     // per-slot terms
  }
  if (c->phot_smem > 200 * 1024) return fail(PAYNE_E_UNSUPPORTED, "photometry hidden width too large");
  CU_TRY(payne::raise_max_dyn_smem(any_band ? (const void*)payne::phot_kernel<true> : (const void*)payne::phot_kernel<false>,
                                    c->phot_smem));
  return PAYNE_OK;
}

// LSF tail (tail_lsf.cuh) for n_total observed pixels: occupancy probe, the vector and the per-CTA scratch.  Once
// per context; the vector is then written by the caller.
int lsf_alloc(PayneCtx* c, long long n_total) {
  using namespace payne;
  if (c->tail.log2N1 > 15) return fail(PAYNE_E_UNSUPPORTED, "LSF broadening is limited to emulator grids of 32768 pixels");
  if (c->lsf.lsf) return PAYNE_OK;
  LsfParams& L = c->lsf;
  L.log2nx_max = std::min(15, c->tail.log2tw);
  const size_t smem = (size_t)4 << std::max(L.log2nx_max, c->tail.log2N1);
  int occ = 0;
  if (!payne::probe_tail_lsf(smem, &occ) || occ < 1) return fail(PAYNE_E_UNSUPPORTED, "LSF tail kernel does not fit on an SM");
  c->lsf_smem = smem; c->lsf_grid = occ * c->sm_count;
  double* d = nullptr;
  CU_TRY(cudaMalloc((void**)&d, (size_t)n_total * sizeof(double))); c->owned.push_back(d); L.lsf = d;
  CU_TRY(cudaMalloc((void**)&d, (size_t)c->lsf_grid * c->D_out * sizeof(double))); c->owned.push_back(d); L.cdf = d;
  CU_TRY(cudaMalloc((void**)&d, (size_t)c->lsf_grid * c->D_out * sizeof(double))); c->owned.push_back(d); L.aux = d;
  CU_TRY(cudaMalloc((void**)&d, ((size_t)c->lsf_grid << L.log2nx_max) * sizeof(double))); c->owned.push_back(d); L.lam = d;
  return PAYNE_OK;
}

// Per-star LSF vectors of payne_ctx_create_stars_opts: every star has one or none does; each is checked as
// payne_ctx_set_lsf checks its vector and they go back to back like the observed pixels.
int set_star_lsf(PayneCtx* c, const PayneObs* obs, const PayneStarOpts* opts) {
  if (!opts) return PAYNE_OK;
  int n_lsf = 0;
  for (int k = 0; k < c->n_stars; ++k) n_lsf += opts[k].lsf != nullptr;
  if (n_lsf == 0) return PAYNE_OK;
  if (n_lsf != c->n_stars)
    return fail(PAYNE_E_UNSUPPORTED, "an LSF vector for every star or for none (the LSF tail and the scalar-R tails are different kernels)");
  if (!c->has_spec) return fail(PAYNE_E_INVALID, "context has no spectrum emulator");
  std::vector<double> all;
  all.reserve((size_t)c->n_obs_total);
  for (int k = 0; k < c->n_stars; ++k)
    for (int j = 0; j < obs[k].n_obs; ++j) {
      if (!(opts[k].lsf[j] > 0.0)) return fail(PAYNE_E_INVALID, "LSF dispersions must be positive (star " + std::to_string(k) + ")");
      all.push_back(opts[k].lsf[j]);
    }
  int rc = lsf_alloc(c, (long long)all.size());
  if (rc) return rc;
  CU_TRY(cudaMemcpy((void*)c->lsf.lsf, all.data(), all.size() * sizeof(double), cudaMemcpyHostToDevice));
  c->lsf_on = true;
  return PAYNE_OK;
}

int ensure_workspace(PayneCtx* c, long long B) {
  const long long need = std::min(B, c->slab);
  if (need <= c->slab_alloc) return PAYNE_OK;
  auto drop = [&](void* p) { if (p) cudaFree(p); };
  drop(c->flux); drop(c->hA); drop(c->hB); drop(c->chi2_sed); drop(c->fast.points); drop(c->rscale);
  c->fast.points = nullptr; c->rscale = nullptr;
  payne::tc_free_acts_x(&c->actA); payne::tc_free_acts_x(&c->actB);
  c->flux = c->hA = c->hB = nullptr; c->chi2_sed = nullptr; c->slab_alloc = 0;
  const long long rows = (need + 127) / 128 * 128;
  if (c->has_spec) {
    const long long hmax = (std::max({c->H[0], c->H[1], c->H[2]}) + 7) / 8 * 8;
    const long long arows = rows * c->n_groups;          // multi-chunk: one block of `rows` rows per chunk net
    c->rows_per_group = rows;
    CU_TRY(cudaMalloc((void**)&c->flux, (size_t)rows * c->ldf * sizeof(float)));
    CU_TRY(cudaMemset(c->flux, 0, (size_t)rows * c->ldf * sizeof(float)));   // the row padding stays zero
    CU_TRY(cudaMalloc((void**)&c->hA, (size_t)arows * hmax * sizeof(float)));
    CU_TRY(cudaMalloc((void**)&c->hB, (size_t)arows * hmax * sizeof(float)));
    CU_TRY(cudaMalloc((void**)&c->rscale, (size_t)rows * sizeof(float)));
    CU_TRY(cudaMalloc(&c->fast.points, (size_t)rows * sizeof(payne::FastPoint)));
    CU_TRY(cudaMemset(c->fast.points, 0, (size_t)rows * sizeof(payne::FastPoint)));   // struct padding is copied too
    int rc = payne::tc_alloc_acts_x(&c->actA, arows, hmax); if (rc) return fail(rc, "tc_alloc_acts");
    rc = payne::tc_alloc_acts_x(&c->actB, arows, hmax); if (rc) return fail(rc, "tc_alloc_acts");
  }
  CU_TRY(cudaMalloc((void**)&c->chi2_sed, (size_t)rows * sizeof(double)));
  // the zero-fills above went to the NULL stream; callers may launch on non-blocking streams that do
  // not order against it, so finish them here (allocation happens once per workspace size)
  CU_TRY(cudaDeviceSynchronize());
  c->slab_alloc = need;
  return PAYNE_OK;
}

// emulator forward for `nb` rows: labels gathered from x (ld) by E -> out [nb, ldo] fp32
// want_depth: the tensor-core modes emit f - 1 (bias shifted by -1 in the epilogue) so that the
// tail keeps ~8 more mantissa bits of the line depth; *is_depth reports what was written.
int run_mlp(PayneCtx* c, const payne::EncodeParams& E, const double* x, long long ld, int nb,
            float* out, long long ldo, bool want_depth, int* is_depth, cudaStream_t st) {
  using namespace payne;
  const int prec = c->lay.precision;
  if (c->multinet) {
    // ---- multi-chunk emulator: G independent 4-layer sigmoid nets, outputs side by side in the flux row
    const int G = c->n_groups, H = c->H[0], P = c->chunk;
    const long long rpg = c->rows_per_group;
    *is_depth = want_depth ? 1 : 0;
    if (prec == PAYNE_PREC_SIMT_FP32) {
      const long long hld = (std::max({c->H[0], c->H[1], c->H[2]}) + 7) / 8 * 8;
      for (int g = 0; g < G; ++g) {
        float* a = c->hA + (size_t)g * rpg * hld; float* b = c->hB + (size_t)g * rpg * hld;
        const long long tot = (long long)nb * H;
        encode_layer1_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(
            E, x, ld, c->W[0] + (size_t)g * H * c->D_in, c->b[0] + (size_t)g * H, a, hld, nb);
        dim3 gh((H + 127) / 128, (nb + 127) / 128);
        sgemm_bias_act_kernel<kActSigmoid><<<gh, 256, 0, st>>>(a, hld, c->W[1] + (size_t)g * H * H, c->b[1] + (size_t)g * H,
                                                                b, hld, nb, H, H, 0.f);
        sgemm_bias_act_kernel<kActSigmoid><<<gh, 256, 0, st>>>(b, hld, c->W[2] + (size_t)g * H * H, c->b[2] + (size_t)g * H,
                                                                a, hld, nb, H, H, 0.f);
        const int ng = g == G - 1 ? c->D_out - (G - 1) * P : P;
        dim3 g4((ng + 127) / 128, (nb + 127) / 128);
        sgemm_bias_act_kernel<kActNone><<<g4, 256, 0, st>>>(a, hld, c->W[3] + (size_t)g * P * H, c->b[3] + (size_t)g * P,
                                                             out + (size_t)g * P, ldo, nb, ng, H, want_depth ? -1.f : 0.f);
        c->launches += 4;
      }
      CU_TRY(cudaGetLastError());
      return PAYNE_OK;
    }
    if (launch_encode_x3(E, x, ld, c->W[0], c->b[0], &c->actA, nb, G, rpg * c->actA.ld, st))
      return fail(PAYNE_E_CUDA, "encode launch");
    c->launches++;
    int rc = tc_run_multinet_x(c->tcw, c->b, H, c->D_out, G, P, &c->actA, &c->actB, rpg, nb, out, ldo,
                             want_depth ? -1.f : 0.f, prec, c->sm_count, st, &c->launches,
                             out == c->flux ? rpg : 0);
    if (rc) return fail(rc, "tensor-core multi-chunk path failed");
    CU_TRY(cudaGetLastError());
    return PAYNE_OK;
  }
  const bool simt = c->legacy || prec == PAYNE_PREC_SIMT_FP32;
  const bool fused_split = !simt && (prec == PAYNE_PREC_PARITY);   // encode + lin1 + slicing in one kernel
  if (fused_split) {
    if (launch_encode_x3(E, x, ld, c->W[0], c->b[0], &c->actA, nb, 1, 0, st)) return fail(PAYNE_E_CUDA, "encode launch");
  } else {
    const long long tot = (long long)nb * c->H[0];
    encode_layer1_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(E, x, ld, c->W[0], c->b[0], c->hA,
                                                                         c->H[0], nb);
  }
  c->launches++;
  *is_depth = 0;
  if (simt) {
    float* cur = c->hA; float* nxt = c->hB;
    const int nl = c->n_layers;
    for (int k = 1; k < nl; ++k) {
      const int K = c->dims_in[k], N = c->dims_out[k];
      dim3 grid((N + 127) / 128, (nb + 127) / 128);
      if (k < nl - 1) {
        if (c->legacy)
          sgemm_bias_act_kernel<kActLeaky><<<grid, 256, 0, st>>>(cur, K, c->W[k], c->b[k], nxt, N, nb, N, K, 0.f);
        else
          sgemm_bias_act_kernel<kActSigmoid><<<grid, 256, 0, st>>>(cur, K, c->W[k], c->b[k], nxt, N, nb, N, K, 0.f);
        std::swap(cur, nxt);
      } else if (c->legacy && c->legacy_tc && prec == PAYNE_PREC_PARITY && (ldo & 3) == 0 && ((uintptr_t)out & 15) == 0) {
        // the wide output layer on the tensor cores: row-scaled exact-accumulation split (mlp_tc.cuh)
        int rc = tc_run_scaled_layer_x(c->tcw[k], c->b[k], cur, K, &c->actA, c->rscale, nb, out, ldo,
                                       want_depth ? -1.f : 0.f, c->sm_count, st, &c->launches);
        if (rc) return fail(rc, "tensor-core output layer failed");
        *is_depth = want_depth ? 1 : 0;
        c->launches--;                       // counted below
      } else {
        sgemm_bias_act_kernel<kActNone><<<grid, 256, 0, st>>>(cur, K, c->W[k], c->b[k], out, ldo, nb, N, K,
                                                              want_depth ? -1.f : 0.f);
        *is_depth = want_depth ? 1 : 0;
      }
      c->launches++;
    }
  } else {
    int rc = tc_run_layers_x(c->tcw, c->b, c->dims_in, c->dims_out, fused_split ? nullptr : c->hA, &c->actA, &c->actB,
                           nb, out, ldo,
                           want_depth ? -1.f : 0.f, prec, c->sm_count, st, &c->launches, c->mapc,
                           out == c->flux ? c->actA.rows : 0, c->use_stack ? &c->stackc : nullptr);
    *is_depth = want_depth ? 1 : 0;
    if (rc) return fail(rc, "tensor-core MLP path failed (precision " + std::to_string(prec) + ")");
  }
  CU_TRY(cudaGetLastError());
  return PAYNE_OK;
}

__global__ void gather_wait_kernel(const unsigned long long* flags, unsigned long long wait_for, int world, int* status);

// A context of several stars needs every point's star: the entries without a star array mean star 0 throughout.
int need_star_array(const PayneCtx* c, const int32_t* star, const char* entry) {
  if (!star && c->n_stars > 1)
    return fail(PAYNE_E_INVALID, "this context holds " + std::to_string(c->n_stars) + " stars: pass every point's star to " + entry);
  return PAYNE_OK;
}

// target: [B] target of every point (payne_ctx_set_targets); the points then name targets and `star` is unused
__global__ void target_star_kernel(const int* target, const int* tfirst, int n_targets, int* star, int n) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int t = target[p];
  star[p] = (t >= 0 && t < n_targets) ? tfirst[t] : -1;
}

// Per-(point, member) records of the fast target tail: at most this many, so the slab of a fast-tail call with targets
// is min(max_batch, kTargetRecords / the largest member count) points (20 MB of records).  The LSF target tail sets its
// members up inside the kernel and has no records.
constexpr long long kTargetRecords = 65536;

// Grows the per-mode buffer *p to at least n zeroed elements, or frees it (n = 0); *have counts what it holds.  Earlier
// calls may still read the old buffer, so the device is synchronised before it is freed.
template <class T>
int resize_buffer(T** p, long long* have, long long n) {
  if (n > 0 ? n <= *have : !*p) return PAYNE_OK;
  CU_TRY(cudaDeviceSynchronize());
  if (*p) cudaFree(*p);
  *p = nullptr; *have = 0;
  if (n > 0) {
    CU_TRY(cudaMalloc((void**)p, (size_t)n * sizeof(T)));
    CU_TRY(cudaMemset(*p, 0, (size_t)n * sizeof(T)));
    CU_TRY(cudaDeviceSynchronize());
    *have = n;
  }
  return PAYNE_OK;
}

// CTAs of the fast tail of `form`: the Point grid from build_tail, the others probed when first needed and capped at
// it (the split kernel's scratch lines exist for that many CTAs).
int form_grid(PayneCtx* c, payne::FastForm form, int* grid) {
  int& g = c->fast_grid[(int)form];
  if (g == 0 && form != payne::FastForm::Point) {
    static const char* const what[] = {"", "target", "binary", "continuum marginalisation"};
    int occ = 0;
    if (!payne::probe_tail_fast(c->tail.log2N1, form, c->fast_smem, &occ) || occ < 1)
      return fail(PAYNE_E_UNSUPPORTED, std::string(what[(int)form]) + " tail kernel does not fit on an SM");
    g = std::min(occ * c->sm_count, c->fast_grid[(int)payne::FastForm::Point]);
  }
  *grid = g;
  return PAYNE_OK;
}

// One call's points and outputs, as an extern "C" entry passes them.
//   star: [B] star index of every point (null: star 0); target: [B] target of every point instead (payne_ctx_set_targets;
//   star is then unused).  binary: every point is a binary (payne_ctx_set_binary): the emulator runs 2 nb rows per slab
//   of nb points.
//   Outputs (null: not wanted): flux [B, ld_flux] model rows; mags; chi2 [B, ld_chi2] the chi2 of every member
//   (targets), or every point's Q (continuum marginalisation, ld_chi2 = 1 for points naming stars); comp [B, 2, ld_flux]
//   a binary's components' spectra; coef [B, ld_coef] c-hat and chol [B, ld_chol] the packed Cholesky factor of every
//   point (payne_ctx_set_cont_marg).
struct Batch {
  const double* theta = nullptr; long long B = 0, ld = 0;
  double* lnl = nullptr;
  const int* star = nullptr;
  const int* target = nullptr;
  bool binary = false;
  double* flux = nullptr; long long ld_flux = 0;
  double* mags = nullptr;
  double* chi2 = nullptr; long long ld_chi2 = 0;
  double* comp = nullptr;
  double* coef = nullptr; long long ld_coef = 0;
  double* chol = nullptr; long long ld_chol = 0;
};

int marg_unsupported(PayneCtx* c);

int run_batch(PayneCtx* c, const Batch& q, cudaStream_t st) {
  using namespace payne;
  const long long B = q.B, ld = q.ld;
  if (B <= 0) return PAYNE_OK;
  const bool marg = c->has_marg;
  if (marg) { int rc = marg_unsupported(c); if (rc) return rc; }
  if (ld < c->ndim_max) return fail(PAYNE_E_INVALID, "ld < ndim (the largest star's with per-star layouts)");
  if (!q.target && q.flux && c->has_spec && q.ld_flux < c->n_obs_max) return fail(PAYNE_E_INVALID, "ld_flux < the largest n_obs");
  const bool records = q.target && !c->lsf_on;           // the fast target tail's per-(point, member) records
  const long long slab = records ? std::min(c->slab, std::max(1LL, kTargetRecords / c->tgt_kmax))
                       : q.binary ? std::max(1LL, c->slab / 2) : c->slab;
  const long long rows = std::min(B, slab);
  int rc = ensure_workspace(c, q.binary ? 2 * B : B);
  if (!rc && q.target) rc = resize_buffer(&c->tgt_star, &c->tgt_star_n, rows);
  if (!rc && records) rc = resize_buffer(&c->tgt_points, &c->tgt_points_n, rows * c->tgt_kmax);
  if (!rc && q.binary) rc = resize_buffer(&c->bin_par, &c->bin_par_n, rows * 3);
  if (rc) return rc;
  // The tail: the LSF-vector tail, else the fast tail in the batch's form (points naming stars may run it
  // cluster-distributed) on line-depth rows, else the general-grid tail (points naming stars only).
  const bool fast_tail = c->has_spec && c->use_fast && c->allow_fast && !c->lsf_on;
  const FastForm form = marg ? FastForm::Marg : q.target ? FastForm::Target : q.binary ? FastForm::Binary : FastForm::Point;
  const bool cluster = form == FastForm::Point && c->use_cluster && c->allow_cluster;
  int fgrid = 0;
  if (fast_tail) { rc = form_grid(c, form, &fgrid); if (rc) return rc; }
  rc = order_after_previous(c, st);
  if (rc) return rc;
  if (c->timing) { c->ms_acc[0] = c->ms_acc[1] = c->ms_acc[2] = 0; c->ms_valid = false; c->pending.clear(); }
  for (long long p0 = 0; p0 < B; p0 += slab) {
    const int nb = (int)std::min(slab, B - p0);
    if (q.target) {
      // the emulators and the photometry see every point as its target's first member
      target_star_kernel<<<(nb + 255) / 256, 256, 0, st>>>(q.target + p0, c->tfirst_dev, c->n_targets, c->tgt_star, nb);
      c->launches++;
    }
    const int* star_s = q.target ? c->tgt_star : q.star ? q.star + p0 : nullptr;   // this slab's star of every point
    const double* th = q.theta + p0 * ld;
    std::array<cudaEvent_t, 4> evs{};
    if (c->timing) {
      for (auto& e : evs) CU_TRY(cudaEventCreate(&e));
      CU_TRY(cudaEventRecord(evs[0], st));
    }
    int is_depth = 0;
    TailParams T = c->tail;
    FastGrid F = c->fast;                                 // the fast tail's, for this slab
    const bool gather_here = c->g_active && c->g_fuse && fast_tail;
    if (c->has_spec) {
      T.theta = th; T.ld = ld; T.flux = c->flux; T.ldf = c->ldf; T.B = nb;
      T.chi2_sed = c->has_phot ? c->chi2_sed : nullptr;
      T.lnl = q.lnl ? q.lnl + p0 : nullptr;
      T.model_out = q.flux ? q.flux + p0 * q.ld_flux : nullptr;
      T.ld_flux = q.ld_flux;
      T.star = star_s;
      T.status = c->status;
      if (q.target) {
        T.target = q.target + p0; T.tfirst = c->tfirst_dev; T.n_targets = c->n_targets; T.kmax = c->tgt_kmax;
        T.chi2_out = q.chi2 ? q.chi2 + p0 * q.ld_chi2 : nullptr; T.ld_chi2 = q.ld_chi2;
      }
      if (q.binary || marg) { T.aj_scratch = c->aj_scratch; T.aj_ld = c->n_obs_max; }
      if (q.binary) {
        T.binary = c->binary_dev; T.bin_par = c->bin_par;
        T.comp_out = q.comp ? q.comp + p0 * 2 * q.ld_flux : nullptr;
      }
      if (marg) {
        T.marg_k = c->marg_k_dev; T.marg_c = c->marg_c_dev;
        T.chi2_out = q.chi2 ? q.chi2 + p0 * q.ld_chi2 : nullptr; T.ld_chi2 = q.ld_chi2;
        T.coef_out = q.coef ? q.coef + p0 * q.ld_coef : nullptr; T.ld_coef = q.ld_coef;
        T.chol_out = q.chol ? q.chol + p0 * q.ld_chol : nullptr; T.ld_chol = q.ld_chol;
      }
      if (gather_here) {
        // all-gather fused into the tail (tail.cuh store_lnl / gather_exit): this slab's slice of every peer's buffer
        T.g_world = c->g_world; T.g_rank = c->g_rank; T.g_done = c->g_done;
        for (int r = 0; r < c->g_world; ++r) {
          T.g_dst[r] = r == c->g_rank ? nullptr : c->g_peer_buf[r] + c->g_bufoff + (size_t)c->g_rank * c->g_slots + p0;
          T.g_flag[r] = c->g_peer_flag[r] + c->g_rank;
        }
        T.g_raise = (p0 + c->slab >= B) ? c->g_raise_to : 0ull;
      }
      if (fast_tail) {
        // the single-CTA forms other than Point's run the split kernel at 65536 samples (the cluster tail has none)
        F.work_start = cluster ? (int)std::min<long long>(c->cluster_n, nb) : std::min(fgrid, nb);
        if (c->grid_cap > 0) F.work_start = std::min(F.work_start, c->grid_cap);
        if (form != FastForm::Point) F.cluster = 0;
        if (q.target) F.points = c->tgt_points;
        if (cluster) F.win_floats = c->cluster_win_floats;
        // per-point setup depends only on theta: fork it beside the emulator GEMMs, join before the tail
        CU_TRY(cudaEventRecord(c->ev_fork, st));
        CU_TRY(cudaStreamWaitEvent(c->side, c->ev_fork, 0));
        if (payne::launch_tail_setup(form, nb, c->side, T, F)) return fail(PAYNE_E_CUDA, "tail_setup launch");
        if (gather_here && p0 == 0 && c->g_wait_for)
          // the buffer the tail is about to write on the peers is free once every rank's previous step has landed here;
          // waited for on the side stream, beside the emulator GEMMs
          gather_wait_kernel<<<1, 32, 0, c->side>>>(c->g_flag, c->g_wait_for, c->g_world, c->status);
        CU_TRY(cudaEventRecord(c->ev_join, c->side));
        c->launches++;
      }
      EncodeParams E = c->enc;
      E.star = star_s;
      if (q.binary) { E.binary = c->binary_dev; E.half = nb; }   // rows [nb, 2 nb): the secondaries
      rc = run_mlp(c, E, th, ld, q.binary ? 2 * nb : nb, c->flux, c->ldf, true, &is_depth, st);
      if (rc) return rc;
      if (c->cont) {
        // modspec *= np.interp(modwave, modcontwave, normalised F_lambda continuum) (predictspec.py:208-226)
        PayneCtx* cc = c->cont;
        cc->slab = c->slab; cc->lay.precision = c->lay.precision;
        rc = ensure_workspace(cc, nb);
        if (rc) return rc;
        int cdepth = 0;
        const long long l0 = cc->launches;
        EncodeParams CE = cc->enc;
        CE.star = E.star;
        rc = run_mlp(cc, CE, th, ld, nb, cc->flux, cc->ldf, true, &cdepth, st);
        if (rc) return rc;
        if (!is_depth) return fail(PAYNE_E_UNSUPPORTED, "continuum multiply expects line-depth rows");
        ContParams C = c->contp;
        C.cont = cc->flux; C.cont_is_depth = cdepth; C.ldc = cc->ldf; C.flux = c->flux; C.ldf = c->ldf; C.B = nb;
        if (payne::launch_continuum(std::min(nb, 8 * c->sm_count), st, C)) return fail(PAYNE_E_CUDA, "continuum launch");
        c->launches += cc->launches - l0 + 1;
      }
    }
    if (c->timing) CU_TRY(cudaEventRecord(evs[1], st));
    if (c->has_phot) {
      PhotParams P = c->phot;
      P.theta = th; P.ld = ld; P.B = nb; P.chi2_sed = c->chi2_sed;
      P.mags_out = q.mags ? q.mags + p0 * P.nb : nullptr;
      P.star = star_s;
      P.status = c->status;
      if (P.band_slot)
        phot_kernel<true><<<(nb + kPhotTile - 1) / kPhotTile, kPhotThreads, c->phot_smem, st>>>(P);
      else
        phot_kernel<false><<<(nb + kPhotTile - 1) / kPhotTile, kPhotThreads, c->phot_smem, st>>>(P);
      c->launches++;
    }
    if (c->timing) CU_TRY(cudaEventRecord(evs[2], st));
    if (c->has_spec) {
      T.flux_is_depth = is_depth;
      if (fast_tail) CU_TRY(cudaStreamWaitEvent(st, c->ev_join, 0));
      if (c->lsf_on) {
        TailParams TL = T;
        TL.col[PAYNE_P_INSTR] = -1;                                   // the vector replaces Inst_R
        TL.fixed[PAYNE_P_INSTR] = std::numeric_limits<double>::quiet_NaN();
        // ... a star's own fixed Inst_R and a per-star layout's Inst_R column too: Rs = NaN, no scalar-R stage
        TL.inst_scale = std::numeric_limits<double>::quiet_NaN();
        const int grid = std::min(c->lsf_grid, nb);
        if (q.target ? payne::launch_tail_lsf_targets(grid, c->lsf_smem, st, TL, c->lsf)
                     : payne::launch_tail_lsf(grid, c->lsf_smem, st, TL, c->lsf))
          return fail(PAYNE_E_CUDA, "tail launch");
      } else if (fast_tail && is_depth) {
        if (cluster ? payne::launch_tail_cluster(T.log2N1, F.work_start, c->cluster_smem, st, T, F)
                    : payne::launch_tail_fast(T.log2N1, form, F.work_start, c->fast_smem, st, T, F))
          return fail(PAYNE_E_CUDA, "tail launch");
        if (gather_here && T.g_raise) c->g_fused = true;
      } else if (form != FastForm::Point) {
        static const char* const what[] = {"", "targets need", "binaries need", "continuum marginalisation needs"};
        return fail(PAYNE_E_UNSUPPORTED, std::string(what[(int)form]) + " the fast tail on line-depth rows");
      } else {
        if (c->tail.log2N1 > 15) return fail(PAYNE_E_UNSUPPORTED, "general-grid tail is limited to 32768-point transforms");
        const int grid = std::min(c->tail_grid, nb);
        if (payne::launch_tail_general(T.log2N1, grid, c->tail_smem, st, T, c->fast.twc)) return fail(PAYNE_E_CUDA, "tail launch");
      }
      c->launches++;
    } else if (q.lnl) {
      lnl_from_sed_kernel<<<(nb + 255) / 256, 256, 0, st>>>(c->chi2_sed, q.lnl + p0, nb);
      c->launches++;
    }
    if (c->timing) { CU_TRY(cudaEventRecord(evs[3], st)); c->pending.push_back(evs); }
    CU_TRY(cudaGetLastError());
  }
  return mark_done(c, st);
}

// Per-star layouts (PayneStarOpts.layout): every rule that does not depend on the device.  A star without a layout
// has the context layout.
int check_star_layouts(const PayneLayout* ctx, const PayneObs* obs, const PayneStarOpts* opts, int n_stars) {
  auto lay_of = [&](int k) { return (opts && opts[k].layout) ? opts[k].layout : ctx; };
  auto has_poly = [](const PayneLayout* L) { return L->modpoly_bool && L->n_poly > 0; };
  for (int k = 0; opts && k < n_stars; ++k) {
    const PayneLayout* L = opts[k].layout;
    if (!L) continue;
    const std::string who = "star " + std::to_string(k) + ": ";
    if (opts[k].fixed) return fail(PAYNE_E_INVALID, who + "give its fixed values in its layout or in PayneStarOpts.fixed, not both");
    if (L->ndim < 0) return fail(PAYNE_E_INVALID, who + "ndim < 0");
    if (L->n_poly < 0 || L->n_poly > PAYNE_MAX_POLY) return fail(PAYNE_E_INVALID, who + "n_poly out of range");
    if (L->spec_bool != ctx->spec_bool) return fail(PAYNE_E_INVALID, who + "spec_bool differs from the context's");
    if (L->precision != ctx->precision) return fail(PAYNE_E_INVALID, who + "precision differs from the context's");
    if (!L->spec_bool && !L->phot_bool) return fail(PAYNE_E_INVALID, who + "nothing to fit");
    if (L->phot_bool && !ctx->phot_bool) return fail(PAYNE_E_INVALID, who + "photometry in a context without a photometry net");
    if (!L->phot_bool && obs[k].nb != 0) return fail(PAYNE_E_INVALID, who + "phot_bool 0 but PayneObs.nb != 0");
    // every sampled column in [0, ndim), none used twice
    std::vector<char> used((size_t)L->ndim, 0);
    auto take = [&](int col, const std::string& what) -> int {
      if (col < 0 || col >= L->ndim) return fail(PAYNE_E_INVALID, who + what + " column " + std::to_string(col) + " outside [0, ndim)");
      if (used[col]) return fail(PAYNE_E_INVALID, who + "column " + std::to_string(col) + " used twice");
      used[col] = 1;
      return PAYNE_OK;
    };
    for (int i = 0; i < PAYNE_NPAR; ++i)
      if (L->col[i] != -1) { int rc = take(L->col[i], "parameter " + std::to_string(i)); if (rc) return rc; }
    for (int i = 0; L->modpoly_bool && i < L->n_poly; ++i) { int rc = take(L->poly_col[i], "pc_" + std::to_string(i)); if (rc) return rc; }
  }
  // The polynomial and the plain final pass round differently ((1 + d) / sigma - o / sigma against d / sigma -
  // (o - 1) / sigma): a star without a polynomial in a polynomial launch would not give its single-star result.
  for (int k = 1; k < n_stars; ++k)
    if (has_poly(lay_of(k)) != has_poly(lay_of(0)))
      return fail(PAYNE_E_UNSUPPORTED, "stars with and without a continuum polynomial (modpoly_bool, n_poly >= 1) in one set (star " +
                  std::to_string(k) + ")");
  return PAYNE_OK;
}

// Device records of the per-star layouts, wired into the consumers.  A star with fewer continuum coefficients than the
// set's largest order gets zeros after its own (tail_setup); that keeps its bits only at finite Chebyshev abscissae, so
// such a star whose abscissae are not all finite (n_obs = 1 or all wavelengths equal: 0/0 in polycalc) is refused.
int upload_star_layouts(PayneCtx* c, const PayneLayout* ctx, const PayneStarOpts* opts, const PayneObs* obs) {
  using namespace payne;
  const int S = c->n_stars;
  std::vector<StarLayout> rec(S);
  int n_poly_max = 0;
  for (int k = 0; k < S; ++k) {
    const PayneLayout* L = opts[k].layout ? opts[k].layout : ctx;
    StarLayout& r = rec[k];
    for (int i = 0; i < PAYNE_NPAR; ++i) r.col[i] = L->col[i];
    r.n_poly = L->modpoly_bool ? L->n_poly : 0;
    for (int i = 0; i < PAYNE_MAX_POLY; ++i) r.poly_col[i] = L->poly_col[i];
    r.photscale = L->photscale_bool;
    n_poly_max = std::max(n_poly_max, r.n_poly);
    c->ndim_max = std::max(c->ndim_max, (int)L->ndim);
  }
  for (int k = 0; k < S && c->has_spec; ++k) {
    if (rec[k].n_poly == n_poly_max) continue;
    const double* w = obs[k].wave;
    const double omin = *std::min_element(w, w + obs[k].n_obs), omax = *std::max_element(w, w + obs[k].n_obs);
    for (int j = 0; j < obs[k].n_obs; ++j)
      if (!std::isfinite(2.0 * ((w[j] - omin) / (omax - omin)) - 1.0))     // append_star_obs's abscissa
        return fail(PAYNE_E_UNSUPPORTED, "star " + std::to_string(k) + ": its continuum order is below the set's largest "
                    "and its Chebyshev abscissae are not finite (n_obs = 1 or all wavelengths equal)");
  }
  int rc = upload_owned(c, &c->star_lay_dev, rec.data(), rec.size());
  if (rc) return rc;
  c->star_lay_h = rec;
  c->tail.n_poly = n_poly_max;       // the final passes evaluate this many coefficients (tail_setup pads with zeros)
  c->tail.star_lay = c->phot.star_lay = c->enc.star_lay = c->star_lay_dev;
  return PAYNE_OK;
}

// The target kernel of the tail the context runs now, probed once: the LSF target tail (its shared-memory opt-in, and
// as many resident CTAs as the star form's grid), or the fast one (its grid).
int probe_targets(PayneCtx* c) {
  int occ = 0;
  if (c->lsf_on) {
    if (c->tgt_lsf_probed) return PAYNE_OK;
    if (!payne::probe_tail_lsf_targets(c->lsf_smem, &occ) || occ * c->sm_count < c->lsf_grid)
      return fail(PAYNE_E_UNSUPPORTED, "LSF target tail kernel does not fit on an SM");
    c->tgt_lsf_probed = true;
    return PAYNE_OK;
  }
  int grid = 0;
  return form_grid(c, payne::FastForm::Target, &grid);
}

// The target entries: targets set, and the context still runs a tail they can use (a one-star context may have
// switched its LSF vector on or off since payne_ctx_set_targets).
int need_targets(PayneCtx* c) {
  if (c->n_targets == 0) return fail(PAYNE_E_INVALID, "no targets: payne_ctx_set_targets first");
  if (c->g_world > 0) return fail(PAYNE_E_UNSUPPORTED, "targets on a context with the fused gather are not supported");
  if (c->lsf_on && !c->tgt_instr_col.empty()) return fail(PAYNE_E_INVALID, c->tgt_instr_col);
  if (!c->lsf_on && !(c->use_fast && c->allow_fast))
    return fail(PAYNE_E_UNSUPPORTED, "targets without LSF vectors need the fast tail");
  return probe_targets(c);
}

// The host-buffer entries: q names host buffers (theta, lnl, and every point's star or target, or neither: star 0),
// which are staged through pinned and device buffers.
int lnlike_host(PayneCtx* c, Batch q) {
  int rc;
  const long long B = q.B, ld = q.ld;
  const bool targets = q.target != nullptr;
  const int32_t* star_host = targets ? q.target : q.star;
  double* lnl_host = q.lnl;
  const int n_idx = targets ? c->n_targets : c->n_stars;
  if (star_host)
    for (int64_t i = 0; i < B; ++i)
      if (star_host[i] < 0 || star_host[i] >= n_idx)
        return fail(PAYNE_E_INVALID, std::string(targets ? "target" : "star") + " index " + std::to_string(star_host[i]) +
                    " of point " + std::to_string(i) + " outside [0, " + std::to_string(n_idx) + ")");
  DeviceGuard dg(c->device);
  if (star_host && B > c->star_cap) {
    if (c->star_pin) cudaFreeHost(c->star_pin);
    if (c->star_stage) cudaFree(c->star_stage);
    c->star_pin = c->star_stage = nullptr; c->star_cap = 0;
    CU_TRY(cudaMallocHost((void**)&c->star_pin, (size_t)B * sizeof(int)));
    CU_TRY(cudaMalloc((void**)&c->star_stage, (size_t)B * sizeof(int)));
    c->star_cap = B;
  }
  if (B > c->stage_cap || ld != c->stage_ld) {
    if (c->theta_pin) cudaFreeHost(c->theta_pin);
    if (c->lnl_pin) cudaFreeHost(c->lnl_pin);
    if (c->theta_stage) cudaFree(c->theta_stage);
    if (c->lnl_stage) cudaFree(c->lnl_stage);
    c->theta_pin = c->lnl_pin = c->theta_stage = c->lnl_stage = nullptr; c->lnl_map = nullptr; c->stage_cap = 0;
    CU_TRY(cudaMallocHost((void**)&c->theta_pin, (size_t)B * ld * sizeof(double)));
    CU_TRY(cudaMallocHost((void**)&c->lnl_pin, (size_t)B * sizeof(double)));
    CU_TRY(cudaMalloc((void**)&c->theta_stage, (size_t)B * ld * sizeof(double)));
    CU_TRY(cudaMalloc((void**)&c->lnl_stage, (size_t)B * sizeof(double)));
    c->stage_cap = B; c->stage_ld = ld;
    // 8 bytes per point: the last kernel writes them into the pinned buffer itself (mapped under unified
    // addressing) instead of a device buffer + a D2H copy behind it (one enqueue and one copy latency per call)
    void* dp = nullptr;
    const char* zenv = getenv("PAYNE_ZERO_COPY_LNL");
    c->lnl_map = (!(zenv && zenv[0] == '0') && cudaHostGetDevicePointer(&dp, c->lnl_pin, 0) == cudaSuccess) ? (double*)dp : nullptr;
    cudaGetLastError();
  }
  std::memcpy(c->theta_pin, q.theta, (size_t)B * ld * sizeof(double));
  CU_TRY(cudaMemcpyAsync(c->theta_stage, c->theta_pin, (size_t)B * ld * sizeof(double),
                         cudaMemcpyHostToDevice, c->stream));
  if (star_host) {
    std::memcpy(c->star_pin, star_host, (size_t)B * sizeof(int));
    CU_TRY(cudaMemcpyAsync(c->star_stage, c->star_pin, (size_t)B * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  }
  q.theta = c->theta_stage;
  (targets ? q.target : q.star) = star_host ? c->star_stage : nullptr;
  q.lnl = c->lnl_map ? c->lnl_map : c->lnl_stage;
  rc = run_batch(c, q, c->stream);
  if (rc) return rc;
  if (!c->lnl_map)
    CU_TRY(cudaMemcpyAsync(c->lnl_pin, c->lnl_stage, (size_t)B * sizeof(double), cudaMemcpyDeviceToHost,
                           c->stream));
  CU_TRY(cudaStreamSynchronize(c->stream));
  std::memcpy(lnl_host, c->lnl_pin, (size_t)B * sizeof(double));
  return PAYNE_OK;
}


// The value of parameter `which` that star k resolves to: its column, or (column -1) its fixed value.
std::pair<int, double> resolve_param(const PayneCtx* c, int k, int which) {
  const int col = c->star_lay_h.empty() ? c->lay.col[which] : c->star_lay_h[k].col[which];
  if (col >= 0) return {col, 0.0};
  return {-1, c->star_fixed_h.empty() ? c->lay.fixed[which] : c->star_fixed_h[(size_t)k * PAYNE_NPAR + which]};
}

// What the binary tail cannot take (payne_ctx_set_binary and every _binary entry: the context may have changed since).
int binary_unsupported(PayneCtx* c) {
  const char* why = !c->has_spec ? "the spectrum emulator is missing"
                  : c->has_phot ? "photometry (phot_bool) is not supported"
                  : c->lsf_on ? "LSF vectors are not supported"
                  : c->cont ? "an attached continuum emulator is not supported"
                  : c->n_targets ? "targets are not supported"
                  : c->star_lay_dev ? "per-star layouts (PayneStarOpts.layout) are not supported"
                  : c->g_world > 0 ? "the fused gather is not supported"
                  : c->has_marg ? "continuum marginalisation is not supported"
                  : !(c->use_fast && c->allow_fast) ? "binaries need the fast tail (an emulator grid uniform in ln wavelength)"
                  : nullptr;
  return why ? fail(PAYNE_E_UNSUPPORTED, std::string("binary: ") + why) : PAYNE_OK;
}

int need_binary(PayneCtx* c) {
  if (!c->has_binary) return fail(PAYNE_E_INVALID, "no binary: payne_ctx_set_binary first");
  return binary_unsupported(c);
}

// What continuum marginalisation cannot take (payne_ctx_set_cont_marg and every entry while it is on).
int marg_unsupported(PayneCtx* c) {
  const char* why = !c->has_spec ? "the spectrum emulator is missing"
                  : c->lsf_on ? "LSF vectors are not supported"
                  : c->has_binary ? "binaries are not supported"
                  : c->cont ? "an attached continuum emulator is not supported"
                  : c->g_world > 0 ? "the fused gather is not supported"
                  : !(c->use_fast && c->allow_fast) ? "it needs the fast tail (an emulator grid uniform in ln wavelength)"
                  : nullptr;
  return why ? fail(PAYNE_E_UNSUPPORTED, std::string("continuum marginalisation: ") + why) : PAYNE_OK;
}

// The _cont entries: the setting is on and the output strides hold the largest star (or target).
int need_marg(PayneCtx* c, bool targets, int64_t ld_coef, int64_t ld_chol) {
  if (!c->has_marg) return fail(PAYNE_E_INVALID, "no continuum marginalisation: payne_ctx_set_cont_marg first");
  long long kc = 0, kl = 0;
  const int n = targets ? c->n_targets : c->n_stars;
  for (int t = 0; t < n; ++t) {
    long long a = 0, b = 0;
    const int k0 = targets ? c->tfirst_h[t] : t, k1 = targets ? c->tfirst_h[t + 1] : t + 1;
    for (int k = k0; k < k1; ++k) { a += c->marg_k_h[k]; b += (long long)c->marg_k_h[k] * (c->marg_k_h[k] + 1) / 2; }
    kc = std::max(kc, a); kl = std::max(kl, b);
  }
  if (ld_coef < kc) return fail(PAYNE_E_INVALID, "ld_coef < " + std::to_string(kc) + " (the largest K" + (targets ? ", summed over a target's members)" : ")"));
  if (ld_chol < kl) return fail(PAYNE_E_INVALID, "ld_chol < " + std::to_string(kl) + " (the largest K (K + 1) / 2" + (targets ? ", summed over a target's members)" : ")"));
  return PAYNE_OK;
}

}  // namespace

extern "C" {

int payne_ctx_set_binary(PayneCtx* c, const PayneBinary* b) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);
  auto drop = [&]() -> int {
    CU_TRY(cudaDeviceSynchronize());                     // earlier calls may still read it
    if (c->binary_dev) cudaFree(c->binary_dev);
    c->binary_dev = nullptr; c->has_binary = false;
    // the a_j scratch is continuum marginalisation's while that is on
    return c->has_marg ? PAYNE_OK : resize_buffer(&c->aj_scratch, &c->aj_scratch_n, 0);
  };
  if (!b) return drop();
  int rc = binary_unsupported(c);
  if (rc) return rc;
  static const char* names[PAYNE_NPAR] = {"Teff", "log(g)", "[Fe/H]", "[a/Fe]", "Vrad", "Vrot", "Vmic", "Inst_R",
                                          "log(R)", "Dist", "log(A)", "Av", "Rv"};
  const int ndim = c->lay.ndim;
  for (int i = 0; i < PAYNE_NPAR; ++i) {
    const bool own = i == PAYNE_P_TEFF || i == PAYNE_P_LOGG || i == PAYNE_P_FEH || i == PAYNE_P_AFE || i == PAYNE_P_VMIC ||
                     i == PAYNE_P_VRAD || i == PAYNE_P_VROT;
    if (!own && (b->col[i] >= 0 || !std::isnan(b->fixed[i])))
      return fail(PAYNE_E_INVALID, std::string("binary: ") + names[i] + " is shared by both components (the secondary "
                  "may have its own Teff, log(g), [Fe/H], [a/Fe], Vmic, Vrad and Vrot only)");
    if (b->col[i] >= ndim)
      return fail(PAYNE_E_INVALID, std::string("binary: ") + names[i] + " column " + std::to_string(b->col[i]) +
                  " outside [0, ndim = " + std::to_string(ndim) + ")");
  }
  if (b->rratio_col >= ndim)
    return fail(PAYNE_E_INVALID, "binary: Rratio column " + std::to_string(b->rratio_col) + " outside [0, ndim = " +
                std::to_string(ndim) + ")");
  if (b->rratio_col < 0 && !std::isfinite(b->rratio_fixed))
    return fail(PAYNE_E_INVALID, "binary: Rratio needs a theta column or a finite fixed value");
  int grid = 0;
  rc = form_grid(c, payne::FastForm::Binary, &grid);
  if (rc) return rc;
  rc = drop();
  if (rc) return rc;
  rc = upload(&c->binary_dev, b, 1);
  if (rc) return rc;
  rc = resize_buffer(&c->aj_scratch, &c->aj_scratch_n, (long long)grid * c->n_obs_max);
  if (rc) return rc;
  c->has_binary = true;
  return PAYNE_OK;
}

int payne_lnlike_batch_binary(PayneCtx* c, const double* theta_dev, const int32_t* star_dev, int64_t B, int64_t ld,
                              double* lnl_dev, void* stream) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B == 0) return PAYNE_OK;
  if (!theta_dev || !lnl_dev) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);
  int rc = need_binary(c);
  if (rc) return rc;
  Batch q{theta_dev, B, ld, lnl_dev, star_dev};
  q.binary = true;
  return run_batch(c, q, (cudaStream_t)stream);
}

int payne_lnlike_batch_binary_host(PayneCtx* c, const double* theta_host, const int32_t* star_host, int64_t B, int64_t ld,
                                   double* lnl_host) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B <= 0) return PAYNE_OK;
  if (!theta_host || !lnl_host) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);
  int rc = need_binary(c);
  if (rc) return rc;
  Batch q{theta_host, B, ld, lnl_host, star_host};
  q.binary = true;
  return lnlike_host(c, q);
}

int payne_model_batch_binary(PayneCtx* c, const double* theta_dev, const int32_t* star_dev, int64_t B, int64_t ld,
                             double* flux_dev, int64_t ld_flux, double* comp_dev, double* lnl_dev, void* stream) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B == 0) return PAYNE_OK;
  if (!theta_dev) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);
  int rc = need_binary(c);
  if (rc) return rc;
  if ((flux_dev || comp_dev) && ld_flux < c->n_obs_max) return fail(PAYNE_E_INVALID, "ld_flux < the largest n_obs");
  Batch q{theta_dev, B, ld, lnl_dev, star_dev};
  q.binary = true;
  q.flux = flux_dev; q.ld_flux = ld_flux; q.comp = comp_dev;
  return run_batch(c, q, (cudaStream_t)stream);
}

int payne_ctx_set_cont_marg(PayneCtx* c, const PayneContMarg* per_star) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);
  auto drop = [&]() -> int {
    CU_TRY(cudaDeviceSynchronize());                     // earlier calls may still read them
    if (c->marg_k_dev) cudaFree(c->marg_k_dev);
    if (c->marg_c_dev) cudaFree(c->marg_c_dev);
    c->marg_k_dev = nullptr; c->marg_c_dev = nullptr; c->has_marg = false;
    c->marg_k_h.clear();
    // the a_j scratch is the binary tail's while binaries are on
    return c->has_binary ? PAYNE_OK : resize_buffer(&c->aj_scratch, &c->aj_scratch_n, 0);
  };
  if (!per_star) return drop();
  const int S = c->n_stars;
  std::vector<int> kk(S);
  std::vector<double> cc(S, 0.0);
  int with = 0;
  for (int k = 0; k < S; ++k) {
    const PayneContMarg& m = per_star[k];
    const std::string who = "continuum marginalisation, star " + std::to_string(k) + ": ";
    if (m.n_coef < 0 || m.n_coef > PAYNE_MAX_POLY)
      return fail(PAYNE_E_INVALID, who + "n_coef " + std::to_string(m.n_coef) + " outside [1, " + std::to_string(PAYNE_MAX_POLY) + "]");
    kk[k] = m.n_coef;
    if (m.n_coef == 0) continue;
    ++with;
    const int np = c->star_lay_h.empty() ? (c->lay.modpoly_bool ? c->lay.n_poly : 0) : c->star_lay_h[k].n_poly;
    if (np > 0) return fail(PAYNE_E_INVALID, who + "its layout samples pc_k as well (modpoly_bool with n_poly > 0)");
    for (int i = 0; i < m.n_coef; ++i) {
      if (!(std::isfinite(m.lo[i]) && std::isfinite(m.hi[i]) && m.lo[i] < m.hi[i]))
        return fail(PAYNE_E_INVALID, who + "the box of coefficient " + std::to_string(i) + " must be finite with lo < hi");
      cc[k] += 0.5 * std::log(2.0 * 3.141592653589793) - std::log(m.hi[i] - m.lo[i]);
    }
  }
  if (with == 0) return fail(PAYNE_E_INVALID, "continuum marginalisation: n_coef outside [1, " + std::to_string(PAYNE_MAX_POLY) + "] for every star");
  if (with != S)
    return fail(PAYNE_E_UNSUPPORTED, "continuum marginalisation: some stars have the setting and others (n_coef 0) do not");
  int rc = marg_unsupported(c);
  if (rc) return rc;
  int grid = 0;
  rc = form_grid(c, payne::FastForm::Marg, &grid);
  if (rc) return rc;
  rc = drop();
  if (rc) return rc;
  rc = upload(&c->marg_k_dev, kk.data(), (size_t)S);
  if (rc) return rc;
  rc = upload(&c->marg_c_dev, cc.data(), (size_t)S);
  if (rc) return rc;
  rc = resize_buffer(&c->aj_scratch, &c->aj_scratch_n, (long long)grid * c->n_obs_max);
  if (rc) return rc;
  c->marg_k_h = kk;
  c->has_marg = true;
  return PAYNE_OK;
}

int payne_cont_batch_stars(PayneCtx* c, const double* theta_dev, const int32_t* star_dev, int64_t B, int64_t ld,
                           double* coef_dev, int64_t ld_coef, double* chol_dev, int64_t ld_chol, double* chi2_dev,
                           double* lnl_dev, void* stream) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B == 0) return PAYNE_OK;
  if (!theta_dev) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);
  int rc = need_marg(c, false, coef_dev ? ld_coef : INT64_MAX, chol_dev ? ld_chol : INT64_MAX);
  if (rc) return rc;
  rc = need_star_array(c, star_dev, "payne_cont_batch_stars");
  if (rc) return rc;
  Batch q{theta_dev, B, ld, lnl_dev, star_dev};
  q.chi2 = chi2_dev; q.ld_chi2 = 1;
  q.coef = coef_dev; q.ld_coef = ld_coef; q.chol = chol_dev; q.ld_chol = ld_chol;
  return run_batch(c, q, (cudaStream_t)stream);
}

int payne_cont_batch_targets(PayneCtx* c, const double* theta_dev, const int32_t* target_dev, int64_t B, int64_t ld,
                             double* coef_dev, int64_t ld_coef, double* chol_dev, int64_t ld_chol, double* chi2_dev,
                             int64_t ld_chi2, double* lnl_dev, void* stream) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B == 0) return PAYNE_OK;
  if (!theta_dev || !target_dev) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);
  int rc = need_targets(c);
  if (rc) return rc;
  rc = need_marg(c, true, coef_dev ? ld_coef : INT64_MAX, chol_dev ? ld_chol : INT64_MAX);
  if (rc) return rc;
  if (chi2_dev && ld_chi2 < c->tgt_kmax) return fail(PAYNE_E_INVALID, "ld_chi2 < the largest member count");
  Batch q{theta_dev, B, ld, lnl_dev};
  q.target = target_dev;
  q.chi2 = chi2_dev; q.ld_chi2 = ld_chi2;
  q.coef = coef_dev; q.ld_coef = ld_coef; q.chol = chol_dev; q.ld_chol = ld_chol;
  return run_batch(c, q, (cudaStream_t)stream);
}

int payne_ctx_set_targets(PayneCtx* c, const int32_t* first, int32_t n_targets) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);
  if (!first) {
    CU_TRY(cudaDeviceSynchronize());                     // earlier calls may still read the table
    if (c->tfirst_dev) cudaFree(c->tfirst_dev);
    c->tfirst_dev = nullptr; c->n_targets = 0; c->tgt_kmax = 0; c->tgt_nobs_max = 0;
    int rc = resize_buffer(&c->tgt_points, &c->tgt_points_n, 0);
    if (!rc) rc = resize_buffer(&c->tgt_star, &c->tgt_star_n, 0);
    if (rc) return rc;
    c->tgt_instr_col.clear();
    c->tfirst_h.clear();
    return PAYNE_OK;
  }
  if (!c->has_spec) return fail(PAYNE_E_UNSUPPORTED, "targets need the spectrum emulator");
  // the LSF tail runs on every grid it accepts; the scalar-R target tail is the fast one
  if (!c->lsf_on && !c->use_fast)
    return fail(PAYNE_E_UNSUPPORTED, "targets need the fast tail (an emulator grid uniform in ln wavelength)");
  if (c->g_world > 0) return fail(PAYNE_E_UNSUPPORTED, "targets on a context with the fused gather are not supported");
  if (n_targets < 1) return fail(PAYNE_E_INVALID, "n_targets must be >= 1");
  if (first[0] != 0 || first[n_targets] != c->n_stars)
    return fail(PAYNE_E_INVALID, "first[0] must be 0 and first[n_targets] n_stars (" + std::to_string(c->n_stars) + ")");
  int kmax = 0;
  long long nobs_max = 0;
  std::string instr_col;
  for (int t = 0; t < n_targets; ++t) {
    if (first[t + 1] <= first[t]) return fail(PAYNE_E_INVALID, "first[] must increase strictly (target " + std::to_string(t) + ")");
    kmax = std::max(kmax, first[t + 1] - first[t]);
    long long no = 0;
    for (int k = first[t]; k < first[t + 1]; ++k) no += c->stars[k].n_obs;
    nobs_max = std::max(nobs_max, no);
    static const char* names[6] = {"Teff", "log(g)", "[Fe/H]", "[a/Fe]", "Vmic", "Vrot"};
    static const int which[6] = {PAYNE_P_TEFF, PAYNE_P_LOGG, PAYNE_P_FEH, PAYNE_P_AFE, PAYNE_P_VMIC, PAYNE_P_VROT};
    for (int k = first[t] + 1; k < first[t + 1]; ++k) {
      const std::string who = "target " + std::to_string(t) + ", member " + std::to_string(k - first[t]) + ": ";
      for (int i = 0; i < 6; ++i) {
        // the emulator row and stage 1 are computed once per point, from these values of the first member
        const auto a = resolve_param(c, first[t], which[i]), b = resolve_param(c, k, which[i]);
        if (a.first != b.first || (a.first < 0 && std::memcmp(&a.second, &b.second, sizeof(double)) != 0))
          return fail(PAYNE_E_INVALID, who + std::string(names[i]) + " differs from the first member's (column or fixed value)");
      }
      if (c->has_phot && c->stars[k].nb > 0)
        return fail(PAYNE_E_INVALID, who + "photometry on a member other than the first");
    }
    // Under an LSF vector no kernel reads Inst_R: a member's Inst_R column would be a sampled dimension without effect.
    for (int k = first[t]; k < first[t + 1] && instr_col.empty(); ++k) {
      const int col = resolve_param(c, k, PAYNE_P_INSTR).first;
      if (col >= 0)
        instr_col = "target " + std::to_string(t) + ", member " + std::to_string(k - first[t]) + ": Inst_R in theta column " +
                    std::to_string(col) + " beside its LSF vector (the vector replaces Inst_R: give Inst_R no column)";
    }
  }
  if (c->lsf_on && !instr_col.empty()) return fail(PAYNE_E_INVALID, instr_col);
  c->tgt_lsf_probed = false;                            // probed again for this context's current tail
  int rc = probe_targets(c);
  if (rc) return rc;
  CU_TRY(cudaDeviceSynchronize());
  if (c->tfirst_dev) cudaFree(c->tfirst_dev);
  c->tfirst_dev = nullptr; c->n_targets = 0;
  rc = upload(&c->tfirst_dev, first, (size_t)n_targets + 1);
  if (rc) return rc;
  if (c->tgt_kmax != kmax) {                             // the record stride changes: reallocate at the next call
    rc = resize_buffer(&c->tgt_points, &c->tgt_points_n, 0);
    if (rc) return rc;
  }
  c->n_targets = n_targets; c->tgt_kmax = kmax; c->tgt_nobs_max = nobs_max; c->tgt_instr_col = instr_col;
  c->tfirst_h.assign(first, first + n_targets + 1);
  return PAYNE_OK;
}

int payne_lnlike_batch_targets(PayneCtx* c, const double* theta_dev, const int32_t* target_dev, int64_t B, int64_t ld,
                               double* lnl_dev, void* stream) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B == 0) return PAYNE_OK;
  if (!theta_dev || !target_dev || !lnl_dev) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);
  int rc = need_targets(c);
  if (rc) return rc;
  Batch q{theta_dev, B, ld, lnl_dev};
  q.target = target_dev;
  return run_batch(c, q, (cudaStream_t)stream);
}

int payne_model_batch_targets(PayneCtx* c, const double* theta_dev, const int32_t* target_dev, int64_t B, int64_t ld,
                              double* flux_dev, int64_t ld_flux, double* chi2_dev, int64_t ld_chi2, double* mags_dev,
                              double* lnl_dev, void* stream) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B == 0) return PAYNE_OK;
  if (!theta_dev || !target_dev) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);
  int rc = need_targets(c);
  if (rc) return rc;
  if (flux_dev && ld_flux < c->tgt_nobs_max) return fail(PAYNE_E_INVALID, "ld_flux < the largest target's pixels (all members)");
  if (chi2_dev && ld_chi2 < c->tgt_kmax) return fail(PAYNE_E_INVALID, "ld_chi2 < the largest member count");
  Batch q{theta_dev, B, ld, lnl_dev};
  q.target = target_dev;
  q.flux = flux_dev; q.ld_flux = ld_flux; q.mags = mags_dev; q.chi2 = chi2_dev; q.ld_chi2 = ld_chi2;
  return run_batch(c, q, (cudaStream_t)stream);
}

int payne_abi_version(void) { return PAYNE_ABI_VERSION; }
const char* payne_last_error(void) { return g_err.c_str(); }

int payne_ctx_create(const PayneSpecNet* spec, const PaynePhotNet* phot, const PayneObs* obs,
                     const PayneLayout* layout, int device, PayneCtx** out) {
  return payne_ctx_create_stars(spec, phot, obs, 1, layout, device, out);
}

int payne_ctx_create_stars(const PayneSpecNet* spec, const PaynePhotNet* phot, const PayneObs* obs, int32_t n_stars,
                           const PayneLayout* layout, int device, PayneCtx** out) {
  return payne_ctx_create_stars_opts(spec, phot, obs, nullptr, n_stars, layout, device, out);
}

int payne_ctx_create_stars_opts(const PayneSpecNet* spec, const PaynePhotNet* phot, const PayneObs* obs,
                                const PayneStarOpts* opts, int32_t n_stars, const PayneLayout* layout, int device,
                                PayneCtx** out) {
  if (!out || !layout || !obs) return fail(PAYNE_E_INVALID, "null argument");
  *out = nullptr;
  if (n_stars < 1) return fail(PAYNE_E_INVALID, "n_stars must be >= 1");
  bool any_band = false, any_fixed = false, any_layout = false;
  for (int k = 0; opts && k < n_stars; ++k) {
    any_band |= opts[k].band != nullptr || opts[k].layout != nullptr;    // a layout may drop the star's photometry
    any_fixed |= opts[k].fixed != nullptr; any_layout |= opts[k].layout != nullptr;
  }
  if (layout->phot_bool && !any_band)
    for (int k = 1; k < n_stars; ++k)
      if (obs[k].nb != obs[0].nb) return fail(PAYNE_E_INVALID, "every star must have the same nb (star " + std::to_string(k) + ")");
  if (layout->spec_bool && !spec) return fail(PAYNE_E_INVALID, "spec_bool set but no spectrum net");
  if (layout->phot_bool && !phot) return fail(PAYNE_E_INVALID, "phot_bool set but no photometry net");
  if (!layout->spec_bool && !layout->phot_bool) return fail(PAYNE_E_INVALID, "nothing to fit");
  if (layout->n_poly < 0 || layout->n_poly > PAYNE_MAX_POLY) return fail(PAYNE_E_INVALID, "n_poly out of range");
  if (any_layout) { int rc = check_star_layouts(layout, obs, opts, n_stars); if (rc) return rc; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(PAYNE_E_CUDA, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(PAYNE_E_INVALID, "bad device ordinal");
  DeviceGuard dg(device);
  cudaDeviceProp prop;
  CU_TRY(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(PAYNE_E_UNSUPPORTED, "built for sm_100a (B200) only");
  PayneCtx* c = new PayneCtx();
  { const char* e = getenv("PAYNE_GEMM_STACK"); c->use_stack = !(e && e[0] == '0'); }
  c->device = device; c->sm_count = prop.multiProcessorCount; c->lay = *layout;
  c->has_spec = layout->spec_bool != 0; c->has_phot = layout->phot_bool != 0;
  c->n_stars = n_stars; c->ndim_max = layout->ndim;
  c->stars.assign(n_stars, payne::ObsStar{});
  int rc = PAYNE_OK;
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) rc = fail(PAYNE_E_CUDA, "stream");
  if (!rc && (cudaStreamCreateWithFlags(&c->side, cudaStreamNonBlocking) != cudaSuccess ||
              cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
              cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming) != cudaSuccess ||
              cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming) != cudaSuccess))
    rc = fail(PAYNE_E_CUDA, "side stream");
  if (!rc && cudaMalloc((void**)&c->status, sizeof(int)) != cudaSuccess) rc = fail(PAYNE_E_NOMEM, "status");
  if (!rc) cudaMemset(c->status, 0, sizeof(int));
  if (!rc && c->has_spec) rc = build_spec(c, spec, obs);
  if (!rc && c->has_phot) rc = build_phot(c, phot, obs, opts);
  if (!rc) rc = set_star_lsf(c, obs, opts);
  if (!rc) rc = upload_owned(c, &c->stars_dev, c->stars.data(), c->stars.size());
  if (!rc && (any_fixed || any_layout)) {
    // star k's row: its own values (PayneStarOpts.fixed or its layout's), or the context layout's where it gives none
    std::vector<double> fx((size_t)n_stars * PAYNE_NPAR);
    for (int k = 0; k < n_stars; ++k)
      std::memcpy(&fx[(size_t)k * PAYNE_NPAR], opts[k].fixed ? opts[k].fixed : opts[k].layout ? opts[k].layout->fixed : layout->fixed,
                  PAYNE_NPAR * sizeof(double));
    rc = upload_owned(c, &c->star_fixed_dev, fx.data(), fx.size());
    c->star_fixed_h = fx;
  }
  if (!rc) {
    c->tail.stars = c->phot.stars = c->stars_dev;
    c->tail.n_stars = c->phot.n_stars = c->enc.n_stars = n_stars;
  }
  if (!rc && any_layout) rc = upload_star_layouts(c, layout, opts, obs);
  if (!rc) c->tail.star_fixed = c->phot.star_fixed = c->enc.star_fixed = c->star_fixed_dev;
  if (rc) { std::string keep = g_err; payne_ctx_destroy(c); g_err = keep; return rc; }
  *out = c;
  return PAYNE_OK;
}

void payne_ctx_destroy(PayneCtx* c) {
  if (!c) return;
  if (c->cont) { payne_ctx_destroy(c->cont); c->cont = nullptr; }
  DeviceGuard dg(c->device);
  cudaDeviceSynchronize();
  for (void* p : c->owned) cudaFree(p);
  auto drop = [&](void* p) { if (p) cudaFree(p); };
  drop(c->flux); drop(c->hA); drop(c->hB); drop(c->chi2_sed); drop(c->fast.points); drop(c->rscale);
  c->fast.points = nullptr; drop(c->status);
  payne::tc_free_acts_x(&c->actA); payne::tc_free_acts_x(&c->actB);
  drop(c->theta_stage); drop(c->lnl_stage); drop(c->star_stage);
  drop(c->tfirst_dev); drop(c->tgt_points); drop(c->tgt_star); drop(c->bin_par); drop(c->aj_scratch);
  drop(c->binary_dev); drop(c->marg_k_dev); drop(c->marg_c_dev);
  if (c->star_pin) cudaFreeHost(c->star_pin);
  for (int r = 0; r < 16; ++r)
    if (c->g_opened[r]) { cudaIpcCloseMemHandle(c->g_peer_buf[r]); cudaIpcCloseMemHandle(c->g_peer_flag[r]); }
  drop(c->g_buf); drop(c->g_flag); drop(c->g_done);
  if (c->theta_pin) cudaFreeHost(c->theta_pin);
  if (c->lnl_pin) cudaFreeHost(c->lnl_pin);
  for (auto& evs : c->pending) for (auto e : evs) cudaEventDestroy(e);
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->side) cudaStreamDestroy(c->side);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->ev_done) cudaEventDestroy(c->ev_done);
  delete c;
}

int payne_lnlike_batch(PayneCtx* c, const double* theta_dev, int64_t B, int64_t ld, double* lnl_dev,
                       void* stream) {
  return payne_lnlike_batch_stars(c, theta_dev, nullptr, B, ld, lnl_dev, stream);
}

int payne_lnlike_batch_stars(PayneCtx* c, const double* theta_dev, const int32_t* star_dev, int64_t B, int64_t ld,
                             double* lnl_dev, void* stream) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B == 0) return PAYNE_OK;                       // an empty batch may come with null buffers
  if (!theta_dev || !lnl_dev) return fail(PAYNE_E_INVALID, "null argument");
  int rc = need_star_array(c, star_dev, "payne_lnlike_batch_stars");
  if (rc) return rc;
  DeviceGuard dg(c->device);
  return run_batch(c, Batch{theta_dev, B, ld, lnl_dev, star_dev}, (cudaStream_t)stream);
}

int payne_model_batch(PayneCtx* c, const double* theta_dev, int64_t B, int64_t ld, double* flux_dev,
                      double* mags_dev, double* lnl_dev, void* stream) {
  return payne_model_batch_stars(c, theta_dev, nullptr, B, ld, flux_dev, c ? c->n_obs_max : 0, mags_dev, lnl_dev, stream);
}

int payne_model_batch_stars(PayneCtx* c, const double* theta_dev, const int32_t* star_dev, int64_t B, int64_t ld,
                            double* flux_dev, int64_t ld_flux, double* mags_dev, double* lnl_dev, void* stream) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B == 0) return PAYNE_OK;
  if (!theta_dev) return fail(PAYNE_E_INVALID, "null argument");
  int rc = need_star_array(c, star_dev, "payne_model_batch_stars");
  if (rc) return rc;
  DeviceGuard dg(c->device);
  Batch q{theta_dev, B, ld, lnl_dev, star_dev};
  q.flux = flux_dev; q.ld_flux = ld_flux; q.mags = mags_dev;
  return run_batch(c, q, (cudaStream_t)stream);
}

int payne_lnlike_batch_host(PayneCtx* c, const double* theta_host, int64_t B, int64_t ld, double* lnl_host) {
  return payne_lnlike_batch_stars_host(c, theta_host, nullptr, B, ld, lnl_host);
}

int payne_lnlike_batch_stars_host(PayneCtx* c, const double* theta_host, const int32_t* star_host, int64_t B, int64_t ld,
                                  double* lnl_host) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B <= 0) return PAYNE_OK;
  if (!theta_host || !lnl_host) return fail(PAYNE_E_INVALID, "null argument");
  int rc = need_star_array(c, star_host, "payne_lnlike_batch_stars_host");
  if (rc) return rc;
  return lnlike_host(c, Batch{theta_host, B, ld, lnl_host, star_host});
}

int payne_lnlike_batch_targets_host(PayneCtx* c, const double* theta_host, const int32_t* target_host, int64_t B,
                                    int64_t ld, double* lnl_host) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B <= 0) return PAYNE_OK;
  if (!theta_host || !target_host || !lnl_host) return fail(PAYNE_E_INVALID, "null argument");
  DeviceGuard dg(c->device);                             // (need_targets may probe a target kernel)
  int rc = need_targets(c);
  if (rc) return rc;
  Batch q{theta_host, B, ld, lnl_host};
  q.target = target_host;
  return lnlike_host(c, q);
}

}  // extern "C"

// ---- all-gather of lnL over peer memory --------------------------------------------------------------------
// One kernel per step instead of a collective library call: thread 0 first waits until every rank's slice of
// the PREVIOUS step has landed here (flags; this also makes the buffer about to be overwritten on the peers free,
// see payne_lnlike_batch_gather), then every thread copies its share of this rank's lnL slice into every rank's
// buffer with plain stores through the NVLink peer mappings; the last CTA to finish raises this rank's flag on
// every rank behind a system-scope fence.
namespace {
struct GatherPush {
  const double* src;                 // this rank's slice [n] (inside its own buffer)
  double* dst[16];                   // every rank's buffer for this step, already offset to this rank's slice
  unsigned long long* flag[16];      // every rank's flag word of THIS rank
  const unsigned long long* local_flags;   // this rank's flag array [world]
  unsigned long long wait_for;       // flags must have reached this value (0: nothing to wait for)
  unsigned long long raise_to;
  int world, rank, n;
  int* status;
};

// One CTA: 32 KB per rank and step is latency, not bandwidth -- a single system-scope fence behind the stores, then the flags.
__global__ void __launch_bounds__(1024) gather_push_kernel(const __grid_constant__ GatherPush G) {
  if (G.wait_for && threadIdx.x < G.world) {
    const volatile unsigned long long* f = G.local_flags + threadIdx.x;
    const long long t0 = clock64();
    while (*f < G.wait_for) {
      if (clock64() - t0 > 20000000000LL) { atomicOr(G.status, 2); break; }     // ~10 s: a peer is gone
      __nanosleep(100);
    }
    __threadfence_system();
  }
  __syncthreads();
  const int n2 = G.n >> 1;                                  // pairs: 16-byte stores (slices are 16-byte aligned when n is even)
  const bool vec = (G.n & 1) == 0;
  if (vec) {
    const double2* s2 = reinterpret_cast<const double2*>(G.src);
    for (int i = threadIdx.x; i < n2; i += blockDim.x) {
      const double2 v = s2[i];
      for (int r = 0; r < G.world; ++r)
        if (r != G.rank) reinterpret_cast<double2*>(G.dst[r])[i] = v;
    }
  } else {
    for (int i = threadIdx.x; i < G.n; i += blockDim.x) {
      const double v = G.src[i];
      for (int r = 0; r < G.world; ++r)
        if (r != G.rank) G.dst[r][i] = v;
    }
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < G.world) {
    __threadfence_system();                                  // (cumulative: orders every thread's stores before the flag)
    *reinterpret_cast<volatile unsigned long long*>(G.flag[threadIdx.x]) = G.raise_to;
  }
}

__global__ void gather_wait_kernel(const unsigned long long* flags, unsigned long long wait_for, int world, int* status) {
  if ((int)threadIdx.x < world) {
    const volatile unsigned long long* f = flags + threadIdx.x;
    const long long t0 = clock64();
    while (*f < wait_for) {
      if (clock64() - t0 > 20000000000LL) { atomicOr(status, 2); break; }
      __nanosleep(200);
    }
    __threadfence_system();
  }
}
}  // namespace

extern "C" {

int payne_gather_create(PayneCtx* c, int world, int rank, int64_t slots, void* handles_out) {
  if (!c || !handles_out) return fail(PAYNE_E_INVALID, "null argument");
  if (world < 1 || world > 16 || rank < 0 || rank >= world || slots < 1) return fail(PAYNE_E_INVALID, "bad world / rank / slots");
  if (c->g_buf) return fail(PAYNE_E_INVALID, "gather already created on this context");
  if (c->n_stars > 1) return fail(PAYNE_E_UNSUPPORTED, "the fused all-gather has no star argument: not available on a context of several stars");
  DeviceGuard dg(c->device);
  c->g_world = world; c->g_rank = rank; c->g_slots = slots; c->g_seq = 0;
  { const char* e = getenv("PAYNE_GATHER_FUSED"); c->g_fuse = !(e && e[0] == '0'); }
  const size_t nb = (size_t)3 * world * slots * sizeof(double);
  CU_TRY(cudaMalloc((void**)&c->g_buf, nb));
  CU_TRY(cudaMemset(c->g_buf, 0, nb));
  CU_TRY(cudaMalloc((void**)&c->g_flag, 16 * sizeof(unsigned long long)));
  CU_TRY(cudaMemset(c->g_flag, 0, 16 * sizeof(unsigned long long)));
  CU_TRY(cudaMalloc((void**)&c->g_done, sizeof(int)));
  CU_TRY(cudaMemset(c->g_done, 0, sizeof(int)));
  CU_TRY(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h[2];
  CU_TRY(cudaIpcGetMemHandle(&h[0], c->g_buf));
  CU_TRY(cudaIpcGetMemHandle(&h[1], c->g_flag));
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size is part of the ABI (PAYNE_GATHER_HANDLE_BYTES)");
  std::memcpy(handles_out, h, sizeof(h));
  c->g_peer_buf[rank] = c->g_buf; c->g_peer_flag[rank] = c->g_flag;
  return PAYNE_OK;
}

int payne_gather_connect(PayneCtx* c, const void* all_handles) {
  if (!c || !all_handles) return fail(PAYNE_E_INVALID, "null argument");
  if (!c->g_buf) return fail(PAYNE_E_INVALID, "payne_gather_create first");
  DeviceGuard dg(c->device);
  const cudaIpcMemHandle_t* h = reinterpret_cast<const cudaIpcMemHandle_t*>(all_handles);
  for (int r = 0; r < c->g_world; ++r) {
    if (r == c->g_rank) continue;
    void *pb = nullptr, *pf = nullptr;
    if (cudaIpcOpenMemHandle(&pb, h[2 * r], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
        cudaIpcOpenMemHandle(&pf, h[2 * r + 1], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      cudaGetLastError();
      return fail(PAYNE_E_UNSUPPORTED, "peer memory of rank " + std::to_string(r) + " cannot be mapped (no P2P path?)");
    }
    c->g_peer_buf[r] = (double*)pb; c->g_peer_flag[r] = (unsigned long long*)pf; c->g_opened[r] = true;
  }
  return PAYNE_OK;
}

int payne_lnlike_batch_gather(PayneCtx* c, const double* theta_dev, int64_t B, int64_t ld, void* stream,
                              double** gathered_prev) {
  if (!c || !theta_dev) return fail(PAYNE_E_INVALID, "null argument");
  if (!c->g_buf) return fail(PAYNE_E_INVALID, "payne_gather_create / payne_gather_connect first");
  if (B != c->g_slots) return fail(PAYNE_E_INVALID, "batch size differs from the gather's slots per rank");
  for (int r = 0; r < c->g_world; ++r)
    if (!c->g_peer_buf[r]) return fail(PAYNE_E_INVALID, "payne_gather_connect first");
  DeviceGuard dg(c->device);
  cudaStream_t st = (cudaStream_t)stream;
  const long long s = c->g_seq;                            // this step
  const size_t per = (size_t)c->g_world * c->g_slots;      // doubles per buffer
  double* mine = c->g_buf + (size_t)(s % 3) * per + (size_t)c->g_rank * c->g_slots;
  // Buffer s % 3 was last read by the consumers of step s - 3, whose reads every rank enqueued before it submitted
  // step s - 2; the push below starts only after every rank's push of step s - 1 has landed here, which on the
  // peer's stream lies behind its submit of step s - 2: nobody still reads what is about to be overwritten.
  c->g_active = true; c->g_fused = false;
  c->g_wait_for = (unsigned long long)s; c->g_raise_to = (unsigned long long)(s + 1);
  c->g_bufoff = (size_t)(s % 3) * per;
  int rc = run_batch(c, Batch{theta_dev, B, ld, mine}, st);
  c->g_active = false;
  if (rc) return rc;
  if (gathered_prev) *gathered_prev = s > 0 ? c->g_buf + (size_t)((s - 1) % 3) * per : nullptr;
  c->g_seq = s + 1;
  if (c->g_fused) return PAYNE_OK;          // the tail stored the slice on the peers and raised the flags itself
  GatherPush G{};
  G.src = mine;
  for (int r = 0; r < c->g_world; ++r) {
    G.dst[r] = c->g_peer_buf[r] + (size_t)(s % 3) * per + (size_t)c->g_rank * c->g_slots;
    G.flag[r] = c->g_peer_flag[r] + c->g_rank;
  }
  G.local_flags = c->g_flag;
  G.wait_for = (unsigned long long)s;                      // step s - 1 complete <=> flags == s
  G.raise_to = (unsigned long long)(s + 1);
  G.world = c->g_world; G.rank = c->g_rank; G.n = (int)B; G.status = c->status;
  gather_push_kernel<<<1, 1024, 0, st>>>(G);
  CU_TRY(cudaGetLastError());
  c->launches++;
  return mark_done(c, st);
}

int payne_gather_flush(PayneCtx* c, void* stream, double** gathered_last) {
  if (!c || !gathered_last) return fail(PAYNE_E_INVALID, "null argument");
  if (!c->g_buf || c->g_seq == 0) return fail(PAYNE_E_INVALID, "nothing submitted");
  DeviceGuard dg(c->device);
  gather_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(c->g_flag, (unsigned long long)c->g_seq, c->g_world, c->status);
  CU_TRY(cudaGetLastError());
  *gathered_last = c->g_buf + (size_t)((c->g_seq - 1) % 3) * (size_t)c->g_world * c->g_slots;
  return PAYNE_OK;
}

int payne_ann_eval(PayneCtx* c, const double* x_dev, int64_t B, float* y_dev, int64_t ldy, void* stream) {
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (B == 0) return PAYNE_OK;
  if (!x_dev || !y_dev) return fail(PAYNE_E_INVALID, "null argument");
  if (!c->has_spec) return fail(PAYNE_E_INVALID, "context has no spectrum emulator");
  if (ldy < c->D_out) return fail(PAYNE_E_INVALID, "ldy < D_out");
  if (!c->legacy && c->lay.precision != PAYNE_PREC_SIMT_FP32 && ((ldy & 3) || ((uintptr_t)y_dev & 15)))
    return fail(PAYNE_E_INVALID, "y_dev must be 16-byte aligned with ldy a multiple of 4 (TMA store)");
  if (B <= 0) return PAYNE_OK;
  DeviceGuard dg(c->device);
  int rc = ensure_workspace(c, B);
  if (rc) return rc;
  rc = order_after_previous(c, (cudaStream_t)stream);
  if (rc) return rc;
  payne::EncodeParams E = c->enc;
  for (int i = 0; i < E.D_in; ++i) E.col[i] = i;
  E.star_fixed = nullptr; E.star_lay = nullptr;
  for (long long p0 = 0; p0 < B; p0 += c->slab) {
    const int nb = (int)std::min<long long>(c->slab, B - p0);
    int isd = 0;
    rc = run_mlp(c, E, x_dev + p0 * c->D_in, c->D_in, nb, y_dev + p0 * ldy, ldy, false, &isd, (cudaStream_t)stream);
    if (rc) return rc;
  }
  return mark_done(c, (cudaStream_t)stream);
}

int payne_ctx_attach_continuum(PayneCtx* c, const PayneSpecNet* cnet) {
  using namespace payne;
  if (!c || !cnet) return fail(PAYNE_E_INVALID, "null argument");
  if (!c->has_spec) return fail(PAYNE_E_INVALID, "context has no spectrum emulator");
  if (cnet->D_out < 2) return fail(PAYNE_E_INVALID, "continuum emulator needs at least two pixels");
  DeviceGuard dg(c->device);
  CU_TRY(cudaDeviceSynchronize());
  if (c->cont) { payne_ctx_destroy(c->cont); c->cont = nullptr; }
  PayneCtx* cc = new PayneCtx();
  cc->device = c->device; cc->sm_count = c->sm_count; cc->lay = c->lay;
  cc->has_spec = true; cc->has_phot = false;
  cc->slab = c->slab;
  int rc = PAYNE_OK;
  if (cudaMalloc((void**)&cc->status, sizeof(int)) != cudaSuccess) rc = fail(PAYNE_E_NOMEM, "status");
  if (!rc) rc = build_spec(cc, cnet, nullptr, /*emulator_only=*/true);
  cc->enc.star_fixed = c->enc.star_fixed; cc->enc.n_stars = c->enc.n_stars;   // labels: the same per-star values
  cc->enc.star_lay = c->enc.star_lay;                                          // ... and columns
  const int nc = cnet->D_out, n = c->D_out;
  cc->ldf = ((long long)nc + 3) / 4 * 4;
  std::vector<double> wc(cnet->wavelength, cnet->wavelength + nc), fac(nc);
  for (int j = 0; j + 1 < nc && !rc; ++j)
    if (!(wc[j + 1] > wc[j])) rc = fail(PAYNE_E_INVALID, "continuum wavelength grid must be strictly increasing");
  // F_nu -> F_lambda factor, speedoflight / (wave * 1e-8)**2 (predictspec.py:219)
  for (int j = 0; j < nc; ++j) { const double x = wc[j] * 1E-8; fac[j] = kSpeedOfLight / (x * x); }
  // np.interp bracket of every emulator pixel in the continuum grid, -1 outside (left = right = nan)
  std::vector<double> w(n);
  std::vector<int> br(n, -1);
  if (!rc) {
    CU_TRY(cudaMemcpy(w.data(), c->tail.w, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) {
      if (w[i] < wc[0] || w[i] > wc[nc - 1] || w[i] != w[i]) continue;
      int j = (int)(std::upper_bound(wc.begin(), wc.end(), w[i]) - wc.begin()) - 1;
      br[i] = std::min(std::max(j, 0), nc - 1);
    }
  }
  double *dfac = nullptr, *dwc = nullptr;
  int* dbr = nullptr;
  if (!rc) rc = upload_owned(cc, &dfac, fac.data(), nc);
  if (!rc) rc = upload_owned(cc, &dwc, wc.data(), nc);
  if (!rc) rc = upload_owned(cc, &dbr, br.data(), n);
  if (rc) { std::string keep = g_err; payne_ctx_destroy(cc); g_err = keep; return rc; }
  ContParams& C = c->contp;
  C.n_c = nc; C.fac = dfac; C.wc = dwc; C.n = n; C.w = c->tail.w; C.bracket = dbr;
  c->cont = cc;
  c->tail.rows_may_nan = 1;          // pixels outside the continuum coverage are NaN from here on
  return PAYNE_OK;
}

int payne_ctx_set_lsf(PayneCtx* c, const double* lsf_host, int64_t n) {
  using namespace payne;
  if (!c) return fail(PAYNE_E_INVALID, "null argument");
  if (!c->has_spec) return fail(PAYNE_E_INVALID, "context has no spectrum emulator");
  if (c->n_stars > 1) return fail(PAYNE_E_UNSUPPORTED, "the LSF vector is per observed pixel: not available on a context of several stars");
  DeviceGuard dg(c->device);
  CU_TRY(cudaDeviceSynchronize());
  if (!lsf_host) { c->lsf_on = false; return PAYNE_OK; }
  if (n != c->tail.n_obs) return fail(PAYNE_E_INVALID, "the LSF vector must have one dispersion per observed pixel");
  if (c->tail.log2N1 > 15) return fail(PAYNE_E_UNSUPPORTED, "LSF broadening is limited to emulator grids of 32768 pixels");
  for (int64_t j = 0; j < n; ++j)
    if (!(lsf_host[j] > 0.0)) return fail(PAYNE_E_INVALID, "LSF dispersions must be positive");
  int rc = lsf_alloc(c, n);
  if (rc) return rc;
  CU_TRY(cudaMemcpy((void*)c->lsf.lsf, lsf_host, (size_t)n * sizeof(double), cudaMemcpyHostToDevice));
  c->lsf_on = true;
  return PAYNE_OK;
}

int64_t payne_ctx_query(PayneCtx* c, const char* key) {
  if (!c || !key) return -1;
  std::string k(key);
  if (k == "n_ann") return c->D_out;
  if (k == "n_obs") return c->n_obs_max;
  if (k == "n_stars") return c->n_stars;
  if (k == "n_targets") return c->n_targets;
  if (k == "binary") return c->has_binary ? 1 : 0;
  if (k == "cont_marg") return c->has_marg ? 1 : 0;
  if (k == "n_obs_total") return c->n_obs_total;
  if (k == "nfft1") return c->has_spec ? (1LL << c->tail.log2N1) : 0;
  if (k == "launches") return c->launches;
  if (k == "grid_loguniform") return c->grid_loguniform;
  if (k == "fast_tail") return c->use_fast && c->allow_fast;
  if (k == "max_batch") return c->slab;
  if (k == "sm_count") return c->sm_count;
  if (k == "tail_grid") return c->tail_grid;
  if (k == "rot_window_floats") return c->fast.win_floats;
  if (k == "tail_cluster") return c->use_fast && c->allow_fast && c->use_cluster && c->allow_cluster;
  if (k == "gemm_stack") return c->use_stack;
  if (k == "tail_clusters") return c->cluster_n;
  if (k == "tail_cluster_ctas_per_sm") return c->cluster_occ;
  if (k == "precision") return c->lay.precision;
  if (k == "legacy_tc") return c->legacy && c->legacy_tc && c->lay.precision == PAYNE_PREC_PARITY;
  if (k == "continuum") return c->cont != nullptr;
  if (k == "lsf") return c->lsf_on;
  if (k == "status") {
    int v = 0;
    DeviceGuard dg(c->device);
    cudaDeviceSynchronize();
    cudaMemcpy(&v, c->status, sizeof(int), cudaMemcpyDeviceToHost);
    return v;
  }
  return -1;
}

int payne_ctx_set(PayneCtx* c, const char* key, int64_t value) {
  if (!c || !key) return fail(PAYNE_E_INVALID, "null argument");
  std::string k(key);
  if (k == "precision") {
    if (value < 0 || value > 4 || value == PAYNE_PREC_BF16) return fail(PAYNE_E_INVALID, "unknown precision");
    if (c->multinet && value != PAYNE_PREC_PARITY && value != PAYNE_PREC_SIMT_FP32)
      return fail(PAYNE_E_UNSUPPORTED, "multi-chunk emulator: precision must be 'parity' or 'simt'");
    if (value == PAYNE_PREC_PARITY && c->has_spec && !c->legacy)
      for (int k = 1; k < (c->multinet ? 4 : 6); ++k)
        if (c->dims_in[k] > payne::kX3MaxK)
          return fail(PAYNE_E_UNSUPPORTED, "parity precision supports hidden widths up to 512");
    c->lay.precision = (int)value;
    return PAYNE_OK;
  }
  if (k == "max_batch") {
    if (value < 1) return fail(PAYNE_E_INVALID, "max_batch must be positive");
    c->slab = value;
    return PAYNE_OK;
  }
  if (k == "timing") { c->timing = value != 0; return PAYNE_OK; }
  if (k == "fast_tail") { c->allow_fast = value != 0; return PAYNE_OK; }
  if (k == "tail_cluster") { c->allow_cluster = value != 0; return PAYNE_OK; }
  if (k == "gemm_stack") { c->use_stack = value != 0; return PAYNE_OK; }
  if (k == "tail_grid_cap") { c->grid_cap = (int)std::max<int64_t>(0, value); return PAYNE_OK; }
  if (k == "discard_rows") { c->tail.discard_rows = value != 0; return PAYNE_OK; }
  if (k == "rows_may_nan") { c->tail.rows_may_nan = value != 0; return PAYNE_OK; }
  // Inst_R column holds the sigma-resolution getspec takes (predictspec.py:255-263) instead of the FWHM
  // resolution the likelihood samples (genmod.py:82-85)
  if (k == "inst_r_is_sigma") { c->tail.inst_scale = value ? 1.0 : payne::kFwhmFit; return PAYNE_OK; }
  return fail(PAYNE_E_INVALID, "unknown key " + k);
}

int payne_gemm_test(const float* A_host, const float* W_host, const float* bias_host, int M, int N, int K,
                    int precision, int device, float* C_host) {
  using namespace payne;
  if (!A_host || !W_host || !bias_host || !C_host || M < 1 || N < 1 || K < 8) return fail(PAYNE_E_INVALID, "bad argument");
  CU_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU_TRY(cudaGetDeviceProperties(&prop, device));
  std::vector<void*> owned;
  TcWeights w;
  int rc = tc_prepare_weights_x(&w, W_host, N, K, &owned);
  TcActs a;
  const long long rows = (M + 127) / 128 * 128, ld = (K + 7) / 8 * 8;
  float *dA = nullptr, *dC = nullptr, *db = nullptr;
  if (!rc) rc = tc_alloc_acts_x(&a, rows, ld);
  if (!rc && (cudaMalloc((void**)&dA, (size_t)M * K * 4) != cudaSuccess ||
              cudaMalloc((void**)&dC, (size_t)M * N * 4) != cudaSuccess ||
              cudaMalloc((void**)&db, (size_t)N * 4) != cudaSuccess)) rc = fail(PAYNE_E_NOMEM, "gemm_test alloc");
  if (!rc) {
    cudaMemcpy(dA, A_host, (size_t)M * K * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(db, bias_host, (size_t)N * 4, cudaMemcpyHostToDevice);
    rc = tc_gemm_test_x(dA, M, N, K, precision, a, w, db, dC, prop.multiProcessorCount);
    if (rc) fail(rc, "gemm_test launch failed");
    if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = fail(PAYNE_E_CUDA, cudaGetErrorString(cudaGetLastError()));
    if (!rc) cudaMemcpy(C_host, dC, (size_t)M * N * 4, cudaMemcpyDeviceToHost);
  }
  tc_free_acts_x(&a);
  if (dA) cudaFree(dA); if (dC) cudaFree(dC); if (db) cudaFree(db);
  for (void* p : owned) cudaFree(p);
  return rc;
}

int payne_fft_test(const float* x_host, int log2N, const float* H_host, int device, float* y_host) {
  if (!x_host || !H_host || !y_host || log2N < 5 || log2N > 15) return fail(PAYNE_E_INVALID, "bad argument");
  CU_TRY(cudaSetDevice(device));
  const int N = 1 << log2N;
  std::vector<float2> tw(N / 2);                       // the tails' table (build_tail) for an N-sample transform
  for (int e = 0; e < N / 2; ++e) tw[e] = unit_round(-2.0 * 3.14159265358979323846 * (double)e / (double)N);
  float *dx = nullptr, *dH = nullptr, *dy = nullptr;
  float2* dtw = nullptr;
  int rc = PAYNE_OK;
  if (cudaMalloc((void**)&dx, (size_t)N * 4) != cudaSuccess || cudaMalloc((void**)&dy, (size_t)N * 4) != cudaSuccess ||
      cudaMalloc((void**)&dH, (size_t)(N / 2 + 1) * 4) != cudaSuccess ||
      cudaMalloc((void**)&dtw, (size_t)(N / 2) * sizeof(float2)) != cudaSuccess)
    rc = fail(PAYNE_E_NOMEM, "fft_test alloc");
  if (!rc) {
    cudaMemcpy(dx, x_host, (size_t)N * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dH, H_host, (size_t)(N / 2 + 1) * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(dtw, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice);
    rc = payne::launch_fft_test(dx, log2N, dH, dtw, dy);
    if (rc) fail(rc, "fft_test launch failed");
    if (!rc && cudaDeviceSynchronize() != cudaSuccess) rc = fail(PAYNE_E_CUDA, cudaGetErrorString(cudaGetLastError()));
    if (!rc) cudaMemcpy(y_host, dy, (size_t)N * 4, cudaMemcpyDeviceToHost);
  }
  if (dx) cudaFree(dx); if (dy) cudaFree(dy); if (dH) cudaFree(dH); if (dtw) cudaFree(dtw);
  return rc;
}

double payne_ctx_last_ms(PayneCtx* c, int which) {
  if (!c || which < 0 || which > 2 || !c->timing) return -1.0;
  if (!c->ms_valid) {
    for (auto& evs : c->pending) {
      if (cudaEventSynchronize(evs[3]) != cudaSuccess) return -1.0;
      for (int i = 0; i < 3; ++i) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, evs[i], evs[i + 1]);
        c->ms_acc[i == 0 ? 0 : (i == 1 ? 2 : 1)] += ms;   // [mlp, phot, tail] -> which {0,2,1}
      }
      for (auto e : evs) cudaEventDestroy(e);
    }
    c->pending.clear();
    c->ms_valid = true;
  }
  return c->ms_acc[which];
}

}  // extern "C"
