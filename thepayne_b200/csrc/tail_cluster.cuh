// Fast fused tail for transforms that do not fit one CTA's shared memory (emulator grids above 16384 pixels:
// N1 = 32768 or 65536 samples), spread over a THREAD-BLOCK CLUSTER of four CTAs.  Same semantics as
// tail_fast.cuh (Payne/predict/predictspec.py:228-289, Payne/utils/smoothing.py:252-314, 588-668); what
// differs is where the transform lives:
//
//   The packed signal z[0, M) (M = N/2 complex points) is cut into four quarters of Q = M/4 points, one per
//   CTA of the cluster (64 KB each at N = 65536, so three CTAs stay resident per SM -- the single-CTA split
//   transform of tail_fast.cuh needs 128 KB and runs one CTA per SM with half the signal in an L2 scratch line).
//   One radix-4 decimation-in-frequency step ACROSS the quarters,
//       u_c[j] = W_M^{jc} * sum_q z[j + qQ] (-i)^{qc},        FFT_Q(u_c)[k'] = Z[4k' + c],
//   sends frequency class c to CTA c: CTA r interpolates the samples of j in [rQ/4, (r+1)Q/4) straight from the
//   emulator row (the regrid of smoothing.py:649-668 fused into the step, as in ct_pass0_regrid), does the
//   butterfly in registers and stores the four results into the four CTAs' buffers through distributed shared
//   memory (st.shared::cluster, coalesced 8-byte stores).  Every CTA then runs the Q-point transform of
//   fft_ct.cuh on its own class entirely in its own shared memory.
//   Filter stage: the pairs (k, M-k) of the real-signal untangling stay inside class 0 (k = 4k': partner
//   Q - k') and class 2 (k = 4k'+2: partner = bitwise complement of k'); classes 1 and 3 pair with EACH OTHER
//   (4k'+1 <-> 4(Q-1-k')+3), so CTA 1 and CTA 3 each take half of those pairs, reading and writing the
//   partner's element through distributed shared memory.
//   The inverse mirrors it: local inverse transforms, then a radix-4 decimation-in-time step across the
//   CTAs leaves CTA q with the natural-order samples [qN/4, (q+1)N/4), and the consumers (regrid back onto the
//   emulator grid; interpolation at the observed pixels + chi2) are split by sample range -- each CTA serves
//   the pixels whose bracketing samples it holds, reading only the one sample beyond its range remotely.
//   The four partial chi2 meet in CTA 0 (st.shared::cluster + cluster barrier, fixed summation order).
//
// All CTAs of a cluster read the same per-point record, so every branch around a cluster barrier is uniform
// across the cluster.  Points are handed out dynamically (CTA 0 claims the cluster's next point from a device counter
// and posts it to its peers, published by the point's last barrier); with the multi-GPU gather on, CTA 0's thread 0
// also stores the point's lnL into the other GPUs' buffers (tail.cuh store_lnl / gather_exit).
// compute-sanitizer (memcheck, racecheck, synccheck, initcheck) is clean on this kernel: profiles/r02_sanitizer.txt.
#pragma once
#include "tail_fast.cuh"

namespace payne {
namespace cl {

constexpr int kCluster = 4;

// -DPAYNE_CLUSTER_PROF: thread 0 of every CTA adds the clocks it spends per phase (barrier waits included)
// into cl_prof[]; payne_debug_cluster_prof() (tail_cluster_tu.cu) reads and clears it.
#ifdef PAYNE_CLUSTER_PROF
__device__ unsigned long long cl_prof[32];
#define CL_PROF_DECL long long prof_t = clock64();
#define CL_PROF(slot)                                                                   \
  do {                                                                                  \
    if (threadIdx.x == 0) {                                                             \
      const long long t_ = clock64();                                                   \
      atomicAdd(&::payne::cl::cl_prof[slot], (unsigned long long)(t_ - prof_t));                     \
      prof_t = t_;                                                                      \
    }                                                                                   \
  } while (0)
#else
#define CL_PROF_DECL
#define CL_PROF(slot) do { } while (0)
#endif

__device__ __forceinline__ unsigned cluster_rank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned cluster_id() { unsigned r; asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned n_clusters() { unsigned r; asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r)); return r; }
// all threads of all CTAs of the cluster; release/acquire at cluster scope (shared::cluster and global writes)
__device__ __forceinline__ void cluster_sync() {
#ifdef PAYNE_CLUSTER_RELAXED_EXPERIMENT   // timing experiment only: no ordering, results may be wrong
  asm volatile("barrier.cluster.arrive.relaxed.aligned;\n\tbarrier.cluster.wait.aligned;" ::: "memory");
#else
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
#endif
}
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t mapa(uint32_t a, unsigned rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
  return r;
}
__device__ __forceinline__ float2 ldc2(uint32_t a) {
  float2 v;
  asm volatile("ld.shared::cluster.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ float ldc1(uint32_t a) {
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void stc2(uint32_t a, float2 v) {
  asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(v.x), "f"(v.y) : "memory");
}
__device__ __forceinline__ void stc_f64(uint32_t a, double v) {
  asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory");
}

// The N real samples of a cluster-distributed transform: sample k lives in CTA k >> log2nq at local index
// k & (nq - 1).  Consumers mostly read their own quarter; the sample just beyond it comes from the neighbour.
struct ZCluster {
  float* zf;
  uint32_t zb;      // shared-window byte address of zf in this CTA
  int rank, log2nq;
  __device__ __forceinline__ float ld(int k) const {
    const int q = k >> log2nq;
    const int off = zidx(k & ((1 << log2nq) - 1));
    if (q == rank) return zf[off];
    return ldc1(mapa(zb, (unsigned)q) + 4u * (unsigned)off);
  }
};

// H restricted to frequency class 0: local k' -> H(4k')
template <class HF>
struct Bins4 {
  const HF& H;
  __device__ __forceinline__ float operator()(int k) const { return H(4 * k); }
};

// Radix-4 DIF step across the cluster with the regrid of the input row fused in (arithmetic of ct_pass0_regrid /
// regrid_in): complex element e = the pair of real samples (2e, 2e+1), sample k = np.interp at row position
// k * num / den.  CTA `rank` makes elements j in [rank Q/4, (rank+1) Q/4) of every class.
template <int LOG2MQ, bool CLEAN>
__device__ __forceinline__ void cross_dif_regrid(uint32_t zb, unsigned rank, const TwTab& tw, int tid,
                                                 const float* __restrict__ row, int num, int den, float invden,
                                                 float c) {
  constexpr int Q = 1 << LOG2MQ, JW = Q / kCluster, NB = JW / kNT;
  static_assert(JW % kNT == 0 && NB >= 1, "quarter too small for the cross step");
  uint32_t rb[kCluster];
#pragma unroll
  for (int q = 0; q < kCluster; ++q) rb[q] = mapa(zb, (unsigned)q);
  const int g0 = (int)rank * JW + tid;
  const long long v0 = 2LL * g0 * num;
  int j = (int)(v0 / den);
  int rem = (int)(v0 - (long long)j * den);
  const long long vi = 2LL * kNT * num, vm = 2LL * Q * num;
  const int ij = (int)(vi / den), ir = (int)(vi - (long long)ij * den);
  const int mj = (int)(vm / den), mr = (int)(vm - (long long)mj * den);
#pragma unroll 2
  for (int i = 0; i < NB; ++i) {
    const int g = g0 + kNT * i;
    // W_M^{g c}, M = 4Q: requested first, they arrive under the row loads
    const float2 w1 = tw_load<LOG2MQ + 2>(tw, g), w2 = tw_load<LOG2MQ + 2>(tw, 2 * g), w3 = tw_load<LOG2MQ + 2>(tw, 3 * g);
    float2 v[kCluster];
    {
      const float* src = row + j;
      int rr = rem;
#pragma unroll
      for (int m = 0; m < kCluster; ++m) {
        float a0 = src[0], a1 = src[1], a2 = src[2];
        if (!CLEAN) {
          if (a0 != a0) a0 = 0.f;
          if (a1 != a1) a1 = 0.f;
          if (a2 != a2) a2 = 0.f;
        }
        const int rem1 = rr + num;
        const bool same = rem1 < den;
        const float lo = same ? a0 : a1, hi = same ? a1 : a2;
        const float d0 = (float)rr * invden, d1 = (float)(same ? rem1 : rem1 - den) * invden;
        v[m].x = fmaf(fmaf(d0 * (d0 - 1.f), c, d0), a1 - a0, a0);
        v[m].y = fmaf(fmaf(d1 * (d1 - 1.f), c, d1), hi - lo, lo);
        rr += mr;
        int adv = mj;
        if (rr >= den) { rr -= den; ++adv; }
        src += adv;
      }
    }
    rem += ir;
    j += ij;
    if (rem >= den) { rem -= den; ++j; }
    dft4<false>(v);
    v[1] = cmul(v[1], w1);
    v[2] = cmul(v[2], w2);
    v[3] = cmul(v[3], w3);
    const uint32_t off = 8u * (unsigned)swz(g);
#pragma unroll
    for (int q = 0; q < kCluster; ++q) stc2(rb[q] + off, v[q]);
  }
}

// Radix-4 DIT step across the cluster (adjoint of the step above): natural-order quarter q ends up in CTA q.
// In place: slot g of every CTA is read and written by exactly one thread of the cluster.
template <int LOG2MQ>
__device__ __forceinline__ void cross_dit(uint32_t zb, unsigned rank, const TwTab& tw, int tid) {
  constexpr int Q = 1 << LOG2MQ, JW = Q / kCluster, NB = JW / kNT;
  uint32_t rb[kCluster];
#pragma unroll
  for (int q = 0; q < kCluster; ++q) rb[q] = mapa(zb, (unsigned)q);
#pragma unroll 2
  for (int i = 0; i < NB; ++i) {
    const int g = (int)rank * JW + tid + kNT * i;
    const uint32_t off = 8u * (unsigned)swz(g);
    const float2 w1 = tw_load<LOG2MQ + 2>(tw, g), w2 = tw_load<LOG2MQ + 2>(tw, 2 * g), w3 = tw_load<LOG2MQ + 2>(tw, 3 * g);
    float2 v[kCluster];
#pragma unroll
    for (int q = 0; q < kCluster; ++q) v[q] = ldc2(rb[q] + off);
    v[1] = cmulc(v[1], w1);
    v[2] = cmulc(v[2], w2);
    v[3] = cmulc(v[3], w3);
    dft4<true>(v);
#pragma unroll
    for (int q = 0; q < kCluster; ++q) stc2(rb[q] + off, v[q]);
  }
}

// Filter stage of frequency class cls in {1, 2, 3} on digit-reversed storage: local index k' stands for
// frequency k = 4k' + cls of the M = 4Q transform; its partner M - k = 4(Q-1-k') + (4 - cls) is the bitwise
// complement of k' in class 4 - cls, i.e. (row', c') = (Mlo-1-row, 15-c) in the buffer `zp` (this CTA's own for
// class 2, CTA 4-cls's for classes 1 and 3).  This CTA takes the pairs whose own element has klo < Mlo/2; for
// classes 1 and 3 the partner CTA takes the others, so every element is touched by one thread of the cluster.
// H(k), k in [0, M], includes the 1/M of the inverse.
template <int LOG2MQ, class HF>
__device__ __forceinline__ void filter_class(float2* z, uint32_t zp, int cls, const TwTab& tw, const HF& H, int tid) {
  using P = CtPlan<LOG2MQ>;
  constexpr int Q = 1 << LOG2MQ, Mlo = Q >> 4, M = 4 * Q;
  constexpr int NITEMS = (Mlo >> 1) << 4;
  const int c = tid & 15;
  // exp(-2 pi i k / N), N = 2M = 8Q, k = 4 klo + cls + 4 c Mlo: the last term is c/32 of a turn, a per-thread
  // constant, and the table factor depends on klo only (two distinct addresses per warp instead of 32)
  const float2 wc = tw_load<5>(tw, c);
  const int sh = tw.log2n - (LOG2MQ + 3);
#pragma unroll 2
  for (int w = tid; w < NITEMS; w += kNT) {
    const int klo = w >> 4;
    const int row = P::row_of(klo);
    const int k = 4 * (klo + (c << (LOG2MQ - 4))) + cls;
    const int pk = swz((row << 4) + c);
    const uint32_t pp = zp + 8u * (unsigned)swz(((Mlo - 1 - row) << 4) + (15 - c));
    const float2 Zk = z[pk], Zp = ldc2(pp);
    const float2 W = cmul(__ldg(tw.tab + ((4 * klo + cls) << sh)), wc);
    const float hk = H(k), hm = H(M - k);
    const float A = 0.5f * (hk + hm), Bc = 0.5f * (hk - hm);
    const float2 E = make_float2(0.5f * (Zk.x + Zp.x), 0.5f * (Zk.y - Zp.y));
    const float2 O = make_float2(0.5f * (Zk.y + Zp.y), -0.5f * (Zk.x - Zp.x));
    const float2 WO = cmul(W, O), WcE = cmulc(E, W);
    const float2 E2 = make_float2(A * E.x + Bc * WO.x, A * E.y + Bc * WO.y);
    const float2 O2 = make_float2(Bc * WcE.x + A * O.x, Bc * WcE.y + A * O.y);
    z[pk] = make_float2(E2.x - O2.y, E2.y + O2.x);
    stc2(pp, make_float2(E2.x + O2.y, O2.x - E2.y));
  }
}

// irfft(rfft(regrid(row)) * H) distributed over the cluster.  On entry no CTA of the cluster reads or writes
// any transform buffer (a cluster barrier lies behind); on return natural-order quarter q sits in CTA q and a
// cluster barrier has published it.
template <int LOG2MQ, class HF>
__device__ __forceinline__ void convolve_regrid(float2* z, uint32_t zb, unsigned rank, const TwTab& tw, const TwConst& tc,
                                                const HF& H, int tid, const float* row, int num, int den,
                                                float invden, float c, bool clean, int slot) {
  CL_PROF_DECL
  if (clean) cross_dif_regrid<LOG2MQ, true>(zb, rank, tw, tid, row, num, den, invden, c);
  else cross_dif_regrid<LOG2MQ, false>(zb, rank, tw, tid, row, num, den, invden, c);
  CL_PROF(slot + 0);
  cluster_sync();
  CL_PROF(slot + 1);
  ct_fwd_all_shared<LOG2MQ>(tw, tid);                    // z is the base of the dynamic shared memory
  CL_PROF(slot + 2);
  cluster_sync();                                       // the partner class is transformed too
  CL_PROF(slot + 3);
  if (rank == 0) ct_filter_pairs<LOG2MQ>(z, tw, Bins4<HF>{H}, tid);
  else filter_class<LOG2MQ>(z, mapa(zb, 4u - rank), (int)rank, tw, H, tid);
  CL_PROF(slot + 4);
  cluster_sync();
  CL_PROF(slot + 5);
  ct_inv_all_shared<LOG2MQ>(tw, tid);
  CL_PROF(slot + 6);
  cluster_sync();
  CL_PROF(slot + 7);
  cross_dit<LOG2MQ>(zb, rank, tw, tid);
  CL_PROF(slot + 8);
  cluster_sync();
  CL_PROF(slot + 9);
}

// Observed pixels whose bracketing sample k = floor(position) lies in this CTA's quarter (pixels left of the
// grid count for CTA 0, right of it for CTA 3: they make the residual NaN, smoothing.py:289).  Pixels
// [jlo, jhi) are scanned; ownership is tested per pixel, so any superset of the owned pixels is correct.
template <bool POLY, bool STARS, class ZV>
__device__ __forceinline__ double final_pass_part(const TailParams& P, const FastGrid& F, const PointSetup& S,
                                                  const FastSetup& FS, const ZV& zv, int tid, int p, int N2,
                                                  int rank, int log2nq, int jlo, int jhi) {
  // Four pixels per trip, loads grouped so that each trip exposes two memory latencies instead of four per pixel:
  // positions -> shared-memory samples -> interpolated depth; then the per-pixel constants -> residuals.  Few
  // values stay live across the groups (the kernel is compiled for 80 registers, and with 3 x 75 KB of shared
  // memory per SM there is next to no L1 to catch spills).
  // POLY: continuum polynomial and / or model output (m = (1 + d) chebval(x), r = m / sigma - flux / sigma;
  // fitutils.py:11-20, likelihood.py:95-97); otherwise r = d / sigma - (flux - 1) / sigma.
  const double nan = CUDART_NAN;
  const double pmax = (double)(N2 - 1);
  const float hdu = S.hdu;
  const double q0 = FS.q0, scale = FS.scale;
  const double* __restrict__ otab = POLY ? P.obs_ot : F.obs_otm1;
  const int off = obs_lo<STARS>(FS.obs);
  double acc = 0.0;
  constexpr int U = 4;
#pragma unroll 1
  for (int j0 = jlo + tid; j0 < jhi; j0 += U * kNT) {
    float d[U];
    unsigned okm = 0, minem = 0;
    {
      double q[U];
#pragma unroll
      for (int u = 0; u < U; ++u) q[u] = (j0 + u * kNT < jhi) ? __ldcg(F.obs_q + j0 + u * kNT) : -1.0;
      float g0[U], g1[U], dl[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const double pp = (q[u] - q0) * scale;
        const bool ok = (pp >= 0.0 && pp <= pmax);           // smoothing.py:289 left/right = nan
        const int k = ok ? min((int)pp, N2 - 2) : 0;
        const int owner = ok ? (k >> log2nq) : ((pp > pmax) ? kCluster - 1 : 0);
        const bool mine = (owner == rank) && (j0 + u * kNT < jhi);
        okm |= (unsigned)ok << u; minem |= (unsigned)mine << u;
        dl[u] = (float)(pp - (double)k);
        const int kk = mine ? k : (rank << log2nq);           // pixels of other CTAs read a harmless local sample
        g0[u] = zv.ld(kk); g1[u] = zv.ld(kk + 1);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) d[u] = fmaf(interp_w(dl[u], hdu), g1[u] - g0[u], g0[u]);
    }
    double is[U], ot[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const bool mine = (minem >> u) & 1u;
      is[u] = mine ? __ldcg(P.obs_inv_s + j0 + u * kNT) : 0.0;
      ot[u] = mine ? __ldcg(otab + j0 + u * kNT) : 0.0;
    }
    if (POLY) {
      double x[U];
#pragma unroll
      for (int u = 0; u < U; ++u) x[u] = (P.n_poly && ((minem >> u) & 1u)) ? __ldcg(P.obs_x + j0 + u * kNT) : 0.0;
      double cv[U];
      if (P.n_poly) chebval_dev4(x, S.poly, P.n_poly, cv);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        double m = ((okm >> u) & 1u) ? 1.0 + (double)d[u] : nan;
        if (P.n_poly) m *= cv[u];
        if ((minem >> u) & 1u) {
          if (P.model_out) P.model_out[(long long)p * P.ld_flux + (j0 + u * kNT - off)] = m;
          const double r = fma(m, is[u], -ot[u]);
          acc = fma(r, r, acc);
        }
      }
    } else {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        double r = fma((double)d[u], is[u], -ot[u]);
        if (!((okm >> u) & 1u)) r = nan;
        if ((minem >> u) & 1u) acc = fma(r, r, acc);
      }
    }
  }
  return acc;
}

}  // namespace cl

// One cluster of four CTAs owns one live point at a time.  LOG2N1 in {15, 16}; every CTA holds N1/8 complex
// points (32 / 64 KB) plus its own copy of the rotation-table window.
// (It keeps its own copies of the record load, the NaN model row, the window staging and the CTA reduction of tail.cuh:
// with those helpers the code of all four instantiations changed -- rot_window alone changed it for STARS -- and the
// 65536-sample single-star kernel's stack and spills went from 144 / 184 / 72 to 136 / 176 / 64 bytes.)
template <int LOG2N1, bool STARS>
__global__ void __launch_bounds__(kNT, 3)
tail_cluster_kernel(const __grid_constant__ TailParams P, const __grid_constant__ FastGrid F) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float2* z = reinterpret_cast<float2*>(smem_raw);
  float* zf = reinterpret_cast<float*>(smem_raw);
  __shared__ FastPoint SP;
  __shared__ double red[kNT / 32];
  __shared__ double cred[cl::kCluster];                  // CTA 0's copy collects the four partial chi2
  PointSetup& S = SP.S;
  FastSetup& FS = SP.FS;
  const int tid = threadIdx.x;
  const TwTab tw{P.tw, P.log2tw, P.twpass};
  const double nan = CUDART_NAN;
  constexpr int N1 = 1 << LOG2N1;
  constexpr int LOG2MQ = LOG2N1 - 3;                      // complex points per CTA
  constexpr int LOG2NQ = LOG2N1 - 2;                      // real samples per CTA
  const unsigned rank = cl::cluster_rank();
  const uint32_t zb = cl::smem_u32(zf);
  float* win = zf + (N1 >> 2);                            // rotation-table window behind the transform buffer
  const FastPoint* points = reinterpret_cast<const FastPoint*>(F.points);
  const ZSmem zs{zf};

  // Dynamic point scheduling: CTA 0 claims the cluster's next point at the top of a point and posts it into every
  // CTA's c_next[parity]; the point's last cluster barrier publishes it.  Two slots: CTA 0 may already be posting
  // point i+1's successor while a slower CTA still reads point i's.
  __shared__ int c_next[2];
  int pn, it = 0, win_have = 0;
  // no CTA touches a peer's shared memory before every CTA of the cluster has started (compute-sanitizer flags the
  // first remote stores otherwise); behind the loop nothing remote is pending: the last access to a peer lies before
  // the last point's final cluster barrier
  cl::cluster_sync();
  for (int p = (int)cl::cluster_id(); p < P.B; p = pn, it ^= 1) {
    float* row = P.flux + (long long)p * P.ldf;
    if (rank == 0 && tid == 0) {
      const int v = F.work_counter ? atomicAdd(F.work_counter, 1) : p + (int)cl::n_clusters();
      const uint32_t a = cl::smem_u32(&c_next[it]);
#pragma unroll
      for (unsigned r = 0; r < cl::kCluster; ++r)
        asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cl::mapa(a, r)), "r"(v) : "memory");
    }
    if (tid < (int)(sizeof(FastPoint) / 16))
      reinterpret_cast<int4*>(&SP)[tid] = __ldg(reinterpret_cast<const int4*>(points + p) + tid);
    __syncthreads();
    if (S.bad) {
      if (rank == 0) {
        if (P.model_out)
          for (int j = tid; j < obs_hi<STARS>(P, FS.obs) - obs_lo<STARS>(FS.obs); j += kNT) P.model_out[(long long)p * P.ld_flux + j] = nan;
        if (tid == 0 && P.lnl) store_lnl(P, p, nan);
      }
      cl::cluster_sync();
      pn = c_next[it];
      continue;
    }
    const int n = P.n;

    // ---------------- stage 1: rotational broadening on the full emulator grid
    if (S.do_rot) {
      const double xt_max = S.vsini_scale * (double)(N1 >> 1);
      float4* win4 = reinterpret_cast<float4*>(win);
      const int nwin = (int)fmin(fmin(xt_max + 2.0, (double)(F.win_floats >> 2)), (double)P.ntab);
      for (int i = win_have + tid; i < nwin; i += kNT) win4[i] = __ldg(P.sbtab + i);     // published by the first cluster barrier
      win_have = max(win_have, nwin);                     // what an earlier point staged stays valid
      const RotHT<2> H{P.sbtab, win4, nwin, S.vsini_scale, P.sb_h, 1.0f / (float)(N1 >> 1), P.ntab, RotHT<2>::fix40(S.vsini_scale)};
      cl::convolve_regrid<LOG2MQ>(z, zb, rank, tw, F.twc, H, tid, row, F.f_num, F.f_den, F.f_invden, F.c_native, S.clean != 0, 0);
      // back onto the emulator grid: this CTA makes the pixels whose left sample floor(i b_num / b_den) it holds
      const int blo = S.use_inst ? max(S.i0 - 1, 0) : 0, bhi = S.use_inst ? min(S.i1 + 1, n - 1) : n - 1;
      const long long nq = 1LL << LOG2NQ;
      const int ilo = (int)(((long long)rank * nq * F.b_den + F.b_num - 1) / F.b_num);
      const int ihi = rank == cl::kCluster - 1 ? n - 1 : (int)(((long long)(rank + 1) * nq * F.b_den + F.b_num - 1) / F.b_num) - 1;
      const cl::ZCluster zc{zf, zb, (int)rank, LOG2NQ};
      CL_PROF_DECL
      regrid_back(row, zc, F, tid, n, N1, max(blo, ilo), min(bhi, ihi));
      CL_PROF(10);
      cl::cluster_sync();                                // the rewritten row is visible to the whole cluster
      CL_PROF(11);
    }

    double acc = 0.0;
    CL_PROF_DECL
    if (S.use_inst) {
      // ---------------- stage 2: mask, regrid, Gaussian broadening
      const int log2N2 = S.log2N2, N2 = 1 << log2N2;
      const int i0 = S.i0;
      const GaussH H{S.taper_a, 2.0f / (float)N2};
      if (log2N2 >= LOG2N1 - 1) {
        const int log2nq2 = log2N2 - 2;
        if (log2N2 == LOG2N1)
          cl::convolve_regrid<LOG2MQ>(z, zb, rank, tw, F.twc, H, tid, row + i0, FS.s_num, FS.s_den, FS.s_invden, F.c_native, S.clean != 0, 12);
        else
          cl::convolve_regrid<LOG2MQ - 1>(z, zb, rank, tw, F.twc, H, tid, row + i0, FS.s_num, FS.s_den, FS.s_invden, F.c_native, S.clean != 0, 12);
        const cl::ZCluster zc{zf, zb, (int)rank, log2nq2};
        int jlo = obs_lo<STARS>(FS.obs), jhi = obs_hi<STARS>(P, FS.obs);   // the point's star
        if (STARS ? FS.jcut[0] >= 0 : F.obs_sorted != 0) {
          if (rank > 0) jlo = FS.jcut[rank - 1];
          if (rank < cl::kCluster - 1) jhi = FS.jcut[rank];
        }
#ifdef PAYNE_CLUSTER_PROF
        prof_t = clock64();
#endif
        if (P.n_poly == 0 && P.model_out == nullptr) acc = cl::final_pass_part<false, STARS>(P, F, S, FS, zc, tid, p, N2, (int)rank, log2nq2, jlo, jhi);
        else acc = cl::final_pass_part<true, STARS>(P, F, S, FS, zc, tid, p, N2, (int)rank, log2nq2, jlo, jhi);
        CL_PROF(22);
      } else if (rank == 0) {
        // small masks (N2 <= N1/4 fits one CTA's buffer): CTA 0 alone, runtime-planned transform
        stage_regrid(S, row, zs, tid, N2, FS.s_num, FS.s_den, i0, FS.s_invden, F.c_native, FS.s_incj, FS.s_incr);
        __syncthreads();
        const Twiddles twr{tw.tab, tw.log2n};
        FftPlan plan; plan.make(log2N2 - 1);
        fft_forward(z, log2N2 - 1, plan, twr, tid, kNT);
        filter_pairs(z, log2N2 - 1, plan, twr, H, tid, kNT);
        fft_inverse(z, log2N2 - 1, plan, twr, tid, kNT);
        acc = (P.n_poly == 0 && P.model_out == nullptr) ? final_pass<false, STARS>(P, F, S, FS, zs, tid, p, N2)
                                                        : final_pass<true, STARS>(P, F, S, FS, zs, tid, p, N2);
      }
    } else {
      // ---------------- no instrumental profile: plain np.interp (predictspec.py:288-289); pixels split evenly
      const double wlo = __ldg(P.w) * S.D, whi = __ldg(P.w + n - 1) * S.D;
      const int off = obs_lo<STARS>(FS.obs), no = obs_hi<STARS>(P, FS.obs) - off;
      const int jlo = off + (int)((long long)no * rank / cl::kCluster), jhi = off + (int)((long long)no * (rank + 1) / cl::kCluster);
      for (int j = jlo + tid; j < jhi; j += kNT) {
        const double x = __ldg(P.obs_w + j);
        double m;
        if (!(x >= wlo && x <= whi)) m = nan;
        else {
          const int g = (int)((__ldg(P.obs_lnw + j) - S.lnD - P.lnw0) * P.inv_dlnw);
          const int jj = locate(P.w, S.D, x, g, 0, n - 2);
          const double wa = __ldg(P.w + jj) * S.D, wb = __ldg(P.w + jj + 1) * S.D;
          const double a = (double)depth_of(row[jj], true, false);
          const double b = (double)depth_of(row[jj + 1], true, false);
          m = 1.0 + np_interp_pair(x, wa, wb, a, b);
        }
        if (P.n_poly) m *= chebval_dev(__ldg(P.obs_x + j), S.poly, P.n_poly);
        if (P.model_out) P.model_out[(long long)p * P.ld_flux + (j - off)] = m;
        const double r = m * __ldg(P.obs_inv_s + j) - __ldg(P.obs_ot + j);
        acc += r * r;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((tid & 31) == 0) red[tid >> 5] = acc;
    __syncthreads();
    if (tid == 0) {
      double c2 = 0.0;
#pragma unroll
      for (int wdx = 0; wdx < kNT / 32; ++wdx) c2 += red[wdx];
      cl::stc_f64(cl::mapa(cl::smem_u32(&cred[rank]), 0u), c2);
    }
    cl::cluster_sync();                                  // partial sums landed; nobody reads a transform buffer any more
    CL_PROF(23);
    pn = c_next[it];
    if (rank == 0 && tid == 0 && P.lnl) {
      double c2 = (cred[0] + cred[1]) + (cred[2] + cred[3]);
      if (P.chi2_sed) c2 += P.chi2_sed[p];
      store_lnl(P, p, -0.5 * c2);
    }
    // the consumed row is dropped from L2 without write-back (tail_fast.cuh); each CTA drops a quarter
    if (P.discard_rows) {
      const int a = (int)((long long)n * rank / cl::kCluster), b = (int)((long long)n * (rank + 1) / cl::kCluster);
      discard_lines(row + a, b - a, tid);
    }
  }
  if (tid == 0) gather_exit(P, gridDim.x);
}

}  // namespace payne
