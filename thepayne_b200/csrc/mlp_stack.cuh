// lin2 .. lin5 of the sigmoid emulator (Payne/train/NNmodels.py:154-162) as ONE launch: a thread-block cluster of
// H/64 CTAs owns a 128-row tile of the batch through all hidden layers.
//
// Layer by layer (tc_gemm_kernel<64, X3, 1>) every hidden layer is a launch of its own: ~12 us each at C2 for 1.7 us
// of tensor-core work -- launch + prologue (barriers, TMEM allocation, descriptor prefetch), the first operand
// fetch, the epilogue and the drain are all exposed four times, and a B = 1 call is a chain of eight
// latency-bound launches.  Here CTA r of the cluster computes output columns [64 r, 64 r + 64) of every layer for
// its row tile: same ring of TMA stages, same six-MMA exact-accumulation split, same register epilogue
// (sigmoid, three bf16 slices, 16-byte stores) as the per-layer kernel -- the results are bit-identical.
// Between two layers the CTAs of a cluster meet at a cluster barrier (release / acquire at cluster scope, plus
// fence.proxy.async on both sides: the next layer's TMA loads read, through the async proxy, the activation
// slices the peers just wrote with ordinary stores).  Row tiles are independent of each other, so there is no
// grid-wide synchronisation, and the weights of the next layer (which do not depend on the barrier) are already
// in flight when it opens: the producer issues their loads into the ring before it arrives.
#pragma once
#include "mlp_tc.cuh"

namespace payne {

template <int kDummy = 0>
__global__ void __launch_bounds__(TcThreads<kModeX3, 1>::value, 1)
tc_hidden_stack_kernel(const __grid_constant__ TcStackMaps T, const __grid_constant__ TcStackArgs G) {
  using Cfg = TcCfg<64, kModeX3>;
  constexpr int BN = 64, NS = Cfg::kStages, NP = 3;
  static_assert(Cfg::kPatchBytes == 0, "the hidden-layer epilogue stays in registers");
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = (unsigned char*)(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
  unsigned char* stages = base;
  uint64_t* bars = (uint64_t*)(base + NS * Cfg::kStageBytes);
  uint64_t* full = bars;                 // [NS]
  uint64_t* empty = bars + NS;           // [NS]
  uint64_t* tfull = bars + 2 * NS;       // [2]
  uint64_t* tempty = bars + 2 * NS + 2;  // [2]
  uint32_t* tmem_ptr = (uint32_t*)(bars + 2 * NS + 4);
  float* sbias = (float*)(bars + 32);    // 256 bytes reserved for barriers
  float* sscale = sbias + BN;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cn = G.H / BN;                                // CTAs per cluster = column tiles of a layer
  const int m0 = ((int)blockIdx.x / cn) * kBM, n0 = ((int)blockIdx.x % cn) * BN;
  const int num_kb = G.H / Cfg::kBK;
  constexpr int kEpiWarps = TcThreads<kModeX3, 1>::kEpiWarps;

  if (warp == 0 && lane == 0) {
    for (int b = 0; b < 2; ++b)
      for (int p = 0; p < NP; ++p) ptx::prefetch_tmap(&T.a[b][p]);
    for (int l = 0; l < G.layers; ++l)
      for (int p = 0; p < NP; ++p) ptx::prefetch_tmap(&T.b[l][p]);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < NS; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { ptx::mbar_init(&tfull[a], 1); ptx::mbar_init(&tempty[a], kEpiWarps); }
    ptx::fence_barrier_init();
  }
  if (warp == 2) ptx::tmem_alloc(tmem_ptr, Cfg::kTmemCols);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // programmatic dependent launch, as in tc_gemm_kernel: the prologue above ran under the previous kernel's drain
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  // ring / accumulator state of the three roles (each role only uses its own)
  int s = 0; uint32_t ph = 0;        // producer and MMA issuer walk the ring in the same order
  int acc = 0; uint32_t aph = 0;     // MMA issuer and epilogue alternate the two accumulators
  int npre = 0;                      // producer: leading stages of this layer whose weight loads are already issued

  for (int l = 0; l < G.layers; ++l) {
    const int src = (G.first + l) & 1, dst = src ^ 1;
    if (warp == 0) {
      // ===================== TMA producer
      if (lane == 0) {
        if (l > 0) asm volatile("fence.proxy.async;" ::: "memory");   // peers' activation stores -> async proxy
        for (int kb = 0; kb < num_kb; ++kb) {
          unsigned char* st = stages + s * Cfg::kStageBytes;
          const int k0 = kb * Cfg::kBK;
          if (kb >= npre) {
            ptx::mbar_wait(&empty[s], ph ^ 1);
            ptx::mbar_expect_tx(&full[s], Cfg::kStageBytes);
#pragma unroll
            for (int p = 0; p < NP; ++p) ptx::tma_load_2d(&T.b[l][p], &full[s], st + NP * Cfg::kABytes + p * Cfg::kBBytes, k0, n0);
          }
#pragma unroll
          for (int p = 0; p < NP; ++p) ptx::tma_load_2d(&T.a[src][p], &full[s], st + p * Cfg::kABytes, k0, m0);
          if (++s == NS) { s = 0; ph ^= 1; }
        }
        // weights of the next layer do not wait for the barrier: into the ring now (slots free up as this layer's
        // MMAs retire), the activation halves of the same stages follow once the barrier has opened
        npre = 0;
        if (l + 1 < G.layers) {
          int ps = s; uint32_t pph = ph;
          const int want = num_kb < NS ? num_kb : NS;
          for (int kb = 0; kb < want; ++kb) {
            unsigned char* st = stages + ps * Cfg::kStageBytes;
            ptx::mbar_wait(&empty[ps], pph ^ 1);
            ptx::mbar_expect_tx(&full[ps], Cfg::kStageBytes);
#pragma unroll
            for (int p = 0; p < NP; ++p)
              ptx::tma_load_2d(&T.b[l + 1][p], &full[ps], st + NP * Cfg::kABytes + p * Cfg::kBBytes, kb * Cfg::kBK, n0);
            if (++ps == NS) { ps = 0; pph ^= 1; }
          }
          npre = want;
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      // ===================== MMA issuer
      if (lane == 0) {
        constexpr uint32_t idesc = umma_idesc(BN, 1u);
        ptx::mbar_wait(&tempty[acc], aph ^ 1);
        ptx::tc_fence_after();
        const uint32_t d_main = tmem_base + (uint32_t)(acc * Cfg::kAccCols);
        const uint32_t d_corr = d_main + BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(&full[s], ph);
          ptx::tc_fence_after();
          const uint32_t st = ptx::smem_u32(stages + s * Cfg::kStageBytes);
          uint64_t da[3], db[3];
#pragma unroll
          for (int p = 0; p < NP; ++p) {
            da[p] = umma_desc_k_sw128(st + p * Cfg::kABytes);
            db[p] = umma_desc_k_sw128(st + NP * Cfg::kABytes + p * Cfg::kBBytes);
          }
#pragma unroll
          for (int ks = 0; ks < Cfg::kBK / Cfg::kUmmaK; ++ks) {
            const uint64_t ko = (uint64_t)((ks * 32) >> 4);
            const uint32_t first = (kb | ks) != 0;
            ptx::mma_bf16(d_main, da[0] + ko, db[0] + ko, idesc, first);       // p1 q1 (exact)
            ptx::mma_bf16(d_corr, da[0] + ko, db[2] + ko, idesc, first);       // p1 q3
            ptx::mma_bf16(d_corr, da[1] + ko, db[1] + ko, idesc, 1);           // p2 q2
            ptx::mma_bf16(d_corr, da[2] + ko, db[0] + ko, idesc, 1);           // p3 q1
            ptx::mma_bf16(d_corr, da[0] + ko, db[1] + ko, idesc, 1);           // p1 q2
            ptx::mma_bf16(d_corr, da[1] + ko, db[0] + ko, idesc, 1);           // p2 q1
          }
          ptx::mma_commit(&empty[s]);
          if (kb == num_kb - 1) ptx::mma_commit(&tfull[acc]);
          if (++s == NS) { s = 0; ph ^= 1; }
        }
        if (++acc == 2) { acc = 0; aph ^= 1; }
      }
      __syncwarp();
    } else if (warp >= 4) {
      // ===================== epilogue: thread = row, 16 columns per warp group (as tc_gemm_kernel, EPI 1)
      const int q = warp & 3;
      constexpr int kEpiThreads = 32 * kEpiWarps;
      ptx::epi_bar_sync_n<kEpiThreads>();            // the previous layer's readers of sbias / sscale are done
      for (int cix = threadIdx.x - 128; cix < BN; cix += kEpiThreads) {
        sbias[cix] = __ldg(G.bias[l] + n0 + cix);
        sscale[cix] = __ldg(G.wscale[l] + n0 + cix);
      }
      ptx::epi_bar_sync_n<kEpiThreads>();
      ptx::mbar_wait(&tfull[acc], aph);
      ptx::tc_fence_after();
      const int grow = m0 + q * 32 + lane;
      const bool rowok = grow < G.M;
      const uint32_t t_main = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * Cfg::kAccCols);
      constexpr int NG = kEpiWarps / 4, CW = BN / NG;
      static_assert(CW == 16, "hidden-layer epilogue: 16 columns per warp group");
      const int cbase = ((warp - 4) >> 2) * CW, col0 = n0 + cbase;
      uint32_t v[CW], c[CW];
      ptx::tmem_ld16_nowait(t_main + (uint32_t)cbase, v);
      ptx::tmem_ld16_nowait(t_main + (uint32_t)(BN + cbase), c);
      ptx::tmem_ld_wait();
      const long long o = (long long)grow * G.ld + col0;
      const float4* b4 = reinterpret_cast<const float4*>(sbias + cbase);
      const float4* s4 = reinterpret_cast<const float4*>(sscale + cbase);
#pragma unroll
      for (int g8 = 0; g8 < CW / 8; ++g8) {
        __align__(16) __nv_bfloat16 q1[8], q2[8], q3[8];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const float4 bb = b4[2 * g8 + h], sc = s4[2 * g8 + h];
          const float bbv[4] = {bb.x, bb.y, bb.z, bb.w}, scv[4] = {sc.x, sc.y, sc.z, sc.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int j = 8 * g8 + 4 * h + e;
            const float val = sigmoidf_exact(fmaf(__uint_as_float(v[j]) + __uint_as_float(c[j]), scv[e], bbv[e]));
            x3_split_act(val, q1[4 * h + e], q2[4 * h + e], q3[4 * h + e]);
          }
        }
        if (rowok) {
          *reinterpret_cast<uint4*>((__nv_bfloat16*)G.plane[dst][0] + o + 8 * g8) = *reinterpret_cast<const uint4*>(q1);
          *reinterpret_cast<uint4*>((__nv_bfloat16*)G.plane[dst][1] + o + 8 * g8) = *reinterpret_cast<const uint4*>(q2);
          *reinterpret_cast<uint4*>((__nv_bfloat16*)G.plane[dst][2] + o + 8 * g8) = *reinterpret_cast<const uint4*>(q3);
        }
      }
      asm volatile("fence.proxy.async;" ::: "memory");   // these stores are read by the peers' TMA loads
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tempty[acc]);
      if (++acc == 2) { acc = 0; aph ^= 1; }
    }
    // every thread of every CTA of the cluster: the row tile's activations of layer l are complete and visible
    if (l + 1 < G.layers) ptx::cluster_sync_all();
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, Cfg::kTmemCols);
}

// The hidden layers tcw[1 .. layers] (all H -> H) from the sliced planes in `a0` ("first" buffer); the output of
// layer l lands in the other buffer, alternating.  Returns PAYNE_E_UNSUPPORTED when the shape does not fit
// (the caller then launches layer by layer).
inline int tc_launch_hidden_stack(const TcWeights* tcw, float* const* bias, int layers, int H, TcActs* a0, TcActs* a1,
                                  int M, cudaStream_t st, TcStackCache* cache) {
  using Cfg = TcCfg<64, kModeX3>;
  if (!cache || layers < 1 || layers > kStackMaxLayers) return PAYNE_E_UNSUPPORTED;
  if (!(H == 64 || H == 128 || H == 256 || H == 512)) return PAYNE_E_UNSUPPORTED;      // cluster of H/64 <= 8 CTAs
  if (a0->ld != a1->ld || a0->rows != a1->rows) return PAYNE_E_UNSUPPORTED;
  for (int l = 0; l < layers; ++l)
    if (tcw[1 + l].N != H || tcw[1 + l].K != H || !tcw[1 + l].xplane[0]) return PAYNE_E_UNSUPPORTED;
  TcStackCache& C = *cache;
  const long long rows = a0->rows >= M ? a0->rows : M;
  const void* key[6 + 3 * kStackMaxLayers] = {};
  for (int p = 0; p < 3; ++p) {
    key[p] = a0->plane[p]; key[3 + p] = a1->plane[p];
    for (int l = 0; l < layers; ++l) key[6 + 3 * l + p] = tcw[1 + l].xplane[p];
  }
  bool hit = C.valid && C.rows == rows && C.lda == a0->ld && C.H == H && C.layers == layers;
  for (int i = 0; i < 6 + 3 * kStackMaxLayers && hit; ++i) hit = C.ptr[i] == key[i];
  if (!hit) {
    C.valid = false;
    for (int p = 0; p < 3; ++p) {
      if (make_tmap(&C.maps.a[0][p], a0->plane[p], rows, H, a0->ld, kBM, 2)) return PAYNE_E_CUDA;
      if (make_tmap(&C.maps.a[1][p], a1->plane[p], rows, H, a1->ld, kBM, 2)) return PAYNE_E_CUDA;
      for (int l = 0; l < kStackMaxLayers; ++l) {
        const TcWeights& W = tcw[1 + (l < layers ? l : 0)];
        if (make_tmap(&C.maps.b[l][p], W.xplane[p], W.N, H, W.Kp, 64, 2)) return PAYNE_E_CUDA;
      }
    }
    for (int i = 0; i < 6 + 3 * kStackMaxLayers; ++i) C.ptr[i] = key[i];
    C.rows = rows; C.lda = a0->ld; C.H = H; C.layers = layers;
    C.valid = true;
  }
  static unsigned long long attr_set = 0;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return PAYNE_E_CUDA;
  if (dev >= 64 || !((attr_set >> dev) & 1ull)) {
    if (cudaFuncSetAttribute(tc_hidden_stack_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmem) != cudaSuccess)
      return PAYNE_E_CUDA;
    if (dev < 64) attr_set |= 1ull << dev;
  }
  TcStackArgs G{};
  for (int l = 0; l < layers; ++l) { G.bias[l] = bias[1 + l]; G.wscale[l] = tcw[1 + l].scale; }
  for (int p = 0; p < 3; ++p) { G.plane[0][p] = a0->plane[p]; G.plane[1][p] = a1->plane[p]; }
  G.ld = a0->ld; G.M = M; G.H = H; G.layers = layers; G.first = 0;
  const int cn = H / 64, num_m = (M + kBM - 1) / kBM;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(num_m * cn)); cfg.blockDim = dim3(TcThreads<kModeX3, 1>::value);
  cfg.dynamicSmemBytes = Cfg::kSmem; cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)cn; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = tc_pdl_enabled() ? 1 : 0;
  cfg.attrs = at; cfg.numAttrs = 2;
  if (cudaLaunchKernelEx(&cfg, tc_hidden_stack_kernel<0>, C.maps, G) != cudaSuccess) { cudaGetLastError(); return PAYNE_E_CUDA; }
  return PAYNE_OK;
}

}  // namespace payne
