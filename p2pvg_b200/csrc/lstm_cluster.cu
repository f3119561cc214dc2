// LSTM-layer scans on thread-block clusters (tensor-core mode): ONE launch runs all timesteps of a layer's recurrence
// (nn.LSTMCell, reference models/lstm.py:41,89).
//
// The recurrence is independent across batch rows, so the batch is cut into slabs of MB = 16*MT rows and each slab is owned
// by one cluster of 8 CTAs; CTA `rank` owns R/8 hidden units.  What makes a step cheap:
//   * the W_hh slice of the CTA never leaves the REGISTER FILE: every warp keeps the mma.sync B fragments of its (n tiles x
//     K range) for the whole sequence (128 registers per thread at R = 256), so a step streams only the 16 x R state
//     through shared memory instead of the 128 KB weight slice;
//   * steps are separated by the hardware cluster barrier (arrive.release / wait.acquire, ~0.2 us) instead of a grid-wide
//     barrier; the exchanged state (h_s forward, dG_s backward) is exactly what the kernel has to write to global memory
//     anyway -- the other 7 CTAs read it back from L2 (measured: DSMEM scatter is limited to ~20 B/clk per SM, slower);
//   * everything that does not depend on the recurrence (input-side pre-activations, saved gates) is requested before
//     the barrier.
// The recurrent product runs as mma.sync m16n8k8 TF32 with fp32 accumulation; activations use MUFU approximations whose
// error (<= 2^-11) is below the TF32 operand rounding.  The exact-fp32 parity mode uses the cooperative kernels of
// lstm_scan.cu instead.
//
//   forward :  gates_s = Pre_s + b_hh + h_{s-1} . W_hh^T ; (i,f,g,o) -> c_s, h_s
//   backward:  dh_s = dHtop_s + dG_{s+1} . W_hh ; cell pointwise backward -> dG_s, dc_{s-1}
#include "common.cuh"

namespace {

constexpr int CS = 8;    // CTAs per cluster
constexpr int NT = 256;  // threads per CTA
constexpr int PAD = 4;

__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void mma_tf32(float* c, const uint32_t* a, const uint32_t* b) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm volatile("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float round_tf32(float x) { return __uint_as_float(to_tf32(x)); }
__device__ __forceinline__ float fast_sigmoid(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float fast_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float4 ld_cg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }

// ------------------------------------------------------------------------------------------------ forward
// Warp w = (kh, ng): K half kh = w >> 2 (R/2 wide), n-tile group ng = w & 3 (TPW = R/64 tiles of 8 gate columns each).
template <int R, int MT>
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(NT, 1)
lstm_cl_fwd_kernel(const float* __restrict__ pre, const float* __restrict__ whh, const float* __restrict__ bhh, float* __restrict__ gates,
                   float* __restrict__ hs, float* __restrict__ cs, int S, int B) {
  constexpr int MB = 16 * MT, UBc = R / CS, NC = 4 * UBc, LD = R + PAD;
  constexpr int TPW = NC / 8 / 4;          // n8 tiles per warp
  constexpr int KS = R / 2 / 8;            // k8 steps per warp
  constexpr int CPT = (MB * UBc + NT - 1) / NT;
  constexpr int GL = NC + 1;
  extern __shared__ __align__(16) float sm[];
  float* Hb = sm;                          // [MB][LD]   h_{s-1} of the slab, TF32-rounded
  float* Gs = Hb + MB * LD;                // [2][MB][GL] partial gate pre-activations of the two K halves
  const int tid = threadIdx.x;
  const uint32_t rank = cluster_rank();
  const int r0 = (blockIdx.x / CS) * MB, u0 = (int)rank * UBc;
  const int warp = tid >> 5, lane = tid & 31, gq = lane >> 2, tq = lane & 3;
  const int kh = warp >> 2, ng = warp & 3;

  // resident B fragments: tile t covers gate columns n = (ng*TPW + t)*8 + gq  ->  W_hh row (n / UBc)*R + u0 + n % UBc
  uint32_t wreg[TPW][KS][2];
#pragma unroll
  for (int t = 0; t < TPW; t++) {
    const int n = (ng * TPW + t) * 8 + gq;
    const float* wrow = whh + (long long)((n / UBc) * R + u0 + (n % UBc)) * R + kh * (R / 2) + tq;
#pragma unroll
    for (int k = 0; k < KS; k++) {
      wreg[t][k][0] = to_tf32(wrow[k * 8]);
      wreg[t][k][1] = to_tf32(wrow[k * 8 + 4]);
    }
  }
  // pointwise cells of this thread: (row, unit) = (ci / UBc, ci % UBc), ci = tid + NT*h
  int crow[CPT], cuu[CPT];
  bool cok[CPT];
  float c_reg[CPT], bh[CPT][4];
#pragma unroll
  for (int h = 0; h < CPT; h++) {
    const int ci = tid + NT * h;
    crow[h] = ci / UBc;
    cuu[h] = ci - crow[h] * UBc;
    cok[h] = ci < MB * UBc && (r0 + crow[h]) < B;
    c_reg[h] = cok[h] ? cs[(long long)(r0 + crow[h]) * R + u0 + cuu[h]] : 0.f;  // cs[0]
#pragma unroll
    for (int g = 0; g < 4; g++) bh[h][g] = cok[h] ? bhh[g * R + u0 + cuu[h]] : 0.f;
  }

#ifdef LSTM_CL_PROFILE
  long long pf[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t0_ = clock64(), t1_;
#define PF(i) do { t1_ = clock64(); pf[i] += t1_ - t0_; t0_ = t1_; } while (0)
#else
#define PF(i)
#endif
  for (int s = 0; s < S; s++) {
    // input-side pre-activations of this step: independent of h, requested (not consumed) before the barrier
    float zp[CPT][4];
#pragma unroll
    for (int h = 0; h < CPT; h++) {
      const long long gbase = ((long long)s * B + r0 + crow[h]) * 4 * R + u0 + cuu[h];
#pragma unroll
      for (int g = 0; g < 4; g++) zp[h][g] = cok[h] ? __ldcs(pre + gbase + (long long)g * R) : 0.f;
    }
    PF(0);
    if (s > 0) cluster_wait();   // h_{s-1} of all 8 CTAs is in global memory / L2
    PF(1);
    // stage h_{s-1} rows [r0, r0+MB) (written by the other CTAs of the cluster: L1-bypassing loads)
    const float* hprev = hs + (long long)s * B * R;
    for (int i = tid; i < MB * (R / 4); i += NT) {
      const int row = i / (R / 4), k4 = i - row * (R / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r0 + row < B) v = ld_cg4(hprev + (long long)(r0 + row) * R + k4 * 4);
      v.x = round_tf32(v.x); v.y = round_tf32(v.y); v.z = round_tf32(v.z); v.w = round_tf32(v.w);
      *reinterpret_cast<float4*>(Hb + row * LD + k4 * 4) = v;
    }
    __syncthreads();
    PF(2);
    {
      float acc[MT][TPW][4];
#pragma unroll
      for (int m = 0; m < MT; m++)
#pragma unroll
        for (int t = 0; t < TPW; t++)
#pragma unroll
          for (int q = 0; q < 4; q++) acc[m][t][q] = 0.f;
      const float* ha = Hb + gq * LD + kh * (R / 2) + tq;
#pragma unroll
      for (int k = 0; k < KS; k++) {
#pragma unroll
        for (int m = 0; m < MT; m++) {
          uint32_t a[4];
          const float* hm = ha + m * 16 * LD + k * 8;
          a[0] = __float_as_uint(hm[0]); a[1] = __float_as_uint(hm[8 * LD]);
          a[2] = __float_as_uint(hm[4]); a[3] = __float_as_uint(hm[8 * LD + 4]);
#pragma unroll
          for (int t = 0; t < TPW; t++) mma_tf32(acc[m][t], a, wreg[t][k]);
        }
      }
      float* o = Gs + kh * MB * GL;
#pragma unroll
      for (int m = 0; m < MT; m++)
#pragma unroll
        for (int t = 0; t < TPW; t++) {
          float* p = o + (m * 16 + gq) * GL + (ng * TPW + t) * 8 + 2 * tq;
          p[0] = acc[m][t][0];
          p[1] = acc[m][t][1];
          p[8 * GL] = acc[m][t][2];
          p[8 * GL + 1] = acc[m][t][3];
        }
    }
    __syncthreads();
    PF(3);
    float outv[CPT][5];
#pragma unroll
    for (int h = 0; h < CPT; h++) {
      if (!cok[h]) continue;
      const int row = crow[h], uu = cuu[h];
      float z[4];
#pragma unroll
      for (int g = 0; g < 4; g++) z[g] = (Gs[row * GL + g * UBc + uu] + Gs[MB * GL + row * GL + g * UBc + uu]) + (zp[h][g] + bh[h][g]);
      const float ig = fast_sigmoid(z[0]), fg = fast_sigmoid(z[1]), gg = fast_tanh(z[2]), og = fast_sigmoid(z[3]);
      const float c = fg * c_reg[h] + ig * gg;
      c_reg[h] = c;
      // the state the other CTAs wait for goes out first
      hs[((long long)(s + 1) * B + r0 + row) * R + u0 + uu] = og * fast_tanh(c);
      outv[h][0] = ig; outv[h][1] = fg; outv[h][2] = gg; outv[h][3] = og; outv[h][4] = c;
    }
    PF(4);
    if (s < S - 1) cluster_arrive();   // release: h_s is visible to the cluster
    PF(5);
#pragma unroll
    for (int h = 0; h < CPT; h++) {
      if (!cok[h]) continue;
      const long long gbase = ((long long)s * B + r0 + crow[h]) * 4 * R + u0 + cuu[h];
      gates[gbase] = outv[h][0];
      gates[gbase + R] = outv[h][1];
      gates[gbase + 2LL * R] = outv[h][2];
      gates[gbase + 3LL * R] = outv[h][3];
      cs[((long long)(s + 1) * B + r0 + crow[h]) * R + u0 + cuu[h]] = outv[h][4];
    }
    PF(6);
  }
#ifdef LSTM_CL_PROFILE
  if (blockIdx.x == 0 && tid == 0)
    printf("fwd MT=%d cycles/step: prefetch %lld wait %lld stage %lld mma %lld pointwise %lld arrive %lld stores %lld\n", MT, pf[0] / S, pf[1] / S,
           pf[2] / S, pf[3] / S, pf[4] / S, pf[5] / S, pf[6] / S);
#endif
}

// ------------------------------------------------------------------------------------------------ backward
// dh_rec[row, uu] = sum_q dG_{s+1}[row, q] . W_hh[q, u0 + uu]   (K = 4R).  Warp w owns the K range [w*4R/8, (w+1)*4R/8) for
// all UBc/8 n tiles; the 8 partial results are summed through shared memory.
template <int R, int MT>
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(NT, 1)
lstm_cl_bwd_kernel(const float* __restrict__ dhtop, const float* __restrict__ whh, const float* __restrict__ gates,
                   const float* __restrict__ cs, float* __restrict__ dG, int S, int B) {
  constexpr int MB = 16 * MT, UBc = R / CS, K4 = 4 * R, LDW = K4 + PAD;
  constexpr int NTL = UBc / 8;             // n8 tiles
  constexpr int KS = K4 / 8 / 8;           // k8 steps per warp
  constexpr int CPT = (MB * UBc + NT - 1) / NT;
  constexpr int PL = UBc + 1;
  extern __shared__ __align__(16) float sm[];
  float* dGb = sm;                         // [MB][LDW]  dG_{s+1} of the slab, TF32-rounded
  float* Ps = dGb + MB * LDW;              // [8][MB][PL] partial products of the 8 K ranges
  const int tid = threadIdx.x;
  const uint32_t rank = cluster_rank();
  const int r0 = (blockIdx.x / CS) * MB, u0 = (int)rank * UBc;
  const int warp = tid >> 5, lane = tid & 31, gq = lane >> 2, tq = lane & 3;

  // resident B fragments: B[k = q][n = uu] = W_hh[q][u0 + uu], q in this warp's K range
  uint32_t wreg[NTL][KS][2];
#pragma unroll
  for (int t = 0; t < NTL; t++) {
    const float* wcol = whh + (long long)(warp * (K4 / 8) + tq) * R + u0 + t * 8 + gq;
#pragma unroll
    for (int k = 0; k < KS; k++) {
      wreg[t][k][0] = to_tf32(wcol[(long long)(k * 8) * R]);
      wreg[t][k][1] = to_tf32(wcol[(long long)(k * 8 + 4) * R]);
    }
  }
  int crow[CPT], cuu[CPT];
  bool cok[CPT];
  float dc_reg[CPT];
#pragma unroll
  for (int h = 0; h < CPT; h++) {
    const int ci = tid + NT * h;
    crow[h] = ci / UBc;
    cuu[h] = ci - crow[h] * UBc;
    cok[h] = ci < MB * UBc && (r0 + crow[h]) < B;
    dc_reg[h] = 0.f;
  }

  for (int it = 0; it < S; it++) {
    const int s = S - 1 - it;
    // saved activations of this thread's cells: independent of the recurrence, requested before the barrier
    float ig[CPT], fg[CPT], gg[CPT], og[CPT], cprev[CPT], cnow[CPT], dht[CPT];
#pragma unroll
    for (int h = 0; h < CPT; h++) {
      ig[h] = fg[h] = gg[h] = og[h] = cprev[h] = cnow[h] = dht[h] = 0.f;
      if (cok[h]) {
        const long long gbase = ((long long)s * B + r0 + crow[h]) * K4 + u0 + cuu[h];
        ig[h] = __ldcs(gates + gbase); fg[h] = __ldcs(gates + gbase + R);
        gg[h] = __ldcs(gates + gbase + 2LL * R); og[h] = __ldcs(gates + gbase + 3LL * R);
        const long long o = ((long long)s * B + r0 + crow[h]) * R + u0 + cuu[h];   // cs[s] = c_{s-1}, cs[s+1] = c_s
        cprev[h] = __ldcs(cs + o);
        cnow[h] = __ldcs(cs + o + (long long)B * R);
        dht[h] = __ldcs(dhtop + o);
      }
    }
    float rec[CPT];
#pragma unroll
    for (int h = 0; h < CPT; h++) rec[h] = 0.f;
    if (it > 0) {
      cluster_wait();   // dG_{s+1} of all 8 CTAs is in global memory / L2
      const float* gnext = dG + (long long)(s + 1) * B * K4;
      for (int i = tid; i < MB * (K4 / 4); i += NT) {
        const int row = i / (K4 / 4), k4 = i - row * (K4 / 4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r0 + row < B) v = ld_cg4(gnext + (long long)(r0 + row) * K4 + k4 * 4);
        v.x = round_tf32(v.x); v.y = round_tf32(v.y); v.z = round_tf32(v.z); v.w = round_tf32(v.w);
        *reinterpret_cast<float4*>(dGb + row * LDW + k4 * 4) = v;
      }
      __syncthreads();
      float acc[MT][NTL][4];
#pragma unroll
      for (int m = 0; m < MT; m++)
#pragma unroll
        for (int t = 0; t < NTL; t++)
#pragma unroll
          for (int q = 0; q < 4; q++) acc[m][t][q] = 0.f;
      const float* ga = dGb + gq * LDW + warp * (K4 / 8) + tq;
#pragma unroll
      for (int k = 0; k < KS; k++) {
#pragma unroll
        for (int m = 0; m < MT; m++) {
          uint32_t a[4];
          const float* gm = ga + m * 16 * LDW + k * 8;
          a[0] = __float_as_uint(gm[0]); a[1] = __float_as_uint(gm[8 * LDW]);
          a[2] = __float_as_uint(gm[4]); a[3] = __float_as_uint(gm[8 * LDW + 4]);
#pragma unroll
          for (int t = 0; t < NTL; t++) mma_tf32(acc[m][t], a, wreg[t][k]);
        }
      }
      float* o = Ps + warp * MB * PL;
#pragma unroll
      for (int m = 0; m < MT; m++)
#pragma unroll
        for (int t = 0; t < NTL; t++) {
          float* p = o + (m * 16 + gq) * PL + t * 8 + 2 * tq;
          p[0] = acc[m][t][0];
          p[1] = acc[m][t][1];
          p[8 * PL] = acc[m][t][2];
          p[8 * PL + 1] = acc[m][t][3];
        }
      __syncthreads();
#pragma unroll
      for (int h = 0; h < CPT; h++) {
        if (!cok[h]) continue;
        float r = 0.f;
#pragma unroll
        for (int p = 0; p < 8; p++) r += Ps[p * MB * PL + crow[h] * PL + cuu[h]];
        rec[h] = r;
      }
    }
#pragma unroll
    for (int h = 0; h < CPT; h++) {
      if (!cok[h]) continue;
      const float dh = dht[h] + rec[h];
      const float tc = fast_tanh(cnow[h]);
      const float dc = dh * og[h] * (1.f - tc * tc) + dc_reg[h];
      dc_reg[h] = dc * fg[h];
      const long long gbase = ((long long)s * B + r0 + crow[h]) * K4 + u0 + cuu[h];
      dG[gbase] = dc * gg[h] * ig[h] * (1.f - ig[h]);
      dG[gbase + R] = dc * cprev[h] * fg[h] * (1.f - fg[h]);
      dG[gbase + 2LL * R] = dc * ig[h] * (1.f - gg[h] * gg[h]);
      dG[gbase + 3LL * R] = dh * tc * og[h] * (1.f - og[h]);
    }
    if (it < S - 1) cluster_arrive();   // release: dG_s is visible to the cluster
  }
}

template <int R, int MT> constexpr size_t fwd_smem() { return (size_t)(16 * MT * (R + PAD) + 2 * 16 * MT * (4 * (R / CS) + 1)) * sizeof(float); }
template <int R, int MT> constexpr size_t bwd_smem() { return (size_t)(16 * MT * (4 * R + PAD) + 8 * 16 * MT * (R / CS + 1)) * sizeof(float); }

template <int R, int MT>
int launch_fwd(const float* pre, const float* whh, const float* bhh, float* gates, float* hs, float* cs, int S, int B, cudaStream_t st) {
  static bool attr = false;
  constexpr size_t smem = fwd_smem<R, MT>();
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(lstm_cl_fwd_kernel<R, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { p2pvg_set_error("lstm_cl_fwd: %s", cudaGetErrorString(e)); return P2PVG_ERR_CUDA; }
    attr = true;
  }
  lstm_cl_fwd_kernel<R, MT><<<CS * cdiv(B, 16 * MT), NT, smem, st>>>(pre, whh, bhh, gates, hs, cs, S, B);
  return p2pvg_check_launch("lstm_cl_fwd");
}
template <int R, int MT>
int launch_bwd(const float* dhtop, const float* whh, const float* gates, const float* cs, float* dG, int S, int B, cudaStream_t st) {
  static bool attr = false;
  constexpr size_t smem = bwd_smem<R, MT>();
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(lstm_cl_bwd_kernel<R, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { p2pvg_set_error("lstm_cl_bwd: %s", cudaGetErrorString(e)); return P2PVG_ERR_CUDA; }
    attr = true;
  }
  lstm_cl_bwd_kernel<R, MT><<<CS * cdiv(B, 16 * MT), NT, smem, st>>>(dhtop, whh, gates, cs, dG, S, B);
  return p2pvg_check_launch("lstm_cl_bwd");
}

}  // namespace

bool p2pvg_lstm_cluster_supported(int R) { return R == 64 || R == 128 || R == 256; }

// diagnostics: cudaOccupancyMaxActiveClusters of the R = 256 scans (clusters of 8): which = 0 fwd MT=1, 1 fwd MT=2, 2 bwd MT=1, 3 bwd MT=2
int p2pvg_lstm_cluster_max_clusters_impl(int which) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(CS * 64);
  cfg.blockDim = dim3(NT);
  int n = -1;
  cudaError_t e;
  if (which == 0) {
    cfg.dynamicSmemBytes = fwd_smem<256, 1>();
    cudaFuncSetAttribute(lstm_cl_fwd_kernel<256, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fwd_smem<256, 1>());
    e = cudaOccupancyMaxActiveClusters(&n, lstm_cl_fwd_kernel<256, 1>, &cfg);
  } else if (which == 1) {
    cfg.dynamicSmemBytes = fwd_smem<256, 2>();
    cudaFuncSetAttribute(lstm_cl_fwd_kernel<256, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fwd_smem<256, 2>());
    e = cudaOccupancyMaxActiveClusters(&n, lstm_cl_fwd_kernel<256, 2>, &cfg);
  } else if (which == 2) {
    cfg.dynamicSmemBytes = bwd_smem<256, 1>();
    cudaFuncSetAttribute(lstm_cl_bwd_kernel<256, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd_smem<256, 1>());
    e = cudaOccupancyMaxActiveClusters(&n, lstm_cl_bwd_kernel<256, 1>, &cfg);
  } else {
    cfg.dynamicSmemBytes = bwd_smem<256, 2>();
    cudaFuncSetAttribute(lstm_cl_bwd_kernel<256, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd_smem<256, 2>());
    e = cudaOccupancyMaxActiveClusters(&n, lstm_cl_bwd_kernel<256, 2>, &cfg);
  }
  if (e != cudaSuccess) { (void)cudaGetLastError(); return -1; }
  return n;
}

// rows per slab: 32 (MT = 2) above this batch size
constexpr int kMt2Above = 128;

// 8 clusters of 8 CTAs are co-resident on a B200 (measured): slabs of 32 rows keep up to 256 rows in one wave
int p2pvg_lstm_cluster_fwd_impl(const float* pre, const float* whh, const float* bhh, float* gates, float* hs, float* cs, int S, int B,
                                int R, cudaStream_t st) {
  if (S <= 0 || B <= 0) return P2PVG_OK;
  const bool two = B > kMt2Above;
  switch (R) {
    case 64: return two ? launch_fwd<64, 2>(pre, whh, bhh, gates, hs, cs, S, B, st) : launch_fwd<64, 1>(pre, whh, bhh, gates, hs, cs, S, B, st);
    case 128: return two ? launch_fwd<128, 2>(pre, whh, bhh, gates, hs, cs, S, B, st) : launch_fwd<128, 1>(pre, whh, bhh, gates, hs, cs, S, B, st);
    case 256: return two ? launch_fwd<256, 2>(pre, whh, bhh, gates, hs, cs, S, B, st) : launch_fwd<256, 1>(pre, whh, bhh, gates, hs, cs, S, B, st);
  }
  p2pvg_set_error("lstm cluster scan: hidden size %d not in {64,128,256}", R);
  return P2PVG_ERR_UNSUPPORTED;
}

int p2pvg_lstm_cluster_bwd_impl(const float* dhtop, const float* whh, const float* gates, const float* cs, float* dG, int S, int B, int R,
                                cudaStream_t st) {
  if (S <= 0 || B <= 0) return P2PVG_OK;
  const bool two = B > kMt2Above;
  switch (R) {
    case 64: return two ? launch_bwd<64, 2>(dhtop, whh, gates, cs, dG, S, B, st) : launch_bwd<64, 1>(dhtop, whh, gates, cs, dG, S, B, st);
    case 128: return two ? launch_bwd<128, 2>(dhtop, whh, gates, cs, dG, S, B, st) : launch_bwd<128, 1>(dhtop, whh, gates, cs, dG, S, B, st);
    case 256: return two ? launch_bwd<256, 2>(dhtop, whh, gates, cs, dG, S, B, st) : launch_bwd<256, 1>(dhtop, whh, gates, cs, dG, S, B, st);
  }
  p2pvg_set_error("lstm cluster scan: hidden size %d not in {64,128,256}", R);
  return P2PVG_ERR_UNSUPPORTED;
}
