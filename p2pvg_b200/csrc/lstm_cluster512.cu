// LSTM-layer scans for hidden size 512 (BASELINE config 5: human3.6m, rnn_size 512) on thread-block clusters of SIXTEEN CTAs.
// Same idea as lstm_cluster.cu (one launch = all timesteps of nn.LSTMCell, reference models/lstm.py:41,89; the W_hh slice of
// a CTA stays on chip for the whole sequence, steps are separated by the hardware cluster barrier), but W_hh is 4 MB here:
// 256 KB per CTA even at cluster size 16 (non-portable size, opt-in) -- more than the register file holds.  Half of every
// warp's mma.sync B fragments therefore live in REGISTERS (128 per thread) and the other half in SHARED MEMORY, stored
// fragment-major so that a warp reads 32 consecutive words (conflict-free).
//
//   forward : each CTA owns 32 hidden units (128 gate columns); the slab's h_{s-1} (32 rows x 512) comes back from L2,
//             gates_s = Pre_s + b_hh + h_{s-1} . W_hh^T, cell update, h_s to global memory (the exchange medium).
//   backward: dh_s = dHtop_s + dG_{s+1} . W_hh.  Splitting the OUTPUT units over the CTAs (lstm_cluster.cu) would need the whole
//             dG_{s+1} slab (16 rows x 2048) staged in every CTA next to a 128 KB weight half: it does not fit.  So the
//             REDUCTION is split instead: a CTA multiplies the dG columns it has just produced itself (its own 4 x 32 gate
//             columns, still in shared memory -- no exchange on the operand side) with W_hh[own rows, all 512 units] and
//             scatters the 16 x 512 partial products to their owners through distributed shared memory (st.shared::cluster,
//             double-buffered receive slots); the owner sums the 16 partials in a fixed order (deterministic).
// TF32 mma.sync m16n8k8 with fp32 accumulation, MUFU activations (error <= 2^-11, below the TF32 operand rounding) exactly
// as in lstm_cluster.cu.
#include <type_traits>

#include "common.cuh"

namespace {

constexpr int R = 512;
constexpr int CS = 16;   // CTAs per cluster (non-portable cluster size)
constexpr int NT = 256;  // threads per CTA
constexpr int PAD = 4;
constexpr int UBc = R / CS;  // 32 hidden units per CTA

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
// address of the same shared-memory variable in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t map_to_cta(const void* local_smem, uint32_t rank) {
  uint32_t l = (uint32_t)__cvta_generic_to_shared(local_smem), r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(l), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster_v2(uint32_t addr, float a, float b) {
  asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a), "f"(b) : "memory");
}

// 16 consecutive 32-bit columns of this thread's tensor-memory lane (lane = 32 * (warp % 4) + lane id): what a thread stores it
// reads back in the same registers
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
               "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]), "r"(v[10]),
               "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
               : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                 "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
               : "r"(taddr)
               : "memory");
}
// tcgen05.wait::ld naming the destination registers of the outstanding load, so that no use of them is scheduled above the wait
__device__ __forceinline__ void tmem_wait_ld16(uint32_t* v) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]), "+r"(v[9]),
                 "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
               :
               : "memory");
}

// ------------------------------------------------------------------------------------------------ forward
// Warp w = (kh, ng): K half kh = w >> 2 (256 wide = 32 k8 steps), n-tile group ng = w & 3 (4 tiles of 8 gate columns).
// k8 steps [0, KR) of a warp are register-resident, [KR, 32) shared-memory-resident.
template <int MT>
__global__ void __launch_bounds__(NT, 1)
lstm_cl16_fwd_kernel(const float* __restrict__ pre, const float* __restrict__ whh, const float* __restrict__ bhh, float* __restrict__ gates,
                     float* __restrict__ hs, float* __restrict__ cs, int S, int B) {
  constexpr int MB = 16 * MT, NC = 4 * UBc, LD = R + PAD;
  constexpr int TPW = NC / 8 / 4;          // 4 n8 tiles per warp
  constexpr int KS = R / 2 / 8;            // 32 k8 steps per warp
  constexpr int KR = 16, KSM = KS - KR;    // register / shared-memory resident steps
  constexpr int CPT = (MB * UBc + NT - 1) / NT;
  constexpr int GL = NC + 1;
  // 48-row slabs (MT = 3): the h slab alone takes what is left beside the weight half, so the partial gate sums are written
  // over the part of the slab that has already been consumed (rows 0..31 -> slab rows 0..15, rows 32..47 -> slab rows 16..23),
  // and the m16 tiles go through the tensor cores in two passes (2 + 1) to keep the accumulators at 32 registers.
  constexpr bool ALIAS = MT > 2;
  static_assert(MT <= 3, "slab rows");
  static_assert(!ALIAS || (2 * 32 * GL == 16 * LD && 2 * 16 * GL == 8 * LD), "aliased partial-sum regions");
  extern __shared__ __align__(16) float sm[];
  float* Wsm = sm;                                   // [8 warps][KSM][TPW][2][32 lanes]
  float* Hb = Wsm + 8 * KSM * TPW * 2 * 32;          // [MB][LD]   h_{s-1} of the slab, TF32-rounded
  float* Gs = ALIAS ? Hb : Hb + MB * LD;             // [2][rows][GL] partial gate pre-activations of the two K halves
  float* bsm = ALIAS ? Hb + MB * LD : Gs + 2 * MB * GL;   // [4][UBc] b_hh of my units
  // line of slab row `row`, K half h, in the partial-sum buffer
  auto gs_line = [&](int row, int h) -> float* {
    if constexpr (ALIAS) return row < 32 ? Gs + (h * 32 + row) * GL : Gs + 16 * LD + (h * 16 + row - 32) * GL;
    else return Gs + (h * MB + row) * GL;
  };
  const int tid = threadIdx.x;
  const uint32_t rank = cluster_rank();
  const int r0 = (blockIdx.x / CS) * MB, u0 = (int)rank * UBc;
  const int warp = tid >> 5, lane = tid & 31, gq = lane >> 2, tq = lane & 3;
  const int kh = warp >> 2, ng = warp & 3;

  // B fragments: tile t covers gate columns n = (ng*TPW + t)*8 + gq  ->  W_hh row (n / UBc)*R + u0 + n % UBc
  uint32_t wreg[TPW][KR][2];
#pragma unroll
  for (int t = 0; t < TPW; t++) {
    const int n = (ng * TPW + t) * 8 + gq;
    const float* wrow = whh + (long long)((n / UBc) * R + u0 + (n % UBc)) * R + kh * (R / 2) + tq;
#pragma unroll
    for (int k = 0; k < KR; k++) {
      wreg[t][k][0] = to_tf32(wrow[k * 8]);
      wreg[t][k][1] = to_tf32(wrow[k * 8 + 4]);
    }
    for (int k = 0; k < KSM; k++) {
      float* dst = Wsm + (((warp * KSM + k) * TPW + t) * 2) * 32 + lane;
      dst[0] = round_tf32(wrow[(KR + k) * 8]);
      dst[32] = round_tf32(wrow[(KR + k) * 8 + 4]);
    }
  }
  // pointwise cells of this thread: (row, unit) = (ci / UBc, ci % UBc), ci = tid + NT*h
  int crow[CPT], cuu[CPT];
  bool cok[CPT];
  float c_reg[CPT];
#pragma unroll
  for (int h = 0; h < CPT; h++) {
    const int ci = tid + NT * h;
    crow[h] = ci / UBc;
    cuu[h] = ci - crow[h] * UBc;
    cok[h] = ci < MB * UBc && (r0 + crow[h]) < B;
    c_reg[h] = cok[h] ? cs[(long long)(r0 + crow[h]) * R + u0 + cuu[h]] : 0.f;  // cs[0]
  }
  if (tid < 4 * UBc) bsm[tid] = bhh[(tid / UBc) * R + u0 + tid % UBc];
  __syncthreads();   // Wsm, bsm complete

  for (int s = 0; s < S; s++) {
    // input-side pre-activations of this step: independent of h, requested (not consumed) before the barrier
    float zp[CPT][4];
#pragma unroll
    for (int h = 0; h < CPT; h++) {
      const long long gbase = ((long long)s * B + r0 + crow[h]) * 4 * R + u0 + cuu[h];
#pragma unroll
      for (int g = 0; g < 4; g++) zp[h][g] = cok[h] ? __ldcs(pre + gbase + (long long)g * R) : 0.f;
    }
    if (s > 0) cluster_wait();   // h_{s-1} of all 16 CTAs is in global memory / L2
    const float* hprev = hs + (long long)s * B * R;
    for (int i = tid; i < MB * (R / 4); i += NT) {
      const int row = i / (R / 4), k4 = i - row * (R / 4);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r0 + row < B) v = ld_cg4(hprev + (long long)(r0 + row) * R + k4 * 4);
      v.x = round_tf32(v.x); v.y = round_tf32(v.y); v.z = round_tf32(v.z); v.w = round_tf32(v.w);
      *reinterpret_cast<float4*>(Hb + row * LD + k4 * 4) = v;
    }
    __syncthreads();
    const float* ha = Hb + gq * LD + kh * (R / 2) + tq;
    const float* wsm = Wsm + (warp * KSM * TPW * 2) * 32 + lane;
    // MC m16 tiles starting at slab row m0: acc = h[m0 .. m0+16 MC) . W_hh^T over this warp's K half and 4 n8 tiles
    auto gate_pass = [&](auto mc_tag, int m0) {
      constexpr int MC = decltype(mc_tag)::value;
      float acc[MC][TPW][4];
#pragma unroll
      for (int m = 0; m < MC; m++)
#pragma unroll
        for (int t = 0; t < TPW; t++)
#pragma unroll
          for (int q = 0; q < 4; q++) acc[m][t][q] = 0.f;
      const float* hp = ha + m0 * LD;
#pragma unroll
      for (int k = 0; k < KR; k++) {
#pragma unroll
        for (int m = 0; m < MC; m++) {
          uint32_t a[4];
          const float* hm = hp + m * 16 * LD + k * 8;
          a[0] = __float_as_uint(hm[0]); a[1] = __float_as_uint(hm[8 * LD]);
          a[2] = __float_as_uint(hm[4]); a[3] = __float_as_uint(hm[8 * LD + 4]);
#pragma unroll
          for (int t = 0; t < TPW; t++) mma_tf32(acc[m][t], a, wreg[t][k]);
        }
      }
#pragma unroll 4
      for (int k = 0; k < KSM; k++) {
        uint32_t b[TPW][2];
#pragma unroll
        for (int t = 0; t < TPW; t++) {
          b[t][0] = __float_as_uint(wsm[((k * TPW + t) * 2) * 32]);
          b[t][1] = __float_as_uint(wsm[((k * TPW + t) * 2 + 1) * 32]);
        }
#pragma unroll
        for (int m = 0; m < MC; m++) {
          uint32_t a[4];
          const float* hm = hp + m * 16 * LD + (KR + k) * 8;
          a[0] = __float_as_uint(hm[0]); a[1] = __float_as_uint(hm[8 * LD]);
          a[2] = __float_as_uint(hm[4]); a[3] = __float_as_uint(hm[8 * LD + 4]);
#pragma unroll
          for (int t = 0; t < TPW; t++) mma_tf32(acc[m][t], a, b[t]);
        }
      }
      if constexpr (ALIAS) {
        if (m0 == 0) __syncthreads();   // every warp is done with slab rows 0..31: their space now takes the partial sums
      }
#pragma unroll
      for (int m = 0; m < MC; m++)
#pragma unroll
        for (int t = 0; t < TPW; t++) {
          float* p = gs_line(m0 + m * 16 + gq, kh) + (ng * TPW + t) * 8 + 2 * tq;
          float* p8 = gs_line(m0 + m * 16 + gq + 8, kh) + (ng * TPW + t) * 8 + 2 * tq;
          p[0] = acc[m][t][0];
          p[1] = acc[m][t][1];
          p8[0] = acc[m][t][2];
          p8[1] = acc[m][t][3];
        }
    };
    if constexpr (MT == 1) gate_pass(std::integral_constant<int, 1>{}, 0);
    else gate_pass(std::integral_constant<int, 2>{}, 0);
    if constexpr (MT == 3) gate_pass(std::integral_constant<int, 1>{}, 32);
    __syncthreads();
    float outv[CPT][5];
#pragma unroll
    for (int h = 0; h < CPT; h++) {
      if (!cok[h]) continue;
      const int row = crow[h], uu = cuu[h];
      float z[4];
#pragma unroll
      for (int g = 0; g < 4; g++) z[g] = (gs_line(row, 0)[g * UBc + uu] + gs_line(row, 1)[g * UBc + uu]) + (zp[h][g] + bsm[g * UBc + uu]);
      const float ig = fast_sigmoid(z[0]), fg = fast_sigmoid(z[1]), gg = fast_tanh(z[2]), og = fast_sigmoid(z[3]);
      const float c = fg * c_reg[h] + ig * gg;
      c_reg[h] = c;
      hs[((long long)(s + 1) * B + r0 + row) * R + u0 + uu] = og * fast_tanh(c);   // the state the other CTAs wait for goes out first
      outv[h][0] = ig; outv[h][1] = fg; outv[h][2] = gg; outv[h][3] = og; outv[h][4] = c;
    }
    if (s < S - 1) cluster_arrive();   // release: h_s is visible to the cluster
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
  }
}

// ------------------------------------------------------------------------------------------------ backward
// Slab of 16 batch rows per cluster.  CTA `rank` owns units [32 rank, 32 rank + 32): the K index kk in [0,128) of its
// product is gate column q = (kk / 32) * R + u0 + kk % 32.  Warp w computes partial[16 rows][64 w .. 64 w + 64) (8 n8 tiles,
// 16 k8 steps: 8 register-resident, 8 shared-memory-resident) and sends it to CTAs 2w and 2w+1.
__global__ void __launch_bounds__(NT, 1)
lstm_cl16_bwd_kernel(const float* __restrict__ dhtop, const float* __restrict__ whh, const float* __restrict__ gates,
                     const float* __restrict__ cs, float* __restrict__ dG, int S, int B) {
  constexpr int MB = 16, K4 = 4 * R, KL = 4 * UBc;     // KL = 128 local reduction columns
  constexpr int NTL = 8;                               // n8 tiles per warp
  constexpr int KS = KL / 8;                           // 16 k8 steps
  constexpr int KR = 8, KSM = KS - KR;
  constexpr int LDA = KL + PAD;
  constexpr int CPT = (MB * UBc) / NT;                 // 2 cells per thread
  extern __shared__ __align__(16) float sm[];
  float* Wsm = sm;                                     // [8 warps][KSM][NTL][2][32 lanes]
  float* recv = Wsm + 8 * KSM * NTL * 2 * 32;          // [2][CS src][MB][UBc]  partial dh_rec for MY units, one slot per source CTA
  float* As = recv + 2 * CS * MB * UBc;                // [MB][LDA]  my dG columns of this step, TF32-rounded
  const int tid = threadIdx.x;
  const uint32_t rank = cluster_rank();
  const int r0 = (blockIdx.x / CS) * MB, u0 = (int)rank * UBc;
  const int warp = tid >> 5, lane = tid & 31, gq = lane >> 2, tq = lane & 3;

  // B fragments: B[k = kk][n] = W_hh[q(kk)][n], n = 64 warp + 8 t + gq
  uint32_t wreg[NTL][KR][2];
#pragma unroll
  for (int t = 0; t < NTL; t++) {
    const int n = warp * 64 + t * 8 + gq;
#pragma unroll
    for (int k = 0; k < KS; k++) {
      const int kk0 = k * 8 + tq, kk1 = kk0 + 4;
      const float w0 = whh[(long long)((kk0 / UBc) * R + u0 + kk0 % UBc) * R + n];
      const float w1 = whh[(long long)((kk1 / UBc) * R + u0 + kk1 % UBc) * R + n];
      if (k < KR) {
        wreg[t][k < KR ? k : 0][0] = to_tf32(w0);
        wreg[t][k < KR ? k : 0][1] = to_tf32(w1);
      } else {
        float* dst = Wsm + (((warp * KSM + (k - KR)) * NTL + t) * 2) * 32 + lane;
        dst[0] = round_tf32(w0);
        dst[32] = round_tf32(w1);
      }
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
    cok[h] = (r0 + crow[h]) < B;
    dc_reg[h] = 0.f;
  }
  // remote receive slots this thread writes: columns [64 warp + 8 t + 2 tq, +1] -> owner CTA (64 warp + 8 t) / 32, unit (8 t + 2 tq) % 32
  uint32_t raddr[2];   // base of recv in CTA 2*warp and 2*warp+1
  raddr[0] = map_to_cta(recv, 2 * warp);
  raddr[1] = map_to_cta(recv, 2 * warp + 1);
  __syncthreads();
  cluster_arrive();   // every CTA of the cluster has started (distributed shared memory may be written from here on)
  cluster_wait();

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
      cluster_wait();   // the 16 partial products for my units have arrived in recv[it & 1]
      const float* rb = recv + (it & 1) * CS * MB * UBc;
#pragma unroll
      for (int h = 0; h < CPT; h++) {
        float r = 0.f;
#pragma unroll
        for (int src = 0; src < CS; src++) r += rb[(src * MB + crow[h]) * UBc + cuu[h]];   // fixed order: deterministic
        rec[h] = r;
      }
    }
#pragma unroll
    for (int h = 0; h < CPT; h++) {
      float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
      if (cok[h]) {
        const float dh = dht[h] + rec[h];
        const float tc = fast_tanh(cnow[h]);
        const float dc = dh * og[h] * (1.f - tc * tc) + dc_reg[h];
        dc_reg[h] = dc * fg[h];
        d0 = dc * gg[h] * ig[h] * (1.f - ig[h]);
        d1 = dc * cprev[h] * fg[h] * (1.f - fg[h]);
        d2 = dc * ig[h] * (1.f - gg[h] * gg[h]);
        d3 = dh * tc * og[h] * (1.f - og[h]);
        const long long gbase = ((long long)s * B + r0 + crow[h]) * K4 + u0 + cuu[h];
        dG[gbase] = d0;
        dG[gbase + R] = d1;
        dG[gbase + 2LL * R] = d2;
        dG[gbase + 3LL * R] = d3;
      }
      float* a = As + crow[h] * LDA + cuu[h];
      a[0] = round_tf32(d0); a[UBc] = round_tf32(d1); a[2 * UBc] = round_tf32(d2); a[3 * UBc] = round_tf32(d3);
    }
    if (it < S - 1) {
      __syncthreads();   // As complete
      float acc[NTL][4];
#pragma unroll
      for (int t = 0; t < NTL; t++)
#pragma unroll
        for (int q = 0; q < 4; q++) acc[t][q] = 0.f;
      const float* ga = As + gq * LDA + tq;
#pragma unroll
      for (int k = 0; k < KR; k++) {
        uint32_t a[4];
        a[0] = __float_as_uint(ga[k * 8]); a[1] = __float_as_uint(ga[8 * LDA + k * 8]);
        a[2] = __float_as_uint(ga[k * 8 + 4]); a[3] = __float_as_uint(ga[8 * LDA + k * 8 + 4]);
#pragma unroll
        for (int t = 0; t < NTL; t++) mma_tf32(acc[t], a, wreg[t][k]);
      }
      const float* wsm = Wsm + (warp * KSM * NTL * 2) * 32 + lane;
#pragma unroll 2
      for (int k = 0; k < KSM; k++) {
        uint32_t a[4];
        a[0] = __float_as_uint(ga[(KR + k) * 8]); a[1] = __float_as_uint(ga[8 * LDA + (KR + k) * 8]);
        a[2] = __float_as_uint(ga[(KR + k) * 8 + 4]); a[3] = __float_as_uint(ga[8 * LDA + (KR + k) * 8 + 4]);
#pragma unroll
        for (int t = 0; t < NTL; t++) {
          uint32_t b[2];
          b[0] = __float_as_uint(wsm[((k * NTL + t) * 2) * 32]);
          b[1] = __float_as_uint(wsm[((k * NTL + t) * 2 + 1) * 32]);
          mma_tf32(acc[t], a, b);
        }
      }
      // scatter: tile t of warp w holds columns n = 64 w + 8 t + 2 tq (+1), rows gq and gq + 8 -> owner 2w + (t >> 2), unit
      // (8 t + 2 tq) & 31, slot [next parity][src = my rank]
      const uint32_t slot = (uint32_t)((((it + 1) & 1) * CS + (int)rank) * MB * UBc) * 4u;
#pragma unroll
      for (int t = 0; t < NTL; t++) {
        const uint32_t base = raddr[t >> 2] + slot + (uint32_t)(((t & 3) * 8 + 2 * tq) * 4);
        st_cluster_v2(base + (uint32_t)(gq * UBc * 4), acc[t][0], acc[t][1]);
        st_cluster_v2(base + (uint32_t)((gq + 8) * UBc * 4), acc[t][2], acc[t][3]);
      }
      cluster_arrive();   // release: my partial products are visible to their owners
    }
  }
}

// ------------------------------------------------------------------------------------------------ backward, 32 / 48-row slabs
// Same algorithm as lstm_cl16_bwd_kernel for slabs of MT m16 tiles.  The receive slots grow with the slab (64 KB per 16 rows,
// double-buffered) and leave no shared memory for a weight half, so the half that does not fit the registers lives in TENSOR
// MEMORY (256 KB per SM, otherwise unused by this kernel): 256 columns, written once with tcgen05.st in the fragment-major order
// the mma.sync B operands need and read back 16 columns per k8 step with tcgen05.ld, double-buffered against the MMAs.  The
// m16 tiles run one after the other (32 accumulator registers).  Why: only 7 clusters of 16 CTAs are resident at a time
// (cudaOccupancyMaxActiveClusters), so 256 rows in 16-row slabs need three passes over the sequence; 48-row slabs need one.
template <int MT>
__global__ void __launch_bounds__(NT, 1)
lstm_cl16_bwd_tm_kernel(const float* __restrict__ dhtop, const float* __restrict__ whh, const float* __restrict__ gates,
                        const float* __restrict__ cs, float* __restrict__ dG, int S, int B) {
  constexpr int MB = 16 * MT, K4 = 4 * R, KL = 4 * UBc;
  constexpr int NTL = 8, KS = KL / 8, KR = 8, KTM = KS - KR;
  constexpr int LDA = KL + PAD;
  constexpr int CPT = (MB * UBc) / NT;                  // 2 MT cells per thread
  constexpr uint32_t TCOLS = 2 * KTM * NTL * 2;          // 256 columns: [warp >> 2][k][tile][2]
  static_assert(KTM % 2 == 0 && TCOLS == 256, "tensor-memory layout");
  extern __shared__ __align__(16) float sm[];
  float* recv = sm;                                     // [2][CS src][MB][UBc]
  float* As = recv + 2 * CS * MB * UBc;                 // [MB][LDA]
  uint32_t* tslot = reinterpret_cast<uint32_t*>(As + MB * LDA);
  const int tid = threadIdx.x;
  const uint32_t rank = cluster_rank();
  const int r0 = (blockIdx.x / CS) * MB, u0 = (int)rank * UBc;
  const int warp = tid >> 5, lane = tid & 31, gq = lane >> 2, tq = lane & 3;

  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(tslot)), "r"(TCOLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tbase = *reinterpret_cast<volatile uint32_t*>(tslot);
  // this warp's lane quarter and column block
  const uint32_t tw = tbase + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)((warp >> 2) * (KTM * NTL * 2));

  // B fragments: B[k = kk][n] = W_hh[q(kk)][n], n = 64 warp + 8 t + gq
  uint32_t wreg[NTL][KR][2];
#pragma unroll
  for (int t = 0; t < NTL; t++) {
    const int n = warp * 64 + t * 8 + gq;
#pragma unroll
    for (int k = 0; k < KR; k++) {
      const int kk0 = k * 8 + tq, kk1 = kk0 + 4;
      wreg[t][k][0] = to_tf32(whh[(long long)((kk0 / UBc) * R + u0 + kk0 % UBc) * R + n]);
      wreg[t][k][1] = to_tf32(whh[(long long)((kk1 / UBc) * R + u0 + kk1 % UBc) * R + n]);
    }
  }
  for (int k = KR; k < KS; k++) {
    uint32_t v[2 * NTL];
    const int kk0 = k * 8 + tq, kk1 = kk0 + 4;
    const float* w0 = whh + (long long)((kk0 / UBc) * R + u0 + kk0 % UBc) * R + warp * 64 + gq;
    const float* w1 = whh + (long long)((kk1 / UBc) * R + u0 + kk1 % UBc) * R + warp * 64 + gq;
#pragma unroll
    for (int t = 0; t < NTL; t++) {
      v[2 * t] = to_tf32(w0[t * 8]);
      v[2 * t + 1] = to_tf32(w1[t * 8]);
    }
    tmem_st16(tw + (uint32_t)((k - KR) * 2 * NTL), v);
  }
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");

  int crow[CPT], cuu[CPT];
  bool cok[CPT];
  float dc_reg[CPT];
#pragma unroll
  for (int h = 0; h < CPT; h++) {
    const int ci = tid + NT * h;
    crow[h] = ci / UBc;
    cuu[h] = ci - crow[h] * UBc;
    cok[h] = (r0 + crow[h]) < B;
    dc_reg[h] = 0.f;
  }
  uint32_t raddr[2];   // base of recv in CTA 2*warp and 2*warp+1
  raddr[0] = map_to_cta(recv, 2 * warp);
  raddr[1] = map_to_cta(recv, 2 * warp + 1);
  __syncthreads();
  cluster_arrive();   // every CTA of the cluster has started (distributed shared memory may be written from here on)
  cluster_wait();

  for (int it = 0; it < S; it++) {
    const int s = S - 1 - it;
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
      cluster_wait();   // the 16 partial products for my units have arrived in recv[it & 1]
      const float* rb = recv + (it & 1) * CS * MB * UBc;
#pragma unroll
      for (int h = 0; h < CPT; h++) {
        float r = 0.f;
#pragma unroll
        for (int src = 0; src < CS; src++) r += rb[(src * MB + crow[h]) * UBc + cuu[h]];   // fixed order: deterministic
        rec[h] = r;
      }
    }
#pragma unroll
    for (int h = 0; h < CPT; h++) {
      float d0 = 0.f, d1 = 0.f, d2 = 0.f, d3 = 0.f;
      if (cok[h]) {
        const float dh = dht[h] + rec[h];
        const float tc = fast_tanh(cnow[h]);
        const float dc = dh * og[h] * (1.f - tc * tc) + dc_reg[h];
        dc_reg[h] = dc * fg[h];
        d0 = dc * gg[h] * ig[h] * (1.f - ig[h]);
        d1 = dc * cprev[h] * fg[h] * (1.f - fg[h]);
        d2 = dc * ig[h] * (1.f - gg[h] * gg[h]);
        d3 = dh * tc * og[h] * (1.f - og[h]);
        const long long gbase = ((long long)s * B + r0 + crow[h]) * K4 + u0 + cuu[h];
        dG[gbase] = d0;
        dG[gbase + R] = d1;
        dG[gbase + 2LL * R] = d2;
        dG[gbase + 3LL * R] = d3;
      }
      float* a = As + crow[h] * LDA + cuu[h];
      a[0] = round_tf32(d0); a[UBc] = round_tf32(d1); a[2 * UBc] = round_tf32(d2); a[3 * UBc] = round_tf32(d3);
    }
    if (it < S - 1) {
      __syncthreads();   // As complete
      const uint32_t slot = (uint32_t)((((it + 1) & 1) * CS + (int)rank) * MB * UBc) * 4u;
      uint32_t b0[2 * NTL], b1[2 * NTL];
      tmem_ld16(tw, b0);   // first tensor-memory step: in flight during the register-resident half
#pragma unroll
      for (int m = 0; m < MT; m++) {
        float acc[NTL][4];
#pragma unroll
        for (int t = 0; t < NTL; t++)
#pragma unroll
          for (int q = 0; q < 4; q++) acc[t][q] = 0.f;
        const float* ga = As + (m * 16 + gq) * LDA + tq;
#pragma unroll
        for (int k = 0; k < KR; k++) {
          uint32_t a[4];
          a[0] = __float_as_uint(ga[k * 8]); a[1] = __float_as_uint(ga[8 * LDA + k * 8]);
          a[2] = __float_as_uint(ga[k * 8 + 4]); a[3] = __float_as_uint(ga[8 * LDA + k * 8 + 4]);
#pragma unroll
          for (int t = 0; t < NTL; t++) mma_tf32(acc[t], a, wreg[t][k]);
        }
#pragma unroll
        for (int k = 0; k < KTM; k += 2) {
          uint32_t a[4];
          tmem_wait_ld16(b0);
          tmem_ld16(tw + (uint32_t)((k + 1) * 2 * NTL), b1);
          a[0] = __float_as_uint(ga[(KR + k) * 8]); a[1] = __float_as_uint(ga[8 * LDA + (KR + k) * 8]);
          a[2] = __float_as_uint(ga[(KR + k) * 8 + 4]); a[3] = __float_as_uint(ga[8 * LDA + (KR + k) * 8 + 4]);
#pragma unroll
          for (int t = 0; t < NTL; t++) mma_tf32(acc[t], a, &b0[2 * t]);
          tmem_wait_ld16(b1);
          if (k + 2 < KTM) tmem_ld16(tw + (uint32_t)((k + 2) * 2 * NTL), b0);
          else if (m + 1 < MT) tmem_ld16(tw, b0);   // first step of the next m16 tile
          a[0] = __float_as_uint(ga[(KR + k + 1) * 8]); a[1] = __float_as_uint(ga[8 * LDA + (KR + k + 1) * 8]);
          a[2] = __float_as_uint(ga[(KR + k + 1) * 8 + 4]); a[3] = __float_as_uint(ga[8 * LDA + (KR + k + 1) * 8 + 4]);
#pragma unroll
          for (int t = 0; t < NTL; t++) mma_tf32(acc[t], a, &b1[2 * t]);
        }
        // scatter: tile t of warp w holds columns n = 64 w + 8 t + 2 tq (+1), rows m*16 + gq (+8) -> owner 2w + (t >> 2), unit
        // (8 t + 2 tq) & 31, slot [next parity][src = my rank]
#pragma unroll
        for (int t = 0; t < NTL; t++) {
          const uint32_t base = raddr[t >> 2] + slot + (uint32_t)(((t & 3) * 8 + 2 * tq) * 4);
          st_cluster_v2(base + (uint32_t)((m * 16 + gq) * UBc * 4), acc[t][0], acc[t][1]);
          st_cluster_v2(base + (uint32_t)((m * 16 + gq + 8) * UBc * 4), acc[t][2], acc[t][3]);
        }
      }
      cluster_arrive();   // release: my partial products are visible to their owners
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tbase), "r"(TCOLS) : "memory");
}
constexpr size_t bwd_tm_smem(int MT) { return (size_t)(2 * CS * 16 * MT * UBc + 16 * MT * (4 * UBc + PAD)) * sizeof(float) + 16; }
static_assert(bwd_tm_smem(3) <= 232448, "backward scan shared memory");

constexpr size_t fwd_smem(int MT) {
  return (size_t)(8 * 16 * 4 * 2 * 32 + 16 * MT * (R + PAD) + (MT > 2 ? 0 : 2 * 16 * MT * (4 * UBc + 1)) + 4 * UBc) * sizeof(float);
}
static_assert(fwd_smem(3) <= 232448 && fwd_smem(2) <= 232448, "forward scan shared memory");
constexpr size_t bwd_smem() { return (size_t)(8 * 8 * 8 * 2 * 32 + 2 * CS * 16 * UBc + 16 * (4 * UBc + PAD)) * sizeof(float); }

template <typename Kern, typename... Args>
int launch_cluster16(Kern kern, const char* what, int grid, size_t smem, cudaStream_t st, bool& attr, Args... args) {
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) { p2pvg_set_error("%s: %s", what, cudaGetErrorString(e)); return P2PVG_ERR_CUDA; }
    attr = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(NT);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = CS;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, args...);
  if (e != cudaSuccess) {
    p2pvg_set_error("%s: launch of %d CTAs in clusters of 16 failed: %s", what, grid, cudaGetErrorString(e));
    (void)cudaGetLastError();
    return P2PVG_ERR_CUDA;
  }
  return P2PVG_OK;
}

}  // namespace

// cudaOccupancyMaxActiveClusters of the cluster-16 scans (which = 0: forward 16-row slabs, 1: 32 rows, 3: 48 rows, 2: backward 16 rows, 4 / 5: backward 32 / 48 rows)
int p2pvg_lstm_cluster512_max_clusters_impl(int which) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(CS * 64);
  cfg.blockDim = dim3(NT);
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = CS;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  int n = -1;
  cudaError_t e;
  if (which == 0) {
    cfg.dynamicSmemBytes = fwd_smem(1);
    cudaFuncSetAttribute(lstm_cl16_fwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fwd_smem(1));
    cudaFuncSetAttribute(lstm_cl16_fwd_kernel<1>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    e = cudaOccupancyMaxActiveClusters(&n, lstm_cl16_fwd_kernel<1>, &cfg);
  } else if (which == 1) {
    cfg.dynamicSmemBytes = fwd_smem(2);
    cudaFuncSetAttribute(lstm_cl16_fwd_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fwd_smem(2));
    cudaFuncSetAttribute(lstm_cl16_fwd_kernel<2>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    e = cudaOccupancyMaxActiveClusters(&n, lstm_cl16_fwd_kernel<2>, &cfg);
  } else if (which == 3) {
    cfg.dynamicSmemBytes = fwd_smem(3);
    cudaFuncSetAttribute(lstm_cl16_fwd_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fwd_smem(3));
    cudaFuncSetAttribute(lstm_cl16_fwd_kernel<3>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    e = cudaOccupancyMaxActiveClusters(&n, lstm_cl16_fwd_kernel<3>, &cfg);
  } else if (which == 4 || which == 5) {
    const int mt = which - 2;   // 2 or 3 m16 tiles per slab
    cfg.dynamicSmemBytes = bwd_tm_smem(mt);
    if (mt == 2) {
      cudaFuncSetAttribute(lstm_cl16_bwd_tm_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd_tm_smem(2));
      cudaFuncSetAttribute(lstm_cl16_bwd_tm_kernel<2>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
      e = cudaOccupancyMaxActiveClusters(&n, lstm_cl16_bwd_tm_kernel<2>, &cfg);
    } else {
      cudaFuncSetAttribute(lstm_cl16_bwd_tm_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd_tm_smem(3));
      cudaFuncSetAttribute(lstm_cl16_bwd_tm_kernel<3>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
      e = cudaOccupancyMaxActiveClusters(&n, lstm_cl16_bwd_tm_kernel<3>, &cfg);
    }
  } else {
    cfg.dynamicSmemBytes = bwd_smem();
    cudaFuncSetAttribute(lstm_cl16_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bwd_smem());
    cudaFuncSetAttribute(lstm_cl16_bwd_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    e = cudaOccupancyMaxActiveClusters(&n, lstm_cl16_bwd_kernel, &cfg);
  }
  if (e != cudaSuccess) { (void)cudaGetLastError(); return -1; }
  return n;
}

// Rows per slab of the forward scan.  Only `maxc` clusters of 16 CTAs are resident at a time (7 on a B200: one per 20-SM GPC),
// a launch with more clusters runs in waves, each wave a complete pass over the S timesteps.  One timestep of a 16*MT-row slab
// costs about 1.5 + 2.8*MT us (measured: 4.3 / 7.1 us for MT = 1 / 2; barrier + L2 round trip, then MMA + pointwise per m16
// tile): pick the MT with the smallest waves * step time.  B = 256: 6 clusters of 48 rows, one wave.
static int fwd_slab_tiles(int B) {
  static const int maxc = [] { const int n = p2pvg_lstm_cluster512_max_clusters_impl(1); return n > 0 ? n : 7; }();
  int best = 1;
  float best_cost = 0.f;
  for (int mt = 1; mt <= 3; mt++) {
    const int clusters = cdiv(B, 16 * mt), waves = cdiv(clusters, maxc);
    const float cost = waves * (1.5f + 2.8f * mt);
    if (mt == 1 || cost < best_cost) best = mt, best_cost = cost;
  }
  return best;
}

int p2pvg_lstm_cluster512_fwd_impl(const float* pre, const float* whh, const float* bhh, float* gates, float* hs, float* cs, int S, int B,
                                   cudaStream_t st) {
  if (S <= 0 || B <= 0) return P2PVG_OK;
  static bool a1 = false, a2 = false, a3 = false;
  const int mt = fwd_slab_tiles(B);
  if (mt == 3) return launch_cluster16(lstm_cl16_fwd_kernel<3>, "lstm_cl16_fwd", CS * cdiv(B, 48), fwd_smem(3), st, a3, pre, whh, bhh, gates, hs, cs, S, B);
  if (mt == 2) return launch_cluster16(lstm_cl16_fwd_kernel<2>, "lstm_cl16_fwd", CS * cdiv(B, 32), fwd_smem(2), st, a2, pre, whh, bhh, gates, hs, cs, S, B);
  return launch_cluster16(lstm_cl16_fwd_kernel<1>, "lstm_cl16_fwd", CS * cdiv(B, 16), fwd_smem(1), st, a1, pre, whh, bhh, gates, hs, cs, S, B);
}

// Rows per slab of the backward scan, same wave model as the forward one.  Measured per timestep: 16-row slabs (weight half in
// shared memory) 5.7 us, 32 / 48-row slabs (weight half in tensor memory) 8.0 / 11.1 us, i.e. about 3.0 + 2.7 us per m16 tile;
// B = 256: one wave of 6 clusters (11.2 us) instead of three waves of 16-row slabs (15.9 us).
static int bwd_slab_tiles(int B) {
  static const int maxc = [] { const int n = p2pvg_lstm_cluster512_max_clusters_impl(2); return n > 0 ? n : 7; }();
  int best = 1;
  float best_cost = 0.f;
  for (int mt = 1; mt <= 3; mt++) {
    const int clusters = cdiv(B, 16 * mt), waves = cdiv(clusters, maxc);
    const float cost = waves * (3.0f + 2.7f * mt);
    if (mt == 1 || cost < best_cost) best = mt, best_cost = cost;
  }
  return best;
}

int p2pvg_lstm_cluster512_bwd_impl(const float* dhtop, const float* whh, const float* gates, const float* cs, float* dG, int S, int B,
                                   cudaStream_t st) {
  if (S <= 0 || B <= 0) return P2PVG_OK;
  static bool a = false, a2 = false, a3 = false;
  const int mt = bwd_slab_tiles(B);
  if (mt == 3) return launch_cluster16(lstm_cl16_bwd_tm_kernel<3>, "lstm_cl16_bwd", CS * cdiv(B, 48), bwd_tm_smem(3), st, a3, dhtop, whh, gates, cs, dG, S, B);
  if (mt == 2) return launch_cluster16(lstm_cl16_bwd_tm_kernel<2>, "lstm_cl16_bwd", CS * cdiv(B, 32), bwd_tm_smem(2), st, a2, dhtop, whh, gates, cs, dG, S, B);
  return launch_cluster16(lstm_cl16_bwd_kernel, "lstm_cl16_bwd", CS * cdiv(B, 16), bwd_smem(), st, a, dhtop, whh, gates, cs, dG, S, B);
}
