// Implicit-GEMM 4x4 / stride-2 / pad-1 convolution family on NHWC bf16 tensors (no im2col / col2im buffers).
// Same persistent tcgen05 skeleton as gemm_tc.cu (TMA -> 128B-swizzled smem -> tcgen05.mma kind::f16 -> TMEM ->
// tcgen05.ld epilogue, double-buffered accumulator); what changes is how an operand tile is fetched:
//
//   "pixel box" tiles: P consecutive NHW pixels of the SMALL map (H x W per image) are a rectangular box
//   {bw = W, bh, bn}; the operand rows for filter tap (kh,kw) are the BIG-map pixels (2y+kh-1, 2x+kw-1), i.e. one
//   4-D TMA load with elementStrides {1,2,2,1} whose out-of-bounds part (the conv padding) is zero-filled by the
//   hardware.  For the transposed direction the rows are SMALL-map pixels (y+dy, x+dx): a stride-1 4-D box.
//
// kind 0  y_small[N,H,W,Cn] = conv_s2(x_big[N,2H,2W,Ck]) . W[Cn, (tap, Ck)]           Conv forward, ConvT data-gradient
// kind 1  g[Cm, (tap, Cn)]  = sum_pix a_small[pix, Cm]^T . gather_s2(b_big)[pix, tap, Cn]   weight gradients (split-K)
// kind 2  y_big[N,2H,2W,Cn] = convT_s2(x_small[N,H,W,Ck]) . W[Ck, (tap, Cn)] + bias + addend   ConvT forward, Conv data-gradient
//         (4 output-parity phases, each a 2x2 stride-1 convolution; `addend` holds the skip-connection half of
//          torch.cat([d, skip]) computed once per distinct source call and is indexed through grp_src)
// kind 3  y[N,H,W,Cn] = conv3x3_s1_p1(x[N,H,W,Ck]) . W[Cn, (tap, Ck)] + bias + addend      vgg layer forward (kind 0 geometry, 9 taps)
// kind 4  g[Cm, (tap, Cn)] = sum_pix a[pix, Cm]^T . gather_3x3(b)[pix, tap, Cn]             vgg weight gradients (kind 1 geometry)
// kind 5  kind 3 with mirrored tap offsets (pixel - (kh-1, kw-1)): the data gradient of a 3x3 convolution
#include <mutex>

#include "tc_common.cuh"

namespace {

using namespace tc;

constexpr int BLOCK_M = 128;
constexpr int NUM_THREADS = 192;
constexpr int A_STAGE_BYTES = BLOCK_M * 128;

template <int BN> struct Cfg {
  static constexpr int B_STAGE_BYTES = BN * 128;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int STAGES = (BN == 256) ? 4 : (BN == 128) ? 6 : 8;  // 128x256 tiles: 87 FLOP per smem-fill byte (L2 -> SM
                                                                        // bandwidth bounds the 128x128 tiles at ~1100 TFLOP/s)
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 512;
};

struct Geom {
  int N, H, W;          // images, small-map height / width
  int Ck, Cn;           // reduction channels / output channels (kind 0,2);  kind 1: Cm = M extent, Cn = gathered channels
  int M;                // GEMM M: kind 0/2: N*H*W pixels; kind 1: Cm
  int Ntot;             // GEMM N: kind 0/2: Cn; kind 1: 16*Cn
  int bh128, bn128;     // pixel box of 128 pixels: {W, bh128, bn128}
  int bh64, bn64;       // pixel box of 64 pixels (kind 1 K-blocks): {bw64, bh64, bn64}; bw64 = 64 < W for 128-wide maps
  int bw64;
  int imgs_per_group;   // addend indexing
  int add_bf16;         // the addend tensor is bf16 (half the epilogue read traffic of the fp32 form)
  int bres;             // kind 0, BN = 64, one channel chunk, <= 9 taps: ALL weight tiles stay resident in shared memory for the whole
                        // kernel (72 KB) and only the A boxes stream through a 7-slot ring -- the 64 -> 64 channel 3x3 layers re-fetched
                        // their 73 KB of weights for every 128-pixel tile (43 FLOP per filled byte -> 65)
  int swap;             // kind 1 with the operand roles swapped: M = taps*Cn (gathered map), N = Cm (few output channels would waste
                        // half of a 128-row MMA tile otherwise); the partial sums are [taps*Cn][Cm] and the reduce kernel transposes
  int ks, st, sgn;      // filter taps per side (4 | 3), stride between the two maps (2 | 1), tap-offset sign (+1 | -1)
};

__device__ __forceinline__ void pix_block(int pb, int P, int H, int W, int bh, int bn, int& n0, int& y0) {
  const int HW = H * W;
  if (HW >= P) {
    const int bpi = HW / P;
    n0 = pb / bpi;
    y0 = (pb - n0 * bpi) * bh;
  } else {
    n0 = pb * bn;
    y0 = 0;
  }
}

// 64 addend columns of one output row into 16-byte registers: 16 loads for fp32, 8 for bf16
__device__ __forceinline__ void addend_load64(float4 (&a4)[16], const float* base, long long elem_off, bool is_bf16) {
  if (is_bf16) {
    const uint4* p = reinterpret_cast<const uint4*>(reinterpret_cast<const bf16*>(base) + elem_off);
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const uint4 r = p[j];
      a4[j] = make_float4(__uint_as_float(r.x), __uint_as_float(r.y), __uint_as_float(r.z), __uint_as_float(r.w));
    }
  } else {
    const float4* p = reinterpret_cast<const float4*>(base + elem_off);
#pragma unroll
    for (int j = 0; j < 16; j++) a4[j] = p[j];
  }
}
// f[0..31] += columns [32 h, 32 h + 32) of what addend_load64 fetched
__device__ __forceinline__ void addend_add32(float (&f)[32], const float4 (&a4)[16], int h, bool is_bf16) {
  if (is_bf16) {
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const float4 r = a4[4 * h + j];
      float v[8];
      unpack16<bf16>(make_uint4(__float_as_uint(r.x), __float_as_uint(r.y), __float_as_uint(r.z), __float_as_uint(r.w)), v);
#pragma unroll
      for (int i = 0; i < 8; i++) f[8 * j + i] += v[i];
    }
  } else {
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const float4 x4 = a4[8 * h + j];
      f[4 * j] += x4.x; f[4 * j + 1] += x4.y; f[4 * j + 2] += x4.z; f[4 * j + 3] += x4.w;
    }
  }
}

template <int KIND, int BN, bool STAT>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, void* __restrict__ Cv, int c_bf16,
                 long long ldc, Geom g, int accumulate, const float* __restrict__ bias, const float* __restrict__ addend,
                 const int* __restrict__ grp_src, float* __restrict__ partial, int kb_per_split, int splits,
                 float2* __restrict__ stat_partial) {
  using C_ = Cfg<BN>;
  constexpr bool A_MN = (KIND == 1), B_MN = (KIND != 0);
  constexpr int UMMA_K = 16;
  constexpr uint32_t TMEM_COLS = 2 * BN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C_::STAGES * C_::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C_::STAGES;
  uint64_t* tmem_full_bar = empty_bar + C_::STAGES;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint64_t* bres_bar = tmem_empty_bar + 2;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bres_bar + 1);
  // resident-weight mode (kind 0, BN = 64): weights at [0, 9 * 8 KB), A ring of 7 x 16 KB behind them
  const bool bres = (KIND == 0) && (BN == 64) && g.bres != 0;
  constexpr int BRES_B_BYTES = 9 * 64 * 128, BRES_STAGES = 7;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_m = (g.M + BLOCK_M - 1) / BLOCK_M, tiles_n = (g.Ntot + BN - 1) / BN;
  const int tiles_mn = tiles_m * tiles_n;
  const int phases = (KIND == 2) ? 4 : 1;
  const int num_tiles = tiles_mn * splits * phases;
  const int cchunks = g.Ck / 64;
  // K blocks: kind 0: 16 taps x Ck/64; kind 2: 4 taps x Ck/64; kind 1: pixel blocks of 64
  const int nkb_total = (KIND == 0) ? g.ks * g.ks * cchunks : (KIND == 2) ? 4 * cchunks : (g.N * g.H * g.W + 63) / 64;

  if (threadIdx.x == 0) {
    for (int s = 0; s < C_::STAGES; s++) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; a++) {
      mbar_init(&tmem_full_bar[a], 1);
      mbar_init(&tmem_empty_bar[a], 4);
    }
    mbar_init(bres_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      uint32_t it = 0;
      if (bres) {   // all weight taps once: [tap][64 output channels][64 input channels]
        mbar_expect_tx(bres_bar, (uint32_t)(g.ks * g.ks) * 64 * 128);
        for (int tap = 0; tap < g.ks * g.ks; tap++) tma_load_2d(&tmB, bres_bar, smem + tap * 64 * 128, tap * 64, 0);
      }
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        // tile decode with as few integer divisions as possible: the producer thread is the latency-critical one
        // kind 2: the output-parity phase is the FASTEST tile index, so that the four phases of one pixel tile run on four
        // CTAs at the same time and share the A tile through L2 (phase-major order re-read A from DRAM once per phase:
        // ncu r01 measured 4.0x the algorithmic A bytes).  Kinds 0 / 2 never split K.
        const int ph = (KIND == 2) ? (t & 3) : 0;
        const int t2 = (KIND == 2) ? (t >> 2) : t;
        const int z = (splits == 1) ? 0 : t2 / tiles_mn, r = t2 - z * tiles_mn;
        const int mt = (tiles_n == 1) ? r : r / tiles_n, nt = (tiles_n == 1) ? 0 : r - mt * tiles_n;
        const int n0 = nt * BN;
        const int kb0 = z * kb_per_split, kb1 = min(kb0 + kb_per_split, nkb_total);
        int pn0 = 0, py0 = 0;
        if (KIND != 1) pix_block(mt, 128, g.H, g.W, g.bh128, g.bn128, pn0, py0);
        const int pa = ph >> 1, pb_ = ph & 1;
        // kind 1: everything that does not depend on the K-block is computed once per tile, the pixel-box coordinates
        // advance incrementally -- the single producer thread must not spend its K-block budget on integer divisions
        int kn0 = 0, ky0 = 0, kx0 = 0;
        int t_kh = 0, t_kw = 0, t_cc = 0;
        int qc0[BN / 64], qdx[BN / 64], qdy[BN / 64];
        int mc0[2] = {0, 0}, mdx[2] = {0, 0}, mdy[2] = {0, 0};
        if (KIND == 1) {
          if (g.bw64 < g.W) {  // a 64-pixel K-block is a fraction of one row
            const int per_row = g.W / g.bw64;
            const int rowi = kb0 / per_row;
            kx0 = (kb0 - rowi * per_row) * g.bw64;
            kn0 = rowi / g.H;
            ky0 = rowi - kn0 * g.H;
          } else {
            pix_block(kb0, 64, g.H, g.W, g.bh64, g.bn64, kn0, ky0);
          }
#pragma unroll
          for (int q = 0; q < BN / 64; q++) {
            const int nb = n0 + 64 * q;
            const int tap = nb / g.Cn;
            const int kh = tap / g.ks;
            qc0[q] = nb - tap * g.Cn;
            qdx[q] = tap - kh * g.ks - 1;
            qdy[q] = kh - 1;
          }
          if (g.swap) {   // the gathered map is the A operand: (tap, channel) of the two 64-row halves of the M tile
#pragma unroll
            for (int q = 0; q < 2; q++) {
              const int mb = mt * BLOCK_M + 64 * q;
              int tap = mb / g.Cn;
              if (tap >= g.ks * g.ks) tap = g.ks * g.ks - 1;   // rows past M are discarded by the epilogue: any in-bounds tap will do
              const int kh = tap / g.ks;
              mc0[q] = mb < g.M ? mb - tap * g.Cn : 0;
              mdx[q] = tap - kh * g.ks - 1;
              mdy[q] = kh - 1;
            }
          }
        }
        for (int kb = kb0; kb < kb1; kb++, it++) {
          // (both divisors are compile-time constants: no runtime division in the single producer / issuer threads)
          const int s = bres ? (int)(it % BRES_STAGES) : (int)(it % C_::STAGES);
          const uint32_t par = (bres ? (it / BRES_STAGES) : (it / C_::STAGES)) & 1;
          mbar_wait(&empty_bar[s], par ^ 1);
          uint8_t* sa = bres ? smem + BRES_B_BYTES + s * A_STAGE_BYTES : smem + s * C_::STAGE_BYTES;
          uint8_t* sb = sa + A_STAGE_BYTES;
          mbar_expect_tx(&full_bar[s], bres ? A_STAGE_BYTES : C_::STAGE_BYTES);
          if (KIND == 0) {
            // (kh, kw, channel chunk) advance incrementally (kinds 0 / 2 never split K: kb starts at 0)
            tma_load_4d(&tmA, &full_bar[s], sa, t_cc * 64, g.sgn * (t_kw - 1), g.st * py0 + g.sgn * (t_kh - 1), pn0);
            if (!bres) tma_load_2d(&tmB, &full_bar[s], sb, kb * 64, n0);   // (tap * Ck + c0) == kb * 64
            if (++t_cc == cchunks) { t_cc = 0; if (++t_kw == g.ks) { t_kw = 0; t_kh++; } }
          } else if (KIND == 2) {
            const int tq = t_kh, c0 = t_cc * 64;   // t_kh doubles as the 2x2 tap index of this phase
            if (++t_cc == cchunks) { t_cc = 0; t_kh++; }
            const int i = tq >> 1, j = tq & 1;
            // phase a: taps (dy=0, ky=a+1) and (dy = a ? +1 : -1, ky = a ? 0 : 3); same along x
            const int dy = i == 0 ? 0 : (pa ? 1 : -1), ky = i == 0 ? pa + 1 : (pa ? 0 : 3);
            const int dx = j == 0 ? 0 : (pb_ ? 1 : -1), kx = j == 0 ? pb_ + 1 : (pb_ ? 0 : 3);
            tma_load_4d(&tmA, &full_bar[s], sa, c0, dx, py0 + dy, pn0);
#pragma unroll
            for (int q = 0; q < BN / 64; q++)
              tma_load_2d(&tmB, &full_bar[s], sb + q * 64 * 128, (ky * 4 + kx) * g.Cn + n0 + 64 * q, c0);
          } else {
            const int m0 = mt * BLOCK_M;
            if (g.swap) {
              tma_load_4d(&tmA, &full_bar[s], sa, mc0[0], g.st * kx0 + mdx[0], g.st * ky0 + mdy[0], kn0);
              tma_load_4d(&tmA, &full_bar[s], sa + 64 * 128, mc0[1], g.st * kx0 + mdx[1], g.st * ky0 + mdy[1], kn0);
#pragma unroll
              for (int q = 0; q < BN / 64; q++) tma_load_2d(&tmB, &full_bar[s], sb + q * 64 * 128, n0 + 64 * q, kb * 64);
            } else {
              tma_load_2d(&tmA, &full_bar[s], sa, m0, kb * 64);
              tma_load_2d(&tmA, &full_bar[s], sa + 64 * 128, m0 + 64, kb * 64);
#pragma unroll
              for (int q = 0; q < BN / 64; q++)
                tma_load_4d(&tmB, &full_bar[s], sb + q * 64 * 128, qc0[q], g.st * kx0 + qdx[q], g.st * ky0 + qdy[q], kn0);
            }
            // next 64-pixel box
            if (g.bw64 < g.W) {
              kx0 += g.bw64;
              if (kx0 >= g.W) { kx0 = 0; if (++ky0 >= g.H) { ky0 = 0; kn0++; } }
            } else if (g.H * g.W >= 64) {
              ky0 += g.bh64;
              if (ky0 >= g.H) { ky0 = 0; kn0++; }
            } else {
              kn0 += g.bn64;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
                             ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
      const uint32_t smem0 = smem_u32(smem);
      const uint64_t da0 = A_MN ? make_desc(smem0, 64 * 128, 1024) : make_desc(smem0, 0, 1024);
      const uint64_t db0 = B_MN ? make_desc(smem0 + A_STAGE_BYTES, 64 * 128, 1024) : make_desc(smem0 + A_STAGE_BYTES, 0, 1024);
      uint32_t it = 0, lt = 0;
      if (bres) {
        mbar_wait(bres_bar, 0);   // the resident weights have landed
        tcgen05_fence_after();
      }
      const uint64_t da0r = make_desc(smem0 + BRES_B_BYTES, 0, 1024), db0r = make_desc(smem0, 0, 1024);
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, lt++) {
        int z = 0;
        if (splits > 1) z = t / tiles_mn;   // only kind 1 splits K (one phase)
        const int kb0 = z * kb_per_split, kb1 = min(kb0 + kb_per_split, nkb_total);
        const uint32_t acc = lt & 1, acc_ph = (lt >> 1) & 1;
        mbar_wait(&tmem_empty_bar[acc], acc_ph ^ 1);
        tcgen05_fence_after();
        const uint32_t tmem_c = tmem_base + acc * BN;
        for (int kb = kb0; kb < kb1; kb++, it++) {
          // (both divisors are compile-time constants: no runtime division in the single producer / issuer threads)
          const int s = bres ? (int)(it % BRES_STAGES) : (int)(it % C_::STAGES);
          const uint32_t par = (bres ? (it / BRES_STAGES) : (it / C_::STAGES)) & 1;
          mbar_wait(&full_bar[s], par);
          tcgen05_fence_after();
          // descriptors of stage 0 / k 0 are built once; the start-address field (bits 0-13, address >> 4) is advanced by
          // plain additions -- the single issuing thread has ~32 clk per 128x64x16 MMA to spend
          const uint64_t stage_off = (uint64_t)((uint32_t)s * (uint32_t)(C_::STAGE_BYTES >> 4));
          const uint64_t a_off = bres ? (uint64_t)((uint32_t)s * (uint32_t)(A_STAGE_BYTES >> 4)) : stage_off;
          const uint64_t b_off = bres ? (uint64_t)((uint32_t)kb * (uint32_t)((64 * 128) >> 4)) : stage_off;   // resident: tap kb
#pragma unroll
          for (int k = 0; k < 64 / UMMA_K; k++) {
            const uint64_t da = (bres ? da0r : da0) + a_off + (uint64_t)(k * ((A_MN ? UMMA_K * 128 : 32) >> 4));
            const uint64_t db = (bres ? db0r : db0) + b_off + (uint64_t)(k * ((B_MN ? UMMA_K * 128 : 32) >> 4));
            umma_bf16(tmem_c, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&empty_bar[s]);
        }
        umma_commit(&tmem_full_bar[acc]);
      }
    }
  } else {
    // ===================== epilogue =====================
    const int q = warp & 3;
    __shared__ float bias_s[2 * BN];
    // BatchNorm forward statistics fused into the epilogue: per-warp column sums (sum y, sum y^2) of the tile, double-
    // buffered by accumulator so that tile t+1 may write while the sums of tile t are still being combined
    __shared__ float2 stat_s[STAT ? 2 * 4 * BN : 1];
    constexpr bool do_stat = STAT;   // a separate instantiation: the statistics cost ~50 registers in this epilogue
    uint32_t lt = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, lt++) {
      const int ph = (KIND == 2) ? (t & 3) : 0;
      const int t2 = (KIND == 2) ? (t >> 2) : t;
      const int z = (splits == 1) ? 0 : t2 / tiles_mn, r = t2 - z * tiles_mn;
      const int mt = (tiles_n == 1) ? r : r / tiles_n, nt = (tiles_n == 1) ? 0 : r - mt * tiles_n;
      const int n0 = nt * BN;
      const uint32_t acc = lt & 1, acc_ph = (lt >> 1) & 1;
      const int rt = q * 32 + lane;  // row within the tile
      long long out_row = (long long)mt * BLOCK_M + rt;
      long long add_row = 0;
      bool row_ok = out_row < g.M;
      if (KIND == 2) {
        // tile row -> small-map pixel -> big-map output pixel of this parity phase
        int pn0, py0;
        pix_block(mt, 128, g.H, g.W, g.bh128, g.bn128, pn0, py0);
        const int HW = g.H * g.W;
        int nn, yy, xx;
        if (HW >= 128) { nn = 0; yy = rt / g.W; xx = rt - yy * g.W; }
        else { nn = rt / HW; const int rem = rt - nn * HW; yy = rem / g.W; xx = rem - yy * g.W; }
        const int n = pn0 + nn, y = py0 + yy;
        row_ok = (n < g.N) && (y < g.H);
        const int oy = 2 * y + (ph >> 1), ox = 2 * xx + (ph & 1);
        out_row = ((long long)n * (2 * g.H) + oy) * (2 * g.W) + ox;
        if (addend && row_ok) {
          const int n2 = grp_src[n / g.imgs_per_group] * g.imgs_per_group + (n % g.imgs_per_group);
          add_row = ((long long)n2 * (2 * g.H) + oy) * (2 * g.W) + ox;
        }
      }
      if (KIND == 0 && addend && row_ok) {
        const int HW = g.H * g.W;
        const int n = (int)(out_row / HW);
        const int n2 = grp_src[n / g.imgs_per_group] * g.imgs_per_group + (n % g.imgs_per_group);
        add_row = (long long)n2 * HW + (out_row - (long long)n * HW);
      }
      // stage the bias slice of this tile in shared memory while the MMAs are still running
      if (bias != nullptr) {
        for (int i = q * 32 + lane; i < BN; i += 128) bias_s[acc * BN + i] = (n0 + i < g.Ntot) ? bias[n0 + i] : 0.f;
        epi_bar_sync();
      }
      const bool use_add = (KIND != 1) && addend != nullptr && row_ok;
      const long long aoff0 = add_row * g.Ntot + n0;   // element offset of this row's first addend column
      const bool abf = g.add_bf16 != 0;
      float4 a4[16];  // addend of the next 64 columns, requested before the accumulator is waited for
      if (use_add) addend_load64(a4, addend, aoff0, abf);
      mbar_wait(&tmem_full_bar[acc], acc_ph);
      tcgen05_fence_after();
#pragma unroll 1
      for (int pr = 0; pr < BN / 64; pr++) {
        // two 32-column chunks per round: both tcgen05.ld in flight before the wait; after the last round the
        // accumulator goes back to the MMA warp *before* the global stores
        uint32_t v2[64];
        const uint32_t taddr = tmem_base + acc * BN + ((uint32_t)(q * 32) << 16) + (uint32_t)(pr * 64);
        tmem_ld32(taddr, v2);
        tmem_ld32(taddr + 32, v2 + 32);
        if (pr > 0 && use_add) addend_load64(a4, addend, aoff0 + pr * 64, abf);
        tmem_ld_wait_dep(v2);
        tmem_ld_wait_dep(v2 + 32);
        if (pr == BN / 64 - 1) {
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
        }
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const int c = pr * 2 + h;
          const uint32_t* v = v2 + 32 * h;
          const int nbase = n0 + c * 32;
          if (nbase >= g.Ntot) continue;             // warp-uniform
          if (!row_ok && !do_stat) continue;         // rows past the end only matter as zeros of the column sums
          if (KIND == 1 && partial != nullptr) {
            float* dst = partial + ((long long)z * g.M + out_row) * g.Ntot + nbase;
#pragma unroll
            for (int j = 0; j < 32; j += 8)   // partial workspace rows are 32-byte aligned (Ntot and nbase are multiples of 32)
              st_global_256(dst + j, v[j], v[j + 1], v[j + 2], v[j + 3], v[j + 4], v[j + 5], v[j + 6], v[j + 7]);
            continue;
          }
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; j++) f[j] = __uint_as_float(v[j]);
          if (bias) {
            const float* bs = bias_s + acc * BN + c * 32;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const float4 b4 = *reinterpret_cast<const float4*>(bs + j);
              f[j] += b4.x; f[j + 1] += b4.y; f[j + 2] += b4.z; f[j + 3] += b4.w;
            }
          }
          if (use_add) addend_add32(f, a4, h, abf);
          if (STAT) {
            // statistics of the tensor AS STORED (bf16-rounded when the output is bf16); all 32 lanes take part
            float s1[32], s2[32];
#pragma unroll
            for (int j = 0; j < 32; j++) {
              const float r = row_ok ? (c_bf16 ? bf16_round(f[j]) : f[j]) : 0.f;
              s1[j] = r;
              s2[j] = r * r;
            }
            const float cs = warp_colsum32(s1, lane), cq = warp_colsum32(s2, lane);
            stat_s[(acc * 4 + q) * BN + c * 32 + lane] = make_float2(cs, cq);
            if (!row_ok) continue;
          }
          if (c_bf16) {
            bf16* crow = reinterpret_cast<bf16*>(Cv) + out_row * ldc + nbase;
            if (accumulate) {
#pragma unroll
              for (int j = 0; j < 32; j++) f[j] += __bfloat162float(crow[j]);
            }
            if ((reinterpret_cast<uintptr_t>(crow) & 31) == 0) {
#pragma unroll
              for (int j = 0; j < 32; j += 16)
                st_global_256(crow + j, pack_bf16x2(f[j], f[j + 1]), pack_bf16x2(f[j + 2], f[j + 3]), pack_bf16x2(f[j + 4], f[j + 5]),
                              pack_bf16x2(f[j + 6], f[j + 7]), pack_bf16x2(f[j + 8], f[j + 9]), pack_bf16x2(f[j + 10], f[j + 11]),
                              pack_bf16x2(f[j + 12], f[j + 13]), pack_bf16x2(f[j + 14], f[j + 15]));
            } else {
#pragma unroll
              for (int j = 0; j < 32; j += 8) {
                uint4 pk;
                pk.x = pack_bf16x2(f[j], f[j + 1]);
                pk.y = pack_bf16x2(f[j + 2], f[j + 3]);
                pk.z = pack_bf16x2(f[j + 4], f[j + 5]);
                pk.w = pack_bf16x2(f[j + 6], f[j + 7]);
                *reinterpret_cast<uint4*>(crow + j) = pk;
              }
            }
          } else {
            float* crow = reinterpret_cast<float*>(Cv) + out_row * ldc + nbase;
            if (accumulate) {
#pragma unroll
              for (int j = 0; j < 32; j++) f[j] += crow[j];
            }
            if ((reinterpret_cast<uintptr_t>(crow) & 31) == 0) {
#pragma unroll
              for (int j = 0; j < 32; j += 8)
                st_global_256(crow + j, __float_as_uint(f[j]), __float_as_uint(f[j + 1]), __float_as_uint(f[j + 2]), __float_as_uint(f[j + 3]),
                              __float_as_uint(f[j + 4]), __float_as_uint(f[j + 5]), __float_as_uint(f[j + 6]), __float_as_uint(f[j + 7]));
            } else {
#pragma unroll
              for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(crow + j) = make_float4(f[j], f[j + 1], f[j + 2], f[j + 3]);
            }
          }
        }
      }
      if (STAT) {
        // combine the four warps' column sums in a fixed order (deterministic) -> one partial row per (pixel tile, phase)
        epi_bar_sync();
        float2* dst = stat_partial + ((long long)mt * phases + ph) * g.Ntot + n0;
        for (int i = q * 32 + lane; i < BN; i += 128) {
          if (n0 + i >= g.Ntot) continue;
          const float2 a = stat_s[(acc * 4 + 0) * BN + i], b = stat_s[(acc * 4 + 1) * BN + i];
          const float2 c2 = stat_s[(acc * 4 + 2) * BN + i], d = stat_s[(acc * 4 + 3) * BN + i];
          dst[i] = make_float2((a.x + b.x) + (c2.x + d.x), (a.y + b.y) + (c2.y + d.y));
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------------------------
// kind 2 with the FOUR output-parity phases fused into one tile (ConvTranspose2d 4x4 / s2 / p1 forward, Conv2d data gradient).
// A tile = 128 small-map pixels x (4 phases x 64 output channels) = 128 x 256 accumulator columns; column block p = 2a + b
// is output parity (a, b).  out[2y+a, 2x+b] = sum over the 2x2 taps of phase (a, b) of x[y+dy, x+dx] . W[ky, kx]:
// the nine shifted pixel boxes (dy, dx) in {-1,0,1}^2 are each fetched ONCE per channel chunk and multiplied (N = 64
// tcgen05.mma) against the weight taps of every phase that uses the shift: (0,0) serves 4 phases, an edge shift 2, a corner
// shift 1 -- 16 (shift, phase) products per chunk like the phase-by-phase kernel, but 9 A tiles instead of 16: 123 FLOP per
// shared-memory fill byte instead of 43 (64 output channels) / 65 (128), i.e. off the L2 -> SM operand-fill limit that held
// those layers at 520 - 660 TFLOP/s (DESIGN.md).  Output channels beyond 64 are further tiles (n-tile nt = channels
// [64 nt, 64 nt + 64)).  Epilogue as in conv_gemm_kernel (bias, fp32 skip addend, bf16 / fp32 store, optional BatchNorm
// statistics), one 64-column round per phase.
__device__ __forceinline__ bool phase_uses(int a, int d) { return d == 0 || (d < 0 ? a == 0 : a == 1); }
__device__ __forceinline__ int phase_tap(int a, int d) { return d == 0 ? a + 1 : (a ? 0 : 3); }
// The accumulator holds the phases in the column-block order [p0, p1, p3, p2]: then the phases served by one shift are
// NEIGHBOURS for the centre shift (all four) and three of the four edge shifts, so one 256- / 128-wide tcgen05.mma covers them
// instead of four / two 64-wide ones (10 instead of 16 MMAs per 16-wide K slice and channel chunk: the single issuing thread
// was the limit of the 64-wide version).  The centre shift comes FIRST in every tile so that all four column blocks start
// accumulating together.
__device__ __forceinline__ int cb_phase(int cb) { return cb == 2 ? 3 : cb == 3 ? 2 : cb; }   // involution: block <-> phase
__device__ __forceinline__ void shift_of(int so, int& dy, int& dx) {
  // 0 centre; 1..4 edges (-1,0) (+1,0) (0,+1) (0,-1); 5..8 corners
  dy = (so == 1 || so == 5 || so == 6) ? -1 : (so == 2 || so == 7 || so == 8) ? 1 : 0;
  dx = (so == 4 || so == 5 || so == 7) ? -1 : (so == 3 || so == 6 || so == 8) ? 1 : 0;
}
__device__ __forceinline__ bool cb_used(int cb, int dy, int dx) {
  const int p = cb_phase(cb);
  return phase_uses(p >> 1, dy) && phase_uses(p & 1, dx);
}

template <bool STAT>
__global__ void __launch_bounds__(NUM_THREADS, 1)
convt4_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, void* __restrict__ Cv, int c_bf16,
              long long ldc, Geom g, const float* __restrict__ bias, const float* __restrict__ addend, const int* __restrict__ grp_src,
              float2* __restrict__ stat_partial) {
  constexpr int BN = 256;
  using C_ = Cfg<BN>;
  constexpr int UMMA_K = 16;
  constexpr int B_TILE_BYTES = 64 * 128;   // 64 reduction channels x 64 output channels (MN-major)
  constexpr uint32_t TMEM_COLS = 2 * BN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C_::STAGES * C_::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C_::STAGES;
  uint64_t* tmem_full_bar = empty_bar + C_::STAGES;
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_m = (g.M + BLOCK_M - 1) / BLOCK_M, tiles_n = g.Cn / 64;
  const int num_tiles = tiles_m * tiles_n;
  const int cchunks = g.Ck / 64;

  if (threadIdx.x == 0) {
    for (int s = 0; s < C_::STAGES; s++) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; a++) {
      mbar_init(&tmem_full_bar[a], 1);
      mbar_init(&tmem_empty_bar[a], 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr_smem)), "r"(TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ===================== TMA producer: one stage = one shifted pixel box + the weight taps of the phases using it
    if (lane == 0) {
      uint32_t it = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int mt = (tiles_n == 1) ? t : t / tiles_n, nt = (tiles_n == 1) ? 0 : t - mt * tiles_n;
        int pn0, py0;
        pix_block(mt, 128, g.H, g.W, g.bh128, g.bn128, pn0, py0);
        for (int cc = 0; cc < cchunks; cc++) {
          const int c0 = cc * 64;
#pragma unroll
          for (int so = 0; so < 9; so++, it++) {
            int dy, dx;
            shift_of(so, dy, dx);
            const int nb = (dy == 0 ? 2 : 1) * (dx == 0 ? 2 : 1);
            const int s = it % C_::STAGES;
            const uint32_t par = (it / C_::STAGES) & 1;
            mbar_wait(&empty_bar[s], par ^ 1);
            uint8_t* sa = smem + s * C_::STAGE_BYTES;
            uint8_t* sb = sa + A_STAGE_BYTES;
            mbar_expect_tx(&full_bar[s], A_STAGE_BYTES + nb * B_TILE_BYTES);
            tma_load_4d(&tmA, &full_bar[s], sa, c0, dx, py0 + dy, pn0);
            int j = 0;
#pragma unroll
            for (int cb = 0; cb < 4; cb++) {   // weight taps in accumulator column-block order
              if (!cb_used(cb, dy, dx)) continue;
              const int p = cb_phase(cb);
              const int ky = phase_tap(p >> 1, dy), kx = phase_tap(p & 1, dx);
              tma_load_2d(&tmB, &full_bar[s], sb + j * B_TILE_BYTES, (ky * 4 + kx) * g.Cn + nt * 64, c0);
              j++;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc0 = (1u << 4) | (1u << 7) | (1u << 10) | (0u << 15) | (1u << 16) | ((uint32_t)(BLOCK_M >> 4) << 24);
      const uint32_t smem0 = smem_u32(smem);
      const uint64_t da0 = make_desc(smem0, 0, 1024);
      const uint64_t db0 = make_desc(smem0 + A_STAGE_BYTES, 64 * 128, 1024);
      uint32_t it = 0, lt = 0;
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, lt++) {
        const uint32_t acc = lt & 1, acc_ph = (lt >> 1) & 1;
        mbar_wait(&tmem_empty_bar[acc], acc_ph ^ 1);
        tcgen05_fence_after();
        for (int cc = 0; cc < cchunks; cc++) {
#pragma unroll
          for (int so = 0; so < 9; so++, it++) {
            int dy, dx;
            shift_of(so, dy, dx);
            const int s = it % C_::STAGES;
            const uint32_t par = (it / C_::STAGES) & 1;
            mbar_wait(&full_bar[s], par);
            tcgen05_fence_after();
            const uint64_t stage_off = (uint64_t)((uint32_t)s * (uint32_t)(C_::STAGE_BYTES >> 4));
            int j = 0;
#pragma unroll
            for (int cb = 0; cb < 4;) {
              if (!cb_used(cb, dy, dx)) { cb++; continue; }
              int len = 1;
              while (cb + len < 4 && cb_used(cb + len, dy, dx)) len++;   // neighbouring column blocks: one wide MMA
              const uint32_t idesc = idesc0 | ((uint32_t)((64 * len) >> 3) << 17);
              const uint32_t tmem_c = tmem_base + acc * BN + cb * 64;
#pragma unroll
              for (int k = 0; k < 64 / UMMA_K; k++) {
                const uint64_t da = da0 + stage_off + (uint64_t)(k * (32 >> 4));
                const uint64_t db = db0 + stage_off + (uint64_t)(j * (B_TILE_BYTES >> 4)) + (uint64_t)(k * ((UMMA_K * 128) >> 4));
                // the centre shift of channel chunk 0 is the first product of every column block of the tile
                umma_bf16(tmem_c, da, db, idesc, (cc > 0 || so > 0 || k > 0) ? 1u : 0u);
              }
              j += len;
              cb += len;
            }
            umma_commit(&empty_bar[s]);
          }
        }
        umma_commit(&tmem_full_bar[acc]);
      }
    }
  } else {
    // ===================== epilogue: one 64-column round per output-parity phase =====================
    const int q = warp & 3;
    __shared__ float bias_s[64];
    __shared__ float2 stat_s[STAT ? 2 * 4 * BN : 1];
    uint32_t lt = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, lt++) {
      const int mt = (tiles_n == 1) ? t : t / tiles_n, nt = (tiles_n == 1) ? 0 : t - mt * tiles_n;
      const int n0 = nt * 64;
      const uint32_t acc = lt & 1, acc_ph = (lt >> 1) & 1;
      const int rt = q * 32 + lane;
      int pn0, py0;
      pix_block(mt, 128, g.H, g.W, g.bh128, g.bn128, pn0, py0);
      const int HW = g.H * g.W;
      int nn, yy, xx;
      if (HW >= 128) { nn = 0; yy = rt / g.W; xx = rt - yy * g.W; }
      else { nn = rt / HW; const int rem = rt - nn * HW; yy = rem / g.W; xx = rem - yy * g.W; }
      const int n = pn0 + nn, y = py0 + yy;
      const bool row_ok = (n < g.N) && (y < g.H);
      int n2 = n;
      if (addend != nullptr && row_ok) n2 = grp_src[n / g.imgs_per_group] * g.imgs_per_group + (n % g.imgs_per_group);
      const bool use_add = addend != nullptr && row_ok;
      epi_bar_sync();   // every warp is done with bias_s of the previous tile
      if (rt < 64) bias_s[rt] = (bias != nullptr) ? bias[n0 + rt] : 0.f;
      epi_bar_sync();
      const bool abf = g.add_bf16 != 0;
      float4 a4[16];
      if (use_add)   // skip addend of the first column block's phase (p0), requested before the accumulator is waited for
        addend_load64(a4, addend, (((long long)n2 * (2 * g.H) + 2 * y) * (2 * g.W) + 2 * xx) * g.Cn + n0, abf);
      mbar_wait(&tmem_full_bar[acc], acc_ph);
      tcgen05_fence_after();
#pragma unroll 1
      for (int cbi = 0; cbi < 4; cbi++) {
        const int p = cb_phase(cbi);   // accumulator column block cbi holds output parity p
        const int oy = 2 * y + (p >> 1), ox = 2 * xx + (p & 1);
        const long long out_row = ((long long)n * (2 * g.H) + oy) * (2 * g.W) + ox;
        uint32_t v2[64];
        const uint32_t taddr = tmem_base + acc * BN + ((uint32_t)(q * 32) << 16) + (uint32_t)(cbi * 64);
        tmem_ld32(taddr, v2);
        tmem_ld32(taddr + 32, v2 + 32);
        if (cbi > 0 && use_add) addend_load64(a4, addend, (((long long)n2 * (2 * g.H) + oy) * (2 * g.W) + ox) * g.Cn + n0, abf);
        tmem_ld_wait_dep(v2);
        tmem_ld_wait_dep(v2 + 32);
        if (cbi == 3) {   // the accumulator goes back to the MMA warp before the last stores
          tcgen05_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tmem_empty_bar[acc]);
        }
#pragma unroll
        for (int h = 0; h < 2; h++) {
          const uint32_t* v = v2 + 32 * h;
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 b4 = *reinterpret_cast<const float4*>(bias_s + 32 * h + j);
            f[j] = __uint_as_float(v[j]) + b4.x; f[j + 1] = __uint_as_float(v[j + 1]) + b4.y;
            f[j + 2] = __uint_as_float(v[j + 2]) + b4.z; f[j + 3] = __uint_as_float(v[j + 3]) + b4.w;
          }
          if (use_add) addend_add32(f, a4, h, abf);
          if (STAT) {
            float s1[32], s2[32];
#pragma unroll
            for (int j = 0; j < 32; j++) {
              const float r = row_ok ? (c_bf16 ? bf16_round(f[j]) : f[j]) : 0.f;
              s1[j] = r;
              s2[j] = r * r;
            }
            const float cs = warp_colsum32(s1, lane), cq = warp_colsum32(s2, lane);
            stat_s[(acc * 4 + q) * BN + p * 64 + h * 32 + lane] = make_float2(cs, cq);
          }
          if (!row_ok) continue;
          if (c_bf16) {
            bf16* crow = reinterpret_cast<bf16*>(Cv) + out_row * ldc + n0 + 32 * h;
#pragma unroll
            for (int j = 0; j < 32; j += 16)
              st_global_256(crow + j, pack_bf16x2(f[j], f[j + 1]), pack_bf16x2(f[j + 2], f[j + 3]), pack_bf16x2(f[j + 4], f[j + 5]),
                            pack_bf16x2(f[j + 6], f[j + 7]), pack_bf16x2(f[j + 8], f[j + 9]), pack_bf16x2(f[j + 10], f[j + 11]),
                            pack_bf16x2(f[j + 12], f[j + 13]), pack_bf16x2(f[j + 14], f[j + 15]));
          } else {
            float* crow = reinterpret_cast<float*>(Cv) + out_row * ldc + n0 + 32 * h;
#pragma unroll
            for (int j = 0; j < 32; j += 8)
              st_global_256(crow + j, __float_as_uint(f[j]), __float_as_uint(f[j + 1]), __float_as_uint(f[j + 2]), __float_as_uint(f[j + 3]),
                            __float_as_uint(f[j + 4]), __float_as_uint(f[j + 5]), __float_as_uint(f[j + 6]), __float_as_uint(f[j + 7]));
          }
        }
      }
      if (STAT) {
        epi_bar_sync();
        for (int i = q * 32 + lane; i < BN; i += 128) {
          const int p = i >> 6, ch = i & 63;
          const float2 a = stat_s[(acc * 4 + 0) * BN + i], b = stat_s[(acc * 4 + 1) * BN + i];
          const float2 c2 = stat_s[(acc * 4 + 2) * BN + i], d = stat_s[(acc * 4 + 3) * BN + i];
          stat_partial[((long long)mt * 4 + p) * g.Cn + n0 + ch] = make_float2((a.x + b.x) + (c2.x + d.x), (a.y + b.y) + (c2.y + d.y));
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// C[M, N] = sum_z partial[z]; transposed != 0: the partials are [z][N][M] (kind 1 with swapped operand roles)
__global__ void conv_splitk_reduce_kernel(const float* __restrict__ partial, int splits, float* __restrict__ C, long long ldc, int M, int N,
                                          int accumulate, int transposed) {
  const long long total = (long long)M * N;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const long long m = idx / N;
    const int n = (int)(idx - m * N);
    const long long pidx = transposed ? (long long)n * M + m : idx;
    float acc = 0.f;
    for (int z = 0; z < splits; z++) acc += partial[(long long)z * total + pidx];
    if (accumulate) acc += C[m * ldc + n];
    C[m * ldc + n] = acc;
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_enc = nullptr;
std::once_flag g_once2;
int g_sms = 148;
int g_attr[2][3][3] = {};
// kind 2 with at most this many output channels: the four parity phases fused into one tile.  Measured (C2 step, B200):
// 64 -> -0.36 ms; 128 -> +0.1 ms (the N = 64 MMAs of the fused tile issue twice as many instructions as the 128-wide phase
// tiles, which outweighs the saved operand fills)
constexpr int kConvt4MaxCn = 64;
int g_convt4_attr[2] = {};

void resolve2() {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0) g_sms = sms;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
    g_enc = reinterpret_cast<EncodeTiledFn>(fn);
  (void)cudaGetLastError();
}

int map2d(CUtensorMap* m, const void* base, long long dim0, long long dim1, long long ld, int box1) {
  cuuint64_t dims[2] = {(cuuint64_t)dim0, (cuuint64_t)dim1};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)box1};
  cuuint32_t es[2] = {1, 1};
  CUresult r = g_enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    p2pvg_set_error("conv_gemm: 2-D tensor map failed (%d)", (int)r);
    return P2PVG_ERR_CUDA;
  }
  return P2PVG_OK;
}

// NHWC [N, Hm, Wm, C] pixel-box map: box {64 ch, bw*s, bh*s, bn} traversed with stride s in x and y
int map4d(CUtensorMap* m, const void* base, int N, int Hm, int Wm, int C, int bw, int bh, int bn, int s) {
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)Wm, (cuuint64_t)Hm, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)Wm * C * 2, (cuuint64_t)Hm * Wm * C * 2};
  cuuint32_t box[4] = {64, (cuuint32_t)(bw * s), (cuuint32_t)(bh * s), (cuuint32_t)bn};
  cuuint32_t es[4] = {1, (cuuint32_t)s, (cuuint32_t)s, 1};
  CUresult r = g_enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    p2pvg_set_error("conv_gemm: 4-D tensor map failed (%d): N=%d H=%d W=%d C=%d box=(%d,%d,%d) s=%d", (int)r, N, Hm, Wm, C, bw, bh, bn, s);
    return P2PVG_ERR_CUDA;
  }
  return P2PVG_OK;
}

bool box_for(int P, int H, int W, int& bh, int& bn) {
  const int HW = H * W;
  if (HW >= P) {
    if (P % W != 0 || (H % (P / W)) != 0) return false;
    bh = P / W;
    bn = 1;
  } else {
    if (P % HW != 0) return false;
    bh = H;
    bn = P / HW;
  }
  return bh * 2 <= 256 && W * 2 <= 256 && bn <= 256;
}

template <int KIND, int BN, bool STAT>
int launch_t(const CUtensorMap& ta, const CUtensorMap& tb, void* C, int c_dtype, long long ldc, const Geom& g, int accumulate,
             const float* bias, const float* addend, const int* grp_src, float* partial, int splits, int kb_per_split, cudaStream_t st,
             float2* stat_partial);

template <int KIND, int BN>
int launch(const CUtensorMap& ta, const CUtensorMap& tb, void* C, int c_dtype, long long ldc, const Geom& g, int accumulate,
           const float* bias, const float* addend, const int* grp_src, float* partial, int splits, int kb_per_split, cudaStream_t st,
           float2* stat_partial = nullptr) {
  if (KIND != 1 && stat_partial != nullptr) return launch_t<KIND, BN, (KIND != 1)>(ta, tb, C, c_dtype, ldc, g, accumulate, bias, addend, grp_src, partial, splits, kb_per_split, st, stat_partial);
  return launch_t<KIND, BN, false>(ta, tb, C, c_dtype, ldc, g, accumulate, bias, addend, grp_src, partial, splits, kb_per_split, st, nullptr);
}

template <int KIND, int BN, bool STAT>
int launch_t(const CUtensorMap& ta, const CUtensorMap& tb, void* C, int c_dtype, long long ldc, const Geom& g, int accumulate,
             const float* bias, const float* addend, const int* grp_src, float* partial, int splits, int kb_per_split, cudaStream_t st,
             float2* stat_partial) {
  auto kern = conv_gemm_kernel<KIND, BN, STAT>;
  int& done = g_attr[STAT][KIND][BN == 256 ? 2 : BN == 128];
  if (!done) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<BN>::SMEM_BYTES);
    if (e != cudaSuccess) {
      p2pvg_set_error("conv_gemm: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return P2PVG_ERR_CUDA;
    }
    done = 1;
  }
  long long tiles = (long long)cdiv(g.M, BLOCK_M) * cdiv(g.Ntot, BN) * splits * (KIND == 2 ? 4 : 1);
  int grid = (int)(tiles < g_sms ? tiles : g_sms);
  kern<<<grid, NUM_THREADS, Cfg<BN>::SMEM_BYTES, st>>>(ta, tb, C, c_dtype == P2PVG_BF16, ldc, g, accumulate, bias, addend, grp_src, partial,
                                                      kb_per_split, splits, stat_partial);
  return p2pvg_check_launch("conv_gemm");
}

int launch_convt4(const CUtensorMap& ta, const CUtensorMap& tb, void* C, int c_dtype, long long ldc, const Geom& g, const float* bias,
                  const float* addend, const int* grp_src, float2* stat_partial, cudaStream_t st) {
  const bool stat = stat_partial != nullptr;
  int& done = g_convt4_attr[stat];
  if (!done) {
    cudaError_t e = stat ? cudaFuncSetAttribute(convt4_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<256>::SMEM_BYTES)
                         : cudaFuncSetAttribute(convt4_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<256>::SMEM_BYTES);
    if (e != cudaSuccess) {
      p2pvg_set_error("conv_gemm (fused phases): cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return P2PVG_ERR_CUDA;
    }
    done = 1;
  }
  const long long tiles = (long long)cdiv(g.M, BLOCK_M) * (g.Cn / 64);
  const int grid = (int)(tiles < g_sms ? tiles : g_sms);
  if (stat)
    convt4_kernel<true><<<grid, NUM_THREADS, Cfg<256>::SMEM_BYTES, st>>>(ta, tb, C, c_dtype == P2PVG_BF16, ldc, g, bias, addend, grp_src, stat_partial);
  else
    convt4_kernel<false><<<grid, NUM_THREADS, Cfg<256>::SMEM_BYTES, st>>>(ta, tb, C, c_dtype == P2PVG_BF16, ldc, g, bias, addend, grp_src, nullptr);
  return p2pvg_check_launch("conv_gemm (fused phases)");
}

}  // namespace

// a, b: see the kind table at the top.  H, W: SMALL-map size.  Returns P2PVG_ERR_UNSUPPORTED when the shape does not
// fit the pixel-box tiling (the caller then uses the explicit im2col / col2im path).
int p2pvg_conv_gemm_impl(int kind, const void* a, const void* b, long long ldb, void* c, int c_dtype, long long ldc, int N, int H, int W,
                         int Ck, int Cn, int Cm, const float* bias, const float* addend, const int* grp_src, int imgs_per_group,
                         int accumulate, void* ws, size_t ws_bytes, void* stat_partial_v, int addend_dtype, cudaStream_t st) {
  float2* stat_partial = reinterpret_cast<float2*>(stat_partial_v);
  std::call_once(g_once2, resolve2);
  P2PVG_REQUIRE(g_enc != nullptr, P2PVG_ERR_UNSUPPORTED, "conv_gemm: cuTensorMapEncodeTiled unavailable");
  P2PVG_REQUIRE(kind >= 0 && kind <= 5, P2PVG_ERR_BAD_ARG, "conv_gemm: bad kind %d", kind);
  if (N <= 0) return P2PVG_OK;
  Geom g;
  g.N = N; g.H = H; g.W = W; g.Ck = Ck; g.Cn = Cn; g.imgs_per_group = imgs_per_group > 0 ? imgs_per_group : 1;
  g.add_bf16 = (addend != nullptr && addend_dtype == P2PVG_BF16) ? 1 : 0;
  g.swap = 0;
  g.bres = 0;
  g.ks = kind >= 3 ? 3 : 4; g.st = kind >= 3 ? 1 : 2; g.sgn = kind == 5 ? -1 : 1;
  const int taps = g.ks * g.ks;
  if (kind == 3 || kind == 5) kind = 0;
  if (kind == 4) kind = 1;
  // kinds 0 / 2 tile the output in 128-pixel boxes, kind 1 reduces over 64-pixel boxes
  g.bh128 = g.bn128 = g.bh64 = g.bn64 = 1;
  g.bw64 = W;
  bool ok;
  if (kind == 1) {
    if (W > 64 && W % 64 == 0 && W * g.st <= 256) { g.bw64 = 64; ok = true; }
    else ok = box_for(64, H, W, g.bh64, g.bn64);
  } else {
    ok = box_for(128, H, W, g.bh128, g.bn128);
  }
  ok = ok && (((uintptr_t)a | (uintptr_t)b | (uintptr_t)c) & 15) == 0;
  if (kind == 1) ok = ok && (Cn % 64 == 0) && (Cm % 8 == 0);
  else ok = ok && (Ck % 64 == 0) && (Cn % 32 == 0) && (ldb % 8 == 0);
  if (kind == 2 || addend != nullptr) ok = ok && (Cn % 64 == 0);
  if (!ok) {
    p2pvg_set_error("conv_gemm: shape not supported by the pixel-box tiling (kind=%d N=%d H=%d W=%d Ck=%d Cn=%d)", kind, N, H, W, Ck, Cn);
    return P2PVG_ERR_UNSUPPORTED;
  }
  CUtensorMap ta, tb;
  int rc;
  const long long pix = (long long)N * H * W;
  if (kind == 0) {
    g.M = (int)pix; g.Ntot = Cn;
    rc = map4d(&ta, a, N, g.st * H, g.st * W, Ck, W, g.bh128, g.bn128, g.st);
    if (rc) return rc;
    const int BN = Cn % 256 == 0 ? 256 : Cn > 64 ? 128 : 64;
    rc = map2d(&tb, b, (long long)taps * Ck, Cn, ldb, BN);
    if (rc) return rc;
    const int nkb = taps * (Ck / 64);
    g.bres = (BN == 64 && Cn == 64 && Ck == 64 && taps <= 9) ? 1 : 0;
    if (BN == 256) return launch<0, 256>(ta, tb, c, c_dtype, ldc, g, accumulate, bias, addend, grp_src, nullptr, 1, nkb, st, stat_partial);
    if (BN == 128) return launch<0, 128>(ta, tb, c, c_dtype, ldc, g, accumulate, bias, addend, grp_src, nullptr, 1, nkb, st, stat_partial);
    return launch<0, 64>(ta, tb, c, c_dtype, ldc, g, accumulate, bias, addend, grp_src, nullptr, 1, nkb, st, stat_partial);
  }
  if (kind == 2) {
    g.M = (int)pix; g.Ntot = Cn;
    rc = map4d(&ta, a, N, H, W, Ck, W, g.bh128, g.bn128, 1);
    if (rc) return rc;
    rc = map2d(&tb, b, 16LL * Cn, Ck, ldb, 64);  // MN-major weight [Ck rows][16*Cn]
    if (rc) return rc;
    const int nkb = 4 * (Ck / 64);
    if (Cn % 64 == 0 && Cn <= kConvt4MaxCn && !accumulate && (ldc % 16 == 0) && (c_dtype == P2PVG_F32 || ldc % 32 == 0) &&
        ((uintptr_t)c & 31) == 0 && (addend == nullptr || ((uintptr_t)addend & 15) == 0))
      return launch_convt4(ta, tb, c, c_dtype, ldc, g, bias, addend, grp_src, stat_partial, st);
    const int BN = Cn % 256 == 0 ? 256 : Cn > 64 ? 128 : 64;
    if (BN == 256) return launch<2, 256>(ta, tb, c, c_dtype, ldc, g, accumulate, bias, addend, grp_src, nullptr, 1, nkb, st, stat_partial);
    if (BN == 128) return launch<2, 128>(ta, tb, c, c_dtype, ldc, g, accumulate, bias, addend, grp_src, nullptr, 1, nkb, st, stat_partial);
    return launch<2, 64>(ta, tb, c, c_dtype, ldc, g, accumulate, bias, addend, grp_src, nullptr, 1, nkb, st, stat_partial);
  }
  // kind 1: weight gradient
  P2PVG_REQUIRE(c_dtype == P2PVG_F32, P2PVG_ERR_BAD_ARG, "conv_gemm kind 1 writes fp32");
  P2PVG_REQUIRE(stat_partial == nullptr, P2PVG_ERR_BAD_ARG, "conv_gemm: BatchNorm statistics belong to the forward / data-gradient kinds");
  g.Ck = 64;
  // 64 output channels would fill only half of a 128-row MMA tile: swap the operand roles (M = taps*Cn from the gathered map,
  // N = Cm); the partial sums are then [taps*Cn][Cm] and the split-K reduce kernel writes the transposed result
  const int nkb = (int)((pix + 63) / 64);
  g.swap = (Cm == 64 && nkb >= 16 && ws != nullptr && (size_t)2 * taps * Cn * Cm * sizeof(float) <= ws_bytes) ? 1 : 0;
  if (g.swap) {
    g.M = taps * Cn; g.Ntot = Cm;
    rc = map4d(&ta, b, N, g.st * H, g.st * W, Cn, g.bw64, g.bh64, g.bn64, g.st);
    if (rc) return rc;
    rc = map2d(&tb, a, Cm, pix, Cm, 64);
    if (rc) return rc;
  } else {
    g.M = Cm; g.Ntot = taps * Cn;
    rc = map2d(&ta, a, Cm, pix, Cm, 64);  // a_small [pix][Cm] as MN-major A
    if (rc) return rc;
    rc = map4d(&tb, b, N, g.st * H, g.st * W, Cn, g.bw64, g.bh64, g.bn64, g.st);
    if (rc) return rc;
  }
  // a wide tile spans several filter taps when Cn == 64
  const int BN = (!g.swap && g.Ntot % 256 == 0) ? 256 : (g.Ntot % 128 == 0) ? 128 : 64;
  const long long tiles = (long long)cdiv(g.M, BLOCK_M) * cdiv(g.Ntot, BN);
  // split-K chosen by a small cost model (units: time of one 128x128x64 k-block on one SM, ~0.22 us): the persistent grid
  // processes ceil(items / SMs) rounds of (k-blocks per item + fixed per-item cost); partial sums cost a write + read
  int splits = g.swap ? 2 : 1;
  {
    double best = 1e300;
    const int maxs = nkb / 8 < 64 ? nkb / 8 : 64;
    const int smin = g.swap ? 2 : 1;
    for (int s = smin; s <= (maxs < smin ? smin : maxs); s++) {
      const int kb = cdiv(nkb, s), se = cdiv(nkb, kb);
      if (se > 1 && (ws == nullptr || (size_t)se * g.M * g.Ntot * sizeof(float) > ws_bytes)) continue;
      const long long rounds = cdiv((long long)tiles * se, g_sms);
      double cost = (double)rounds * (kb + 8.0);
      if (se > 1) cost += (double)se * g.M * g.Ntot * 8.0 / 6.0e12 / (0.22e-6 * BN / 128);
      if (cost < best) { best = cost; splits = se; }
    }
  }
  int kbps = cdiv(nkb, splits);
  splits = cdiv(nkb, kbps);
  float* partial = splits > 1 ? reinterpret_cast<float*>(ws) : nullptr;
  if (BN == 256) rc = launch<1, 256>(ta, tb, c, c_dtype, ldc, g, accumulate, nullptr, nullptr, nullptr, partial, splits, kbps, st);
  else if (BN == 128) rc = launch<1, 128>(ta, tb, c, c_dtype, ldc, g, accumulate, nullptr, nullptr, nullptr, partial, splits, kbps, st);
  else rc = launch<1, 64>(ta, tb, c, c_dtype, ldc, g, accumulate, nullptr, nullptr, nullptr, partial, splits, kbps, st);
  if (rc) return rc;
  if (splits > 1) {
    long long total = (long long)Cm * taps * Cn;
    int blocks = (int)((total + 255) / 256 > 1184 ? 1184 : (total + 255) / 256);
    conv_splitk_reduce_kernel<<<blocks, 256, 0, st>>>(partial, splits, (float*)c, ldc, Cm, taps * Cn, accumulate, g.swap);
    return p2pvg_check_launch("conv_splitk_reduce");
  }
  P2PVG_REQUIRE(!g.swap, P2PVG_ERR_UNSUPPORTED, "conv_gemm kind 1 (swapped roles) needs the split-K workspace");
  return P2PVG_OK;
}
