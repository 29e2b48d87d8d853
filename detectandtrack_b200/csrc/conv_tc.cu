// Conv3d / Conv2d / FC as ONE implicit-GEMM kernel on the 5th-gen tensor cores (tcgen05),
// NDHWC activations, fused AffineChannel (+bias) + residual / top-down-upsample add + ReLU.
//
// Replaces, on the reference's hot path:
//   Caffe2 Conv / ConvNd engine=CUDNN        (lib/modeling/detector.py:318-322,410-436 and every
//                                             call site listed in SURVEY.md §2.3 K5)
//   AffineChannelNdOp<float,CUDAContext>     (lib/ops/affine_channel_nd_op.cu:19-70)  -> epilogue
//   Relu / Sum (residual)                    (lib/modeling/ResNet3D.py:37,47,147-152) -> epilogue
//   UpsampleNearest + Sum (FPN top-down)     (lib/modeling/FPN3D.py:211-222)          -> epilogue
//   FC (cuBLAS)                              (lib/modeling/head_builder.py:33-36)     -> kT=kH=kW=1
//
// GEMM view: D[m, n] = sum_{tap, c} A[m @ tap, c] * W[tap, n, c]
//   m = output position (img, t, ho, wo) tiled as TH x TW spatial patches (TH*TW <= 128 rows)
//   n = output channel, BLOCK_N in {32, 64, 128, 256};  k-block = one tap x 128 bytes of channels
//   A tile: one 5-D TMA box (C=128B, TW, TH, 1, 1) at the tap-shifted coordinate; out-of-bounds
//           elements (spatial / temporal zero padding, ragged edge tiles, channel tail) are
//           zero-filled by the TMA unit, so padding costs no instructions and no branches.  Taps of the outermost
//           filter dimension whose box lies wholly in that fill are not issued at all (tap_range).
//   W tile: 3-D TMA box (C=128B, BLOCK_N, 1) of the pre-packed [tap][Cout][Cin] weights.
//   Both land in the 128B-swizzled K-major layout tcgen05.mma reads directly.
// Roles (640 threads, 1 CTA / SM, persistent over tiles):
//   warp 0, 19: TMA producers (activation / weight tiles; one elected lane each)   smem ring: full[]/empty[]
//   warp 1    : TMEM allocator + MMA issuer (one lane)   tcgen05.mma -> TMEM, tcgen05.commit
//   warp 2    : TMA store warp                           staged output chunks -> global, recycles staging slots
//   warps 3-18: epilogue; TMEM -> registers (tcgen05.ld), scale/bias/residual/ReLU in fp32, staged in
//               128B-swizzled smem chunks.  Two TMEM accumulator stages overlap it with the next tile's MMAs.
// Everything is handed over through mbarriers; there is no block-wide barrier inside the tile loop.
#include "common.cuh"
#include "tc_common.cuh"
#include "../../include/dt_b200.h"
#include <cuda_bf16.h>
#include <stdlib.h>

namespace dt {

using namespace tc;

// division by a run-time constant without the ~100-cycle integer-division sequence (valid for x < 2^31)
struct FastDiv {
  uint32_t mul, shr, d;
};
static FastDiv make_fastdiv(int d) {
  FastDiv f; f.d = (uint32_t)d; f.mul = 0; f.shr = 0;
  if (d > 1) {
    int l = 0;
    while ((1u << l) < (uint32_t)d) ++l;
    const int pw = 31 + l;
    f.mul = (uint32_t)((((unsigned long long)1 << pw) + (unsigned long long)d - 1) / (unsigned long long)d);
    f.shr = (uint32_t)(l - 1);
  }
  return f;
}
__device__ __forceinline__ uint32_t fdiv(uint32_t x, const FastDiv& f) { return f.d == 1 ? x : (__umulhi(x, f.mul) >> f.shr); }

struct ConvKernelParams {
  // output geometry
  int N, To, Ho, Wo, Cout;
  // filter
  int kT, kH, kW, sT, sH, sW, pT, pH, pW;
  int kchunks;                 // ceil(Cin / BK)
  // tiling
  int TH, TW, TT, TB;          // rows of one M tile = TB images x TT frames x TH x TW positions (<= 128)
  int tiles_h, tiles_w, tiles_t, tiles_b, tiles_n, total_tiles;
  FastDiv fd_n, fd_w, fd_h, fd_t;    // tile index -> (column tile, w, h, t, image) tile coordinates
  uint32_t a_bytes;            // TB*TT*TH*TW*128
  // epilogue
  const float* scale;          // [Cout] or null (1)
  const float* bias;           // [Cout] or null (0)
  const void* residual;        // same dtype as out, or null
  int res_mode;                // 0 none, 1 same shape, 2 nearest-2x upsample of (Ho/2, Wo/2)
  int res_ld;
  int relu;
  int out_f32;                 // 1: fp32 output, 0: bf16
  // 3xTF32 ("fp32-accurate") mode: activations / weights are stored as [hi | lo] tf32 pairs along the
  // channel axis; D = A_hi*B_hi + A_lo*B_hi + A_hi*B_lo (the lo*lo term is below fp32 resolution).
  int split_in;                // 1: three k-blocks per (tap, channel chunk) with the offsets below
  int nsub;                    // k-blocks per (tap, channel chunk): 1 plain, 3 split operands (hi*hi, lo*hi, hi*lo),
                               // 2 split conv1 (the blob pixel carries [hi3 | lo3]: one block against [W_hi | W_hi], one against [W_lo | 0])
  int a_lo_off, b_lo_off;      // element offsets of the lo halves in the x rows / packed weight rows
  int split_out;               // 1: write hi at channel c and lo at out_lo_off + c (fp32)
  int out_lo_off, res_lo_off;  // lo-half offsets of the output / residual rows
  int nstages, ncbuf;          // smem split chosen per layer: operand ring depth / output staging buffers
  int ks;                      // k-blocks per ring stage
  int ktab;                    // entries of the k-block schedule (kiters + 1 padding, even)
  int t_first;                 // first output frame computed (frames before it are skipped)
  int Ti, Hi;                  // input frames / rows (the extents tap_range tests a tap's box against)
  int tap_skip;                // 1: each tile walks only the taps of tap_range (0: every tap)
  int row_planes;              // conv1: input rows de-interleaved by parity, filter row kh -> plane kh & 1, row + kh >> 1
  int nrbuf;                   // > 0: bf16 residual chunks arrive by TMA in a ring of this many staged chunks
  int res_up;                  // with nrbuf > 0: the residual is the (Ho/2, Wo/2) map of the FPN top-down add;
                               // its (TH/2 x TW/2) box is loaded and every row is read by its four children
  int ab_format;               // tcgen05 kind::f16 operand format: 1 bf16, 0 fp16 (kind::tf32: 2)
  int round_tf32;              // fp32 output is rounded (RNE) to tf32 so the next tcgen05 kind::tf32 MMA,
                               // which TRUNCATES its 32-bit operands, sees exactly representable values
};

__device__ __forceinline__ float round_to_tf32(float v) {
  uint32_t u = __float_as_uint(v);
  u += 0xFFFu + ((u >> 13) & 1u);
  return __uint_as_float(u & 0xFFFFE000u);
}

constexpr int EPI_WARPS = 16;                         // 4 TMEM lane groups x 4 column quarters
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int CONV_THREADS = 128 + EPI_THREADS;       // + two TMA producer warps, the MMA issuer and the TMA store warp
constexpr int B_WARP = 3 + EPI_WARPS;                 // weight-tile producer (warps 3 .. 3+EPI_WARPS-1 are the epilogue)

template <int BN>
struct ConvCfg {
  static constexpr int A_BYTES = 128 * 128;            // 128 rows x 128 B
  static constexpr int B_BYTES = BN * 128;
  static constexpr int KB_BYTES = A_BYTES + B_BYTES;   // one k-block of both operands
  static constexpr int MAX_STAGES = 8;
  static constexpr int TMEM_COLS = (2 * BN < 32) ? 32 : 2 * BN;
  static constexpr int C_BYTES = 128 * 128;            // one staged output chunk: 128 rows x 128 B
  static constexpr int BAR_BYTES = 384;                // mbarriers + TMEM base pointer
  static constexpr int FIXED_BYTES = BAR_BYTES;
  static constexpr int BUDGET = 227 * 1024;
  // K-heavy layers want a deep operand ring; K-light (HBM-bound) layers want output staging buffers so the
  // epilogue never waits for a TMA store to drain, and (with a residual) a ring of prefetched residual chunks.
  static int tab_bytes(int kiters) { return ((kiters + 2) * 24 + 127) / 128 * 128; }   // k-block schedule
  static void split(int kiters, bool res_tma, bool split_out, bool out_f32, int* stages, int* ks, int* ncbuf, int* nrbuf) {
    const int chunks = BN / (out_f32 ? 32 : 64);        // staged chunks per tile
    int c = (kiters >= 12 && !split_out) ? ((BN >= 256) ? 1 : 2) : 4;   // split (hi, lo) output: two slots of two buffers
    if (!split_out && c > 2 * chunks) c = chunks >= 1 ? 2 * chunks : 2;   // two tiles of staging are enough
    const int r = res_tma ? ((kiters >= 12 || split_out) ? 2 : 4) : 0;      // split output: a residual slot is a chunk pair
    const int rb = split_out ? 2 * r : r;
    // narrow tiles retire a k-block's MMAs faster than one producer / issuer round trip through the
    // mbarriers: let a ring stage carry two k-blocks there (same bytes in flight, half the handshakes)
    const int avail = BUDGET - FIXED_BYTES - tab_bytes(kiters) - (c + rb) * C_BYTES;
    const int k = (BN <= 128 && kiters >= 2 && avail / (2 * KB_BYTES) >= 3) ? 2 : 1;
    int st = avail / (k * KB_BYTES);
    if (st > MAX_STAGES) st = MAX_STAGES;
    *stages = st; *ks = k; *ncbuf = c; *nrbuf = r;
  }
  static int smem_bytes(int kiters, int stages, int ks, int ncbuf, int nrbuf, bool split_out) {
    return stages * ks * KB_BYTES + (ncbuf + (split_out ? 2 : 1) * nrbuf) * C_BYTES + FIXED_BYTES + tab_bytes(kiters);
  }
};

struct TileCoord { int nt, twi, thi, tti, tbi; };
__device__ __forceinline__ TileCoord decode_tile(const ConvKernelParams& p, int tile) {
  TileCoord c;
  uint32_t m = fdiv((uint32_t)tile, p.fd_n);  c.nt = tile - (int)m * p.tiles_n;
  uint32_t q = fdiv(m, p.fd_w);               c.twi = (int)m - (int)q * p.tiles_w;  m = q;
  q = fdiv(m, p.fd_h);                        c.thi = (int)m - (int)q * p.tiles_h;  m = q;
  q = fdiv(m, p.fd_t);                        c.tti = (int)m - (int)q * p.tiles_t;
  c.tbi = (int)q;
  return c;
}

// Schedule entries [kb, ke) one tile issues.  The schedule is tap-major with kt outermost, so the taps of the
// outermost filter dimension with more than one tap (kt, else kh) are contiguous runs of kiters / extent entries.
// Tap k of that dimension reads input positions base + k + j*s, j in [0, n) (n = TT frames or TH rows of the tile's
// box); when none of them lies inside [0, lim) the box is all TMA zero fill and its products are exact zeros, so
// those taps are left out.  Skipping zero products and keeping the order of the others leaves every sum unchanged.
// An empty range (a tile wholly in the padding) issues everything, so the accumulator is always written.
struct KRange { int kb, ke; };
__device__ __forceinline__ KRange tap_range(const ConvKernelParams& p, const TileCoord& tc, int kiters) {
  KRange r = {0, kiters};
  if (!p.tap_skip) return r;
  int ext, base, n, s, lim;
  if (p.kT > 1) {
    ext = p.kT; base = (tc.tti * p.TT + p.t_first) * p.sT - p.pT; n = p.TT; s = p.sT; lim = p.Ti;
  } else if (p.kH > 1) {
    ext = p.kH; base = tc.thi * p.TH * p.sH - p.pH; n = p.TH; s = p.sH; lim = p.Hi;
  } else {
    return r;
  }
  const int k0 = max(0, -(base + (n - 1) * s));
  const int k1 = min(ext, lim - base);
  if (k0 < k1) {
    const int per = kiters / ext;
    r.kb = k0 * per; r.ke = k1 * per;
  }
  return r;
}

#ifdef DT_CONV_TRACE
__device__ long long g_conv_trace[64 * 16];
#define TRACE(ti, k) do { if (blockIdx.x == 0 && (ti) < 64) g_conv_trace[(ti) * 16 + (k)] = clock64(); } while (0)
#define TRACE_ADD(ti, k, v) do { if (blockIdx.x == 0 && (ti) < 64) g_conv_trace[(ti) * 16 + (k)] += (v); } while (0)
#else
#define TRACE(ti, k) do {} while (0)
#define TRACE_ADD(ti, k, v) do {} while (0)
#endif

// SPLIT: the output (and the residual) rows are [hi | lo] pairs (the x3 modes' intermediate activations); a template
// parameter so that the plain kernels do not carry the pair logic's registers (the epilogue sits at the 96-register cap).
template <int BN, bool TF32, bool SPLIT>
__global__ void __launch_bounds__(CONV_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmR,
               const ConvKernelParams p) {
  using Cfg = ConvCfg<BN>;
  const int STAGES = p.nstages;
  constexpr int BK = TF32 ? 32 : 64;                 // elements per 128-byte k-block
  // SWIZZLE_128B operands need 1024-byte aligned tiles: the dynamic window is declared with that alignment
  // (no static shared memory in this kernel) and checked once below instead of spending a kilobyte on slack
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* cbuf = smem + STAGES * p.ks * Cfg::KB_BYTES;              // [NCBUF][128 rows][128 B], 128B-swizzled
  uint8_t* rbuf = cbuf + p.ncbuf * Cfg::C_BYTES;                     // [NRBUF] residual chunks, same layout
  constexpr uint32_t rslot_bytes = SPLIT ? 2u * Cfg::C_BYTES : (uint32_t)Cfg::C_BYTES;   // split: (hi, lo) chunk pair
  uint64_t* bars = reinterpret_cast<uint64_t*>(rbuf + p.nrbuf * rslot_bytes);
  uint64_t* full = bars;                       // [STAGES]  operands landed
  uint64_t* empty = bars + STAGES;             // [STAGES]  operands consumed by the MMAs
  uint64_t* tmem_full = bars + 2 * STAGES;     // [2]       accumulator complete
  uint64_t* tmem_empty = tmem_full + 2;        // [2]       accumulator read out
  uint64_t* r_full = tmem_full + 4;            // [4]       residual chunk landed
  uint64_t* r_empty = tmem_full + 8;           // [4]       residual chunk consumed
  uint64_t* c_full = tmem_full + 12;           // [4]       output chunk staged by all epilogue warps
  uint64_t* c_free = tmem_full + 16;           // [4]       staging slot read out by its TMA store
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(tmem_full + 20);
  // k-block schedule of one tile: what the producers add to the tile's base coordinates for k-block j.
  // Built once; walking taps / channel chunks with carry logic in the producer loop costs more cycles per
  // k-block than a narrow tile's MMAs take.
  int4* tabA = reinterpret_cast<int4*>(reinterpret_cast<uint8_t*>(bars) + Cfg::BAR_BYTES);   // {c, dw, dh, dt}
  int2* tabB = reinterpret_cast<int2*>(tabA + p.ktab);                                        // {c, tap}
  if (threadIdx.x == 0 && (smem_u32(smem) & 1023u) != 0) __trap();
  {
    const int nsub = p.nsub;
    const int kit = p.kT * p.kH * p.kW * p.kchunks * nsub;
    for (int j = threadIdx.x; j < p.ktab; j += blockDim.x) {
      const int jj = min(j, kit - 1);                   // padding entries repeat the last k-block (never issued)
      const int sub = jj % nsub;
      int r = jj / nsub;
      const int kc = r % p.kchunks; r /= p.kchunks;
      const int tap = r;
      const int kw = r % p.kW; r /= p.kW;
      const int kh = r % p.kH;
      const int kt = r / p.kH;
      // sub 0: A_hi x B_hi, 1: A_lo x B_hi, 2: A_hi x B_lo
      const int ca = kc * BK + (sub == 1 ? p.a_lo_off : 0);
      const int cb = kc * BK + (sub == 2 ? p.b_lo_off : 0);
      if (p.row_planes) {          // conv1: one box per filter row; split mode: weight blocks 2*kh (hi) and 2*kh + 1 (lo)
        tabA[j] = make_int4(0, 0, kh >> 1, kh & 1);
        tabB[j] = make_int2(0, tap * nsub + sub);
      } else {
        tabA[j] = make_int4(ca, kw, kh, kt);
        tabB[j] = make_int2(cb, tap);
      }
    }
  }

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    prefetch_tmap(&tmC);
    if (p.nrbuf > 0) prefetch_tmap(&tmR);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 2); mbar_init(&empty[s], 1); }    // full: A and B producers
    for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], EPI_WARPS); }
    for (int s = 0; s < 4; ++s) {
      mbar_init(&r_full[s], 1); mbar_init(&r_empty[s], EPI_WARPS);
      mbar_init(&c_full[s], EPI_WARPS); mbar_init(&c_free[s], 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_base_smem);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_base_smem;
  // Programmatic dependent launch: everything above (barrier init, TMEM allocation, tensor-map prefetch, the k-block
  // schedule) touched only kernel parameters and shared memory, so it may overlap the tail of the previous kernel of
  // the stream; no global data is read or written before this wait.  The trigger lets the NEXT kernel's prologue do
  // the same under this one's tail (its CTAs become resident as this kernel's CTAs retire: 1 CTA / SM by shared memory).
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  const int taps = p.kT * p.kH * p.kW;
  const int kiters = taps * p.kchunks * p.nsub;

  if (warp == 0 || warp == B_WARP) {
    // ===================== TMA producers =====================
    // Two warps: warp 0 loads the activation tiles (and the residual ring), warp B_WARP the weight tiles; both
    // arm the same full[] barrier with their own byte count.  One warp doing both spends ~500 cycles per
    // k-block on scalar bookkeeping + TMA issue, more than a 128-column tile's MMAs take (256 cycles).
    // The whole warp runs the loop (warp-uniform control flow and addresses, so descriptors / coordinates
    // stay in uniform registers); one elected lane issues.  A divergent `if (lane == 0)` around the loop
    // makes the compiler wrap every UTMALDG / UTCHMMA in an elect-broadcast "waterfall" loop.
    const bool load_b = warp != 0;
    int stage = 0; uint32_t phase = 0;
    int rslot = 0; uint32_t rphase = 0;
    const uint32_t smem_u = smem_u32(smem) + (load_b ? (uint32_t)Cfg::A_BYTES : 0u);
    const uint32_t full_u = smem_u32(full), empty_u = smem_u32(empty);
    const int KS = p.ks;                                  // k-blocks per ring stage (one mbarrier round trip)
    const uint32_t stage_bytes = (uint32_t)KS * Cfg::KB_BYTES;
    const uint32_t kb_tx = load_b ? (uint32_t)Cfg::B_BYTES : p.a_bytes;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(p, tile);
      const int n = tc.tbi * p.TB;
      const int w_base = tc.twi * p.TW * p.sW - p.pW;
      const int h_base = tc.thi * p.TH * p.sH - p.pH;
      const int t_base = p.row_planes ? 0 : (tc.tti * p.TT + p.t_first) * p.sT - p.pT;
      const int n_base = tc.nt * BN;
      const KRange kr = tap_range(p, tc, kiters);
#ifdef DT_CONV_TRACE
      long long acc_wait = 0, acc_issue = 0;
#endif
      if (lane == 0 && !load_b) TRACE(tile / gridDim.x, 0);
      for (int ki = kr.kb; ki < kr.ke; ki += KS) {
        const int nk = min(KS, kr.ke - ki);
        // this stage's k-blocks from the schedule (uniform loads), then ONE elected issue block
        int x0[2], x1[2], x2[2], x3[2];
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          if (load_b) {
            const int2 e = tabB[ki + q];
            x0[q] = e.x; x1[q] = n_base; x2[q] = e.y; x3[q] = 0;
          } else {
            const int4 e = tabA[ki + q];
            x0[q] = e.x; x1[q] = w_base + e.y; x2[q] = h_base + e.z; x3[q] = t_base + e.w;
          }
        }
#ifdef DT_CONV_TRACE
        const long long tw0 = clock64();
#endif
        mbar_wait_u(empty_u + stage * 8, phase ^ 1);
#ifdef DT_CONV_TRACE
        acc_wait += clock64() - tw0;
        const long long tw2 = clock64();
#endif
        if (elect_one()) {
          const uint32_t bar = full_u + stage * 8;
          const uint32_t dst = smem_u + stage * stage_bytes;
          mbar_expect_tx_u(bar, (uint32_t)nk * kb_tx);
          if (load_b) {
            tma_load_3d_u(dst, &tmB, bar, x0[0], x1[0], x2[0]);
            if (nk > 1) tma_load_3d_u(dst + Cfg::KB_BYTES, &tmB, bar, x0[1], x1[1], x2[1]);
          } else {
            tma_load_5d_u(dst, &tmA, bar, x0[0], x1[0], x2[0], x3[0], n);
            if (nk > 1) tma_load_5d_u(dst + Cfg::KB_BYTES, &tmA, bar, x0[1], x1[1], x2[1], x3[1], n);
          }
        }
#ifdef DT_CONV_TRACE
        acc_issue += clock64() - tw2;
#endif
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (lane == 0 && !load_b) TRACE(tile / gridDim.x, 1);
#ifdef DT_CONV_TRACE
      if (lane == 0 && !load_b) { TRACE_ADD(tile / gridDim.x, 10, acc_wait); TRACE_ADD(tile / gridDim.x, 12, acc_issue); }
#endif
      if (p.nrbuf > 0 && !load_b) {
        // residual chunks of this tile (bf16, same box as the output chunks), consumed in order by the epilogue
        const int ncols = min(BN, p.Cout - n_base);
        for (int cc = 0; cc < ncols; cc += 64) {
          mbar_wait(&r_empty[rslot], rphase ^ 1);
          if (elect_one()) {
            const uint32_t bar = smem_u32(&r_full[rslot]);
            const uint32_t rbytes = p.res_up ? p.a_bytes >> 2 : p.a_bytes;
            mbar_expect_tx_u(bar, SPLIT ? 2u * rbytes : rbytes);
            tma_load_5d_u(smem_u32(rbuf) + rslot * rslot_bytes, &tmR, bar, n_base + cc, (tc.twi * p.TW) >> p.res_up,
                          (tc.thi * p.TH) >> p.res_up, tc.tti * p.TT, n);
            if (SPLIT)
              tma_load_5d_u(smem_u32(rbuf) + rslot * rslot_bytes + Cfg::C_BYTES, &tmR, bar, n_base + cc + p.res_lo_off,
                            (tc.twi * p.TW) >> p.res_up, (tc.thi * p.TH) >> p.res_up, tc.tti * p.TT, n);
          }
          if (++rslot == p.nrbuf) { rslot = 0; rphase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp, one elected lane issues) =====================
    const uint32_t idesc = make_idesc(128, BN, TF32 ? 2 : p.ab_format);
    const uint32_t smem_u = smem_u32(smem);
    const uint32_t full_u = smem_u32(full);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const int KS = p.ks;
    const uint32_t stage_bytes = (uint32_t)KS * Cfg::KB_BYTES;
    int stage = 0; uint32_t phase = 0;
    int as = 0; uint32_t aphase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      mbar_wait(&tmem_empty[as], aphase ^ 1);
      tcgen05_fence_after();
      const uint32_t d_tmem = tmem_u + as * BN;
      const KRange kr = tap_range(p, decode_tile(p, tile), kiters);     // the producers' range: the rings stay in step
      if (lane == 0) TRACE(tile / gridDim.x, 2);
#ifdef DT_CONV_TRACE
      long long acc_wf = 0;
#endif
      for (int ki = kr.kb; ki < kr.ke; ki += KS) {
        const int nk = min(KS, kr.ke - ki);
#ifdef DT_CONV_TRACE
        const long long tw1 = clock64();
#endif
        mbar_wait_u(full_u + stage * 8, phase);
#ifdef DT_CONV_TRACE
        acc_wf += clock64() - tw1;
#endif
        tcgen05_fence_after();
        const uint32_t a_addr = smem_u + stage * stage_bytes;
        if (elect_one()) {
          for (int q = 0; q < nk; ++q) {
            const uint64_t adesc = make_sw128_kmajor_desc(a_addr + q * Cfg::KB_BYTES);
            const uint64_t bdesc = make_sw128_kmajor_desc(a_addr + q * Cfg::KB_BYTES + Cfg::A_BYTES);
#pragma unroll
            for (int k = 0; k < 4; ++k)          // 4 x 32 B = one 128-byte swizzle row of K
              umma<TF32>(d_tmem, adesc + 2 * k, bdesc + 2 * k, idesc, (ki != kr.kb || q || k) ? 1u : 0u);
          }
          umma_commit(&empty[stage]);            // frees the smem slot when these MMAs retire
          if (ki + nk >= kr.ke) umma_commit(&tmem_full[as]);   // accumulator ready for the epilogue
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (lane == 0) TRACE(tile / gridDim.x, 3);
#ifdef DT_CONV_TRACE
      if (lane == 0) TRACE_ADD(tile / gridDim.x, 11, acc_wf);
#endif
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  } else if (warp == 2) {
    // ===================== TMA store warp =====================
    // Waits until all epilogue warps have staged a chunk (c_full), stores it (one elected lane, which also owns
    // the bulk async-groups) and hands staging slots back (c_free) once their store has read them out.  Keeping
    // this off the epilogue warps removes every block-wide barrier from the epilogue.
    constexpr bool split_out = SPLIT;
    const int CW = p.out_f32 ? 32 : 64;
    const int nslots = split_out ? p.ncbuf / 2 : p.ncbuf;     // split output: a slot is a (hi, lo) buffer pair
    const uint32_t slot_bytes = split_out ? 2u * Cfg::C_BYTES : (uint32_t)Cfg::C_BYTES;
    const uint32_t cbuf_u32 = smem_u32(cbuf);
    int slot = 0, prev_slot = 0; uint32_t sphase = 0;
    int issued = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(p, tile);
      const int nbase = tc.nt * BN;
      const int ncols = min(BN, p.Cout - nbase);
      const int cw0 = tc.twi * p.TW, ch0 = tc.thi * p.TH, ct0 = tc.tti * p.TT, cn0 = tc.tbi * p.TB;
      for (int cc = 0; cc < ncols; cc += CW) {
        mbar_wait(&c_full[slot], sphase);
        if (elect_one()) {
          const uint32_t buf = cbuf_u32 + (uint32_t)slot * slot_bytes;
          tma_store_5d(&tmC, buf, nbase + cc, cw0, ch0, ct0, cn0);
          if (split_out) tma_store_5d(&tmC, buf + Cfg::C_BYTES, nbase + cc + p.out_lo_off, cw0, ch0, ct0, cn0);
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
        // hand back the slot of the PREVIOUS chunk as soon as its store has read it out (at most this chunk's
        // store stays pending), so the epilogue warps may run nslots - 1 chunks ahead of the slowest one
        if (nslots == 1) {
          if (elect_one()) { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); mbar_arrive(&c_free[0]); }
        } else if (issued > 0) {
          if (elect_one()) { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); mbar_arrive(&c_free[prev_slot]); }
        }
        prev_slot = slot;
        ++issued;
        if (++slot == nslots) { slot = 0; sphase ^= 1; }
        __syncwarp();
      }
    }
    if (elect_one()) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  } else {
    // ===================== epilogue (warps 3..18) =====================
    // TMEM -> registers -> fp32 epilogue -> 128B-swizzled smem chunk -> TMA store (store warp).
    // Sixteen warps (four per scheduler): warp w reads TMEM lane group (w & 3) and owns column quarter
    // ((w - 3) >> 2) of every staged 128-byte row (32 bytes: 16 bf16 or 8 fp32 outputs).  No block-wide
    // barriers: staging slots are handed over through mbarriers (c_full / c_free), scale / bias are uniform
    // 16-byte loads through L1, ReLU rides on the bf16 pack (cvt.rn.relu), the TMEM load of chunk c+1 is issued
    // as soon as chunk c's accumulators have been consumed, and the accumulator is released to the MMA warp
    // right after its last column has been read.  The TMA store writes whole 128-byte lines and clips rows /
    // channels outside the tensor, so ragged tiles need no predication on the store side.
    const int lg = warp & 3;                   // TMEM lane group this warp may access
    const int part = (warp - 3) >> 2;          // which 32-byte quarter of the staged row this warp fills
    const int row = lg * 32 + lane;            // accumulator row == TMEM lane == staging row
    int rr = row;
    const int tw = rr % p.TW; rr /= p.TW;
    const int th = rr % p.TH; rr /= p.TH;
    const int tl = rr % p.TT;
    const int nl = rr / p.TT;                  // >= TB for the unused tail rows of a short tile
    const bool out_f32 = p.out_f32 != 0;
    constexpr bool split_out = SPLIT;
    const bool relu = p.relu != 0;
    const int res_mode = p.res_mode;
    const int Cout = p.Cout;
    const int CW = out_f32 ? 32 : 64;          // output columns per 128-byte staged row
    const int colw = out_f32 ? 8 : 16;         // columns this warp owns per chunk
    const int nslots = split_out ? p.ncbuf / 2 : p.ncbuf;
    const uint32_t slot_bytes = split_out ? 2u * Cfg::C_BYTES : (uint32_t)Cfg::C_BYTES;
    const uint32_t cbuf_u32 = smem_u32(cbuf);
    const uint32_t rbuf_u32 = smem_u32(rbuf);
    const bool res_tma = p.nrbuf > 0;
    const bool res_ldg = res_mode != 0 && !res_tma;
    // residual row of this thread inside a ring slot: its own row, or (top-down add) the row of its parent
    // position in the (TH/2 x TW/2) box of the coarser map
    const int rrow = p.res_up ? ((nl * p.TT + tl) * (p.TH >> 1) + (th >> 1)) * (p.TW >> 1) + (tw >> 1) : row;
    const uint32_t rrow_smem = (uint32_t)rrow * 128u;
    const uint32_t rswz = (uint32_t)(rrow & 7);
    const uint32_t rq0 = (((uint32_t)(2 * part)) ^ rswz) << 4, rq1 = (((uint32_t)(2 * part + 1)) ^ rswz) << 4;
    int rslot = 0; uint32_t rphase = 0;
    const uint32_t row_smem = (uint32_t)row * 128u;
    const uint32_t swz = (uint32_t)(row & 7);
    const uint32_t q0 = (((uint32_t)(2 * part)) ^ swz) << 4, q1 = (((uint32_t)(2 * part + 1)) ^ swz) << 4;
    const float* __restrict__ g_scale = p.scale;
    const float* __restrict__ g_bias = p.bias;
    int as = 0; uint32_t aphase = 0;
    int slot = 0; uint32_t sphase = 0;
    for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(p, tile);
      bool valid = true;
      size_t rpos = 0;
      if (res_ldg) {                           // per-thread residual row (fp32 / upsample-add paths only)
        const int ho = tc.thi * p.TH + th, wo = tc.twi * p.TW + tw;
        const int t = tc.tti * p.TT + tl, n = tc.tbi * p.TB + nl;
        valid = (nl < p.TB) && (ho < p.Ho) && (wo < p.Wo) && (t < p.To) && (n < p.N);
        rpos = (res_mode == 2) ? ((size_t)(n * p.To + t) * (p.Ho >> 1) + (ho >> 1)) * (p.Wo >> 1) + (wo >> 1)
                               : ((size_t)(n * p.To + t) * p.Ho + ho) * p.Wo + wo;
      }
      const int nbase = tc.nt * BN;
      const int ncols = min(BN, Cout - nbase);     // live output columns of this tile
      if (threadIdx.x == 96) TRACE(tile / gridDim.x, 4);

      mbar_wait(&tmem_full[as], aphase);
      if (threadIdx.x == 96) TRACE(tile / gridDim.x, 5);
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + as * BN + ((uint32_t)(lg * 32) << 16) + (uint32_t)(colw * part);
      uint32_t r[16];
      if (out_f32) tmem_ld_32x32b_x8_lo(taddr, r); else tmem_ld_32x32b_x16(taddr, r);
#pragma unroll 1
      for (int cc = 0; cc < ncols; cc += CW) {
        const int c0 = cc + colw * part;           // first column (inside the tile) this warp handles
        const int cbase = nbase + c0;
        const bool more = cc + CW < ncols;
        // AffineChannel scale / bias of this warp's columns: uniform 16-byte loads (L1 hits after first touch)
        float sc[16], bi[16];
        if (cbase + colw <= Cout) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (q < (colw >> 2)) {
              const float4 s4 = g_scale ? __ldg(reinterpret_cast<const float4*>(g_scale + cbase) + q) : make_float4(1.f, 1.f, 1.f, 1.f);
              const float4 b4 = g_bias ? __ldg(reinterpret_cast<const float4*>(g_bias + cbase) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
              sc[4 * q] = s4.x; sc[4 * q + 1] = s4.y; sc[4 * q + 2] = s4.z; sc[4 * q + 3] = s4.w;
              bi[4 * q] = b4.x; bi[4 * q + 1] = b4.y; bi[4 * q + 2] = b4.z; bi[4 * q + 3] = b4.w;
            }
          }
        } else {                                   // ragged channel tail
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const bool in = j < colw && cbase + j < Cout;
            sc[j] = (in && g_scale) ? __ldg(g_scale + cbase + j) : 1.f;
            bi[j] = (in && g_bias) ? __ldg(g_bias + cbase + j) : 0.f;
          }
        }
        float v[16];
        if (out_f32) {
          // ---- fp32 output: this warp owns 8 columns = 32 bytes
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = fmaf(__uint_as_float(r[j]), sc[j], bi[j]);
          if (more) {
            tmem_ld_32x32b_x8_lo(taddr + cc + CW, r);
          } else {                                 // accumulator fully read: release it to the MMA warp
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[as]);
          }
          if (res_mode != 0 && valid) {
            const float* rp = reinterpret_cast<const float*>(p.residual) + rpos * p.res_ld + cbase;
            if (cbase + 8 <= Cout) {
#pragma unroll
              for (int j = 0; j < 8; j += 4) {
                const float4 q = __ldg(reinterpret_cast<const float4*>(rp + j));
                v[j] += q.x; v[j + 1] += q.y; v[j + 2] += q.z; v[j + 3] += q.w;
                if (split_out) {                                     // residual = hi + lo
                  const float4 ql = __ldg(reinterpret_cast<const float4*>(rp + p.res_lo_off + j));
                  v[j] += ql.x; v[j + 1] += ql.y; v[j + 2] += ql.z; v[j + 3] += ql.w;
                }
              }
            } else {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                if (cbase + j < Cout) v[j] += __ldg(rp + j) + (split_out ? __ldg(rp + p.res_lo_off + j) : 0.f);
            }
          }
          if (relu) {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaxf(v[j], 0.f);
          }
        } else {
          // ---- bf16 output: this warp owns 16 columns = 32 bytes
          // residual rows first: the global loads overlap the TMEM wait
          uint4 resq[2];
          const bool res_on = res_ldg && valid;
          const bool res_vec = res_on && (cbase + 16 <= Cout);
          const __nv_bfloat16* rp = reinterpret_cast<const __nv_bfloat16*>(p.residual) + rpos * p.res_ld + cbase;
          if (res_vec) {
            resq[0] = __ldg(reinterpret_cast<const uint4*>(rp));
            resq[1] = __ldg(reinterpret_cast<const uint4*>(rp + 8));
          }
          // the producer warp prefetched this chunk's residual rows (zero-filled outside the tensor) into the swizzled ring
          if (res_tma) mbar_wait(&r_full[rslot], rphase);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaf(__uint_as_float(r[j]), sc[j], bi[j]);
          if (more) {
            tmem_ld_32x32b_x16(taddr + cc + CW, r);
          } else {                                 // accumulator fully read: release it to the MMA warp
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[as]);
          }
          auto add16 = [&](const uint4& a, const uint4& b) {          // 16 bf16 residual values onto v
            const uint32_t w8[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              v[2 * e] += __uint_as_float(w8[e] << 16);
              v[2 * e + 1] += __uint_as_float(w8[e] & 0xffff0000u);
            }
          };
          if (res_tma) {
            // read this thread's 32 bytes (hi, then the lo chunk in the slot's second buffer), then hand the slot back
            const uint32_t src = rbuf_u32 + (uint32_t)rslot * rslot_bytes + rrow_smem;
            add16(lds_u4(src + rq0), lds_u4(src + rq1));
            if (SPLIT) add16(lds_u4(src + Cfg::C_BYTES + rq0), lds_u4(src + Cfg::C_BYTES + rq1));
            __syncwarp();
            if (lane == 0) mbar_arrive(&r_empty[rslot]);
            if (++rslot == p.nrbuf) { rslot = 0; rphase ^= 1; }
          } else if (res_vec) {
            add16(resq[0], resq[1]);
            if (SPLIT)                                                // residual = hi + lo (bf16 pairs)
              add16(__ldg(reinterpret_cast<const uint4*>(rp + p.res_lo_off)), __ldg(reinterpret_cast<const uint4*>(rp + p.res_lo_off + 8)));
          } else if (res_on) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (cbase + j < Cout) v[j] += __bfloat162float(rp[j]) + (SPLIT ? __bfloat162float(rp[p.res_lo_off + j]) : 0.f);
          }
        }

        // staging slot: the TMA store that used it last must have read it out (c_free)
        mbar_wait(&c_free[slot], sphase ^ 1);
        if (threadIdx.x == 96) TRACE(tile / gridDim.x, 6);
        const uint32_t dst = cbuf_u32 + (uint32_t)slot * slot_bytes + row_smem;
        if (out_f32) {
          if (split_out) {
            float lo[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) { const float hi = round_to_tf32(v[j]); lo[j] = round_to_tf32(v[j] - hi); v[j] = hi; }
            const uint32_t dst_lo = dst + Cfg::C_BYTES;               // the lo chunk uses the slot's second buffer
            sts_f4(dst_lo + q0, lo[0], lo[1], lo[2], lo[3]);
            sts_f4(dst_lo + q1, lo[4], lo[5], lo[6], lo[7]);
          } else if (p.round_tf32) {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = round_to_tf32(v[j]);
          }
          sts_f4(dst + q0, v[0], v[1], v[2], v[3]);
          sts_f4(dst + q1, v[4], v[5], v[6], v[7]);
        } else {
          uint32_t h[8];
          if (split_out) {
            // bf16 pair storage: hi = bf16(v), lo = bf16(v - hi) (v - hi is exact in fp32); hi + lo carries 16
            // mantissa bits, which three bf16 MMAs per k-block turn into an fp32-accurate product
            uint32_t l[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float a = v[2 * j], b = v[2 * j + 1];
              if (relu) { a = fmaxf(a, 0.f); b = fmaxf(b, 0.f); }
              h[j] = pack_bf16x2(a, b);
              l[j] = pack_bf16x2(a - __uint_as_float(h[j] << 16), b - __uint_as_float(h[j] & 0xffff0000u));
            }
            const uint32_t dst_lo = dst + Cfg::C_BYTES;
            sts_b4(dst_lo + q0, l[0], l[1], l[2], l[3]);
            sts_b4(dst_lo + q1, l[4], l[5], l[6], l[7]);
          } else if (relu) {
#pragma unroll
            for (int j = 0; j < 8; ++j) h[j] = pack_bf16x2_relu(v[2 * j], v[2 * j + 1]);
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) h[j] = pack_bf16x2(v[2 * j], v[2 * j + 1]);
          }
          sts_b4(dst + q0, h[0], h[1], h[2], h[3]);
          sts_b4(dst + q1, h[4], h[5], h[6], h[7]);
        }
        // generic-proxy smem writes -> visible to the async proxy, then this warp's arrival on the slot
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&c_full[slot]);
        if (threadIdx.x == 96) TRACE(tile / gridDim.x, 7);
        if (++slot == nslots) { slot = 0; sphase ^= 1; }
      }
      if (threadIdx.x == 96) TRACE(tile / gridDim.x, 9);
      if (++as == 2) { as = 0; aphase ^= 1; }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
}

// ------------------------------------------------------------------ host side (encode_map: tc_common.cuh)
// M tile = TB images x TT frames x TH x TW output positions (<= 128 rows).  Small feature maps (14x14 RoI
// heads, 25x42 res5) would waste a quarter of every 128-row MMA with purely spatial tiles; stacking frames /
// images fills the rows.  Among the shapes within 4 % of the best useful-row fraction a purely spatial tile
// wins (the fullest, then the widest); otherwise the widest stacked tile (longest runs per TMA box).
struct TileShape { int th, tw, tt, tb; };
static TileShape pick_tile(int Ho, int Wo, int To, int N, int max_w, int max_h, bool stack_t) {
  TileShape best = {8, 16, 1, 1};
  double best_eff = -1;
  long best_rank = -1;
  for (int pass = 0; pass < 2; ++pass)
    for (int tw = 1; tw <= 128 && tw <= max_w && tw <= Wo; ++tw)
      for (int th = 1; th * tw <= 128 && th <= max_h && th <= Ho; ++th) {
        const int rem = 128 / (tw * th);
        for (int tt = 1; tt <= rem && tt <= To && (tt == 1 || stack_t); ++tt)
          for (int tb = 1; tb * tt <= rem && tb <= N; ++tb) {
            const double tiles = (double)cdiv(Wo, tw) * cdiv(Ho, th) * cdiv(To, tt) * cdiv(N, tb);
            const double eff = (double)Ho * Wo * To * N / (tiles * 128.0);
            if (pass == 0) { if (eff > best_eff) best_eff = eff; continue; }
            if (eff < best_eff - 0.04) continue;
            const bool plain = tt == 1 && tb == 1;
            const long e = (long)(eff * 1e6);
            const long rank = plain ? (1L << 40) + e * 1000L + tw : (long)tw * 10000000L + e;
            if (rank > best_rank) { best_rank = rank; best = {th, tw, tt, tb}; }
          }
      }
  return best;
}

// Output map: dims (Cout, Wo, Ho, To, N) of the NDHWC result, box = one staged chunk (128 B of channels x one M tile).
static int encode_out_map(CUtensorMap* m, void* y, int out_f32, int Cout, int Wo, int Ho, int To, int N, int out_ld,
                          const TileShape& ts, bool time_major = false) {
  const uint64_t oesz = out_f32 ? 4 : 2;
  uint64_t d[5] = {(uint64_t)Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)To, (uint64_t)N};
  const uint64_t frame = (uint64_t)out_ld * oesz * Wo * Ho;
  uint64_t st[4] = {(uint64_t)out_ld * oesz, (uint64_t)out_ld * oesz * Wo, time_major ? frame * N : frame,
                    time_major ? frame : frame * To};
  uint32_t b[5] = {(uint32_t)(128 / oesz), (uint32_t)ts.tw, (uint32_t)ts.th, (uint32_t)ts.tt, (uint32_t)ts.tb};
  uint32_t e[5] = {1, 1, 1, 1, 1};
  return encode_map(m, out_f32 != 0 ? 1 : 0, 5, y, d, st, b, e);
}

template <int BN, bool TF32, bool SPLIT>
static int launch_conv1(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const CUtensorMap& tmR,
                       const ConvKernelParams& p, int grid, cudaStream_t stream) {
  using Cfg = ConvCfg<BN>;
  static DynSmemGrant grant;
  DT_CHECK_CUDA(grant_dyn_smem(conv_tc_kernel<BN, TF32, SPLIT>, Cfg::BUDGET, &grant));
  ConvKernelParams q = p;
  const int kiters = p.kT * p.kH * p.kW * p.kchunks * p.nsub;
  DT_CHECK_ARG(kiters <= 2048, "conv: %d k-blocks per tile exceed the schedule table", kiters);
  Cfg::split(kiters, p.nrbuf > 0, p.split_out != 0, p.out_f32 != 0, &q.nstages, &q.ks, &q.ncbuf, &q.nrbuf);
  q.ktab = (kiters + 2) & ~1;
  const int smem = Cfg::smem_bytes(kiters, q.nstages, q.ks, q.ncbuf, q.nrbuf, p.split_out != 0);
  DT_CHECK_ARG(q.nstages >= 2 && smem <= Cfg::BUDGET, "conv: smem split failed (%d stages, %d B)", q.nstages, smem);
  // DT_PDL=1 in the environment launches with programmatic stream serialization (the kernel waits on griddepcontrol
  // before its first global access).  Measured on B200 (profiles/r02_pdl_ab.md): no gain inside the captured step
  // (126.0 vs 126.3 clips/s bf16x3, 329.6 vs 330.4 bf16) — the replayed graph has no launch gaps left to hide — so plain
  // stream order stays the default.
  static const bool pdl = [] { const char* e = getenv("DT_PDL"); return e && e[0] == '1'; }();
  cudaLaunchConfig_t lc;
  memset(&lc, 0, sizeof(lc));
  lc.gridDim = dim3((unsigned)grid); lc.blockDim = dim3(CONV_THREADS); lc.dynamicSmemBytes = (size_t)smem; lc.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  lc.attrs = at; lc.numAttrs = pdl ? 1 : 0;
  DT_CHECK_CUDA(cudaLaunchKernelEx(&lc, conv_tc_kernel<BN, TF32, SPLIT>, tmA, tmB, tmC, tmR, q));
  return 0;
}

template <int BN, bool TF32>
static int launch_conv(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const CUtensorMap& tmR,
                       const ConvKernelParams& p, int grid, cudaStream_t stream) {
  return p.split_out ? launch_conv1<BN, TF32, true>(tmA, tmB, tmC, tmR, p, grid, stream)
                     : launch_conv1<BN, TF32, false>(tmA, tmB, tmC, tmR, p, grid, stream);
}

}  // namespace dt

#ifdef DT_CONV_TRACE
extern "C" int dt_conv_trace_write(const long long* in) { return cudaMemcpyToSymbol(dt::g_conv_trace, in, sizeof(long long) * 64 * 16) != cudaSuccess; }
extern "C" int dt_conv_trace_read(long long* out) { return cudaMemcpyFromSymbol(out, dt::g_conv_trace, sizeof(long long) * 64 * 16) != cudaSuccess; }
#endif

using namespace dt;

extern "C" int dt_conv3d(const dt_conv_desc* d, const void* x, const void* w, const float* scale, const float* bias,
                         const void* residual, void* y, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DT_CHECK_ARG(d != nullptr, "dt_conv3d: null descriptor");
  DT_CHECK_ARG(d->dtype == DT_DTYPE_BF16 || d->dtype == DT_DTYPE_TF32 || d->dtype == DT_DTYPE_F16, "dt_conv3d: dtype %d not in {BF16, TF32, F16}", d->dtype);
  const bool tf32 = d->dtype == DT_DTYPE_TF32;
  const bool f16 = d->dtype == DT_DTYPE_F16;          // fp16 x and w (11-bit operands, one MMA per product); outputs stay bf16 / fp32
  DT_CHECK_ARG(!f16 || (!(d->x3 & 1) && d->res_mode == 0), "dt_conv3d: DT_DTYPE_F16 inputs are plain rows and take no residual");
  const int in_dt = tf32 ? 1 : (f16 ? 2 : 0);
  const int esz = tf32 ? 4 : 2;
  const int BK = tf32 ? 32 : 64;
  DT_CHECK_ARG(d->N >= 1 && d->Ti >= 1 && d->Hi >= 1 && d->Wi >= 1 && d->Cin >= 1 && d->Cout >= 1,
               "dt_conv3d: bad input shape N=%d T=%d H=%d W=%d Cin=%d Cout=%d", d->N, d->Ti, d->Hi, d->Wi, d->Cin, d->Cout);
  DT_CHECK_ARG(d->kT >= 1 && d->kH >= 1 && d->kW >= 1 && d->sT >= 1 && d->sH >= 1 && d->sW >= 1 && d->pT >= 0 &&
                   d->pH >= 0 && d->pW >= 0, "dt_conv3d: bad filter geometry");
  const int To_full = (d->Ti + 2 * d->pT - d->kT) / d->sT + 1;
  DT_CHECK_ARG(d->out_t_first >= 0 && d->out_t_count >= 0 && d->out_t_first + d->out_t_count <= (To_full > 0 ? To_full : 0),
               "dt_conv3d: output frame range [%d, +%d) outside the %d output frames", d->out_t_first, d->out_t_count, To_full);
  DT_CHECK_ARG(d->out_t_count == 0 || d->res_mode == 0, "dt_conv3d: an output frame range cannot be combined with a residual");
  const int To = d->out_t_count > 0 ? d->out_t_count : To_full;
  const int Ho = (d->Hi + 2 * d->pH - d->kH) / d->sH + 1;
  const int Wo = (d->Wi + 2 * d->pW - d->kW) / d->sW + 1;
  DT_CHECK_ARG(To >= 1 && Ho >= 1 && Wo >= 1, "dt_conv3d: empty output (%d,%d,%d)", To, Ho, Wo);
  const int in_ld = d->in_ld > 0 ? d->in_ld : d->Cin;
  const int w_ld = d->w_ld > 0 ? d->w_ld : d->Cin;
  const int out_ld = d->out_ld > 0 ? d->out_ld : d->Cout;
  const int res_ld = d->res_ld > 0 ? d->res_ld : d->Cout;
  DT_CHECK_ARG((in_ld * esz) % 16 == 0 && (w_ld * esz) % 16 == 0,
               "dt_conv3d: channel strides must be multiples of 16 bytes (in_ld=%d, w_ld=%d, %d B/elem)", in_ld, w_ld, esz);
  DT_CHECK_ARG(in_ld >= d->Cin && w_ld >= d->Cin && out_ld >= d->Cout, "dt_conv3d: leading dims smaller than channels");
  DT_CHECK_ARG(x && w && y, "dt_conv3d: null tensor pointer");
  DT_CHECK_ARG(((uintptr_t)x % 16) == 0 && ((uintptr_t)w % 16) == 0 && ((uintptr_t)y % 16) == 0,
               "dt_conv3d: tensors must be 16-byte aligned");
  DT_CHECK_ARG(d->res_mode >= 0 && d->res_mode <= 2 && (d->res_mode == 0 || residual), "dt_conv3d: bad residual mode/pointer");
  DT_CHECK_ARG(d->res_mode != 2 || (Ho % 2 == 0 && Wo % 2 == 0), "dt_conv3d: upsample-add needs even output size, got %dx%d", Ho, Wo);
  const int out_f32 = d->out_f32;
  const int oesz = out_f32 ? 4 : 2;
  // vector stores need 16-byte aligned rows
  DT_CHECK_ARG((out_ld * oesz) % 16 == 0 && (d->res_mode == 0 || (res_ld * oesz) % 16 == 0),
               "dt_conv3d: out_ld/res_ld rows must be 16-byte multiples");

  // stacking frames inside one TMA box needs unit temporal stride (pointwise convs fold strides into the map)
  const bool pointwise = d->kT == 1 && d->kH == 1 && d->kW == 1 && d->pT == 0 && d->pH == 0 && d->pW == 0;
  const TileShape ts = pick_tile(Ho, Wo, To, d->N, pointwise ? 256 : 256 / d->sW, pointwise ? 256 : 256 / d->sH,
                                 pointwise || d->sT == 1);
  const int TH = ts.th, TW = ts.tw;
  ConvKernelParams p;
  memset(&p, 0, sizeof(p));
  p.N = d->N; p.To = To; p.Ho = Ho; p.Wo = Wo; p.Cout = d->Cout;
  p.kT = d->kT; p.kH = d->kH; p.kW = d->kW; p.pT = d->pT; p.pH = d->pH; p.pW = d->pW;
  p.sT = d->sT; p.sH = d->sH; p.sW = d->sW;
  p.kchunks = cdiv(d->Cin, BK);
  p.TH = TH; p.TW = TW; p.TT = ts.tt; p.TB = ts.tb;
  p.tiles_h = cdiv(Ho, TH); p.tiles_w = cdiv(Wo, TW); p.tiles_t = cdiv(To, ts.tt); p.tiles_b = cdiv(d->N, ts.tb);
  p.a_bytes = (uint32_t)(TH * TW * ts.tt * ts.tb) * 128u;
  p.scale = scale; p.bias = bias; p.residual = residual; p.res_mode = d->res_mode; p.res_ld = res_ld;
  p.relu = d->relu; p.out_f32 = out_f32; p.round_tf32 = d->out_round_tf32;
  // 3xTF32 split operands / outputs
  p.split_in = (d->x3 & 1) ? 1 : 0;
  p.split_out = (d->x3 & 2) ? 1 : 0;
  p.nsub = p.split_in ? 3 : 1;
  p.ab_format = f16 ? 0 : 1;
  DT_CHECK_ARG(!p.split_in || d->Cin % BK == 0, "dt_conv3d: x3 inputs need Cin %% %d == 0 (Cin=%d)", BK, d->Cin);
  DT_CHECK_ARG(!p.split_out || ((tf32 ? out_f32 : !out_f32) && d->Cout % (out_f32 ? 32 : 64) == 0),
               "dt_conv3d: x3 outputs are fp32 pairs (TF32) / bf16 pairs (BF16) with Cout %% %d == 0 (Cout=%d)", out_f32 ? 32 : 64, d->Cout);
  p.a_lo_off = d->in_lo_off > 0 ? d->in_lo_off : in_ld / 2;
  p.b_lo_off = w_ld / 2;
  p.out_lo_off = d->out_lo_off > 0 ? d->out_lo_off : out_ld / 2;
  p.res_lo_off = d->res_lo_off > 0 ? d->res_lo_off : res_ld / 2;
  DT_CHECK_ARG(!p.split_in || (p.a_lo_off + d->Cin <= in_ld && p.b_lo_off >= d->Cin), "dt_conv3d: x3 lo halves do not fit the rows");
  DT_CHECK_ARG(!p.split_out || p.out_lo_off + d->Cout <= out_ld, "dt_conv3d: x3 output lo half does not fit the row");

  int BN = d->Cout >= 256 ? 256 : (d->Cout > 64 ? 128 : (d->Cout > 32 ? 64 : 32));
  if (d->Cout > 128 && d->Cout < 256) BN = 128;
  // bf16 same-shape residual: its chunks are prefetched by TMA into a shared-memory ring (coalesced 128-byte
  // rows instead of one 32-byte global load per thread).  The ring needs room, so these layers use 128-wide
  // column tiles (they are the K-light 1x1 expansions of the bottlenecks: HBM-bound, not MMA-bound).
  // The FPN top-down add (res_mode 2) goes the same way when the tile is even-sized (tile origins are then even
  // too): the (TH/2 x TW/2) box of the coarser map is loaded and each row serves its four children.
  const bool res_even = (TH % 2 == 0) && (TW % 2 == 0);
  const bool res_tma = (d->res_mode == 1 || (d->res_mode == 2 && res_even)) && !out_f32 && !tf32 &&
                       ((uintptr_t)residual % 16) == 0;
  if (res_tma && BN > 128) BN = 128;
  p.t_first = d->out_t_count > 0 ? d->out_t_first : 0;
  p.Ti = d->Ti; p.Hi = d->Hi;
  // DT_CONV_TAP_SKIP=0 in the environment issues every tap of every tile (the same results, for A/B timing); read on
  // each call, unlike DT_PDL, so that one process can run a conv both ways
  {
    const char* e = getenv("DT_CONV_TAP_SKIP");
    p.tap_skip = (e && e[0] == '0') ? 0 : 1;
  }
  p.nrbuf = res_tma ? 1 : 0;                         // ring depth is chosen with the smem split at launch
  p.res_up = (res_tma && d->res_mode == 2) ? 1 : 0;
  p.tiles_n = cdiv(d->Cout, BN);
  p.fd_n = make_fastdiv(p.tiles_n); p.fd_w = make_fastdiv(p.tiles_w); p.fd_h = make_fastdiv(p.tiles_h); p.fd_t = make_fastdiv(p.tiles_t);
  const long long total = (long long)p.tiles_b * p.tiles_t * p.tiles_h * p.tiles_w * p.tiles_n;
  DT_CHECK_ARG(total < (1ll << 31), "dt_conv3d: too many tiles");
  p.total_tiles = (int)total;

  // ---- tensor maps -------------------------------------------------------------
  // A: dims (C, W, H, T, N) of the NDHWC input.  Pointwise strided convs (1x1x1, stride s, no
  // padding) fold the stride into the global strides so no element-stride traversal is needed;
  // other strided convs use TMA element strides (box covers s*TW input columns, every s-th kept).
  CUtensorMap tmA, tmB;
  uint64_t dims[5], strides[4]; uint32_t box[5], estr[5] = {1, 1, 1, 1, 1};
  const uint64_t sC = (uint64_t)in_ld * esz, sW = sC * d->Wi, sH = sW * d->Hi, sT = sH * d->Ti;
  const uint64_t cdim = p.split_in ? (uint64_t)in_ld : (uint64_t)d->Cin;
  if (pointwise) {
    dims[0] = cdim; dims[1] = Wo; dims[2] = Ho; dims[3] = To_full; dims[4] = d->N;
    strides[0] = sC * d->sW; strides[1] = sW * d->sH; strides[2] = sH * d->sT; strides[3] = sT;
    box[0] = BK; box[1] = TW; box[2] = TH; box[3] = ts.tt; box[4] = ts.tb;
    p.sT = p.sH = p.sW = 1;
  } else {
    dims[0] = cdim; dims[1] = d->Wi; dims[2] = d->Hi; dims[3] = d->Ti; dims[4] = d->N;
    strides[0] = sC; strides[1] = sW; strides[2] = sH; strides[3] = sT;
    box[0] = BK; box[1] = (uint32_t)TW * d->sW; box[2] = (uint32_t)TH * d->sH; box[3] = ts.tt; box[4] = ts.tb;
    estr[1] = d->sW; estr[2] = d->sH;
    DT_CHECK_ARG(box[1] <= 256 && box[2] <= 256, "dt_conv3d: strided tile too large for a TMA box");
  }
  if (encode_map(&tmA, in_dt, 5, x, dims, strides, box, estr)) return 1;
  {
    const int taps = d->kT * d->kH * d->kW;
    uint64_t wd[3] = {p.split_in ? (uint64_t)w_ld : (uint64_t)d->Cin, (uint64_t)d->Cout, (uint64_t)taps};
    uint64_t ws[2] = {(uint64_t)w_ld * esz, (uint64_t)w_ld * esz * d->Cout};
    uint32_t wb[3] = {(uint32_t)BK, (uint32_t)BN, 1};
    uint32_t we[3] = {1, 1, 1};
    if (encode_map(&tmB, in_dt, 3, w, wd, ws, wb, we)) return 1;
  }
  CUtensorMap tmC, tmR;
  if (encode_out_map(&tmC, y, out_f32, p.split_out ? out_ld : d->Cout, Wo, Ho, To, d->N, out_ld, ts, d->out_time_major != 0)) return 1;
  if (res_tma && p.res_up) {
    const TileShape half = {ts.th / 2, ts.tw / 2, ts.tt, ts.tb};
    if (encode_out_map(&tmR, const_cast<void*>(residual), 0, p.split_out ? res_ld : d->Cout, Wo / 2, Ho / 2, To, d->N, res_ld, half)) return 1;
  } else if (res_tma) {
    if (encode_out_map(&tmR, const_cast<void*>(residual), 0, p.split_out ? res_ld : d->Cout, Wo, Ho, To, d->N, res_ld, ts)) return 1;
  } else {
    tmR = tmC;
  }
  int dev = 0, sms = 148;
  DT_CHECK_CUDA(cudaGetDevice(&dev));
  DT_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int grid = p.total_tiles < sms ? p.total_tiles : sms;
#define DT_LAUNCH(BNv)                                                                      \
  return tf32 ? launch_conv<BNv, true>(tmA, tmB, tmC, tmR, p, grid, stream) : launch_conv<BNv, false>(tmA, tmB, tmC, tmR, p, grid, stream)
  switch (BN) {
    case 256: DT_LAUNCH(256);
    case 128: DT_LAUNCH(128);
    case 64: DT_LAUNCH(64);
    default: DT_LAUNCH(32);
  }
#undef DT_LAUNCH
}


// Planning query: MIRRORS the choices of dt_conv3d above (tile picker, column tile, residual ring, smem split) without
// touching the device, so that the host logic is testable without a GPU (tests/test_conv_plan.py).
template <int BN>
static void plan_split(int kiters, bool res_tma, bool split_out, bool out_f32, dt_conv_plan_t* o) {
  using Cfg = ConvCfg<BN>;
  Cfg::split(kiters, res_tma, split_out, out_f32, &o->stages, &o->ks, &o->ncbuf, &o->nrbuf);
  o->smem_bytes = Cfg::smem_bytes(kiters, o->stages, o->ks, o->ncbuf, o->nrbuf, split_out);
}

extern "C" int dt_conv_plan(const dt_conv_desc* d, int residual_aligned, dt_conv_plan_t* o) {
  DT_CHECK_ARG(d != nullptr && o != nullptr, "dt_conv_plan: null pointer");
  DT_CHECK_ARG(d->dtype == DT_DTYPE_BF16 || d->dtype == DT_DTYPE_TF32, "dt_conv_plan: dtype %d not in {BF16, TF32}", d->dtype);
  DT_CHECK_ARG(d->N >= 1 && d->Ti >= 1 && d->Hi >= 1 && d->Wi >= 1 && d->Cin >= 1 && d->Cout >= 1 && d->kT >= 1 && d->kH >= 1 &&
                   d->kW >= 1 && d->sT >= 1 && d->sH >= 1 && d->sW >= 1 && d->pT >= 0 && d->pH >= 0 && d->pW >= 0,
               "dt_conv_plan: bad shape");
  const bool tf32 = d->dtype == DT_DTYPE_TF32;
  const int BK = tf32 ? 32 : 64;
  const int To_full = (d->Ti + 2 * d->pT - d->kT) / d->sT + 1;
  const int To = d->out_t_count > 0 ? d->out_t_count : To_full;
  const int Ho = (d->Hi + 2 * d->pH - d->kH) / d->sH + 1;
  const int Wo = (d->Wi + 2 * d->pW - d->kW) / d->sW + 1;
  DT_CHECK_ARG(To >= 1 && Ho >= 1 && Wo >= 1, "dt_conv_plan: empty output (%d,%d,%d)", To, Ho, Wo);
  const bool pointwise = d->kT == 1 && d->kH == 1 && d->kW == 1 && d->pT == 0 && d->pH == 0 && d->pW == 0;
  const TileShape ts = pick_tile(Ho, Wo, To, d->N, pointwise ? 256 : 256 / d->sW, pointwise ? 256 : 256 / d->sH,
                                 pointwise || d->sT == 1);
  int BN = d->Cout >= 256 ? 256 : (d->Cout > 64 ? 128 : (d->Cout > 32 ? 64 : 32));
  if (d->Cout > 128 && d->Cout < 256) BN = 128;
  const bool res_even = (ts.th % 2 == 0) && (ts.tw % 2 == 0);
  const bool res_tma = (d->res_mode == 1 || (d->res_mode == 2 && res_even)) && !d->out_f32 && !tf32 && residual_aligned;
  if (res_tma && BN > 128) BN = 128;
  const bool split_in = (d->x3 & 1) != 0, split_out = (d->x3 & 2) != 0;
  memset(o, 0, sizeof(*o));
  o->BN = BN; o->TH = ts.th; o->TW = ts.tw; o->TT = ts.tt; o->TB = ts.tb;
  o->kiters = d->kT * d->kH * d->kW * cdiv(d->Cin, BK) * (split_in ? 3 : 1);
  const long long mt = (long long)cdiv(Wo, ts.tw) * cdiv(Ho, ts.th) * cdiv(To, ts.tt) * cdiv(d->N, ts.tb);
  o->tiles = (int)(mt * cdiv(d->Cout, BN));
  o->useful_rows = (double)Ho * Wo * To * d->N / ((double)mt * 128.0);
  switch (BN) {
    case 256: plan_split<256>(o->kiters, res_tma, split_out, d->out_f32 != 0, o); break;
    case 128: plan_split<128>(o->kiters, res_tma, split_out, d->out_f32 != 0, o); break;
    case 64: plan_split<64>(o->kiters, res_tma, split_out, d->out_f32 != 0, o); break;
    default: plan_split<32>(o->kiters, res_tma, split_out, d->out_f32 != 0, o); break;
  }
  return 0;
}


// conv1 of the ResNet bodies: 7x7 stride 2 pad 3 on a 3-channel image (lib/modeling/ResNet3D.py:258-261,
// ResNet.py).  With Cin = 3 a per-tap k-block would waste 61/64 of every MMA, so the taps of one filter
// ROW are packed into K instead: the image blob is channel-padded to Cp (8 bf16 / 4 fp32 = 16 bytes per
// pixel) and carries physical zero borders (3 rows top/bottom, 4 pixels left/right, written by
// dt_prep_clip), so the 7-pixel window of output column wo is ONE contiguous 112-byte run starting at
// padded pixel 2*wo + 1.  The A tensor map is an overlapping strided view
//   dim0 = 8 pixels x Cp (128 B, the 8th pixel meets zero weights), dim1 = wo (stride 2 pixels = 32 B),
//   dim2 = rows of one parity plane, dim3 = plane, dim4 = frames
// (the blob's padded rows are de-interleaved by parity, so the stride-2 row walk of filter row kh is a
// unit-stride box in plane kh & 1 starting at row ho + (kh >> 1); TMA element strides halve its throughput)
// and the conv is 7 k-blocks (one per filter row) of K = 128 bytes: 3*7/ (8*8) = 33 % useful MACs instead
// of 4.7 %.  w [7][Cout][8*Cp] (kw-major, channel-minor).  y [F, Hp/2, Wp/2, out_ld].
extern "C" int dt_conv1_7x7s2(const void* x_padded, int F, int Hp, int Wp, int Cp, const void* w, int Cout,
                              const float* scale, const float* bias, int relu, int dtype, int out_f32,
                              int out_round_tf32, int x3, void* y, int out_ld, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DT_CHECK_ARG(dtype == DT_DTYPE_BF16 || dtype == DT_DTYPE_TF32, "dt_conv1_7x7s2: bad dtype %d", dtype);
  const bool tf32 = dtype == DT_DTYPE_TF32;
  const int esz = tf32 ? 4 : 2;
  DT_CHECK_ARG(Cp * esz == 16, "dt_conv1_7x7s2: the blob must carry 16 bytes per pixel (Cp=%d, %d B/elem)", Cp, esz);
  DT_CHECK_ARG(F >= 1 && Hp >= 2 && Wp >= 2 && Hp % 2 == 0 && Wp % 2 == 0 && Cout >= 1 && Cout <= 64,
               "dt_conv1_7x7s2: bad shape F=%d Hp=%d Wp=%d Cout=%d", F, Hp, Wp, Cout);
  DT_CHECK_ARG(x_padded && w && y, "dt_conv1_7x7s2: null pointer");
  // x3 (bf16 only): the blob pixel is [hi(3) | lo(3) | 0 0] (dt_prep_clip out mode 3), w holds 14 blocks
  // [2*kh]: [W_hi | W_hi] per pixel, [2*kh + 1]: [W_lo | 0], and y rows are [hi(Cout) | lo(Cout)] bf16 pairs
  DT_CHECK_ARG(!x3 || (!tf32 && !out_f32 && Cout == 64), "dt_conv1_7x7s2: x3 needs DT_DTYPE_BF16, bf16 pair output and Cout == 64");
  const int oesz = out_f32 ? 4 : 2;
  if (out_ld <= 0) out_ld = x3 ? 2 * Cout : Cout;
  DT_CHECK_ARG((out_ld * oesz) % 16 == 0 && out_ld >= (x3 ? 2 * Cout : Cout), "dt_conv1_7x7s2: bad out_ld %d", out_ld);
  const int Ho = Hp / 2, Wo = Wp / 2;
  const int BKe = 128 / esz;                       // elements per k-block
  const TileShape ts = pick_tile(Ho, Wo, 1, 1, 256, 128, false);      // spatial tiles only
  const int TH = ts.th, TW = ts.tw;
  ConvKernelParams p;
  memset(&p, 0, sizeof(p));
  p.N = F; p.To = 1; p.Ho = Ho; p.Wo = Wo; p.Cout = Cout;
  p.kT = 1; p.kH = 7; p.kW = 1; p.sT = 1; p.sH = 1; p.sW = 1; p.pT = 0; p.pH = 0; p.pW = 0;
  p.row_planes = 1;
  p.kchunks = 1;
  p.ab_format = 1;
  p.nsub = x3 ? 2 : 1;
  p.split_out = x3 ? 1 : 0;
  p.out_lo_off = out_ld / 2;
  p.TH = TH; p.TW = TW; p.TT = 1; p.TB = 1; p.tiles_h = cdiv(Ho, TH); p.tiles_w = cdiv(Wo, TW); p.tiles_t = 1; p.tiles_b = F;
  p.tiles_n = 1;
  p.a_bytes = (uint32_t)TH * TW * 128u;
  p.scale = scale; p.bias = bias; p.relu = relu; p.out_f32 = out_f32;
  p.round_tf32 = out_round_tf32;
  p.fd_n = make_fastdiv(1); p.fd_w = make_fastdiv(p.tiles_w); p.fd_h = make_fastdiv(p.tiles_h); p.fd_t = make_fastdiv(1);
  const long long total = (long long)F * p.tiles_h * p.tiles_w;
  DT_CHECK_ARG(total < (1ll << 31), "dt_conv1_7x7s2: too many tiles");
  p.total_tiles = (int)total;
  // padded rows are stored de-interleaved (dt_prep_clip row_planes): filter row kh of output row ho reads
  // padded row 2*ho + kh = plane (kh & 1), plane row ho + (kh >> 1) -> unit-stride boxes, the plane is dim 3
  const uint64_t pix = 16, row = (uint64_t)(Wp + 8) * pix, plane = row * ((Hp + 6) / 2), frame = 2 * plane;
  CUtensorMap tmA, tmB;
  {
    uint64_t dims[5] = {(uint64_t)BKe, (uint64_t)Wo, (uint64_t)((Hp + 6) / 2), 2, (uint64_t)F};
    uint64_t strides[4] = {2 * pix, row, plane, frame};
    uint32_t box[5] = {(uint32_t)BKe, (uint32_t)TW, (uint32_t)TH, 1, 1};
    uint32_t estr[5] = {1, 1, 1, 1, 1};
    if (encode_map(&tmA, tf32 ? 1 : 0, 5, (const char*)x_padded + pix, dims, strides, box, estr)) return 1;
  }
  {
    uint64_t wd[3] = {(uint64_t)BKe, (uint64_t)Cout, (uint64_t)(x3 ? 14 : 7)};
    uint64_t ws[2] = {128, (uint64_t)128 * Cout};
    uint32_t wb[3] = {(uint32_t)BKe, 64, 1};
    uint32_t we[3] = {1, 1, 1};
    if (encode_map(&tmB, tf32 ? 1 : 0, 3, w, wd, ws, wb, we)) return 1;
  }
  CUtensorMap tmC;
  if (encode_out_map(&tmC, y, out_f32, x3 ? out_ld : Cout, Wo, Ho, 1, F, out_ld, ts)) return 1;
  int dev = 0, sms = 148;
  DT_CHECK_CUDA(cudaGetDevice(&dev));
  DT_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int grid = p.total_tiles < sms ? p.total_tiles : sms;
  return tf32 ? launch_conv<64, true>(tmA, tmB, tmC, tmC, p, grid, stream) : launch_conv<64, false>(tmA, tmB, tmC, tmC, p, grid, stream);
}
