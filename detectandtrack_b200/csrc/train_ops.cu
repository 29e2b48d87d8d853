// Training-step kernels of the data-parallel path (BASELINE.json configs[4]; the reference builds these with
// model.AddGradientOperators + add_parameter_update_ops, lib/modeling/model_builder.py:908-985):
//
//   dt_wgrad            Conv / ConvNd filter gradient on the tcgen05 tensor cores:
//                         dW[tap][co][ci] = sum over positions of gz[pos, co] * x[pos @ tap, ci]
//                       a GEMM whose K axis is the position axis.  Both operands are read from CHANNEL-MAJOR PLANES
//                       ([N, T, C, plane], plane = the zero-bordered (H+2p) x (W+2p) map flattened), so a position run is
//                       contiguous (a K-major operand for tcgen05, staged by TMA with the 128B swizzle) and a filter ROW
//                       offset (kh) is a constant offset along the flattened plane (rows are padded to a multiple of 8
//                       positions, so the offset keeps TMA's 16-byte alignment of the innermost coordinate; the physical
//                       zero border supplies the padding, TMA's out-of-bounds zero fill the plane ends and the temporal
//                       padding).  A +-1 COLUMN offset (kw) would break that alignment, so the input planes are stored kW
//                       times, copy kw pre-shifted by kw - pW positions (dt_to_planes wshift).  Split-K over positions
//                       across CTAs, fp32 partial sums reduced into dW with vector red.global.
//   dt_to_planes        NDHWC activation / gradient -> those planes (tiled transpose through shared memory, optional
//                       spatial subsampling for the strided 1x1 convs).
//   dt_bwd_pointwise    the elementwise part of a block's backward: gz = (g1 + g2) * [y > 0] * scale[c]
//                       (Relu / Sum / AffineChannelNd gradients, lib/ops/affine_channel_nd_op.cu:73-92: dX = dY * scale;
//                       the affine parameters themselves are frozen in Detectron-style fine-tuning)
//   dt_upsample_add_bwd FPN top-down join backward (lib/modeling/FPN3D.py:186-222): the coarser level receives the 2x2 sum
//   dt_scatter_stride2  dgrad of a stride-2 pointwise conv: values land on the even positions of a zeroed map
//   dt_sgd_update       MomentumSGDUpdate with weight decay (model_builder.py:954-985) on fp32 master weights kept in the
//                       packed [tap][Cout][Cin] order, re-emitting the bf16 forward weights and the (flipped, transposed)
//                       bf16 dgrad weights in the same pass
#include "common.cuh"
#include "tc_common.cuh"
#include "../../include/dt_b200.h"
#include "../../include/dt_b200_train3d.h"
#include <cuda_bf16.h>
#include <stdlib.h>

namespace dt {

using namespace tc;

// ------------------------------------------------------------------------------------------------ wgrad
struct WgradParams {
  int Cout, Cin, taps;
  int kT, kH, kW, pT, pH, pW;
  int Wp;                 // row length of the padded plane (W + 2*pW rounded up to 8)
  int T, N;               // frames, images
  int kchunks;            // 64-position chunks per plane
  int tiles_m, tiles_n, ksplit;
  float* dW;              // [taps][Cout][Cin] fp32, accumulated into (caller zeroes)
};

constexpr int WG_THREADS = 192;       // warp 0 TMA producer, warp 1 TMEM + MMA issuer, warps 2-5 epilogue
constexpr int WG_STAGES = 4;

template <int BN>
__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_kernel(const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmX, const WgradParams p) {
  constexpr int A_BYTES = 128 * 128, B_BYTES = BN * 128, ST_BYTES = A_BYTES + B_BYTES;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + WG_STAGES * ST_BYTES);
  uint64_t* empty = full + WG_STAGES;
  uint64_t* acc_full = empty + WG_STAGES;
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(acc_full + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    prefetch_tmap(&tmG); prefetch_tmap(&tmX);
    for (int s = 0; s < WG_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<(BN < 32 ? 32 : BN)>(tmem_base_smem);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_base_smem;

  // work item: (tap, m tile, n tile, k split)
  int w = blockIdx.x;
  const int ks = w % p.ksplit; w /= p.ksplit;
  const int nt = w % p.tiles_n; w /= p.tiles_n;
  const int mt = w % p.tiles_m;
  const int tap = w / p.tiles_m;
  const int kw = tap % p.kW, kh = (tap / p.kW) % p.kH, kt = tap / (p.kW * p.kH);
  const int shift = (kh - p.pH) * p.Wp;          // filter-row offset along the flattened padded plane (multiple of 8: 16-byte
                                                 // aligned TMA coordinate); the column offset selects the pre-shifted copy kw
  const int dt_ = kt - p.pT;
  // k-blocks = (image, frame, chunk) triples; frames whose tap-shifted source frame is outside the clip contribute zero
  // (temporal zero padding) and are skipped by producer and issuer alike
  const long long total = (long long)p.N * p.T * p.kchunks;
  const long long k0 = total * ks / p.ksplit, k1 = total * (ks + 1) / p.ksplit;

  if (warp == 0) {
    int stage = 0; uint32_t phase = 0;
    long long r = k0 / p.kchunks;
    int chunk = (int)(k0 - r * p.kchunks);
    int t = (int)(r % p.T), n = (int)(r / p.T);
    for (long long kb = k0; kb < k1; ++kb) {
      const int ts = t + dt_;
      if (ts >= 0 && ts < p.T) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (elect_one()) {
          const uint32_t dst = smem_u32(smem) + stage * ST_BYTES;
          const uint32_t bar = smem_u32(&full[stage]);
          mbar_expect_tx_u(bar, (uint32_t)ST_BYTES);
          // A: gz planes, box (64 positions, 128 channels); B: x planes at the tap-shifted position / frame
          asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                       ::"r"(dst), "l"(reinterpret_cast<uint64_t>(&tmG)), "r"(bar), "r"(chunk * 64), "r"(mt * 128), "r"(t), "r"(n) : "memory");
          asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
                       ::"r"(dst + A_BYTES), "l"(reinterpret_cast<uint64_t>(&tmX)), "r"(bar), "r"(chunk * 64 + shift), "r"(nt * BN), "r"(ts), "r"(n), "r"(kw) : "memory");
        }
        if (++stage == WG_STAGES) { stage = 0; phase ^= 1; }
      }
      if (++chunk == p.kchunks) { chunk = 0; if (++t == p.T) { t = 0; ++n; } }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(128, BN, 1);
    int stage = 0; uint32_t phase = 0;
    long long r = k0 / p.kchunks;
    int chunk = (int)(k0 - r * p.kchunks);
    int t = (int)(r % p.T);
    uint32_t first = 1;
    for (long long kb = k0; kb < k1; ++kb) {
      const int ts = t + dt_;
      if (ts >= 0 && ts < p.T) {
        mbar_wait(&full[stage], phase);
        tcgen05_fence_after();
        const uint32_t a_addr = smem_u32(smem) + stage * ST_BYTES;
        if (elect_one()) {
          const uint64_t adesc = make_sw128_kmajor_desc(a_addr);
          const uint64_t bdesc = make_sw128_kmajor_desc(a_addr + A_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma<false>(tmem_base, adesc + 2 * k, bdesc + 2 * k, idesc, (first && k == 0) ? 0u : 1u);
          umma_commit(&empty[stage]);
        }
        first = 0;
        if (++stage == WG_STAGES) { stage = 0; phase ^= 1; }
      }
      if (++chunk == p.kchunks) { chunk = 0; if (++t == p.T) t = 0; }
    }
    if (elect_one()) umma_commit(acc_full);          // fires when every MMA above has retired (immediately if none)
  } else {
    // epilogue warps 2..5: TMEM lane group (warp & 3), 32 rows each.  While the MMAs run these warps are idle, so they
    // replay the k-block walk to learn whether this CTA accumulated anything at all (a range made only of temporally
    // padded frames leaves the accumulator unwritten).
    bool nothing = true;
    {
      long long r = k0 / p.kchunks;
      int chunk = (int)(k0 - r * p.kchunks);
      int t = (int)(r % p.T);
      for (long long kb = k0; kb < k1 && nothing; ) {
        const int ts = t + dt_;
        if (ts >= 0 && ts < p.T) nothing = false;
        const long long step = p.kchunks - chunk;           // jump to the next frame
        kb += step; chunk = 0; if (++t == p.T) t = 0;
      }
    }
    mbar_wait(acc_full, 0);
    tcgen05_fence_after();
    const int lg = warp & 3;
    const int row = mt * 128 + lg * 32 + lane;
    if (!nothing) {
      float* out = p.dW + ((size_t)tap * p.Cout + row) * p.Cin + nt * BN;
      for (int c0 = 0; c0 < BN; c0 += 16) {
        uint32_t r[16];
        tmem_ld_32x32b_x16(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)c0, r);
        tmem_ld_wait();
        if (row < p.Cout) {
          const int col = nt * BN + c0;
          if (col + 16 <= p.Cin && (p.Cin & 3) == 0) {
#pragma unroll
            for (int q = 0; q < 4; ++q)
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(out + c0 + 4 * q), "f"(__uint_as_float(r[4 * q])),
                           "f"(__uint_as_float(r[4 * q + 1])), "f"(__uint_as_float(r[4 * q + 2])), "f"(__uint_as_float(r[4 * q + 3])) : "memory");
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (col + j < p.Cin) atomicAdd(out + c0 + j, __uint_as_float(r[j]));
          }
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<(BN < 32 ? 32 : BN)>(tmem_base);
}

template <int BN>
static int launch_wgrad(const CUtensorMap& tmG, const CUtensorMap& tmX, const WgradParams& p, cudaStream_t stream) {
  constexpr int smem = WG_STAGES * (128 * 128 + BN * 128) + 256;
  static DynSmemGrant grant;
  DT_CHECK_CUDA(grant_dyn_smem(wgrad_kernel<BN>, smem, &grant));
  const long long grid = (long long)p.taps * p.tiles_m * p.tiles_n * p.ksplit;
  DT_CHECK_ARG(grid < (1ll << 31), "dt_wgrad: grid too large");
  wgrad_kernel<BN><<<(unsigned)grid, WG_THREADS, smem, stream>>>(tmG, tmX, p);
  DT_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------------ wgrad, NDHWC operands
// The same GEMM read STRAIGHT from the NDHWC tensors (no channel-major copies): a TMA box (64 channels = 128 B, TW, TH, TT, TB)
// of 64 positions lands in shared memory as 64 rows of 128 bytes — positions down the rows, 64 channels along each swizzled
// row.  Read as an MN-MAJOR tcgen05 operand (instruction descriptor bits 15 / 16) that is exactly the canonical layout
// ((8,8,m),(8,k)):((1,8,LBO),(64,SBO)) with K = the position axis: 8 positions x 128 B per swizzle atom (SBO = 1024 B between
// 8-position groups) and LBO = 8 KB between 64-channel groups.  The filter tap is a coordinate shift of the input box (TMA
// zero fill = the conv's padding), exactly as in the forward kernel, so kw needs no pre-shifted copies.
struct WgradNParams {
  int Cout, Cin, taps;
  int kT, kH, kW, pT, pH, pW;
  int TW, TH, TT, TB;
  int nW, nH, nT, nN;       // position tiles per axis
  int T;                    // frames (temporal bounds of the tap shift when TT == 1)
  int tiles_m, tiles_n, ksplit;
  float* dW;
};

__device__ __forceinline__ uint64_t make_sw128_mnmajor_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);        // start address
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;   // LBO: stride between 64-element groups along M / N
  d |= (uint64_t)(1024 >> 4) << 32;                   // SBO: stride between 8-row groups along K
  d |= (uint64_t)1 << 46;                             // version
  d |= (uint64_t)2 << 61;                             // SWIZZLE_128B
  return d;
}

template <int BN>
__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_nhwc_kernel(const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmX, const WgradNParams p) {
  constexpr int GRP = 64 * 128;                                    // one (64 positions x 64 channels) box
  constexpr int A_BYTES = 2 * GRP, B_BYTES = (BN / 64) * GRP, ST_BYTES = A_BYTES + B_BYTES;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + WG_STAGES * ST_BYTES);
  uint64_t* empty = full + WG_STAGES;
  uint64_t* acc_full = empty + WG_STAGES;
  uint32_t* tmem_base_smem = reinterpret_cast<uint32_t*>(acc_full + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    prefetch_tmap(&tmG); prefetch_tmap(&tmX);
    for (int s = 0; s < WG_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<(BN < 32 ? 32 : BN)>(tmem_base_smem);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_base_smem;

  int w = blockIdx.x;
  const int ks = w % p.ksplit; w /= p.ksplit;
  const int nt = w % p.tiles_n; w /= p.tiles_n;
  const int mt = w % p.tiles_m;
  const int tap = w / p.tiles_m;
  const int kw = tap % p.kW, kh = (tap / p.kW) % p.kH, kt = tap / (p.kW * p.kH);
  const int dw = kw - p.pW, dh = kh - p.pH, dt_ = kt - p.pT;
  const long long total = (long long)p.nN * p.nT * p.nH * p.nW;
  const long long k0 = total * ks / p.ksplit, k1 = total * (ks + 1) / p.ksplit;
  // a k-block whose tap-shifted frames all lie outside the clip contributes zero: skipped by producer and issuer alike
  auto live = [&](int it) -> bool { const int t0 = it * p.TT + dt_; return t0 + p.TT > 0 && t0 < p.T; };
  auto decode = [&](long long kb, int& iw, int& ih, int& it, int& in) {
    iw = (int)(kb % p.nW); kb /= p.nW;
    ih = (int)(kb % p.nH); kb /= p.nH;
    it = (int)(kb % p.nT); in = (int)(kb / p.nT);
  };

  if (warp == 0) {
    int stage = 0; uint32_t phase = 0;
    int iw, ih, it, in;
    decode(k0, iw, ih, it, in);
    for (long long kb = k0; kb < k1; ++kb) {
      if (live(it)) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (elect_one()) {
          const uint32_t dst = smem_u32(smem) + stage * ST_BYTES;
          const uint32_t bar = smem_u32(&full[stage]);
          mbar_expect_tx_u(bar, (uint32_t)ST_BYTES);
          const int w0 = iw * p.TW, h0 = ih * p.TH, t0 = it * p.TT, n0 = in * p.TB;
#pragma unroll
          for (int g = 0; g < 2; ++g)
            asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
                         ::"r"(dst + g * GRP), "l"(reinterpret_cast<uint64_t>(&tmG)), "r"(bar), "r"(mt * 128 + g * 64), "r"(w0), "r"(h0), "r"(t0), "r"(n0) : "memory");
#pragma unroll
          for (int g = 0; g < BN / 64; ++g)
            asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
                         ::"r"(dst + A_BYTES + g * GRP), "l"(reinterpret_cast<uint64_t>(&tmX)), "r"(bar), "r"(nt * BN + g * 64), "r"(w0 + dw), "r"(h0 + dh),
                           "r"(t0 + dt_), "r"(n0) : "memory");
        }
        if (++stage == WG_STAGES) { stage = 0; phase ^= 1; }
      }
      if (++iw == p.nW) { iw = 0; if (++ih == p.nH) { ih = 0; if (++it == p.nT) { it = 0; ++in; } } }
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc(128, BN, 1) | (1u << 15) | (1u << 16);      // A and B MN-major
    int stage = 0; uint32_t phase = 0;
    int iw, ih, it, in;
    decode(k0, iw, ih, it, in);
    uint32_t first = 1;
    for (long long kb = k0; kb < k1; ++kb) {
      if (live(it)) {
        mbar_wait(&full[stage], phase);
        tcgen05_fence_after();
        const uint32_t a_addr = smem_u32(smem) + stage * ST_BYTES;
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k) {                                // 16 positions (2 swizzle atoms of 8 rows) per MMA
            const uint64_t adesc = make_sw128_mnmajor_desc(a_addr + k * 2048, GRP);
            const uint64_t bdesc = make_sw128_mnmajor_desc(a_addr + A_BYTES + k * 2048, GRP);
            umma<false>(tmem_base, adesc, bdesc, idesc, (first && k == 0) ? 0u : 1u);
          }
          umma_commit(&empty[stage]);
        }
        first = 0;
        if (++stage == WG_STAGES) { stage = 0; phase ^= 1; }
      }
      if (++iw == p.nW) { iw = 0; if (++ih == p.nH) { ih = 0; if (++it == p.nT) { it = 0; ++in; } } }
    }
    if (elect_one()) umma_commit(acc_full);
  } else {
    bool nothing = true;
    {
      int iw, ih, it, in;
      decode(k0, iw, ih, it, in);
      for (long long kb = k0; kb < k1 && nothing; ++kb) {
        if (live(it)) nothing = false;
        if (++iw == p.nW) { iw = 0; if (++ih == p.nH) { ih = 0; if (++it == p.nT) { it = 0; ++in; } } }
      }
    }
    mbar_wait(acc_full, 0);
    tcgen05_fence_after();
    const int lg = warp & 3;
    const int row = mt * 128 + lg * 32 + lane;
    if (!nothing) {
      float* out = p.dW + ((size_t)tap * p.Cout + row) * p.Cin + nt * BN;
      for (int c0 = 0; c0 < BN; c0 += 16) {
        uint32_t r[16];
        tmem_ld_32x32b_x16(tmem_base + ((uint32_t)(lg * 32) << 16) + (uint32_t)c0, r);
        tmem_ld_wait();
        if (row < p.Cout) {
          const int col = nt * BN + c0;
          if (col + 16 <= p.Cin && (p.Cin & 3) == 0) {
#pragma unroll
            for (int q = 0; q < 4; ++q)
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(out + c0 + 4 * q), "f"(__uint_as_float(r[4 * q])),
                           "f"(__uint_as_float(r[4 * q + 1])), "f"(__uint_as_float(r[4 * q + 2])), "f"(__uint_as_float(r[4 * q + 3])) : "memory");
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (col + j < p.Cin) atomicAdd(out + c0 + j, __uint_as_float(r[j]));
          }
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<(BN < 32 ? 32 : BN)>(tmem_base);
}

template <int BN>
static int launch_wgrad_nhwc(const CUtensorMap& tmG, const CUtensorMap& tmX, const WgradNParams& p, cudaStream_t stream) {
  constexpr int smem = WG_STAGES * (2 + BN / 64) * 64 * 128 + 256;
  static DynSmemGrant grant;
  DT_CHECK_CUDA(grant_dyn_smem(wgrad_nhwc_kernel<BN>, smem, &grant));
  const long long grid = (long long)p.taps * p.tiles_m * p.tiles_n * p.ksplit;
  DT_CHECK_ARG(grid < (1ll << 31), "dt_wgrad_nhwc: grid too large");
  wgrad_nhwc_kernel<BN><<<(unsigned)grid, WG_THREADS, smem, stream>>>(tmG, tmX, p);
  DT_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------------ planes
// x [N*T frames, H, W, ldx] (first C channels) -> planes [copies][N*T, C, Pld]: plane position ((h / sh) + pH) * Wp + (w / sw) + pW
// for h % sh == 0, w % sw == 0; border and row tail zero.  Copy j holds the plane shifted by wshift0 + j columns (column c of
// the copy = pixel column c + shift; the wgrad input operand: one copy per filter column).  Tile: 64 plane positions (+ the
// shift halo) x 64 channels staged ONCE in shared memory, every copy written from it.
constexpr int TP_HALO = 3;
__global__ void __launch_bounds__(256)
to_planes_kernel(const __nv_bfloat16* __restrict__ x, int F, int H, int W, int C, int ldx, int sh, int sw, int pH, int pW,
                 int wshift0, int ncopies, int Ho, int Wo, int Pld, long long copy_stride, __nv_bfloat16* __restrict__ out) {
  __shared__ __nv_bfloat16 tile[64 + 2 * TP_HALO][66];
  const int Wp = (Wo + 2 * pW + 7) / 8 * 8;
  const int plane = (Ho + 2 * pH) * Wp;
  const int p0 = blockIdx.x * 64, c0 = blockIdx.y * 64, f = blockIdx.z;
  // load the UNSHIFTED plane positions p0 - HALO .. p0 + 64 + HALO: thread -> (position, 16-byte channel group)
  for (int i = threadIdx.x; i < (64 + 2 * TP_HALO) * 8; i += blockDim.x) {
    const int pp = i >> 3, cg = (i & 7) * 8;
    const int pos = p0 - TP_HALO + pp;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (pos >= 0 && pos < plane && c0 + cg < C) {
      const int hp = pos / Wp, wp = pos - hp * Wp;
      const int ho = hp - pH, wo = wp - pW;
      if (ho >= 0 && ho < Ho && wo >= 0 && wo < Wo)
        v = *reinterpret_cast<const uint4*>(x + (((size_t)f * H + (size_t)ho * sh) * W + (size_t)wo * sw) * ldx + c0 + cg);
    }
    const __nv_bfloat16* e = reinterpret_cast<const __nv_bfloat16*>(&v);
#pragma unroll
    for (int j = 0; j < 8; ++j) tile[pp][cg + j] = e[j];
  }
  __syncthreads();
  // store: thread -> (copy, channel, 8 consecutive positions).  Copy with shift d at column wp shows the pixel of column
  // wp + d, i.e. the staged position + d, unless that column falls outside the padded row (then zero: rows do not wrap).
  const __nv_bfloat16 zero = __float2bfloat16_rn(0.f);
  for (int i = threadIdx.x; i < ncopies * 64 * 8; i += blockDim.x) {
    const int cp = i / 512, rem = i - cp * 512;
    const int cc = rem >> 3, pg = (rem & 7) * 8;
    if (c0 + cc >= C || p0 + pg >= Pld) continue;
    const int d = wshift0 + cp;
    __align__(16) __nv_bfloat16 v[8];
    const int hp0 = (p0 + pg) / Wp, wp0 = (p0 + pg) - hp0 * Wp;       // Wp % 8 == 0: the 8 positions share a row
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int wsrc = wp0 + j + d;
      v[j] = (wsrc >= 0 && wsrc < Wp) ? tile[pg + j + d + TP_HALO][cc] : zero;
    }
    *reinterpret_cast<uint4*>(out + (size_t)cp * copy_stride + ((size_t)f * C + c0 + cc) * Pld + p0 + pg) = *reinterpret_cast<const uint4*>(v);
  }
}

// ------------------------------------------------------------------------------------------------ pointwise backward
__global__ void bwd_pointwise_kernel(const __nv_bfloat16* __restrict__ g1, const __nv_bfloat16* __restrict__ g2,
                                     const __nv_bfloat16* __restrict__ y, const float* __restrict__ scale, long long rows,
                                     int C, __nv_bfloat16* __restrict__ out, const float* __restrict__ scale2,
                                     __nv_bfloat16* __restrict__ out2) {
  const int cv = C / 8;
  const long long total = rows * cv;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % cv) * 8;
    const size_t off = (size_t)(idx / cv) * C + c;
    const uint4 a = *reinterpret_cast<const uint4*>(g1 + off);
    const __nv_bfloat16* ae = reinterpret_cast<const __nv_bfloat16*>(&a);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __bfloat162float(ae[j]);
    if (g2) {
      const uint4 b = *reinterpret_cast<const uint4*>(g2 + off);
      const __nv_bfloat16* be = reinterpret_cast<const __nv_bfloat16*>(&b);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += __bfloat162float(be[j]);
    }
    if (y) {
      const uint4 m = *reinterpret_cast<const uint4*>(y + off);
      const __nv_bfloat16* me = reinterpret_cast<const __nv_bfloat16*>(&m);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __bfloat162float(me[j]) > 0.f ? v[j] : 0.f;
    }
    __align__(16) __nv_bfloat16 o[8];
    if (out2) {                                           // second consumer of the same masked sum (its own channel scale, or none)
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = __float2bfloat16_rn(scale2 ? v[j] * scale2[c + j] : v[j]);
      *reinterpret_cast<uint4*>(out2 + off) = *reinterpret_cast<const uint4*>(o);
    }
    if (scale) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] *= scale[c + j];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = __float2bfloat16_rn(v[j]);
    *reinterpret_cast<uint4*>(out + off) = *reinterpret_cast<const uint4*>(o);
  }
}

// coarse_out[f, h, w, c] = coarse_in[f, h, w, c] (optional) + sum of the 2x2 children of fine[f, 2h.., 2w.., c]
__global__ void upsample_add_bwd_kernel(const __nv_bfloat16* __restrict__ fine, const __nv_bfloat16* __restrict__ coarse_in,
                                        int F, int Hc, int Wc, int C, __nv_bfloat16* __restrict__ out) {
  const int cv = C / 8;
  const long long total = (long long)F * Hc * Wc * cv;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % cv) * 8;
    long long r = idx / cv;
    const int w = (int)(r % Wc); r /= Wc;
    const int h = (int)(r % Hc);
    const int f = (int)(r / Hc);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = 0.f;
    for (int dy = 0; dy < 2; ++dy)
      for (int dx = 0; dx < 2; ++dx) {
        const uint4 a = *reinterpret_cast<const uint4*>(fine + (((size_t)f * 2 * Hc + 2 * h + dy) * (2 * Wc) + 2 * w + dx) * C + c);
        const __nv_bfloat16* ae = reinterpret_cast<const __nv_bfloat16*>(&a);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] += __bfloat162float(ae[j]);
      }
    const size_t off = (((size_t)f * Hc + h) * Wc + w) * C + c;
    if (coarse_in) {
      const uint4 a = *reinterpret_cast<const uint4*>(coarse_in + off);
      const __nv_bfloat16* ae = reinterpret_cast<const __nv_bfloat16*>(&a);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += __bfloat162float(ae[j]);
    }
    __align__(16) __nv_bfloat16 o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = __float2bfloat16_rn(v[j]);
    *reinterpret_cast<uint4*>(out + off) = *reinterpret_cast<const uint4*>(o);
  }
}

// out [F, 2*Hs, 2*Ws (cropped to H, W), C]: out[f, 2h, 2w] = src[f, h, w], zero elsewhere
__global__ void scatter_stride2_kernel(const __nv_bfloat16* __restrict__ src, int F, int Hs, int Ws, int H, int W, int C,
                                       __nv_bfloat16* __restrict__ out) {
  const int cv = C / 8;
  const long long total = (long long)F * H * W * cv;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % cv) * 8;
    long long r = idx / cv;
    const int w = (int)(r % W); r /= W;
    const int h = (int)(r % H);
    const int f = (int)(r / H);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (!(h & 1) && !(w & 1) && (h >> 1) < Hs && (w >> 1) < Ws)
      v = *reinterpret_cast<const uint4*>(src + (((size_t)f * Hs + (h >> 1)) * Ws + (w >> 1)) * C + c);
    *reinterpret_cast<uint4*>(out + (((size_t)f * H + h) * W + w) * C + c) = v;
  }
}

// out [B, T, P, C]: frame c = src [B, P, C], every other frame zero (backward of the slice-center body/head link)
__global__ void embed_frame_kernel(const uint4* __restrict__ src, long long per_frame_v, int B, int T, int c, uint4* __restrict__ out) {
  const long long total = (long long)B * T * per_frame_v;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long e = i % per_frame_v;
    const long long bt = i / per_frame_v;
    const int t = (int)(bt % T);
    out[i] = (t == c) ? src[(bt / T) * per_frame_v + e] : make_uint4(0, 0, 0, 0);
  }
}

// ------------------------------------------------------------------------------------------------ SGD
// Caffe2 MomentumSGDUpdate (non-Nesterov): g' = lr * (grad_scale * g + wd * w) + momentum * m;  m = g';  w -= g'
// w / g / m [taps][Cout][Cin] fp32.  Re-emits wf [taps][Cout][Cin] bf16 (forward operand) and wd_ [taps][Cin][Cout] bf16
// with the taps FLIPPED (dgrad of a stride-1 "same" conv is the conv of the gradient with the flipped, transposed filter).
// grid (ci tiles of 32, co tiles of 32, taps), block (32, 8): coalesced fp32 reads / writes along Cin, the transposed dgrad
// filter written through a shared-memory tile so that its stores are coalesced along Cout as well
__global__ void __launch_bounds__(256)
sgd_update_kernel(float* __restrict__ w, const float* __restrict__ g, float* __restrict__ m, int taps, int Cout, int Cin, float lr,
                  float momentum, float wd, float grad_scale, __nv_bfloat16* __restrict__ wf, __nv_bfloat16* __restrict__ wdg) {
  __shared__ float tile[32][33];
  const int tap = blockIdx.z, co0 = blockIdx.y * 32, ci0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int co = co0 + r, ci = ci0 + tx;
    float nw = 0.f;
    if (co < Cout && ci < Cin) {
      const size_t i = ((size_t)tap * Cout + co) * Cin + ci;
      const float wi = w[i];
      const float adj = lr * (grad_scale * g[i] + wd * wi) + momentum * m[i];
      m[i] = adj;
      nw = wi - adj;
      w[i] = nw;
      if (wf) wf[i] = __float2bfloat16_rn(nw);
    }
    tile[r][tx] = nw;
  }
  if (!wdg) return;
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int ci = ci0 + r, co = co0 + tx;
    if (ci < Cin && co < Cout) wdg[((size_t)(taps - 1 - tap) * Cin + ci) * Cout + co] = __float2bfloat16_rn(tile[tx][r]);
  }
}

// Every parameter tensor of the model in ONE launch: a table of items (device memory, built once by the trainer) and the
// exclusive prefix of their 32x32 tile counts; a block finds its item by binary search and runs the same tile update.
struct SgdItem {
  float* w; const float* g; float* m; __nv_bfloat16* wf; __nv_bfloat16* wdg;
  int taps, Cout, Cin, tiles_ci, tiles_co;
  float lr_mult, wd_mult;
};

__global__ void __launch_bounds__(256)
sgd_update_multi_kernel(const SgdItem* __restrict__ items, const int* __restrict__ first_block, int n_items, float lr, float momentum,
                        float wd, float grad_scale) {
  __shared__ float tile[32][33];
  int lo = 0, hi = n_items - 1;
  while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (first_block[mid] <= (int)blockIdx.x) lo = mid; else hi = mid - 1; }
  const SgdItem it = items[lo];
  int t = (int)blockIdx.x - first_block[lo];
  const int tci = t % it.tiles_ci; t /= it.tiles_ci;
  const int tco = t % it.tiles_co;
  const int tap = t / it.tiles_co;
  const int co0 = tco * 32, ci0 = tci * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const float lr_i = lr * it.lr_mult, wd_i = wd * it.wd_mult;
  for (int r = ty; r < 32; r += 8) {
    const int co = co0 + r, ci = ci0 + tx;
    float nw = 0.f;
    if (co < it.Cout && ci < it.Cin) {
      const size_t i = ((size_t)tap * it.Cout + co) * it.Cin + ci;
      const float wi = it.w[i];
      const float adj = lr_i * (grad_scale * it.g[i] + wd_i * wi) + momentum * it.m[i];
      it.m[i] = adj;
      nw = wi - adj;
      it.w[i] = nw;
      if (it.wf) it.wf[i] = __float2bfloat16_rn(nw);
    }
    tile[r][tx] = nw;
  }
  if (!it.wdg) return;
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int ci = ci0 + r, co = co0 + tx;
    if (ci < it.Cin && co < it.Cout) it.wdg[((size_t)(it.taps - 1 - tap) * it.Cin + ci) * it.Cout + co] = __float2bfloat16_rn(tile[tx][r]);
  }
}

// ------------------------------------------------------------------------------------------------ bias gradient, RPN losses
// db[c] += sum over rows of g[row, c]   (Conv bias gradient; biases of the FPN / RPN / head convs are trainable)
// block (32 channel groups of 8, 8 row lanes): 16-byte loads, fp32 partial sums, shared-memory reduction, one atomic per channel
__global__ void __launch_bounds__(256)
bias_grad_kernel(const __nv_bfloat16* __restrict__ g, long long rows, int C, int ld, float* __restrict__ db) {
  __shared__ float part[8][32][9];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c0 = (blockIdx.y * 32 + tx) * 8;
  const long long per = (rows + gridDim.x - 1) / gridDim.x;
  const long long r0 = per * blockIdx.x, r1 = min(rows, r0 + per);
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  if (c0 < C) {
    for (long long r = r0 + ty; r < r1; r += 8) {
      const uint4 v = *reinterpret_cast<const uint4*>(g + (size_t)r * ld + c0);
      const __nv_bfloat16* e = reinterpret_cast<const __nv_bfloat16*>(&v);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += __bfloat162float(e[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) part[ty][tx][j] = acc[j];
  __syncthreads();
  // 256 threads -> 256 channels of this block
  const int cc = threadIdx.x;                      // channel inside the 256-channel tile
  const int c = blockIdx.y * 256 + cc;
  if (c < C && r1 > r0) {
    float s = 0.f;
#pragma unroll
    for (int y = 0; y < 8; ++y) s += part[y][cc >> 3][cc & 7];
    atomicAdd(db + c, s);
  }
}

// FPN RPN losses and their gradients at one level (lib/modeling/FPN.py:282-321 with the Detectron ops
// SigmoidCrossEntropyLoss(normalize=0, scale=s_cls) and SmoothL1Loss(beta, scale=s_box), the latter divided by the batch size):
//   out rows [rows, ld_o] fp32 = [A logits | 4A deltas (a*4 + k)];  labels [rows, A] int32 (-1 = ignore);
//   targets / inside / outside weights [rows, 4A] fp32.  grad rows [rows, ld_g] bf16 in the same channel order (padding 0).
//   loss[0] += cls loss, loss[1] += bbox loss.
__global__ void rpn_loss_grad_kernel(const float* __restrict__ out, int ld_o, const int* __restrict__ labels,
                                     const float* __restrict__ targets, const float* __restrict__ iw, const float* __restrict__ ow,
                                     long long rows, int A, float s_cls, float s_box, float beta, __nv_bfloat16* __restrict__ grad,
                                     int ld_g, float* __restrict__ loss) {
  float lc = 0.f, lb = 0.f;
  const long long total = rows * ld_g;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int ch = (int)(idx % ld_g);
    const long long r = idx / ld_g;
    float gv = 0.f;
    if (ch < A) {
      const int t = labels[r * A + ch];
      if (t >= 0) {
        const float x = out[r * ld_o + ch];
        // -x*(t - [x>=0]) + log(1 + exp(x - 2x[x>=0]))   (the op's stable form)
        lc += s_cls * (-x * ((float)t - (x >= 0.f ? 1.f : 0.f)) + log1pf(expf(x - 2.f * x * (x >= 0.f ? 1.f : 0.f))));
        gv = s_cls * (1.f / (1.f + expf(-x)) - (float)t);
      }
    } else if (ch < 5 * A) {
      const int j = ch - A;
      const float w_in = iw[r * 4 * A + j], w_out = ow[r * 4 * A + j];
      const float d = w_in * (out[r * ld_o + ch] - targets[r * 4 * A + j]);
      const float ad = fabsf(d);
      lb += s_box * w_out * (ad < beta ? 0.5f * d * d / beta : ad - 0.5f * beta);
      gv = s_box * w_out * w_in * (ad < beta ? d / beta : (d > 0.f ? 1.f : -1.f));
    }
    grad[idx] = __float2bfloat16_rn(gv);
  }
  for (int o = 16; o > 0; o >>= 1) { lc += __shfl_xor_sync(0xffffffffu, lc, o); lb += __shfl_xor_sync(0xffffffffu, lb, o); }
  if ((threadIdx.x & 31) == 0 && loss) { if (lc != 0.f) atomicAdd(loss, lc); if (lb != 0.f) atomicAdd(loss + 1, lb); }
}

// The normaliser of Detectron's SigmoidCrossEntropyLoss with its default normalize=1: max(#labels >= 0, 1e-5) over the
// whole label blob.  One CTA (the single-level tube RPN has a few 10^4 labels per GPU).
__global__ void __launch_bounds__(1024) label_count_kernel(const int* __restrict__ labels, long long n, float* __restrict__ norm) {
  __shared__ int part[32];
  int c = 0;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) c += labels[i] >= 0;
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += part[w];
    norm[0] = fmaxf((float)s, 1e-5f);
  }
}

// Tube RPN losses (model_builder.py add_rpn_outputs(nd=True) + add_rpn_losses(time_dim=T)) read from the per-frame head
// output out [B, T, HW, ld_o] fp32 = [A logits | 4A deltas (a*4 + k)] per frame:
//   cls   TimePool avg of the logits over T, SigmoidCrossEntropyLoss(scale = s_cls) / norm[0]   labels [B, HW, A]
//   bbox  SmoothL1Loss(beta, scale = s_box) on the frame-folded deltas: channel a*4 + k of frame t is column
//         a*4T + t*4 + k of targets / inside / outside [B, HW, 4TA]
// grad [B, T, HW, ld_g] bf16 in the per-frame layout: the TimePool backward puts the logit gradient / T on every frame.
__global__ void rpn_tube_loss_grad_kernel(const float* __restrict__ out, int ld_o, const int* __restrict__ labels,
                                          const float* __restrict__ targets, const float* __restrict__ iw, const float* __restrict__ ow,
                                          int B, int T, long long HW, int A, float s_cls, float s_box, float beta,
                                          const float* __restrict__ norm, __nv_bfloat16* __restrict__ grad, int ld_g, float* __restrict__ loss) {
  float lc = 0.f, lb = 0.f;
  const long long total = (long long)B * T * HW * ld_g;
  const float sc = s_cls / norm[0];
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int ch = (int)(idx % ld_g);
    const long long q = idx / ld_g;
    const long long p = q % HW;
    const int t = (int)((q / HW) % T), b = (int)(q / HW / T);
    const long long pix = (long long)b * HW + p;
    float gv = 0.f;
    if (ch < A) {
      const int lab = labels[pix * A + ch];
      if (lab >= 0) {
        const float* o = out + ((size_t)b * T * HW + p) * ld_o + ch;
        float x = o[0];
        for (int u = 1; u < T; ++u) x += o[(size_t)u * HW * ld_o];
        x /= (float)T;
        if (t == 0) lc += sc * (-x * ((float)lab - (x >= 0.f ? 1.f : 0.f)) + log1pf(expf(x - 2.f * x * (x >= 0.f ? 1.f : 0.f))));
        gv = sc * (1.f / (1.f + expf(-x)) - (float)lab) / (float)T;
      }
    } else if (ch < 5 * A) {
      const int j = ch - A;
      const size_t col = (size_t)pix * 4 * T * A + (j >> 2) * 4 * T + t * 4 + (j & 3);
      const float w_in = iw[col], w_out = ow[col];
      const float d = w_in * (out[(size_t)q * ld_o + ch] - targets[col]);
      const float ad = fabsf(d);
      lb += s_box * w_out * (ad < beta ? 0.5f * d * d / beta : ad - 0.5f * beta);
      gv = s_box * w_out * w_in * (ad < beta ? d / beta : (d > 0.f ? 1.f : -1.f));
    }
    grad[idx] = __float2bfloat16_rn(gv);
  }
  for (int o = 16; o > 0; o >>= 1) { lc += __shfl_xor_sync(0xffffffffu, lc, o); lb += __shfl_xor_sync(0xffffffffu, lb, o); }
  if ((threadIdx.x & 31) == 0 && loss) { if (lc != 0.f) atomicAdd(loss, lc); if (lb != 0.f) atomicAdd(loss + 1, lb); }
}

// Backward of the two ReduceBackMeans (W, then H) of the res5 RoI head, fused with the pointwise step that follows it:
// out[n, p, c] = g[n, c] / HW * [y > 0] * scale[c]; out2 = the same masked value * scale2[c] (or unscaled).  y, scale, out2
// may be NULL (plain broadcast).  The [N, HW, C] broadcast itself is never stored.
__global__ void spatial_mean_bwd_kernel(const __nv_bfloat16* __restrict__ g, long long N, int HW, int C, const __nv_bfloat16* __restrict__ y,
                                        const float* __restrict__ scale, __nv_bfloat16* __restrict__ out, const float* __restrict__ scale2,
                                        __nv_bfloat16* __restrict__ out2) {
  const int cv = C / 8;
  const long long total = N * HW * cv;
  const float inv = 1.f / (float)HW;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % cv) * 8;
    const long long row = idx / cv;
    const size_t off = (size_t)row * C + c;
    const uint4 a = *reinterpret_cast<const uint4*>(g + (size_t)(row / HW) * C + c);
    const __nv_bfloat16* ae = reinterpret_cast<const __nv_bfloat16*>(&a);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __bfloat162float(ae[j]) * inv;
    if (y) {
      const uint4 m = *reinterpret_cast<const uint4*>(y + off);
      const __nv_bfloat16* me = reinterpret_cast<const __nv_bfloat16*>(&m);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __bfloat162float(me[j]) > 0.f ? v[j] : 0.f;
    }
    __align__(16) __nv_bfloat16 o[8];
    if (out2) {
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = __float2bfloat16_rn(scale2 ? v[j] * scale2[c + j] : v[j]);
      *reinterpret_cast<uint4*>(out2 + off) = *reinterpret_cast<const uint4*>(o);
    }
    if (scale) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] *= scale[c + j];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = __float2bfloat16_rn(v[j]);
    *reinterpret_cast<uint4*>(out + off) = *reinterpret_cast<const uint4*>(o);
  }
}


// ------------------------------------------------------------------------------------------------ RoI heads (backward)
// out = bf16(g + acc)
__global__ void grad_join_f32_kernel(const __nv_bfloat16* __restrict__ g, const float* __restrict__ acc, long long n8,
                                     __nv_bfloat16* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    const float4 a0 = reinterpret_cast<const float4*>(acc)[2 * i], a1 = reinterpret_cast<const float4*>(acc)[2 * i + 1];
    float v[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
    if (g) {
      const uint4 gv = reinterpret_cast<const uint4*>(g)[i];
      const __nv_bfloat16* ge = reinterpret_cast<const __nv_bfloat16*>(&gv);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += __bfloat162float(ge[j]);
    }
    __align__(16) __nv_bfloat16 o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = __float2bfloat16_rn(v[j]);
    reinterpret_cast<uint4*>(out)[i] = *reinterpret_cast<const uint4*>(o);
  }
}

struct RoiBwdLevels {
  float* dfeat[8];
  int H[8], W[8];
  float scale[8];
};

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// the forward's bilinear sample (dense_ops.cu bilinear_acc) transposed: v[8] * weight into the four corners
__device__ __forceinline__ void bilinear_scatter(float* __restrict__ d, int H, int W, int C, float y, float x, const float* v, float wgt) {
  if (!(y >= -1.f && y <= (float)H && x >= -1.f && x <= (float)W)) return;      // also for a non-finite RoI (diverged weights)
  if (y <= 0.f) y = 0.f;
  if (x <= 0.f) x = 0.f;
  int yl = (int)y, xl = (int)x, yh, xh;
  if (yl >= H - 1) { yh = yl = H - 1; y = (float)yl; } else yh = yl + 1;
  if (xl >= W - 1) { xh = xl = W - 1; x = (float)xl; } else xh = xl + 1;
  const float ly = y - yl, lx = x - xl, hy = 1.f - ly, hx = 1.f - lx;
  const float w4[4] = {hy * hx * wgt, hy * lx * wgt, ly * hx * wgt, ly * lx * wgt};
  float* p4[4] = {d + ((size_t)yl * W + xl) * C, d + ((size_t)yl * W + xh) * C, d + ((size_t)yh * W + xl) * C, d + ((size_t)yh * W + xh) * C};
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    if (w4[q] == 0.f) continue;
    red_add_v4(p4[q], v[0] * w4[q], v[1] * w4[q], v[2] * w4[q], v[3] * w4[q]);
    red_add_v4(p4[q] + 4, v[4] * w4[q], v[5] * w4[q], v[6] * w4[q], v[7] * w4[q]);
  }
}

// grid (R*T, P); threads over (pw, 8-channel vectors) exactly like roi_align_kernel
__global__ void roi_align_bwd_kernel(RoiBwdLevels lv, int kmin, const float* __restrict__ rois, int ldr, const int* __restrict__ n_dev,
                                     int R, int T, const int* __restrict__ levels, int C, int P, int sampling,
                                     const __nv_bfloat16* __restrict__ grad) {
  const int rt = blockIdx.x, ph = blockIdx.y;
  const int r = rt / T, t = rt - r * T;
  const int n = n_dev ? min(*n_dev, R) : R;
  if (r >= n) return;
  const int cv = C / 8;
  const float* roi = rois + (size_t)r * ldr;
  const int l = levels ? (levels[r] - kmin) : 0;
  const int H = lv.H[l], W = lv.W[l];
  const float sc = lv.scale[l];
  const int img = (int)roi[0] * T + t;
  float* d = lv.dfeat[l] + (size_t)img * H * W * C;
  const float x1 = roi[1 + 4 * t] * sc, y1 = roi[2 + 4 * t] * sc, x2 = roi[3 + 4 * t] * sc, y2 = roi[4 + 4 * t] * sc;
  const float rw = fmaxf(x2 - x1, 1.f), rh = fmaxf(y2 - y1, 1.f);
  const float bh = rh / (float)P, bw = rw / (float)P;
  const int gh = sampling > 0 ? sampling : (int)ceilf(rh / P), gw = sampling > 0 ? sampling : (int)ceilf(rw / P);
  const float inv_cnt = 1.f / (float)(gh * gw);
  const __nv_bfloat16* gbase = grad + ((size_t)rt * P + ph) * P * C;
  for (int i = threadIdx.x; i < P * cv; i += blockDim.x) {
    const int pw = i / cv, c = (i - pw * cv) * 8;
    const uint4 gv = *reinterpret_cast<const uint4*>(gbase + (size_t)pw * C + c);
    const __nv_bfloat16* ge = reinterpret_cast<const __nv_bfloat16*>(&gv);
    float v[8];
    bool any = false;
#pragma unroll
    for (int j = 0; j < 8; ++j) { v[j] = __bfloat162float(ge[j]); any |= v[j] != 0.f; }
    if (!any) continue;
    for (int iy = 0; iy < gh; ++iy) {
      const float y = y1 + ph * bh + (iy + 0.5f) * bh / (float)gh;
      for (int ix = 0; ix < gw; ++ix) {
        const float x = x1 + pw * bw + (ix + 0.5f) * bw / (float)gw;
        bilinear_scatter(d + c, H, W, C, y, x, v, inv_cnt);
      }
    }
  }
}

// one thread per RoI (C is small).  A RoI owns T consecutive rows of `out` / `grad`, one per frame, each [C logits |
// 4C deltas (c*4 + k)]; T = 1 is the 2-D head.  For T > 1 the fold of dt_fold_tube_heads is applied on the fly (logits =
// mean over the frames, box column c*4T + t*4 + k of targets / weights) and its backward is fused into the gradient
// write: every frame row receives the logit gradient / T and its own frame's box gradient.  With T = 1 every
// expression reduces exactly (x / 1.f == x) to the 2-D head's.
__device__ __forceinline__ float tube_logit(const float* o, int ld_o, int T, int j) {
  float a = o[j];
  for (int t = 1; t < T; ++t) a += o[(size_t)t * ld_o + j];
  return a / (float)T;
}

__global__ void frcnn_loss_grad_kernel(const float* __restrict__ out, int ld_o, const int* __restrict__ labels,
                                       const float* __restrict__ targets, const float* __restrict__ iw, const float* __restrict__ ow,
                                       int rows, int T, int C, const float* __restrict__ totals, float s_cls, float s_box,
                                       __nv_bfloat16* __restrict__ grad, int ld_g, float* __restrict__ loss, float* __restrict__ acc) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  float lc = 0.f, lb = 0.f, hit = 0.f;
  if (r < rows) {
    __nv_bfloat16* g = grad + (size_t)r * T * ld_g;
    const int lbl = labels[r];
    const float N = totals[0];
    if (lbl < 0 || !(N > 0.f)) {
      for (int j = 0; j < T * ld_g; ++j) g[j] = __float2bfloat16_rn(0.f);
    } else {
      const float* o = out + (size_t)r * T * ld_o;
      const int C4T = 4 * C * T;
      float m = tube_logit(o, ld_o, T, 0); int am = 0;
      for (int j = 1; j < C; ++j) { const float v = tube_logit(o, ld_o, T, j); if (v > m) { m = v; am = j; } }
      float se = 0.f;
      for (int j = 0; j < C; ++j) se += expf(tube_logit(o, ld_o, T, j) - m);
      const float lse = logf(se);
      lc = -(tube_logit(o, ld_o, T, lbl) - m - lse) * s_cls / N;
      hit = am == lbl ? 1.f : 0.f;
      for (int j = 0; j < C; ++j) {
        const float pj = expf(tube_logit(o, ld_o, T, j) - m - lse);
        const __nv_bfloat16 gj = __float2bfloat16_rn((pj - (j == lbl ? 1.f : 0.f)) * s_cls / N / (float)T);
        for (int t = 0; t < T; ++t) g[(size_t)t * ld_g + j] = gj;
      }
      for (int t = 0; t < T; ++t) {
        const float* ot = o + (size_t)t * ld_o;
        __nv_bfloat16* gt = g + (size_t)t * ld_g;
        for (int j = 0; j < 4 * C; ++j) {
          const size_t col = (size_t)r * C4T + (j >> 2) * 4 * T + t * 4 + (j & 3);
          const float w_in = iw[col], w_out = ow[col];
          const float d = w_in * (ot[C + j] - targets[col]);
          const float ad = fabsf(d);
          lb += w_out * (ad < 1.f ? 0.5f * d * d : ad - 0.5f) * s_box / N;
          gt[C + j] = __float2bfloat16_rn(w_out * w_in * (ad < 1.f ? d : (d > 0.f ? 1.f : -1.f)) * s_box / N);
        }
        for (int j = 5 * C; j < ld_g; ++j) gt[j] = __float2bfloat16_rn(0.f);
      }
    }
  }
  for (int o2 = 16; o2 > 0; o2 >>= 1) {
    lc += __shfl_xor_sync(0xffffffffu, lc, o2); lb += __shfl_xor_sync(0xffffffffu, lb, o2); hit += __shfl_xor_sync(0xffffffffu, hit, o2);
  }
  if ((threadIdx.x & 31) == 0) {
    if (loss) { if (lc != 0.f) atomicAdd(loss, lc); if (lb != 0.f) atomicAdd(loss + 1, lb); }
    if (acc && hit != 0.f) atomicAdd(acc, hit);
  }
}

// one CTA per (RoI d, joint k): 2S x 2S map -> bilinear 2x -> spatial softmax loss -> gradient back to the packed layout
__global__ void __launch_bounds__(256)
kps_loss_grad_kernel(const float* __restrict__ low, int ld, int S, int K, const int* __restrict__ loc, const float* __restrict__ wts,
                     const float* __restrict__ totals, float scale, __nv_bfloat16* __restrict__ grad, int ld_g, float* __restrict__ loss) {
  extern __shared__ float sm[];
  const int d = blockIdx.x, k = blockIdx.y;
  const int S2 = 2 * S, M = 4 * S;
  float* Lm = sm;                       // [S2][S2]
  float* U = Lm + S2 * S2;              // [M][M] upsampled logits, then their gradient
  __shared__ float red[32];
  __shared__ float s_max, s_sum;
  const float w = wts[(size_t)d * K + k];
  const float tw = totals[1];
  __nv_bfloat16* gd = grad + (size_t)d * S * S * ld_g;
  if (!(w > 0.f) || !(tw > 0.f)) {      // no target: zero gradient for this joint's four sub-pixel channels
    for (int i = threadIdx.x; i < S * S * 4; i += blockDim.x) gd[(size_t)(i >> 2) * ld_g + (i & 3) * K + k] = __float2bfloat16_rn(0.f);
    return;
  }
  const float* ld_ = low + (size_t)d * S * S * ld;
  for (int i = threadIdx.x; i < S2 * S2; i += blockDim.x) {
    const int Y = i / S2, X = i - Y * S2;
    Lm[i] = ld_[((size_t)(Y >> 1) * S + (X >> 1)) * ld + ((Y & 1) * 2 + (X & 1)) * K + k];
  }
  __syncthreads();
  const float f4[4] = {0.25f, 0.75f, 0.75f, 0.25f};
  // ConvTranspose k4 s2 p1: U[o] = sum_i L[i] * f[o - 2i + 1]  -> i in {(o-2)/2 .. (o+1)/2}
  float mx = -3.4e38f;
  for (int i = threadIdx.x; i < M * M; i += blockDim.x) {
    const int Y = i / M, X = i - Y * M;
    float acc = 0.f;
    for (int iy = (Y - 2 + 1) >> 1; iy <= (Y + 1) >> 1; ++iy) {
      if (iy < 0 || iy >= S2) continue;
      const int ky = Y - 2 * iy + 1;
      if (ky < 0 || ky > 3) continue;
      for (int ix = (X - 2 + 1) >> 1; ix <= (X + 1) >> 1; ++ix) {
        if (ix < 0 || ix >= S2) continue;
        const int kx = X - 2 * ix + 1;
        if (kx < 0 || kx > 3) continue;
        acc += Lm[iy * S2 + ix] * f4[ky] * f4[kx];
      }
    }
    U[i] = acc;
    mx = fmaxf(mx, acc);
  }
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) { float m = red[0]; for (int i = 1; i < (int)(blockDim.x >> 5); ++i) m = fmaxf(m, red[i]); s_max = m; }
  __syncthreads();
  mx = s_max;
  float se = 0.f;
  for (int i = threadIdx.x; i < M * M; i += blockDim.x) se += expf(U[i] - mx);
  for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = se;
  __syncthreads();
  if (threadIdx.x == 0) { float s = 0.f; for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i]; s_sum = s; }
  __syncthreads();
  const float lse = logf(s_sum);
  const int target = loc[(size_t)d * K + k];
  const float gs = w * scale / tw;
  if (threadIdx.x == 0 && loss) atomicAdd(loss, -(U[target] - mx - lse) * gs);
  __syncthreads();
  for (int i = threadIdx.x; i < M * M; i += blockDim.x) U[i] = (expf(U[i] - mx - lse) - (i == target ? 1.f : 0.f)) * gs;
  __syncthreads();
  // dL[i] = sum_o dU[o] * f[o - 2i + 1], o in 2i-1 .. 2i+2
  for (int i = threadIdx.x; i < S2 * S2; i += blockDim.x) {
    const int iy = i / S2, ix = i - iy * S2;
    float acc = 0.f;
#pragma unroll
    for (int ky = 0; ky < 4; ++ky) {
      const int Y = 2 * iy - 1 + ky;
      if (Y < 0 || Y >= M) continue;
#pragma unroll
      for (int kx = 0; kx < 4; ++kx) {
        const int X = 2 * ix - 1 + kx;
        if (X < 0 || X >= M) continue;
        acc += U[Y * M + X] * f4[ky] * f4[kx];
      }
    }
    gd[((size_t)(iy >> 1) * S + (ix >> 1)) * ld_g + ((iy & 1) * 2 + (ix & 1)) * K + k] = __float2bfloat16_rn(acc);
  }
}

__global__ void subpixel_grad_fix_kernel(float* __restrict__ gW, float* __restrict__ gb, int K, int Cin, int ldc) {
  const long long total = 9ll * ldc * Cin;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int co = (int)((i / Cin) % ldc), tap = (int)(i / ((long long)Cin * ldc));
    bool live = co < 4 * K;
    if (live) {
      const int sub = co / K, py = sub >> 1, px = sub & 1;
      const int dy = tap / 3 - 1, dx = tap % 3 - 1;
      const int ky = py + 1 - 2 * dy, kx = px + 1 - 2 * dx;
      live = ky >= 0 && ky <= 3 && kx >= 0 && kx <= 3;
    }
    if (!live) gW[i] = 0.f;
  }
  if (gb && blockIdx.x == 0) {
    for (int k = threadIdx.x; k < ldc; k += blockDim.x) {
      if (k < K) {
        const float s = gb[k] + gb[K + k] + gb[2 * K + k] + gb[3 * K + k];
        gb[k] = s; gb[K + k] = s; gb[2 * K + k] = s; gb[3 * K + k] = s;
      } else if (k >= 4 * K) {
        gb[k] = 0.f;
      }
    }
  }
}

}  // namespace dt

using namespace dt;

static int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  const long long cap = 148ll * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

extern "C" int dt_planes_ld(int Ho, int Wo, int pH, int pW) { return (Ho + 2 * pH) * ((Wo + 2 * pW + 7) / 8 * 8); }

extern "C" int dt_to_planes(const void* x, int F, int H, int W, int C, int ldx, int sh, int sw, int pH, int pW, int wshift,
                            int ncopies, void* out, void* stream) {
  DT_CHECK_ARG(F >= 0 && H >= 1 && W >= 1 && C >= 8 && C % 8 == 0 && ldx >= C && ldx % 8 == 0 && sh >= 1 && sw >= 1 && pH >= 0 && pW >= 0,
               "dt_to_planes: bad shape F=%d H=%d W=%d C=%d ldx=%d", F, H, W, C, ldx);
  DT_CHECK_ARG(ncopies >= 1 && wshift >= -pW && wshift + ncopies - 1 <= pW && pW <= TP_HALO,
               "dt_to_planes: shifts %d..%d outside [-%d, %d] (pW <= %d)", wshift, wshift + ncopies - 1, pW, pW, TP_HALO);
  if (F == 0) return 0;
  DT_CHECK_ARG(x && out, "dt_to_planes: null pointer");
  const int Ho = (H + sh - 1) / sh, Wo = (W + sw - 1) / sw;
  const int Pld = dt_planes_ld(Ho, Wo, pH, pW);
  dim3 grid((Pld + 63) / 64, (C + 63) / 64, F);
  to_planes_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, F, H, W, C, ldx, sh, sw, pH, pW, wshift, ncopies, Ho, Wo, Pld,
                                                           (long long)F * C * Pld, (__nv_bfloat16*)out);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_wgrad(const void* gz_planes, const void* x_planes, int N, int T, int Ho, int Wo, int Cout, int Cin, int kT, int kH,
                        int kW, float* dW, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DT_CHECK_ARG(N >= 1 && T >= 1 && Ho >= 1 && Wo >= 1 && Cout >= 1 && Cin >= 8 && Cin % 8 == 0 && kT >= 1 && kH >= 1 && kW >= 1 &&
                   (kT & 1) && (kH & 1) && (kW & 1),
               "dt_wgrad: bad shape N=%d T=%d %dx%d Cout=%d Cin=%d k=%dx%dx%d (odd 'same' kernels, Cin %% 8 == 0)", N, T, Ho, Wo, Cout, Cin, kT, kH, kW);
  DT_CHECK_ARG(gz_planes && x_planes && dW, "dt_wgrad: null pointer");
  const int pT = kT / 2, pH = kH / 2, pW = kW / 2;
  const int Pld = dt_planes_ld(Ho, Wo, pH, pW);
  const int Wp = (Wo + 2 * pW + 7) / 8 * 8, plane = Pld;
  WgradParams p;
  memset(&p, 0, sizeof(p));
  p.Cout = Cout; p.Cin = Cin; p.taps = kT * kH * kW; p.kT = kT; p.kH = kH; p.kW = kW; p.pT = pT; p.pH = pH; p.pW = pW;
  p.Wp = Wp; p.T = T; p.N = N; p.kchunks = cdiv(plane, 64); p.dW = dW;
  const int BN = Cin >= 256 ? 256 : (Cin > 64 ? 128 : 64);
  p.tiles_m = cdiv(Cout, 128); p.tiles_n = cdiv(Cin, BN);
  const long long units = (long long)p.taps * p.tiles_m * p.tiles_n;
  const long long kblocks = (long long)N * T * p.kchunks;
  long long ksplit = (148 * 3 + units - 1) / units;               // ~3 waves of CTAs
  if (ksplit > kblocks / 4) ksplit = kblocks / 4;
  if (ksplit < 1) ksplit = 1;
  p.ksplit = (int)ksplit;
  CUtensorMap tmG, tmX;
  {
    uint64_t d[4] = {(uint64_t)plane, (uint64_t)Cout, (uint64_t)T, (uint64_t)N};
    uint64_t s[3] = {(uint64_t)Pld * 2, (uint64_t)Pld * 2 * Cout, (uint64_t)Pld * 2 * Cout * T};
    uint32_t b[4] = {64, 128, 1, 1}, e[4] = {1, 1, 1, 1};
    if (encode_map(&tmG, 0, 4, gz_planes, d, s, b, e)) return 1;
  }
  {   // x planes: kW pre-shifted copies [kW][N*T, Cin, Pld]
    uint64_t d[5] = {(uint64_t)plane, (uint64_t)Cin, (uint64_t)T, (uint64_t)N, (uint64_t)kW};
    uint64_t s[4] = {(uint64_t)Pld * 2, (uint64_t)Pld * 2 * Cin, (uint64_t)Pld * 2 * Cin * T, (uint64_t)Pld * 2 * Cin * T * N};
    uint32_t b[5] = {64, (uint32_t)BN, 1, 1, 1}, e[5] = {1, 1, 1, 1, 1};
    if (encode_map(&tmX, 0, 5, x_planes, d, s, b, e)) return 1;
  }
  switch (BN) {
    case 256: return launch_wgrad<256>(tmG, tmX, p, stream);
    case 128: return launch_wgrad<128>(tmG, tmX, p, stream);
    default: return launch_wgrad<64>(tmG, tmX, p, stream);
  }
}

extern "C" int dt_wgrad_nhwc(const void* gz, int ld_g, const void* x, int ld_x, int N, int T, int Ho, int Wo, int Hi, int Wi, int Cout,
                             int Cin, int kT, int kH, int kW, int sH, int sW, float* dW, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  DT_CHECK_ARG(N >= 1 && T >= 1 && Ho >= 1 && Wo >= 1 && Cout >= 1 && Cin >= 8 && Cin % 4 == 0 && kT >= 1 && kH >= 1 && kW >= 1 && (kT & 1) &&
                   (kH & 1) && (kW & 1) && ld_g >= Cout && ld_g % 8 == 0 && ld_x >= Cin && ld_x % 8 == 0 && sH >= 1 && sW >= 1,
               "dt_wgrad_nhwc: bad shape N=%d T=%d %dx%d Cout=%d (ld %d) Cin=%d (ld %d) k=%dx%dx%d", N, T, Ho, Wo, Cout, ld_g, Cin, ld_x, kT, kH, kW);
  const bool strided = sH != 1 || sW != 1;
  DT_CHECK_ARG(!strided || (kT == 1 && kH == 1 && kW == 1), "dt_wgrad_nhwc: only pointwise convs may be strided");
  DT_CHECK_ARG(strided ? (Ho == (Hi + sH - 1) / sH && Wo == (Wi + sW - 1) / sW) : (Ho == Hi && Wo == Wi), "dt_wgrad_nhwc: output %dx%d does not match input %dx%d / stride", Ho, Wo, Hi, Wi);
  DT_CHECK_ARG(gz && x && dW, "dt_wgrad_nhwc: null pointer");
  WgradNParams p;
  memset(&p, 0, sizeof(p));
  p.Cout = Cout; p.Cin = Cin; p.taps = kT * kH * kW; p.kT = kT; p.kH = kH; p.kW = kW; p.pT = kT / 2; p.pH = kH / 2; p.pW = kW / 2;
  p.T = T; p.dW = dW;
  // 64-position tile (TW, TH, TT, TB), powers of two: the largest useful fraction, then the widest rows
  {
    double best = -1.0;
    for (int tw = 64; tw >= 1; tw >>= 1)
      for (int th = 64 / tw; th >= 1; th >>= 1)
        for (int tt = 64 / (tw * th); tt >= 1; tt >>= 1) {
          const int tb = 64 / (tw * th * tt);
          if (tt > 1 && kT > 1) continue;                                   // temporal taps shift whole frames: one frame per box
          const double cover = (double)cdiv(Wo, tw) * tw * cdiv(Ho, th) * th * cdiv(T, tt) * tt * (double)cdiv(N, tb) * tb;
          const double eff = (double)Wo * Ho * T * N / cover;
          if (eff > best + 1e-9) { best = eff; p.TW = tw; p.TH = th; p.TT = tt; p.TB = tb; }
        }
  }
  p.nW = cdiv(Wo, p.TW); p.nH = cdiv(Ho, p.TH); p.nT = cdiv(T, p.TT); p.nN = cdiv(N, p.TB);
  const int BN = Cin >= 256 ? 256 : (Cin > 64 ? 128 : 64);
  p.tiles_m = cdiv(Cout, 128); p.tiles_n = cdiv(Cin, BN);
  const long long units = (long long)p.taps * p.tiles_m * p.tiles_n;
  const long long kblocks = (long long)p.nW * p.nH * p.nT * p.nN;
  // K split: every CTA adds its 128 x BN partial tile into dW with red.global, so the split count is also the atomic
  // traffic multiplier.  DT_WGRAD_WAVES overrides the wave count (tuning knob of tools/bench_wgrad.py).
  // Measured on B200 (tools/bench_wgrad.py, profiles/wgrad_waves_r02.md): pointwise layers are fastest with ONE wave of CTAs
  // (a 1x1 filter has few (tap, tile) units, so 3 waves meant ~100 partial tiles added per output tile), multi-tap layers with 2.
  static const int waves_env = [] { const char* e = getenv("DT_WGRAD_WAVES"); const int v = e ? atoi(e) : 0; return v >= 1 && v <= 16 ? v : 0; }();
  const int waves = waves_env ? waves_env : (p.taps == 1 ? 1 : 2);
  long long ksplit = (148 * waves + units - 1) / units;
  if (ksplit > kblocks / 4) ksplit = kblocks / 4;
  if (ksplit < 1) ksplit = 1;
  p.ksplit = (int)ksplit;
  CUtensorMap tmG, tmX;
  const uint32_t box[5] = {64, (uint32_t)p.TW, (uint32_t)p.TH, (uint32_t)p.TT, (uint32_t)p.TB}, e[5] = {1, 1, 1, 1, 1};
  {
    uint64_t d[5] = {(uint64_t)Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)T, (uint64_t)N};
    const uint64_t sC = (uint64_t)ld_g * 2;
    uint64_t st[4] = {sC, sC * Wo, sC * Wo * Ho, sC * Wo * Ho * T};
    if (encode_map(&tmG, 0, 5, gz, d, st, box, e)) return 1;
  }
  {   // strided pointwise convs: the stride is folded into the global strides (positions of the OUTPUT grid)
    uint64_t d[5] = {(uint64_t)Cin, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)T, (uint64_t)N};
    const uint64_t sC = (uint64_t)ld_x * 2;
    uint64_t st[4] = {sC * sW, sC * Wi * sH, sC * Wi * Hi, sC * Wi * Hi * T};
    if (encode_map(&tmX, 0, 5, x, d, st, box, e)) return 1;
  }
  switch (BN) {
    case 256: return launch_wgrad_nhwc<256>(tmG, tmX, p, stream);
    case 128: return launch_wgrad_nhwc<128>(tmG, tmX, p, stream);
    default: return launch_wgrad_nhwc<64>(tmG, tmX, p, stream);
  }
}

extern "C" int dt_bwd_pointwise(const void* g1, const void* g2, const void* y, const float* scale, long long rows, int C, void* out,
                                void* stream) {
  return dt_bwd_pointwise2(g1, g2, y, scale, rows, C, out, nullptr, nullptr, stream);
}

extern "C" int dt_bwd_pointwise2(const void* g1, const void* g2, const void* y, const float* scale, long long rows, int C, void* out,
                                 const float* scale2, void* out2, void* stream) {
  DT_CHECK_ARG(rows >= 0 && C >= 8 && C % 8 == 0, "dt_bwd_pointwise: bad shape rows=%lld C=%d (C %% 8 == 0)", rows, C);
  if (rows == 0) return 0;
  DT_CHECK_ARG(g1 && out, "dt_bwd_pointwise: null pointer");
  bwd_pointwise_kernel<<<grid_for(rows * (C / 8), 256), 256, 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)g1, (const __nv_bfloat16*)g2, (const __nv_bfloat16*)y, scale, rows, C, (__nv_bfloat16*)out, scale2,
      (__nv_bfloat16*)out2);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_upsample_add_bwd(const void* fine, const void* coarse_in, int F, int Hc, int Wc, int C, void* out, void* stream) {
  DT_CHECK_ARG(F >= 0 && Hc >= 1 && Wc >= 1 && C >= 8 && C % 8 == 0, "dt_upsample_add_bwd: bad shape");
  if (F == 0) return 0;
  DT_CHECK_ARG(fine && out, "dt_upsample_add_bwd: null pointer");
  upsample_add_bwd_kernel<<<grid_for((long long)F * Hc * Wc * (C / 8), 256), 256, 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)fine, (const __nv_bfloat16*)coarse_in, F, Hc, Wc, C, (__nv_bfloat16*)out);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_scatter_stride2(const void* src, int F, int Hs, int Ws, int H, int W, int C, void* out, void* stream) {
  DT_CHECK_ARG(F >= 0 && Hs >= 1 && Ws >= 1 && H >= 1 && W >= 1 && (H + 1) / 2 == Hs && (W + 1) / 2 == Ws && C >= 8 && C % 8 == 0,
               "dt_scatter_stride2: bad shape %dx%d -> %dx%d C=%d", Hs, Ws, H, W, C);
  if (F == 0) return 0;
  DT_CHECK_ARG(src && out, "dt_scatter_stride2: null pointer");
  scatter_stride2_kernel<<<grid_for((long long)F * H * W * (C / 8), 256), 256, 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)src, F, Hs, Ws, H, W, C, (__nv_bfloat16*)out);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_embed_frame(const void* src, int B, int T, long long frame_elems, int c, void* out, void* stream) {
  DT_CHECK_ARG(B >= 0 && T >= 1 && c >= 0 && c < T && frame_elems >= 8 && frame_elems % 8 == 0, "dt_embed_frame: bad shape B=%d T=%d c=%d elems=%lld", B, T, c, frame_elems);
  if (B == 0) return 0;
  DT_CHECK_ARG(src && out, "dt_embed_frame: null pointer");
  embed_frame_kernel<<<grid_for((long long)B * T * (frame_elems / 8), 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)src, frame_elems / 8, B, T, c, (uint4*)out);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_sgd_update(float* w, const float* g, float* m, int taps, int Cout, int Cin, float lr, float momentum, float wd,
                             float grad_scale, void* w_fwd_bf16, void* w_dgrad_bf16, void* stream) {
  DT_CHECK_ARG(taps >= 1 && taps <= 65535 && Cout >= 1 && Cin >= 1 && (Cout + 31) / 32 <= 65535, "dt_sgd_update: bad shape");
  DT_CHECK_ARG(w && g && m, "dt_sgd_update: null pointer");
  dim3 grid((Cin + 31) / 32, (Cout + 31) / 32, taps);
  sgd_update_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(w, g, m, taps, Cout, Cin, lr, momentum, wd, grad_scale,
                                                            (__nv_bfloat16*)w_fwd_bf16, (__nv_bfloat16*)w_dgrad_bf16);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_sgd_update_multi(const void* items, const int* first_block, int n_items, int total_blocks, float lr, float momentum,
                                   float wd, float grad_scale, void* stream) {
  DT_CHECK_ARG(n_items >= 1 && total_blocks >= 1, "dt_sgd_update_multi: empty table (n_items=%d, blocks=%d)", n_items, total_blocks);
  DT_CHECK_ARG(items && first_block, "dt_sgd_update_multi: null pointer");
  static_assert(sizeof(SgdItem) == 72, "dt_sgd_item layout");
  sgd_update_multi_kernel<<<total_blocks, 256, 0, (cudaStream_t)stream>>>((const SgdItem*)items, first_block, n_items, lr, momentum, wd, grad_scale);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_bias_grad(const void* g, long long rows, int C, int ld, float* db, void* stream) {
  DT_CHECK_ARG(rows >= 0 && C >= 8 && C % 8 == 0 && ld >= C && ld % 8 == 0, "dt_bias_grad: bad shape rows=%lld C=%d ld=%d (multiples of 8)", rows, C, ld);
  if (rows == 0) return 0;
  DT_CHECK_ARG(g && db, "dt_bias_grad: null pointer");
  long long gx = rows / 128; if (gx < 1) gx = 1; if (gx > 148 * 8) gx = 148 * 8;
  dim3 grid((unsigned)gx, (C + 255) / 256);
  bias_grad_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)g, rows, C, ld, db);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_rpn_loss_grad(const float* out, int ld_o, const int* labels, const float* targets, const float* inside_w,
                                const float* outside_w, long long rows, int A, float scale_cls, float scale_box, float beta,
                                void* grad, int ld_g, float* loss, void* stream) {
  DT_CHECK_ARG(rows >= 0 && A >= 1 && ld_o >= 5 * A && ld_g >= 5 * A && beta > 0.f, "dt_rpn_loss_grad: bad shape rows=%lld A=%d ld_o=%d ld_g=%d", rows, A, ld_o, ld_g);
  if (rows == 0) return 0;
  DT_CHECK_ARG(out && labels && targets && inside_w && outside_w && grad, "dt_rpn_loss_grad: null pointer");
  rpn_loss_grad_kernel<<<grid_for(rows * ld_g, 256), 256, 0, (cudaStream_t)stream>>>(out, ld_o, labels, targets, inside_w, outside_w, rows, A,
                                                                                  scale_cls, scale_box, beta, (__nv_bfloat16*)grad, ld_g, loss);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_grad_join_f32(const void* g, const float* acc, long long n, void* out, void* stream) {
  DT_CHECK_ARG(n >= 0 && n % 8 == 0, "dt_grad_join_f32: n=%lld must be a multiple of 8", n);
  if (n == 0) return 0;
  DT_CHECK_ARG(acc && out, "dt_grad_join_f32: null pointer");
  grad_join_f32_kernel<<<grid_for(n / 8, 256), 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)g, acc, n / 8, (__nv_bfloat16*)out);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_roi_align_bwd(const void* grad, float* const* dfeats, const int* Hs, const int* Ws, const float* scales, int nlevels,
                                int k_min, int C, const float* rois, int ldr, const int* n_dev, int R, int T, const int* levels, int P,
                                int sampling_ratio, void* stream) {
  DT_CHECK_ARG(nlevels >= 1 && nlevels <= 8 && C >= 8 && C % 8 == 0 && R >= 0 && T >= 1 && P >= 1 && ldr >= 4 * T + 1,
               "dt_roi_align_bwd: bad shape (C=%d must be a multiple of 8)", C);
  DT_CHECK_ARG(nlevels == 1 || levels, "dt_roi_align_bwd: multi-level pooling needs the per-RoI level array");
  if (R == 0) return 0;
  DT_CHECK_ARG(grad && dfeats && Hs && Ws && scales && rois, "dt_roi_align_bwd: null pointer");
  RoiBwdLevels lv;
  for (int l = 0; l < nlevels; ++l) {
    DT_CHECK_ARG(dfeats[l], "dt_roi_align_bwd: null accumulator for level %d", l);
    lv.dfeat[l] = dfeats[l]; lv.H[l] = Hs[l]; lv.W[l] = Ws[l]; lv.scale[l] = scales[l];
  }
  dim3 grid(R * T, P);
  roi_align_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(lv, k_min, rois, ldr, n_dev, R, T, levels, C, P, sampling_ratio,
                                                              (const __nv_bfloat16*)grad);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_frcnn_loss_grad(const float* out, int ld_o, const int* labels, const float* targets, const float* inside_w,
                                  const float* outside_w, int rows, int C, const float* totals, float scale_cls, float scale_box,
                                  void* grad, int ld_g, float* loss, float* accuracy, void* stream) {
  DT_CHECK_ARG(rows >= 0 && C >= 2 && ld_o >= 5 * C && ld_g >= 5 * C, "dt_frcnn_loss_grad: bad shape rows=%d C=%d ld_o=%d ld_g=%d", rows, C, ld_o, ld_g);
  if (rows == 0) return 0;
  DT_CHECK_ARG(out && labels && targets && inside_w && outside_w && totals && grad, "dt_frcnn_loss_grad: null pointer");
  frcnn_loss_grad_kernel<<<(rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(out, ld_o, labels, targets, inside_w, outside_w, rows, 1, C,
                                                                             totals, scale_cls, scale_box, (__nv_bfloat16*)grad, ld_g, loss, accuracy);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_frcnn_tube_loss_grad(const float* out, int ld_o, const int* labels, const float* targets, const float* inside_w,
                                       const float* outside_w, int R, int T, int C, const float* totals, float scale_cls, float scale_box,
                                       void* grad, int ld_g, float* loss, float* accuracy, void* stream) {
  DT_CHECK_ARG(R >= 0 && T >= 1 && T <= DT_MAX_T && C >= 2 && ld_o >= 5 * C && ld_g >= 5 * C,
               "dt_frcnn_tube_loss_grad: bad shape R=%d T=%d C=%d ld_o=%d ld_g=%d", R, T, C, ld_o, ld_g);
  if (R == 0) return 0;
  DT_CHECK_ARG(out && labels && targets && inside_w && outside_w && totals && grad, "dt_frcnn_tube_loss_grad: null pointer");
  frcnn_loss_grad_kernel<<<(R + 127) / 128, 128, 0, (cudaStream_t)stream>>>(out, ld_o, labels, targets, inside_w, outside_w, R, T, C,
                                                                          totals, scale_cls, scale_box, (__nv_bfloat16*)grad, ld_g, loss, accuracy);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_rpn_tube_loss_grad(const float* out, int ld_o, const int* labels, const float* targets, const float* inside_w,
                                     const float* outside_w, int B, int T, int H, int W, int A, float scale_cls, float scale_box, float beta,
                                     float* normalizer, void* grad, int ld_g, float* loss, void* stream) {
  DT_CHECK_ARG(B >= 0 && T >= 1 && T <= DT_MAX_T && H >= 1 && W >= 1 && A >= 1 && ld_o >= 5 * A && ld_g >= 5 * A && beta > 0.f,
               "dt_rpn_tube_loss_grad: bad shape B=%d T=%d %dx%d A=%d ld_o=%d ld_g=%d", B, T, H, W, A, ld_o, ld_g);
  if (B == 0) return 0;
  DT_CHECK_ARG(out && labels && targets && inside_w && outside_w && normalizer && grad, "dt_rpn_tube_loss_grad: null pointer");
  const long long HW = (long long)H * W;
  label_count_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(labels, (long long)B * HW * A, normalizer);
  DT_CHECK_LAUNCH();
  rpn_tube_loss_grad_kernel<<<grid_for((long long)B * T * HW * ld_g, 256), 256, 0, (cudaStream_t)stream>>>(
      out, ld_o, labels, targets, inside_w, outside_w, B, T, HW, A, scale_cls, scale_box, beta, normalizer, (__nv_bfloat16*)grad, ld_g, loss);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_spatial_mean_bwd(const void* g, long long N, int H, int W, int C, const void* y, const float* scale, void* out,
                                   const float* scale2, void* out2, void* stream) {
  DT_CHECK_ARG(N >= 0 && H >= 1 && W >= 1 && C >= 8 && C % 8 == 0, "dt_spatial_mean_bwd: bad shape N=%lld %dx%d C=%d (C %% 8 == 0)", N, H, W, C);
  if (N == 0) return 0;
  DT_CHECK_ARG(g && out, "dt_spatial_mean_bwd: null pointer");
  spatial_mean_bwd_kernel<<<grid_for(N * H * W * (C / 8), 256), 256, 0, (cudaStream_t)stream>>>(
      (const __nv_bfloat16*)g, N, H * W, C, (const __nv_bfloat16*)y, scale, (__nv_bfloat16*)out, scale2, (__nv_bfloat16*)out2);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_kps_loss_grad(const float* low, int ld, int S, int K, int D, const int* locations, const float* weights,
                                const float* totals, float scale, void* grad, int ld_g, float* loss, void* stream) {
  DT_CHECK_ARG(S >= 1 && S <= 32 && K >= 1 && D >= 0 && ld >= 4 * K && ld_g >= 4 * K, "dt_kps_loss_grad: bad shape S=%d K=%d D=%d ld=%d ld_g=%d", S, K, D, ld, ld_g);
  if (D == 0) return 0;
  DT_CHECK_ARG(low && locations && weights && totals && grad, "dt_kps_loss_grad: null pointer");
  const size_t smem = (size_t)(4 * S * S + 16 * S * S) * sizeof(float);
  static DynSmemGrant grant;
  DT_CHECK_CUDA(grant_dyn_smem(kps_loss_grad_kernel, (int)smem, &grant));
  dim3 grid(D, K);
  kps_loss_grad_kernel<<<grid, 256, smem, (cudaStream_t)stream>>>(low, ld, S, K, locations, weights, totals, scale, (__nv_bfloat16*)grad, ld_g, loss);
  DT_CHECK_LAUNCH();
  return 0;
}

extern "C" int dt_subpixel_grad_fix(float* gW, float* gb, int K, int Cin, int ldc, void* stream) {
  DT_CHECK_ARG(K >= 1 && Cin >= 1 && ldc >= 4 * K, "dt_subpixel_grad_fix: bad shape K=%d Cin=%d ldc=%d", K, Cin, ldc);
  DT_CHECK_ARG(gW, "dt_subpixel_grad_fix: null pointer");
  subpixel_grad_fix_kernel<<<grid_for(9ll * ldc * Cin, 256), 256, 0, (cudaStream_t)stream>>>(gW, gb, K, Cin, ldc);
  DT_CHECK_LAUNCH();
  return 0;
}
