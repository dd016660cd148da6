// flmr_scan_plaid_kernel.cuh — the fused late-interaction scan over a corpus kept COMPRESSED in HBM (PLAID /
// ColBERTv2 residual codec: one centroid code + nbits per dimension per token, plus one fp32 inverse norm per
// token stored at corpus creation).  Results are bit-identical to decoding the index into bf16 first
// (flmr_plaid_decode) and scanning that with flmr_scan_kernel: the decode arithmetic below is the one
// flmr_plaid_decode_kernel uses, and every stage after the B-operand tile is the bf16 kernel's.
//
// Structure (one persistent CTA per SM, 16 warps; single-CTA passes only):
//   warps 0..7   : epilogue, two warpgroups — as flmr_scan_kernel.
//   warp 8       : reducer — as flmr_scan_kernel.
//   warp 9       : bulk-copy producer.  Streams each 96-token tile's codes, inverse norms and packed residuals
//                  (cp.async.bulk, no tensor map) through a ring of compressed stages in shared memory.
//   warps 10..11 : tcgen05.mma issuers — as flmr_scan_kernel (queries stationary in TMEM).
// The issuer, epilogue and reducer sections below are a copy of flmr_scan_kernel's (without its debug and CTA-pair
// branches): that kernel must stay byte-identical, so they cannot be shared.  A change there must be ported here;
// tests/test_plaid_resident_host.py pins flmr_scan_kernel.cuh's hash to flag it.
//   warps 12..15 : decoders.  Each turns 24 rows of a compressed stage into the 128B-swizzled bf16 B-operand
//                  D stage: bf16((centroid[code][i] + bucket_weight[idx]) * inv_norm), centroid rows from L2,
//                  bucket weights from shared memory; then fence.proxy.async (the MMA reads the stage through
//                  the async proxy) and one arrive per warp on the stage's "full" barrier.
//
// Row layout: the bf16 corpus' padded order (passages padded to a multiple of 4 rows by repeating the last
// token's code, residual and inverse norm), so the partition, the tile end masks, the pass plan, the reducer,
// the merge and the sharded exchange are the same.  The compressed arrays carry kTileN extra zero rows (code 0,
// inverse norm 0) so the last tile of the last CTA never reads past them; those rows decode to zeros and, as
// with the bf16 kernel's out-of-range rows, never reach a score (no passage ends after them).
#pragma once
#include <cuda_bf16.h>

#include "flmr_scan_kernel.cuh"

namespace flmr {

// ---- PLAID residual codec, shared by flmr_plaid_decode_kernel, the corpus packer, the gather and the scan ----
// Bucket index of the `pos`-th field of a packed residual byte (the reference packs each index LSB-first into
// big-endian bytes: residual.py:188-204 binarize, :51-73 reversed_bit_map).
__device__ __forceinline__ uint32_t plaid_bucket(uint32_t byte, int pos, int nbits) {
  const uint32_t field = (byte >> (8 - nbits * (pos + 1))) & ((1u << nbits) - 1u);
  return __brev(field) >> (32 - nbits);
}

// Un-normalised value of dims 4*lane .. 4*lane+3 of one token (one warp per token): centroid + bucket weight.
__device__ __forceinline__ void plaid_lane_values(const float4 c, const uint8_t* __restrict__ row,
                                                  const float* s_w, int nbits, int lane, float (&v)[4]) {
  const int keys = 8 / nbits;   // bucket indices per packed byte
  v[0] = c.x;
  v[1] = c.y;
  v[2] = c.z;
  v[3] = c.w;
#pragma unroll
  for (int dd = 0; dd < 4; ++dd) {
    const int i = 4 * lane + dd;
    v[dd] += s_w[plaid_bucket(__ldg(row + i / keys), i % keys, nbits)];
  }
}

// Warp-collective inverse L2 norm of the token whose dims the warp's lanes hold four at a time
// (torch.nn.functional.normalize, eps = 1e-12, as index_storage.py:173 applies it).
// The sum of squares is spelled out as the FMA chain nvcc made of `v0*v0 + v1*v1 + v2*v2 + v3*v3` in the decode
// kernel, so no call site is left to a contraction choice of its own.
__device__ __forceinline__ float plaid_inv_norm(const float (&v)[4]) {
  float ss = __fmaf_rn(v[3], v[3], __fmaf_rn(v[2], v[2], __fmaf_rn(v[0], v[0], __fmul_rn(v[1], v[1]))));
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
  return 1.0f / fmaxf(sqrtf(ss), 1e-12f);
}

// One decoded, normalised dim before bf16 rounding.
__device__ __forceinline__ float plaid_value(float centroid, float weight, float inv) {
  return __fmul_rn(__fadd_rn(centroid, weight), inv);
}

// ---- bulk copies + proxy fence (not in flmr_device.cuh, which the bf16 kernels share unchanged) ----
__device__ __forceinline__ void bulk_load(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar,
                                          uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

struct PlaidParams {
  const int32_t* codes;       // [n_rows + kTileN] padded order
  const uint8_t* residuals;   // [n_rows + kTileN][16 * nbits]
  const float* inv_norm;      // [n_rows + kTileN]
  const float* centroids;     // [n_centroids][128]
  const float* weights;       // [2^nbits]
};

constexpr int kDecWarps = 4;                       // warps 12..15
constexpr int kWarpDec = kWarpMma + kMmaWarps;     // 12
constexpr int kPlaidThreads = (kWarpDec + kDecWarps) * 32;   // 512
constexpr int kDecRows = kTileN / kDecWarps;       // 24 rows of every tile per decode warp
constexpr int kPDStages = 4;                       // bf16 D stages (the bf16 kernel has 7: filled from L2 there)
static_assert(kTileN % kDecWarps == 0 && (kDecRows * 16) % 32 == 0, "decode split");

template <int NBITS>
struct PlaidSmem {
  static constexpr int kResBytes = kTileN * 16 * NBITS;                 // packed residuals of one tile
  static constexpr int kCStageBytes = kTileN * 8 + kResBytes;           // codes + inverse norms + residuals
  static constexpr int kOffD = 0;
  static constexpr int kOffPartial = kOffD + kPDStages * kDTileBytes;
  static constexpr int kOffLanePart = kOffPartial + ScanSmem::kPartialBytes;
  static constexpr int kOffKeys = kOffLanePart + ScanSmem::kLanePartBytes;
  static constexpr int kOffMinKey = kOffKeys + ScanSmem::kKeysBytes;
  static constexpr int kOffMinPos = kOffMinKey + kNqMax * 8;
  static constexpr int kOffCarry = kOffMinPos + kNqMax * 4;
  static constexpr int kOffW = kOffCarry + kMtMax * kTileM * 4;         // float[256] bucket weights
  static constexpr int kOffC = (kOffW + 256 * 4 + 127) / 128 * 128;     // compressed ring
  static constexpr int kFixed = kOffC + 1024 + 16 + 8 * (1 + 2 * kPDStages + 2 * kMaxAccStages + 4 + kMtMax * 4);
  // as many compressed stages as fit (each bar pair 16 B), at most 8
  static constexpr int kCStagesFit = (232448 - kFixed) / (kCStageBytes + 16);
  static constexpr int kCStages = kCStagesFit > 8 ? 8 : kCStagesFit;
  static constexpr int kOffBars = kOffC + kCStages * kCStageBytes;
  static constexpr int kNumBars = 1 + 2 * kPDStages + 2 * kMaxAccStages + 4 + kMtMax * 4 + 2 * kCStages;
  static constexpr int kOffTmemPtr = kOffBars + kNumBars * 8;
  static constexpr int kBytes = kOffTmemPtr + 16 + 1024;
  static_assert(kCStages >= 2, "compressed ring needs two stages");
  static_assert(kBytes <= 232448, "exceeds 227 KiB of shared memory per CTA");
};

template <int NBITS>
__global__ void __launch_bounds__(kPlaidThreads, 1)
flmr_scan_plaid_kernel(const __grid_constant__ ScanParams p, const __grid_constant__ PlaidParams q) {
  using S = PlaidSmem<NBITS>;
  constexpr int kCStages = S::kCStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t smem_base = smem_u32(smem);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cta = static_cast<int>(blockIdx.x);

  const uint32_t bar_base = smem_base + S::kOffBars;
  const uint32_t bar_q_full = bar_base;
  auto bar_d_full = [&](int s) { return bar_base + 8u * (1 + s); };
  auto bar_d_empty = [&](int s) { return bar_base + 8u * (1 + kPDStages + s); };
  auto bar_t_full = [&](int s) { return bar_base + 8u * (1 + 2 * kPDStages + s); };
  auto bar_t_empty = [&](int s) { return bar_base + 8u * (1 + 2 * kPDStages + kMaxAccStages + s); };
  auto bar_p_full = [&](int b) { return bar_base + 8u * (1 + 2 * kPDStages + 2 * kMaxAccStages + b); };
  auto bar_p_empty = [&](int b) { return bar_base + 8u * (1 + 2 * kPDStages + 2 * kMaxAccStages + 2 + b); };
  auto bar_carry = [&](int mt, int quad) {
    return bar_base + 8u * (1 + 2 * kPDStages + 2 * kMaxAccStages + 4 + mt * 4 + quad);
  };
  constexpr int kBarC = 1 + 2 * kPDStages + 2 * kMaxAccStages + 4 + kMtMax * 4;
  auto bar_c_full = [&](int s) { return bar_base + 8u * (kBarC + s); };
  auto bar_c_empty = [&](int s) { return bar_base + 8u * (kBarC + kCStages + s); };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + S::kOffTmemPtr);

  const int32_t row_begin = p.cta_row_begin[cta];
  const int64_t tile_base = p.cta_tile_base[cta];
  const int n_tiles = static_cast<int>(p.cta_tile_base[cta + 1] - tile_base);
  const int n_mtiles = p.n_mtiles;
  const uint32_t acc_stages = static_cast<uint32_t>(scan_acc_stages(n_mtiles));
  const uint32_t stage_mask = acc_stages - 1u, stage_shift = (acc_stages == 4u) ? 2u : 1u;
  const uint32_t acc_col0 = static_cast<uint32_t>(kQCols * n_mtiles);

  // ---- one-time setup --------------------------------------------------------------------------
  if (warp == kWarpProducer && lane == 0) {
    mbar_init(bar_q_full, 4);
    for (int s = 0; s < kPDStages; ++s) {
      mbar_init(bar_d_full(s), kDecWarps);   // one arrive per decode warp
      mbar_init(bar_d_empty(s), kMmaWarps);
    }
    for (int s = 0; s < kCStages; ++s) {
      mbar_init(bar_c_full(s), 1);
      mbar_init(bar_c_empty(s), kDecWarps);
    }
    for (int s = 0; s < kMaxAccStages; ++s) {
      mbar_init(bar_t_full(s), 1);
      mbar_init(bar_t_empty(s), 4);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(bar_p_full(b), kEpiWarps);
      mbar_init(bar_p_empty(b), kRedWarps);
    }
    for (int i = 0; i < kMtMax * 4; ++i) mbar_init(bar_carry(i >> 2, i & 3), 1);
    mbar_fence_init();
  }
  if (warp == kWarpMma) tmem_alloc<512>(smem_base + S::kOffTmemPtr);
  if (warp < kWarpProducer) {
    const int et = threadIdx.x;
    constexpr int kInitThreads = kEpiThreads + kRedWarps * 32;
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem + S::kOffKeys);
    for (int i = et; i < kNqMax * kMaxK; i += kInitThreads) keys[i] = 0ull;
    if (et < kNqMax) {
      reinterpret_cast<uint64_t*>(smem + S::kOffMinKey)[et] = 0ull;
      reinterpret_cast<int*>(smem + S::kOffMinPos)[et] = 0;
    }
    float* carry0 = reinterpret_cast<float*>(smem + S::kOffCarry);
    for (int i = et; i < kMtMax * kTileM; i += kInitThreads) carry0[i] = p.init_val;
  }
  if (warp >= kWarpDec) {
    float* s_w = reinterpret_cast<float*>(smem + S::kOffW);
    for (int i = threadIdx.x - kWarpDec * 32; i < (1 << NBITS); i += kDecWarps * 32) s_w[i] = q.weights[i];
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == kWarpProducer) {
    // ===================== bulk-copy producer =====================
    for (int t = 0; t < n_tiles; ++t) {
      const int s = t % kCStages;
      const uint32_t ph = (t / kCStages) & 1;
      mbar_wait(bar_c_empty(s), ph ^ 1u, p.status, kDevTimeoutProducer);
      if (elect_one_sync()) {
        mbar_arrive_expect_tx(bar_c_full(s), S::kCStageBytes);
        const uint32_t dst = smem_base + S::kOffC + s * S::kCStageBytes;
        const int64_t row = static_cast<int64_t>(row_begin) + static_cast<int64_t>(t) * kTileN;
        bulk_load(dst, q.codes + row, kTileN * 4, bar_c_full(s), kPolicyEvictFirst);
        bulk_load(dst + kTileN * 4, q.inv_norm + row, kTileN * 4, bar_c_full(s), kPolicyEvictFirst);
        bulk_load(dst + kTileN * 8, q.residuals + row * (16 * NBITS), S::kResBytes, bar_c_full(s),
                  kPolicyEvictFirst);
      }
      __syncwarp();
    }
  } else if (warp >= kWarpDec) {
    // ===================== decoders =====================
    // Lane item i (12 per lane per tile) = (row, 16-byte chunk) of this warp's 24 rows: 8 dims, i.e. NBITS bytes
    // of packed residual, two float4 of the centroid row, one 16-byte swizzled store into the D stage.
    const int dw = warp - kWarpDec;
    const float* s_w = reinterpret_cast<const float*>(smem + S::kOffW);
    constexpr int kKeys = 8 / NBITS;
    for (int t = 0; t < n_tiles; ++t) {
      const int cs = t % kCStages;
      const uint32_t cph = (t / kCStages) & 1;
      const int ds = t % kPDStages;
      const uint32_t dph = (t / kPDStages) & 1;
      mbar_wait(bar_c_full(cs), cph, p.status, kDevTimeoutProducer);
      mbar_wait(bar_d_empty(ds), dph ^ 1u, p.status, kDevTimeoutProducer);
      const uint8_t* cst = smem + S::kOffC + cs * S::kCStageBytes;
      const int32_t* s_codes = reinterpret_cast<const int32_t*>(cst);
      const float* s_inv = reinterpret_cast<const float*>(cst + kTileN * 4);
      const uint8_t* s_res = cst + kTileN * 8;
      uint8_t* dstage = smem + S::kOffD + ds * kDTileBytes;
#pragma unroll 2
      for (int it = 0; it < kDecRows * 16 / 32; ++it) {
        const int item = it * 32 + lane;
        const int r = dw * kDecRows + (item >> 4);
        const int j = item & 15;                        // 16-byte chunk: dims 8j .. 8j+7
        const int32_t code = s_codes[r];
        const float inv = s_inv[r];
        const float4* crow = reinterpret_cast<const float4*>(q.centroids + static_cast<int64_t>(code) * kDim + 8 * j);
        const float4 c0 = __ldg(crow), c1 = __ldg(crow + 1);
        uint64_t word;
        if constexpr (NBITS == 8) word = *reinterpret_cast<const uint64_t*>(s_res + r * 128 + j * 8);
        else if constexpr (NBITS == 4) word = *reinterpret_cast<const uint32_t*>(s_res + r * 64 + j * 4);
        else if constexpr (NBITS == 2) word = *reinterpret_cast<const uint16_t*>(s_res + r * 32 + j * 2);
        else word = s_res[r * 16 + j];
        const float c[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
        float v[8];
#pragma unroll
        for (int dd = 0; dd < 8; ++dd) {
          const uint32_t byte = static_cast<uint32_t>(word >> (8 * (dd / kKeys))) & 0xFFu;
          v[dd] = plaid_value(c[dd], s_w[plaid_bucket(byte, dd % kKeys, NBITS)], inv);
        }
        uint32_t w[4];
#pragma unroll
        for (int h = 0; h < 4; ++h) {
          __nv_bfloat162 b2 = __floats2bfloat162_rn(v[2 * h], v[2 * h + 1]);
          w[h] = *reinterpret_cast<uint32_t*>(&b2);
        }
        // 128B swizzle (as the TMA writes it): chunk jj of row r sits at chunk jj ^ (r & 7) of its 128-B row
        const int kb = j >> 3, jj = j & 7;
        *reinterpret_cast<uint4*>(dstage + kb * kDKBlockBytes + r * 128 + ((jj ^ (r & 7)) << 4)) =
            make_uint4(w[0], w[1], w[2], w[3]);
      }
      fence_proxy_async_smem();   // generic-proxy stores -> visible to tcgen05.mma (async proxy)
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar_d_full(ds));
        mbar_arrive(bar_c_empty(cs));
      }
    }
  } else if (warp >= kWarpMma) {
    // ===================== MMA issuers (as flmr_scan_kernel) =====================
    const uint32_t iw = static_cast<uint32_t>(warp - kWarpMma);
    constexpr uint32_t idesc = make_idesc_bf16_f32(kTileM, kTileN);
    mbar_wait(bar_q_full, 0, p.status, kDevTimeoutMma);
    tc_fence_after_sync();
    for (int t = 0; t < n_tiles; ++t) {
      const int s = t % kPDStages;
      const uint32_t ph = (t / kPDStages) & 1;
      mbar_wait(bar_d_full(s), ph, p.status, kDevTimeoutMma);
      tc_fence_after_sync();
      const uint64_t b_desc0 = make_kmajor_sw128_desc(smem_base + S::kOffD + s * kDTileBytes);
      const uint32_t a_first = static_cast<uint32_t>(t) * n_mtiles;
      const bool rot = ((n_mtiles & t) & 1) != 0;
#pragma unroll 1
      for (uint32_t a = a_first + ((a_first ^ iw) & 1u); a < a_first + n_mtiles; a += 2) {
        const uint32_t j = a - a_first;
        const uint32_t mt = rot ? (j == 0 ? static_cast<uint32_t>(n_mtiles) - 1u : j - 1u) : j;
        const uint32_t as = a & stage_mask, aph = (a >> stage_shift) & 1u;
        mbar_wait(bar_t_empty(as), aph ^ 1u, p.status, kDevTimeoutMma);
        tc_fence_after_sync();
        const uint32_t d_tmem = tmem_base + acc_col0 + as * kTileN;
        const uint32_t a_tmem = tmem_base + mt * kQCols;
        if (elect_one_sync()) {
#pragma unroll
          for (int k = 0; k < kDim / 16; ++k) {
            const uint64_t b_desc =
                b_desc0 + static_cast<uint64_t>(((k >> 2) * kDKBlockBytes + (k & 3) * 32) >> 4);
            tc_mma_ts(d_tmem, a_tmem + k * 8, b_desc, idesc, k > 0 ? 1u : 0u);
          }
          tc_commit(bar_t_full(as));
        }
        __syncwarp();
      }
      if (elect_one_sync()) tc_commit(bar_d_empty(s));
      __syncwarp();
    }
  } else if (warp < kEpiWarps) {
    // ===================== epilogue (as flmr_scan_kernel) =====================
    const int wg = warp >> 2;
    const int quad = warp & 3;
    const uint32_t lane_base = static_cast<uint32_t>(quad * 32) << 16;
    float* partial = reinterpret_cast<float*>(smem + S::kOffPartial);
    float* lane_part = reinterpret_cast<float*>(smem + S::kOffLanePart) + lane;
    float* carry = reinterpret_cast<float*>(smem + S::kOffCarry) + quad * 32 + lane;
    const bool carry_crosses = (n_mtiles & 1) != 0;
    const float init = p.init_val;

    if (wg == 0) {
      for (int mt = 0; mt < n_mtiles; ++mt) {
        const uint4* src = p.q_pad + (static_cast<int64_t>(mt) * kTileM + quad * 32 + lane) * 16;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          uint32_t w[32];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const uint4 x = __ldg(src + h * 8 + i);
            w[4 * i] = x.x;
            w[4 * i + 1] = x.y;
            w[4 * i + 2] = x.z;
            w[4 * i + 3] = x.w;
          }
          FLMR_TMEM_ST32(tmem_base + lane_base + mt * kQCols + h * 32, w);
        }
      }
      tmem_wait_st();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_q_full);
    }

    uint32_t mask_next = (n_tiles > 0) ? __ldg(p.tile_end_mask + tile_base) : 0u;
    for (int t = 0; t < n_tiles; ++t) {
      const uint32_t mask = mask_next;
      if (t + 1 < n_tiles) mask_next = __ldg(p.tile_end_mask + tile_base + t + 1);
      const int buf = t & 1;
      mbar_wait(bar_p_empty(buf), ((static_cast<uint32_t>(t) >> 1) & 1u) ^ 1u, p.status, kDevTimeoutEpilogue);
      const uint32_t a_first = static_cast<uint32_t>(t) * n_mtiles;
      const bool rot = ((n_mtiles & t) & 1) != 0;
#pragma unroll 1
      for (uint32_t a = a_first + ((a_first ^ static_cast<uint32_t>(wg)) & 1u); a < a_first + n_mtiles; a += 2) {
        const int j = static_cast<int>(a - a_first);
        const int mt = rot ? (j == 0 ? n_mtiles - 1 : j - 1) : j;
        const bool crosses = carry_crosses && mt == n_mtiles - 1;
        const uint32_t as = a & stage_mask, aph = (a >> stage_shift) & 1u;
        if (crosses && t > 0)
          mbar_wait(bar_carry(mt, quad), static_cast<uint32_t>(t - 1) & 1u, p.status, kDevTimeoutEpilogue);
        float m = carry[mt * kTileM];
        mbar_wait(bar_t_full(as), aph, p.status, kDevTimeoutEpilogue);
        tc_fence_after_sync();
        {
          const uint32_t taddr = tmem_base + lane_base + acc_col0 + as * kTileN;
          uint32_t v[kChunks][32];
          float* partial_rb = partial + (buf * kRbMax + mt * 4 + quad) * kSlots;
          float* lane_part_rb = lane_part + ((buf * kFastSlots) * kRbMax + mt * 4 + quad) * kLaneStride;
          int slot = 0;
          FLMR_TMEM_LD32(v[0], taddr);
          FLMR_TMEM_WAIT_LD32(v[0]);
#pragma unroll
          for (int c = 1; c < kChunks; ++c) FLMR_TMEM_LD32(v[c], taddr + 32 * c);
          process_chunk(v[0], mask & 0xFFu, m, init, partial_rb, lane_part_rb, slot, lane);
#pragma unroll
          for (int c = 1; c < kChunks; ++c) FLMR_TMEM_WAIT_LD32(v[c]);
          tc_fence_before_sync();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_t_empty(as));
#pragma unroll
          for (int c = 1; c < kChunks; ++c)
            process_chunk(v[c], (mask >> (8 * c)) & 0xFFu, m, init, partial_rb, lane_part_rb, slot, lane);
        }
        carry[mt * kTileM] = m;
        if (crosses) {
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_carry(mt, quad));
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_p_full(buf));
    }
    tc_fence_before_sync();
  } else {
    // ===================== reducer (as flmr_scan_kernel) =====================
    const float* partial = reinterpret_cast<const float*>(smem + S::kOffPartial);
    uint64_t* keys = reinterpret_cast<uint64_t*>(smem + S::kOffKeys);
    uint64_t* minkey_s = reinterpret_cast<uint64_t*>(smem + S::kOffMinKey);
    int* minpos_s = reinterpret_cast<int*>(smem + S::kOffMinPos);
    uint32_t mask_next = 0;
    int32_t fpid_next = 0;
    if (n_tiles > 0) {
      mask_next = __ldg(p.tile_end_mask + tile_base);
      fpid_next = __ldg(p.tile_first_pid + tile_base);
    }
    for (int t = 0; t < n_tiles; ++t) {
      const uint32_t mask = mask_next;
      const int32_t first_pid = fpid_next;
      if (t + 1 < n_tiles) {
        mask_next = __ldg(p.tile_end_mask + tile_base + t + 1);
        fpid_next = __ldg(p.tile_first_pid + tile_base + t + 1);
      }
      const int buf = t & 1;
      mbar_wait(bar_p_full(buf), (static_cast<uint32_t>(t) >> 1) & 1u, p.status, kDevTimeoutEpilogue);
      const int n_slots = __popc(mask);
      const float* lane_part0 = reinterpret_cast<const float*>(smem + S::kOffLanePart);
#pragma unroll 1
      for (int slot = 0; slot < n_slots; ++slot) {
        const int64_t pid = static_cast<int64_t>(first_pid) + slot;
        const float* lp_slot = lane_part0 + ((buf * kFastSlots + slot) * kRbMax) * kLaneStride;
        if (slot < kFastSlots && p.rbq <= p.lane_mode_max_rbq) {
#pragma unroll 1
          for (int b0 = 0; b0 < p.nq_pass; b0 += 32) {
            const int b = b0 + lane;
            const bool valid = b < p.nq_pass;
            float sc = 0.f;
            uint64_t key = 0ull;
            if (valid) {
              const float* lp = lp_slot + (b * p.rbq) * kLaneStride;
              for (int r = 0; r < p.rbq; ++r) {
#pragma unroll 8
                for (int j = 0; j < 32; ++j) sc += lp[r * kLaneStride + j];
              }
              const int64_t gi = static_cast<int64_t>(b) * p.n_passages + pid;
              if (p.acc_in) sc += __ldg(p.acc_in + gi);
              if (p.acc_out) p.acc_out[gi] = sc;
              key = (static_cast<uint64_t>(float_to_ordered(sc)) << 32) |
                    static_cast<uint64_t>(0xFFFFFFFFu - static_cast<uint32_t>(pid));
            }
            if (p.k > 0) {
              uint32_t hits = __ballot_sync(0xffffffffu, valid && key > minkey_s[valid ? b : 0]);
              while (hits) {
                const int src = __ffs(hits) - 1;
                hits &= hits - 1;
                const uint64_t cand = shfl64(key, src);
                const int cb = b0 + src;
                uint64_t minkey = minkey_s[cb];
                int minpos = minpos_s[cb];
                if (cand > minkey) {
                  topk_replace_min(keys + cb * kMaxK, p.k, cand, minkey, minpos, lane);
                  if (lane == 0) {
                    minkey_s[cb] = minkey;
                    minpos_s[cb] = minpos;
                  }
                  __syncwarp();
                }
              }
            }
          }
        } else {
#pragma unroll 1
          for (int b = 0; b < p.nq_pass; ++b) {
            float sc = 0.f;
            if (slot < kFastSlots) {
              const float* lp = lp_slot + (b * p.rbq) * kLaneStride + lane;
#pragma unroll 2
              for (int r = 0; r < p.rbq; ++r) sc += lp[r * kLaneStride];
              sc = warp_sum(sc);
            } else {
              const float* pr = partial + (buf * kRbMax + b * p.rbq) * kSlots + slot;
#pragma unroll 2
              for (int r = 0; r < p.rbq; ++r) sc += pr[r * kSlots];
            }
            const int64_t gi = static_cast<int64_t>(b) * p.n_passages + pid;
            if (p.acc_in) sc += __ldg(p.acc_in + gi);
            if (p.acc_out && lane == 0) p.acc_out[gi] = sc;
            if (p.k > 0) {
              const uint64_t key = (static_cast<uint64_t>(float_to_ordered(sc)) << 32) |
                                   static_cast<uint64_t>(0xFFFFFFFFu - static_cast<uint32_t>(pid));
              uint64_t minkey = minkey_s[b];
              if (key > minkey) {
                int minpos = minpos_s[b];
                topk_replace_min(keys + b * kMaxK, p.k, key, minkey, minpos, lane);
                if (lane == 0) {
                  minkey_s[b] = minkey;
                  minpos_s[b] = minpos;
                }
                __syncwarp();
              }
            }
          }
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_p_empty(buf));
    }
    if (p.k > 0) {
      __syncwarp();
      for (int b = 0; b < p.nq_pass; ++b) {
        uint64_t* dst = p.cand_keys + (static_cast<int64_t>(cta) * p.cand_q_stride + p.cand_q_first + b) * p.k;
        for (int i = lane; i < p.k; i += 32) dst[i] = keys[b * kMaxK + i];
      }
    }
  }

  // ---- teardown -----------------------------------------------------------------------------------
  __syncthreads();
  if (warp == kWarpMma) {
    tc_fence_after_sync();
    tmem_dealloc<512>(tmem_base);
  }
}

// ---- helper kernels of the compressed corpus --------------------------------------------------------------

// Corpus creation, one chunk of whole passages at a time: passages [p_begin, p_begin + p_count), whose packed source
// rows start at row src_row_base of the global packed order (soff) and sit at `codes` / `residuals` row 0, go to
// rows poff[p] .. poff[p+1] of the padded layout, the last token repeated over the padding rows; every row also gets
// its inverse norm, computed exactly as flmr_plaid_decode_kernel normalises.  A code outside [0, n_centroids) sets
// *bad_code and its row is left as code 0 / inverse norm 0 (the creation then fails).  One warp per passage.
__global__ void flmr_plaid_pack_kernel(const int32_t* __restrict__ codes, const uint8_t* __restrict__ residuals,
                                       const int64_t* __restrict__ soff, const int64_t* __restrict__ poff,
                                       int64_t p_begin, int64_t p_count, int64_t src_row_base,
                                       const float* __restrict__ centroids, int64_t n_centroids,
                                       const float* __restrict__ bucket_weights, int nbits,
                                       int32_t* __restrict__ out_codes, uint8_t* __restrict__ out_residuals,
                                       float* __restrict__ out_inv, int* __restrict__ bad_code) {
  __shared__ float s_w[256];
  for (int i = threadIdx.x; i < (1 << nbits); i += blockDim.x) s_w[i] = bucket_weights[i];
  __syncthreads();
  const int64_t w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= p_count) return;
  const int64_t p = p_begin + w;
  const int packed = kDim * nbits / 8;
  const int64_t s0 = soff[p] - src_row_base, len = soff[p + 1] - soff[p];
  const int64_t d0 = poff[p], plen = poff[p + 1] - d0;
  for (int64_t j = 0; j < plen; ++j) {
    const int64_t t = s0 + (j < len ? j : len - 1);
    const int64_t d = d0 + j;
    const int32_t code = codes[t];
    const uint8_t* row = residuals + t * packed;
    for (int b = lane; b < packed; b += 32) out_residuals[d * packed + b] = row[b];
    if (code < 0 || code >= n_centroids) {
      if (lane == 0) {
        out_codes[d] = 0;
        out_inv[d] = 0.f;
        *bad_code = 1;
      }
      continue;
    }
    const float4 c = __ldg(reinterpret_cast<const float4*>(centroids + static_cast<int64_t>(code) * kDim) + lane);
    float v[4];
    plaid_lane_values(c, row, s_w, nbits, lane, v);
    const float inv = plaid_inv_norm(v);
    if (lane == 0) {
      out_codes[d] = code;
      out_inv[d] = inv;
    }
  }
}

// flmr_corpus_gather on a compressed corpus: decode the requested rows (one warp per output row, lane = 4 dims).
__global__ void flmr_gather_plaid_kernel(const int32_t* __restrict__ codes, const uint8_t* __restrict__ residuals,
                                         const float* __restrict__ inv_norm, const float* __restrict__ centroids,
                                         const float* __restrict__ bucket_weights, int nbits,
                                         const int64_t* __restrict__ poff, const int32_t* __restrict__ doclen,
                                         const int64_t* __restrict__ pids, int64_t n_pids, int nd_max,
                                         int64_t n_passages, int64_t pid_base, uint2* __restrict__ out,
                                         uint8_t* __restrict__ mask) {
  __shared__ float s_w[256];
  for (int i = threadIdx.x; i < (1 << nbits); i += blockDim.x) s_w[i] = bucket_weights[i];
  __syncthreads();
  const int64_t w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= n_pids * nd_max) return;
  const int64_t slot = w / nd_max;
  const int j = static_cast<int>(w % nd_max);
  const int64_t p = pids[slot] - pid_base;
  uint2 o = make_uint2(0u, 0u);
  bool real = false;
  if (p >= 0 && p < n_passages && j < doclen[p]) {
    const int64_t r = poff[p] + j;
    const int keys = 8 / nbits;
    const float inv = inv_norm[r];
    const float4 c = __ldg(reinterpret_cast<const float4*>(centroids + static_cast<int64_t>(codes[r]) * kDim) + lane);
    const uint8_t* row = residuals + r * (kDim * nbits / 8);
    const float cc[4] = {c.x, c.y, c.z, c.w};
    float v[4];
#pragma unroll
    for (int dd = 0; dd < 4; ++dd) {
      const int i = 4 * lane + dd;
      v[dd] = plaid_value(cc[dd], s_w[plaid_bucket(__ldg(row + i / keys), i % keys, nbits)], inv);
    }
    __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]);
    __nv_bfloat162 hi = __floats2bfloat162_rn(v[2], v[3]);
    o.x = *reinterpret_cast<uint32_t*>(&lo);
    o.y = *reinterpret_cast<uint32_t*>(&hi);
    real = true;
  }
  out[w * 32 + lane] = o;
  if (mask && lane == 0) mask[w] = real ? 1 : 0;
}

}  // namespace flmr
