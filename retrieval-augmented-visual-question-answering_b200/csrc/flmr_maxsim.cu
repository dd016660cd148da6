// flmr_maxsim.cu — C-ABI implementation (include/flmr_maxsim.h) of the B200-native FLMR/ColBERT
// MaxSim + top-k path.  Host logic: corpus residency + partition metadata, query staging, pass
// planning, launches.  Device code: the fused scan kernel (flmr_scan_kernel.cuh) plus four small
// helper kernels (query staging, candidate merge, corpus repack, SIMT cross-check).
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
// No libcuda link dependency: cuTensorMapEncodeTiled is resolved through the runtime's
// cudaGetDriverEntryPoint, so the library loads (and its symbols can be checked) without a GPU.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <limits>
#include <mutex>
#include <new>
#include <cerrno>
#include <ctime>
#include <string>
#include <thread>
#include <vector>

#include "../../include/flmr_maxsim.h"
#include "flmr_scan_kernel.cuh"
#include "flmr_scan_plaid_kernel.cuh"
#include "flmr_scan3_kernel.cuh"
#include "flmr_train_kernels.cuh"
#include "flmr_train_tc_kernel.cuh"

namespace {

using namespace flmr;

static_assert(kMaxK == FLMR_MAX_K, "header / kernel top-k capacity mismatch");
static_assert(kGroup == FLMR_TOKEN_GROUP, "header / kernel token group mismatch");
static_assert(kDim == FLMR_DIM, "header / kernel dim mismatch");

// ---- error plumbing -----------------------------------------------------------------------------
thread_local std::string g_last_error;
thread_local int64_t g_launches = 0;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define FLMR_CUDA(expr)                                                                     \
  do {                                                                                      \
    cudaError_t e__ = (expr);                                                               \
    if (e__ != cudaSuccess)                                                                 \
      return fail(e__ == cudaErrorMemoryAllocation ? FLMR_ERR_OOM : FLMR_ERR_CUDA,          \
                  "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = false;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) return;
    ok = (cudaSetDevice(dev) == cudaSuccess);
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// ---- TMA descriptor encoding through the runtime-resolved driver entry point ------------------------
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                   const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                   const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int get_encode_fn(EncodeTiledFn* out) {
  static EncodeTiledFn fn = nullptr;
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    FLMR_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || !p)
      return fail(FLMR_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  *out = fn;
  return FLMR_OK;
}

// bf16 [rows, 128] row-major matrix, box = 64 columns (128 B, one swizzle span) x box_rows rows.
int encode_rows_map(CUtensorMap* map, const void* base, uint64_t rows, uint32_t box_rows) {
  EncodeTiledFn enc = nullptr;
  int rc = get_encode_fn(&enc);
  if (rc) return rc;
  const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(kDim), static_cast<cuuint64_t>(rows)};
  const cuuint64_t gstride[1] = {static_cast<cuuint64_t>(kDim) * 2};
  const cuuint32_t box[2] = {64u, box_rows};
  const cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride,
                   box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(FLMR_ERR_CUDA, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
  return FLMR_OK;
}

// ---- helper kernels --------------------------------------------------------------------------------

// Stage the resident queries of EVERY pass of a call in one launch (blockIdx.y = pass): each query padded
// with zero rows to rbq*32 rows, the pass's block padded with zero rows to n_mtiles*128 rows, pass i at
// qpad + i * kMtMax*128 rows.  One thread per 16 bytes.
constexpr int kStageMaxPasses = 64;
struct StagePass {
  int32_t q_first, n_q, row0, rows, rbq, n_rows_pad;
};
struct StageParams {
  StagePass pass[kStageMaxPasses];
};
__global__ void flmr_stage_queries_kernel(const uint4* __restrict__ q, uint4* __restrict__ qpad,
                                          int nq_total_rows, const __grid_constant__ StageParams sp) {
  const StagePass& ps = sp.pass[blockIdx.y];
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = idx >> 4, c = idx & 15;
  if (r >= ps.n_rows_pad) return;
  const int rows_q = ps.rbq * 32;
  const int b = r / rows_q, i = r % rows_q;
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  if (b < ps.n_q && i < ps.rows)
    v = q[(static_cast<int64_t>(ps.q_first + b) * nq_total_rows + ps.row0 + i) * 16 + c];
  qpad[static_cast<int64_t>(blockIdx.y) * (kMtMax * kTileM * 16) + idx] = v;
}

// Copy passages into the padded layout: passage p occupies rows [poff[p], poff[p+1]) of dst, its
// last token repeated over the padding rows.  One warp per passage, 2 rows per iteration.
__global__ void flmr_repack_kernel(const uint4* __restrict__ src, const int64_t* __restrict__ soff,
                                   const int64_t* __restrict__ poff, uint4* __restrict__ dst,
                                   int64_t p_begin, int64_t p_count, int64_t src_row_base) {
  const int64_t w = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= p_count) return;
  const int64_t p = p_begin + w;
  const int64_t s0 = soff[p], len = soff[p + 1] - s0;
  const int64_t d0 = poff[p], plen = poff[p + 1] - d0;
  const int half = lane >> 4, c = lane & 15;
  for (int64_t j = half; j < plen; j += 2) {
    const int64_t sj = j < len ? j : len - 1;
    dst[(d0 + j) * 16 + c] = src[(s0 - src_row_base + sj) * 16 + c];
  }
}

// Streamed corpus load: rows [s0, s0 + n) of the PACKED source order (staged at `src`) go to their place in the
// padded layout; the last token of a passage is also copied over its padding rows.  Chunks need not start or end
// on passage boundaries.  One half-warp per row; the passage of a row is found by binary search in `soff`.
__global__ void flmr_scatter_rows_kernel(const uint4* __restrict__ src, const int64_t* __restrict__ soff,
                                         const int64_t* __restrict__ poff, uint4* __restrict__ dst,
                                         int64_t s0, int64_t n, int64_t n_passages) {
  const int64_t r = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 4;
  const int c = threadIdx.x & 15;
  if (r >= n) return;
  const int64_t srow = s0 + r;
  int64_t lo = 0, hi = n_passages;          // largest p with soff[p] <= srow
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (soff[mid] <= srow) lo = mid; else hi = mid;
  }
  const uint4 v = src[r * 16 + c];
  const int64_t d = poff[lo] + (srow - soff[lo]);
  dst[d * 16 + c] = v;
  if (srow == soff[lo + 1] - 1)             // last token: fill the group padding with copies
    for (int64_t j = d + 1; j < poff[lo + 1]; ++j) dst[j * 16 + c] = v;
}

// Independent plain-SIMT MaxSim (test infrastructure): one block per (passage, query), one thread
// per query token (looping if nq > blockDim), fp32 FMA over bf16 inputs, fixed-order block sum.
__global__ void flmr_simt_maxsim_kernel(const __nv_bfloat16* __restrict__ d, const int64_t* poff,
                                        const int32_t* doclen, const __nv_bfloat16* __restrict__ q,
                                        int nq, float init, float* __restrict__ out,
                                        int64_t n_passages) {
  __shared__ float drow[kDim];
  __shared__ float red[256];
  const int64_t p = blockIdx.x;
  const int b = blockIdx.y;
  const int len = doclen[p];
  const __nv_bfloat16* dp = d + poff[p] * kDim;
  float total = 0.f;
  for (int i0 = 0; i0 < nq; i0 += blockDim.x) {
    const int i = i0 + threadIdx.x;
    float m = init;
    const __nv_bfloat16* qi = q + (static_cast<int64_t>(b) * nq + (i < nq ? i : 0)) * kDim;
    for (int j = 0; j < len; ++j) {
      __syncthreads();
      if (threadIdx.x < kDim) drow[threadIdx.x] = __bfloat162float(dp[j * kDim + threadIdx.x]);
      __syncthreads();
      float acc = 0.f;
#pragma unroll 16
      for (int c = 0; c < kDim; ++c) acc = fmaf(__bfloat162float(qi[c]), drow[c], acc);
      m = fmaxf(m, acc);
    }
    if (i < nq) total += m;
  }
  red[threadIdx.x] = total;
  __syncthreads();
  for (int s = blockDim.x / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[static_cast<int64_t>(b) * n_passages + p] = red[0];
}

// PLAID residual decode (SURVEY.md 8f-3): emb[t][i] = centroids[code[t]][i] + bucket_weights[idx(t, i)],
// idx = the nbits-wide field of dim i in the token's packed residual bytes, bit-reversed (the
// reference packs each bucket index LSB-first into big-endian bytes: residual.py:188-204 binarize,
// :51-73 reversed_bit_map, :77-93 lookup table; decode loop decompress_residuals.cpp:27-78), then the
// row is L2-normalised (index_storage.py:173) and stored as bf16.  HBM-bound byte work: one warp per
// token, lane = 4 dims, centroid rows come from L2, bucket weights from shared memory.  The arithmetic is
// flmr_scan_plaid_kernel.cuh's plaid_* functions, so a compressed corpus decodes to the same bits.
__global__ void flmr_plaid_decode_kernel(const int32_t* __restrict__ codes,
                                         const uint8_t* __restrict__ residuals,
                                         const float* __restrict__ centroids,
                                         const float* __restrict__ bucket_weights, int nbits,
                                         int normalize, int64_t n_tokens, int64_t n_centroids,
                                         uint2* __restrict__ out, int* __restrict__ bad_code) {
  __shared__ float s_w[256];
  for (int i = threadIdx.x; i < (1 << nbits); i += blockDim.x) s_w[i] = bucket_weights[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = (static_cast<int64_t>(gridDim.x) * blockDim.x) >> 5;
  const int packed_dim = kDim * nbits / 8;    // bytes per token
  for (int64_t t = warp0; t < n_tokens; t += n_warps) {
    const int32_t code = codes[t];
    if (code < 0 || code >= n_centroids) {    // corrupt index: flag, never read out of bounds
      if (lane == 0) {
        *reinterpret_cast<volatile int*>(bad_code) = 1;
        __threadfence_system();
      }
      continue;
    }
    const float4 c = __ldg(reinterpret_cast<const float4*>(centroids + static_cast<int64_t>(code) * kDim) + lane);
    const uint8_t* row = residuals + t * packed_dim;
    float v[4];
    plaid_lane_values(c, row, s_w, nbits, lane, v);
    if (normalize) {
      const float inv = plaid_inv_norm(v);
#pragma unroll
      for (int dd = 0; dd < 4; ++dd) v[dd] *= inv;
    }
    __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]);
    __nv_bfloat162 hi = __floats2bfloat162_rn(v[2], v[3]);
    uint2 w;
    w.x = *reinterpret_cast<uint32_t*>(&lo);
    w.y = *reinterpret_cast<uint32_t*>(&hi);
    out[t * 32 + lane] = w;
  }
}

// Candidate merge: per query, select the k_out best of n candidates by (score desc, pid asc).
// Candidates come either as packed keys written by the scan kernel (keys != null; pid = pid_base +
// ~low32) or as (score, pid) arrays laid out [list][query][k_in].  One 1024-thread block per query,
// up to kMergePer candidates per thread in registers, k_out selection rounds.
constexpr int kMergeThreads = 1024;
constexpr int kMergePer = 20;
constexpr int64_t kPidEmpty = 0x7fffffffffffffffll;

struct Cand {
  uint32_t ord;  // ordered score; 0 = empty
  int64_t pid;
};
__device__ __forceinline__ bool cand_better(const Cand& a, const Cand& b) {
  return a.ord > b.ord || (a.ord == b.ord && a.pid < b.pid);
}

__global__ void __launch_bounds__(kMergeThreads)
flmr_merge_kernel(const uint64_t* __restrict__ keys, const float* __restrict__ in_scores,
                  const int64_t* __restrict__ in_pids, int n_lists, int n_queries, int k_in,
                  int k_out, int64_t pid_base, float* __restrict__ out_scores,
                  int64_t* __restrict__ out_pids, int q_offset) {
  __shared__ uint32_t s_ord[32];
  __shared__ int64_t s_pid[32];
  __shared__ uint32_t w_ord;
  __shared__ int64_t w_pid;
  const int b = q_offset + blockIdx.x;   // n_queries = stride of the per-list arrays; blocks cover [q_offset, q_offset + grid)
  const int n = n_lists * k_in;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  Cand c[kMergePer];
#pragma unroll
  for (int i = 0; i < kMergePer; ++i) {
    const int idx = threadIdx.x + i * kMergeThreads;
    c[i].ord = 0u;
    c[i].pid = kPidEmpty;
    if (idx < n) {
      const int l = idx / k_in, j = idx % k_in;
      const int64_t g = (static_cast<int64_t>(l) * n_queries + b) * k_in + j;
      if (keys) {
        const uint64_t key = keys[g];
        if (key != 0ull) {
          c[i].ord = static_cast<uint32_t>(key >> 32);
          c[i].pid = pid_base + (0xFFFFFFFFu - static_cast<uint32_t>(key));
        }
      } else {
        const int64_t pid = in_pids[g];
        if (pid >= 0) {
          c[i].ord = float_to_ordered(in_scores[g]);
          c[i].pid = pid;
        }
      }
    }
  }
  for (int r = 0; r < k_out; ++r) {
    Cand best = c[0];
#pragma unroll
    for (int i = 1; i < kMergePer; ++i)
      if (cand_better(c[i], best)) best = c[i];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
      Cand o;
      o.ord = __shfl_xor_sync(0xffffffffu, best.ord, off);
      o.pid = __shfl_xor_sync(0xffffffffu, best.pid, off);
      if (cand_better(o, best)) best = o;
    }
    if (lane == 0) {
      s_ord[warp] = best.ord;
      s_pid[warp] = best.pid;
    }
    __syncthreads();
    if (warp == 0) {
      Cand x;
      x.ord = s_ord[lane];
      x.pid = s_pid[lane];
#pragma unroll
      for (int off = 16; off >= 1; off >>= 1) {
        Cand o;
        o.ord = __shfl_xor_sync(0xffffffffu, x.ord, off);
        o.pid = __shfl_xor_sync(0xffffffffu, x.pid, off);
        if (cand_better(o, x)) x = o;
      }
      if (lane == 0) {
        w_ord = x.ord;
        w_pid = x.pid;
        const bool empty = (x.ord == 0u);
        out_scores[static_cast<int64_t>(b) * k_out + r] =
            empty ? -INFINITY : ordered_to_float(x.ord);
        out_pids[static_cast<int64_t>(b) * k_out + r] = empty ? -1 : x.pid;
      }
    }
    __syncthreads();
    const uint32_t wo = w_ord;
    const int64_t wp = w_pid;
    if (wo != 0u) {
#pragma unroll
      for (int i = 0; i < kMergePer; ++i)
        if (c[i].ord == wo && c[i].pid == wp) {
          c[i].ord = 0u;
          c[i].pid = kPidEmpty;
        }
    }
    // (w_ord/w_pid are rewritten only after the next round's first __syncthreads)
  }
}

// Top-k selection over a dense score row for k beyond the fused capacity (SURVEY 8a a10:
// Searcher.dense_search accepts any k).  One 1024-thread block per query:
//   1. 4-pass MSB radix select (8 bits per pass, 256-bin histogram in shared memory) over the
//      order-preserving uint32 image of the scores -> key T of the k-th best score, and how many keys
//      are strictly better;
//   2. order-preserving compaction: every thread owns a contiguous slice of the row, block-wide
//      exclusive scans place the keys > T, then as many keys == T (ascending pid) as still fit;
//   3. bitonic sort of the k survivors by (score desc, pid asc) in shared memory.
constexpr int kSelectThreads = 1024;
constexpr int kSelectMaxK = 2048;

__global__ void __launch_bounds__(kSelectThreads)
flmr_select_kernel(const float* __restrict__ scores, int64_t n, int k, int64_t pid_base,
                   float* __restrict__ out_scores, int64_t* __restrict__ out_pids) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t s_prefix, s_need, s_gt_total;
  __shared__ uint32_t scan_gt[kSelectThreads], scan_eq[kSelectThreads];
  __shared__ uint32_t sel_ord[kSelectMaxK];
  __shared__ uint32_t sel_pid[kSelectMaxK];
  const int tid = threadIdx.x;
  const float* row = scores + static_cast<int64_t>(blockIdx.x) * n;
  const int kk = static_cast<int>(n < k ? n : k);
  // ---- 1. radix select of the kk-th largest ordered key ----
  if (tid == 0) {
    s_prefix = 0u;
    s_need = static_cast<uint32_t>(kk);
  }
  uint32_t mask_hi = 0u;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = tid; i < 256; i += kSelectThreads) hist[i] = 0u;
    __syncthreads();
    const uint32_t prefix = s_prefix;
    for (int64_t i = tid; i < n; i += kSelectThreads) {
      const uint32_t key = float_to_ordered(row[i] + 0.0f);
      if ((key & mask_hi) == prefix) atomicAdd(&hist[(key >> shift) & 0xFFu], 1u);
    }
    __syncthreads();
    if (tid == 0) {
      uint32_t need = s_need, bin = 255;
      for (;; --bin) {                       // from the largest digit down
        if (hist[bin] >= need || bin == 0) break;
        need -= hist[bin];
      }
      s_need = need;                         // still to take inside this bin
      s_prefix = prefix | (bin << shift);
    }
    __syncthreads();
    mask_hi |= 0xFFu << shift;
  }
  const uint32_t T = s_prefix;               // key of the kk-th best; s_need of the keys == T are taken
  // ---- 2. order-preserving compaction ----
  const int64_t per = (n + kSelectThreads - 1) / kSelectThreads;
  const int64_t i0 = static_cast<int64_t>(tid) * per, i1 = (i0 + per < n) ? i0 + per : n;
  uint32_t c_gt = 0, c_eq = 0;
  for (int64_t i = i0; i < i1; ++i) {
    const uint32_t key = float_to_ordered(row[i] + 0.0f);
    c_gt += key > T;
    c_eq += key == T;
  }
  scan_gt[tid] = c_gt;
  scan_eq[tid] = c_eq;
  __syncthreads();
  for (int off = 1; off < kSelectThreads; off <<= 1) {   // Hillis-Steele inclusive scans
    const uint32_t a = tid >= off ? scan_gt[tid - off] : 0u, b = tid >= off ? scan_eq[tid - off] : 0u;
    __syncthreads();
    scan_gt[tid] += a;
    scan_eq[tid] += b;
    __syncthreads();
  }
  if (tid == kSelectThreads - 1) s_gt_total = scan_gt[tid];
  __syncthreads();
  const uint32_t gt_total = s_gt_total;
  uint32_t o_gt = scan_gt[tid] - c_gt, o_eq = gt_total + scan_eq[tid] - c_eq;
  for (int64_t i = i0; i < i1; ++i) {
    const uint32_t key = float_to_ordered(row[i] + 0.0f);
    if (key > T) {
      sel_ord[o_gt] = key;
      sel_pid[o_gt++] = static_cast<uint32_t>(i);
    } else if (key == T) {
      if (o_eq < static_cast<uint32_t>(kk)) {
        sel_ord[o_eq] = key;
        sel_pid[o_eq] = static_cast<uint32_t>(i);
      }
      ++o_eq;
    }
  }
  // ---- 3. bitonic sort (descending score, ascending pid) over the next power of two ----
  int m = 1;
  while (m < kk) m <<= 1;
  __syncthreads();
  for (int i = kk + tid; i < m; i += kSelectThreads) {
    sel_ord[i] = 0u;                         // empty entries sort last
    sel_pid[i] = 0xFFFFFFFFu;
  }
  __syncthreads();
  auto before = [&](int a, int b) {          // true if entry a must come before entry b
    return sel_ord[a] > sel_ord[b] || (sel_ord[a] == sel_ord[b] && sel_pid[a] < sel_pid[b]);
  };
  for (int size = 2; size <= m; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < m; i += kSelectThreads) {
        const int j = i ^ stride;
        if (j > i) {
          const bool up = (i & size) == 0;   // ascending position = better entries first
          if (up ? before(j, i) : before(i, j)) {
            const uint32_t to = sel_ord[i], tp = sel_pid[i];
            sel_ord[i] = sel_ord[j];
            sel_pid[i] = sel_pid[j];
            sel_ord[j] = to;
            sel_pid[j] = tp;
          }
        }
      }
      __syncthreads();
    }
  }
  for (int i = tid; i < k; i += kSelectThreads) {
    const bool ok = i < kk;
    out_scores[static_cast<int64_t>(blockIdx.x) * k + i] = ok ? ordered_to_float(sel_ord[i]) : -INFINITY;
    out_pids[static_cast<int64_t>(blockIdx.x) * k + i] = ok ? pid_base + sel_pid[i] : -1;
  }
}

}  // namespace

// ---- handles -----------------------------------------------------------------------------------------
struct flmr_corpus {
  int device = 0;
  int64_t n_passages = 0, n_tokens = 0, n_rows = 0, pid_base = 0;
  int n_ctas = 0;
  int64_t n_tiles = 0;
  bool adopted = false;
  int64_t hbm_bytes = 0;
  __nv_bfloat16* d_tokens = nullptr;   // [n_rows, 128] padded layout
  int64_t* d_poff = nullptr;           // [n_passages + 1] stored-row offsets
  int32_t* d_doclen = nullptr;         // [n_passages] real lengths
  int32_t* d_cta_row_begin = nullptr;  // [n_ctas + 1]
  int64_t* d_cta_tile_base = nullptr;  // [n_ctas + 1]
  uint32_t* d_tile_end_mask = nullptr; // [n_tiles]
  int32_t* d_tile_first_pid = nullptr; // [n_tiles]
  CUtensorMap tmap_d;
  // CTA-pair experiment (flmr_debug_set_scan_variant(4)): n_pairs contiguous ranges, one per pair of CTAs, and a
  // tensor map with a half-tile box
  int n_pairs = 0;
  int sm_count = 0;
  int64_t n_tiles_pair = 0;
  int32_t* d_pair_row_begin = nullptr;
  int64_t* d_pair_tile_base = nullptr;
  uint32_t* d_pair_end_mask = nullptr;
  int32_t* d_pair_first_pid = nullptr;
  CUtensorMap tmap_half;
  // compressed (PLAID) residency, flmr_corpus_create_plaid: nbits != 0 and d_tokens == nullptr.  Rows in the
  // padded order above plus kTileN zero rows; the scan decodes them (flmr_scan_plaid_kernel.cuh)
  int nbits = 0;
  int64_t n_centroids = 0;
  int32_t* d_codes = nullptr;          // [n_rows + kTileN]
  uint8_t* d_residuals = nullptr;      // [n_rows + kTileN][16 * nbits]
  float* d_inv_norm = nullptr;         // [n_rows + kTileN]
  float* d_centroids = nullptr;        // [n_centroids][128]
  float* d_weights = nullptr;          // [2^nbits]
};

// Streaming corpus construction (index load): the padded token matrix is allocated once, packed rows arrive in
// order through two pinned staging buffers (host fill of one overlaps the DMA of the other).
struct flmr_corpus_builder {
  flmr_corpus* corpus = nullptr;        // under construction (owned until finish)
  std::vector<int64_t> soff, poff;
  std::vector<int32_t> doclens;
  bool aligned = true;                  // every doclen a multiple of kGroup: rows land in place, no scatter
  int64_t rows_done = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  static constexpr int kBufs = 2;
  static constexpr int64_t kBufRows = (64ll << 20) / (kDim * 2);   // 64 MB of rows per staging buffer
  void* h_pin[kBufs] = {nullptr, nullptr};
  uint4* d_stage[kBufs] = {nullptr, nullptr};   // device staging (unaligned corpora only)
  cudaEvent_t free_ev[kBufs] = {nullptr, nullptr};
  int64_t *d_soff = nullptr, *d_poff = nullptr;
  int next = 0;
  double fill_s = 0.0;                  // host time spent filling the pinned buffers (read / memcpy)
};

// Chunked construction of a compressed corpus (flmr_corpus_plaid_builder_*): the handle's arrays are allocated once
// from the doclens, then chunks of whole passages are packed into them in order, so a load holds no more than the
// resident arrays plus the caller's current chunk.
struct flmr_corpus_plaid_builder {
  flmr_corpus* corpus = nullptr;        // under construction (owned until finish)
  std::vector<int64_t> soff, poff;
  std::vector<int32_t> doclens;
  int64_t passages_done = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  int64_t *d_soff = nullptr, *d_poff = nullptr;
  int* d_bad = nullptr;                 // set by the pack kernel when a code is out of range
};

struct flmr_workspace {
  const flmr_corpus* corpus = nullptr;
  int device = 0;
  int max_queries = 0, max_nq = 0;
  __nv_bfloat16* d_qpad = nullptr;     // [kStageMaxPasses][kMtMax*128, 128] staged (zero-padded) queries, one slot per pass
  uint64_t* d_cand_keys = nullptr;     // [n_ctas][max_queries][k] candidate keys of one call chunk
  float* d_acc = nullptr;              // [group][n_passages] lazily allocated (row-sliced queries)
  int64_t acc_capacity = 0;            // floats allocated at d_acc
  int* h_status = nullptr;             // pinned + mapped: readable by the host even after a device trap
  int* d_status = nullptr;             // device alias of h_status
  int dbg_mode = 0, dbg_lane_rbq = 4;  // -DFLMR_DEBUG builds: FLMR_DEBUG_MODE / FLMR_LANE_RBQ, read once at creation
};

// NCCL is resolved at RUN time (dlopen): the library has no link dependency on it, loads on a box without
// NCCL, and shares the libnccl the host process already loaded (torch ships its own) when there is one.
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, /* ncclUniqueId by value: 128 bytes */ struct NcclId, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  int (*CommCount)(void*, int*) = nullptr;
  int (*CommUserRank)(void*, int*) = nullptr;
};
struct NcclId {
  char internal[128];
};

struct flmr_comm {
  void* nccl = nullptr;   // ncclComm_t
  int rank = 0, world = 1, device = 0;
  bool owned = false;     // created by flmr_comm_create (destroyed with the handle) vs adopted
  // exchange buffers, grown on demand: this rank's [B, k] lists and everybody's [world, B, k]
  float* d_send_s = nullptr;
  int64_t* d_send_p = nullptr;
  float* d_recv_s = nullptr;
  int64_t* d_recv_p = nullptr;
  int64_t capacity = 0;   // entries (B * k) the send buffers hold
};

namespace {

int load_nccl(const NcclApi** out) {
  static NcclApi api;
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  if (!api.handle) {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // the copy the process already uses, if any
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return fail(FLMR_ERR_UNSUPPORTED, "NCCL is not available (dlopen libnccl.so.2: %s)", dlerror());
    NcclApi a;
    a.handle = h;
    a.GetUniqueId = reinterpret_cast<decltype(a.GetUniqueId)>(dlsym(h, "ncclGetUniqueId"));
    a.CommInitRank = reinterpret_cast<decltype(a.CommInitRank)>(dlsym(h, "ncclCommInitRank"));
    a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
    a.AllGather = reinterpret_cast<decltype(a.AllGather)>(dlsym(h, "ncclAllGather"));
    a.GroupStart = reinterpret_cast<decltype(a.GroupStart)>(dlsym(h, "ncclGroupStart"));
    a.GroupEnd = reinterpret_cast<decltype(a.GroupEnd)>(dlsym(h, "ncclGroupEnd"));
    a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
    a.CommCount = reinterpret_cast<decltype(a.CommCount)>(dlsym(h, "ncclCommCount"));
    a.CommUserRank = reinterpret_cast<decltype(a.CommUserRank)>(dlsym(h, "ncclCommUserRank"));
    if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.AllGather || !a.GroupStart || !a.GroupEnd ||
        !a.GetErrorString || !a.CommCount || !a.CommUserRank)
      return fail(FLMR_ERR_UNSUPPORTED, "libnccl.so.2 lacks an expected entry point");
    api = a;
  }
  *out = &api;
  return FLMR_OK;
}

#define FLMR_NCCL(api, expr)                                                                          \
  do {                                                                                                \
    int r__ = (expr);                                                                                 \
    if (r__ != 0)                                                                                     \
      return fail(FLMR_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, (api)->GetErrorString(r__), __FILE__, __LINE__); \
  } while (0)

constexpr int kNcclInt64 = 4, kNcclFloat32 = 7;   // ncclDataType_t values (nccl.h: ncclInt64 = 4, ncclFloat32 = 7)

thread_local bool g_profiling = false;
// which scan kernel a search on this thread launches: 0 = chosen per pass (launch_scan), 2 = flmr_scan_kernel (two
// epilogue warpgroups), 3 = flmr_scan3_kernel (three, static query-tile assignment); flmr_debug_set_scan_variant
thread_local int g_scan_variant = 0;
struct EventPair {
  cudaEvent_t a, b;
};
thread_local std::vector<EventPair> g_scan_events;

template <typename T>
int dev_upload(T** dptr, const std::vector<T>& h, int64_t* bytes_acc) {
  const size_t bytes = std::max<size_t>(h.size(), 1) * sizeof(T);
  FLMR_CUDA(cudaMalloc(reinterpret_cast<void**>(dptr), bytes));
  if (!h.empty()) FLMR_CUDA(cudaMemcpy(*dptr, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  if (bytes_acc) *bytes_acc += static_cast<int64_t>(bytes);
  return FLMR_OK;
}

// FLMR_OK if every pointer is device memory of `device` (or managed).
int check_device_ptrs(std::initializer_list<const void*> ptrs, int device) {
  for (const void* ptr : ptrs) {
    cudaPointerAttributes attr{};
    const bool ok = cudaPointerGetAttributes(&attr, ptr) == cudaSuccess &&
                    ((attr.type == cudaMemoryTypeDevice && attr.device == device) ||
                     attr.type == cudaMemoryTypeManaged);
    cudaGetLastError();
    if (!ok) return fail(FLMR_ERR_INVALID_ARG, "PLAID arrays must be device pointers on device %d", device);
  }
  return FLMR_OK;
}

// Token-balanced split of the passages into n_ctas contiguous ranges + per-tile metadata.
void build_partition(const std::vector<int64_t>& poff, int n_ctas, int tile_n,
                     std::vector<int32_t>* cta_row_begin, std::vector<int64_t>* cta_tile_base,
                     std::vector<uint32_t>* tile_end_mask, std::vector<int32_t>* tile_first_pid) {
  const int64_t n = static_cast<int64_t>(poff.size()) - 1;
  const int64_t rows = poff[n];
  std::vector<int64_t> pbeg(n_ctas + 1);
  pbeg[0] = 0;
  for (int c = 1; c < n_ctas; ++c) {
    const int64_t target = rows * c / n_ctas;
    int64_t p = std::lower_bound(poff.begin(), poff.end(), target) - poff.begin();
    p = std::min<int64_t>(std::max<int64_t>(p, pbeg[c - 1]), n);
    pbeg[c] = p;
  }
  pbeg[n_ctas] = n;
  cta_row_begin->resize(n_ctas + 1);
  cta_tile_base->resize(n_ctas + 1);
  int64_t tiles = 0;
  for (int c = 0; c <= n_ctas; ++c) {
    (*cta_row_begin)[c] = static_cast<int32_t>(poff[pbeg[c]]);
    (*cta_tile_base)[c] = tiles;
    if (c < n_ctas) tiles += (poff[pbeg[c + 1]] - poff[pbeg[c]] + tile_n - 1) / tile_n;
  }
  tile_end_mask->assign(tiles, 0u);
  tile_first_pid->assign(tiles, 0);
  for (int c = 0; c < n_ctas; ++c) {
    const int64_t r0 = poff[pbeg[c]];
    const int64_t tb = (*cta_tile_base)[c];
    const int64_t nt = (*cta_tile_base)[c + 1] - tb;
    std::vector<char> seen(nt, 0);
    for (int64_t p = pbeg[c]; p < pbeg[c + 1]; ++p) {
      const int64_t last = poff[p + 1] - 1 - r0;  // last stored row of p, relative to the CTA
      const int64_t t = last / tile_n;
      const int g = static_cast<int>((last % tile_n) / kGroup);
      (*tile_end_mask)[tb + t] |= (1u << g);
      if (!seen[t]) {
        seen[t] = 1;
        (*tile_first_pid)[tb + t] = static_cast<int32_t>(p);
      }
    }
  }
}

// ---- pass planning (pure host logic; exported for tests as flmr_debug_plan_passes) -------------------
// One pass = one launch of the scan kernel over the whole shard with up to kRbMax 32-row blocks of
// queries resident (kNqMax queries at most).
enum : int { kPassAccIn = 1, kPassAccOut = 2, kPassFinal = 4, kPassPair = 8 };
struct PassPlan {
  int q_first, n_q;        // queries [q_first, q_first + n_q) are resident (pair pass: n_q PER CTA, the pass covers
                           // [q_first, q_first + 2 n_q), CTA r of every pair the r-th half)
  int row0, rows;          // their rows [row0, row0 + rows)
  int rbq, n_mtiles;       // 32-row blocks per query, 128-row MMA tiles of the pass (per CTA)
  int flags;               // kPassAccIn: add the partial scores of earlier slices; kPassAccOut: store
                           // partial scores; kPassFinal: scores complete -> top-k (+ all-scores output);
                           // kPassPair: CTA-pair pass (clusters of two CTAs share a token range)
  int group_first, acc_slot;  // row of the partial-score buffer: query group_first + acc_slot (+ i)
};

// allow_pair: CTA-pair passes (run_search decides: shards that span every SM) for as many queries as fill them —
// every CTA of a pair keeps exactly the residency a normal pass would give it, so a pair pass serves twice the
// queries per corpus pass; with fewer than four 128-row tiles per CTA pairs measured slower and are not planned.
// Pair passes always cover a PREFIX of the queries (*n_pair_queries_out); the rest gets normal passes.
void plan_passes(int n_queries, int nq, bool allow_pair, std::vector<PassPlan>* out, int* group_out,
                 int* n_pair_queries_out) {
  out->clear();
  int n_pair_q = 0;
  const int rbq_total = (nq + 31) / 32;
  if (rbq_total <= kRbMax) {
    const int qpp_max = std::min(kNqMax, kRbMax / rbq_total);
    if (allow_pair && qpp_max * rbq_total * 32 >= 4 * kTileM) {
      for (; n_pair_q + 2 * qpp_max <= n_queries; n_pair_q += 2 * qpp_max)
        out->push_back({n_pair_q, qpp_max, 0, nq, rbq_total, (qpp_max * rbq_total * 32 + kTileM - 1) / kTileM,
                        kPassFinal | kPassPair, n_pair_q, 0});
    }
    // whole queries resident: as many per pass as fit, spread evenly over the passes that takes (64
    // queries of one row block: 4 passes of 16 rather than 20+20+20+4, whose short last pass would be
    // HBM-bound while the others are tensor-bound)
    const int rest = n_queries - n_pair_q;
    const int n_passes = (rest + qpp_max - 1) / qpp_max;
    const int qpp = n_passes ? (rest + n_passes - 1) / n_passes : 1;
    for (int b0 = n_pair_q; b0 < n_queries; b0 += qpp) {
      const int nqp = std::min(qpp, n_queries - b0);
      out->push_back({b0, nqp, 0, nq, rbq_total, (nqp * rbq_total * 32 + kTileM - 1) / kTileM, kPassFinal,
                      b0, 0});
    }
    *group_out = 1;
    if (n_pair_queries_out) *n_pair_queries_out = n_pair_q;
    return;
  }
  // queries longer than one pass holds: rows sliced over several passes, partial scores carried through
  // HBM.  Full slices take one pass per query (pair pass: per two queries, one in each CTA); the TAIL slices of up
  // to `group` queries share one pass (Nq = 832: 3 queries = 3 full passes + 1 tail pass instead of 6; with pairs
  // 6 queries = 3 full pair passes + 1 tail pair pass).
  const int rows_per_slice = kRbMax * 32;
  const int n_slices = (nq + rows_per_slice - 1) / rows_per_slice;
  const int tail_row0 = (n_slices - 1) * rows_per_slice;
  const int tail_rows = nq - tail_row0;
  const int tail_rbq = (tail_rows + 31) / 32;
  const int g_max = std::max(1, std::min(kNqMax, kRbMax / tail_rbq));
  int group_used = 0;
  if (allow_pair) {
    const int G = 2 * g_max;                    // queries per pair group; a query's slot in the partial-score
    for (; n_pair_q + G <= n_queries; n_pair_q += G) {   // buffer = its index in the group
      const int b0 = n_pair_q;
      for (int j = 0; j < g_max; ++j)           // queries b0 + 2j (CTA 0) and b0 + 2j + 1 (CTA 1)
        for (int sl = 0; sl + 1 < n_slices; ++sl)
          out->push_back({b0 + 2 * j, 1, sl * rows_per_slice, rows_per_slice, kRbMax, rows_per_slice / kTileM,
                          kPassAccOut | (sl > 0 ? kPassAccIn : 0) | kPassPair, b0, 2 * j});
      out->push_back({b0, g_max, tail_row0, tail_rows, tail_rbq, (g_max * tail_rbq * 32 + kTileM - 1) / kTileM,
                      kPassAccIn | kPassFinal | kPassPair, b0, 0});
      group_used = G;
    }
  }
  const int rest = n_queries - n_pair_q;
  const int group = std::max(1, std::min(g_max, rest));
  for (int b0 = n_pair_q; b0 < n_queries; b0 += group) {
    const int g = std::min(group, n_queries - b0);
    for (int b = 0; b < g; ++b)
      for (int sl = 0; sl + 1 < n_slices; ++sl)
        out->push_back({b0 + b, 1, sl * rows_per_slice, rows_per_slice, kRbMax, rows_per_slice / kTileM,
                        kPassAccOut | (sl > 0 ? kPassAccIn : 0), b0, b});
    out->push_back({b0, g, tail_row0, tail_rows, tail_rbq, (g * tail_rbq * 32 + kTileM - 1) / kTileM,
                    kPassAccIn | kPassFinal, b0, 0});
    group_used = std::max(group_used, g);
  }
  *group_out = std::max(1, group_used);
  if (n_pair_queries_out) *n_pair_queries_out = n_pair_q;
}

int launch_scan(const flmr_corpus* c, flmr_workspace* ws, ScanParams p, bool pair, cudaStream_t st) {
  // three epilogue warpgroups pay off exactly where they buy a third TMEM accumulator stage and one accumulator
  // per warpgroup and D tile: passes with three resident query tiles (one Nq = 320 query: +12 % in short runs, +4 %
  // sustained); with five tiles (2 / 2 / 1 accumulators per warpgroup, still two stages) they measured 7 % slower
  // than strict two-warpgroup alternation, with one, two or four tiles the same (profiles/r02_scan_variant_probe.md)
  const bool three = !pair && ((g_scan_variant == 3) || (g_scan_variant == 0 && p.n_mtiles == 3));
#ifdef FLMR_DEBUG
  auto kern = p.debug_mode ? flmr_scan_kernel<true> : flmr_scan_kernel<false>;
  const bool use3 = three && !p.debug_mode;
#else
  auto kern = flmr_scan_kernel<false>;
  const bool use3 = three;
#endif
  EventPair ev{};
  if (g_profiling) {
    FLMR_CUDA(cudaEventCreate(&ev.a));
    FLMR_CUDA(cudaEventCreate(&ev.b));
    FLMR_CUDA(cudaEventRecord(ev.a, st));
  }
  (void)ws;
  if (c->nbits) {
    // compressed corpus: the decoding kernel, single-CTA passes on the two-warpgroup structure (never planned as
    // pairs: n_pairs = 0), whatever the scan variant
    const PlaidParams q{c->d_codes, c->d_residuals, c->d_inv_norm, c->d_centroids, c->d_weights};
    switch (c->nbits) {
      case 1: flmr_scan_plaid_kernel<1><<<c->n_ctas, kPlaidThreads, PlaidSmem<1>::kBytes, st>>>(p, q); break;
      case 2: flmr_scan_plaid_kernel<2><<<c->n_ctas, kPlaidThreads, PlaidSmem<2>::kBytes, st>>>(p, q); break;
      case 4: flmr_scan_plaid_kernel<4><<<c->n_ctas, kPlaidThreads, PlaidSmem<4>::kBytes, st>>>(p, q); break;
      default: flmr_scan_plaid_kernel<8><<<c->n_ctas, kPlaidThreads, PlaidSmem<8>::kBytes, st>>>(p, q); break;
    }
  } else if (pair) {
    // clusters of two CTAs share one of the n_pairs token ranges; the tensor map has a half-tile box
    p.cta_row_begin = c->d_pair_row_begin;
    p.cta_tile_base = c->d_pair_tile_base;
    p.tile_end_mask = c->d_pair_end_mask;
    p.tile_first_pid = c->d_pair_first_pid;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(2 * c->n_pairs));
    cfg.blockDim = dim3(kScanThreads);
    cfg.dynamicSmemBytes = ScanSmem::kBytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    FLMR_CUDA(cudaLaunchKernelEx(&cfg, flmr_scan_kernel<false, true>, c->tmap_half, p));
  } else if (use3) {
    flmr_scan3_kernel<<<c->n_ctas, kScan3Threads, ScanSmem::kBytes, st>>>(c->tmap_d, p);
  } else {
    kern<<<c->n_ctas, kScanThreads, ScanSmem::kBytes, st>>>(c->tmap_d, p);
  }
  FLMR_CUDA(cudaGetLastError());
  ++g_launches;
  if (g_profiling) {
    FLMR_CUDA(cudaEventRecord(ev.b, st));
    g_scan_events.push_back(ev);
  }
  return FLMR_OK;
}

// One launch stages `count` zero-padded query blocks (slot i of the workspace's staging buffer <- sp.pass[i]).
int stage_queries(flmr_workspace* ws, const void* d_q, int nq, const StageParams& sp, int count, cudaStream_t st) {
  const int threads = 256;
  dim3 grid((kMtMax * kTileM * 16 + threads - 1) / threads, static_cast<unsigned>(count));
  flmr_stage_queries_kernel<<<grid, threads, 0, st>>>(reinterpret_cast<const uint4*>(d_q),
                                                      reinterpret_cast<uint4*>(ws->d_qpad), nq, sp);
  FLMR_CUDA(cudaGetLastError());
  ++g_launches;
  return FLMR_OK;
}

// Queries [q0, q0 + nq) of a chunk of `stride` queries; `n_lists` = candidate lists per query (CTAs, or CTA pairs
// for queries that went through pair passes).  d_out_* point at the chunk's first query.
int launch_merge_keys(const flmr_corpus* c, flmr_workspace* ws, int n_lists, int stride, int q0, int nq, int k,
                      float* d_out_scores, int64_t* d_out_pids, cudaStream_t st) {
  if (nq <= 0) return FLMR_OK;
  if (static_cast<int64_t>(n_lists) * k > kMergeThreads * kMergePer)
    return fail(FLMR_ERR_UNSUPPORTED, "n_lists*k = %lld exceeds merge capacity %d",
                (long long)n_lists * k, kMergeThreads * kMergePer);
  flmr_merge_kernel<<<nq, kMergeThreads, 0, st>>>(ws->d_cand_keys, nullptr, nullptr, n_lists, stride, k, k,
                                                  c->pid_base, d_out_scores, d_out_pids, q0);
  FLMR_CUDA(cudaGetLastError());
  ++g_launches;
  return FLMR_OK;
}

// Partial-score rows of row-sliced (Nq > 640) queries: grown on demand, never shrunk.
int ensure_acc(flmr_workspace* ws, int64_t floats) {
  if (ws->acc_capacity >= floats) return FLMR_OK;
  if (ws->d_acc) cudaFree(ws->d_acc);
  ws->d_acc = nullptr;
  ws->acc_capacity = 0;
  FLMR_CUDA(cudaMalloc(reinterpret_cast<void**>(&ws->d_acc), static_cast<size_t>(floats) * sizeof(float)));
  ws->acc_capacity = floats;
  return FLMR_OK;
}

// Shared driver of flmr_maxsim_scores / flmr_maxsim_topk.
int run_search(const flmr_corpus* c, flmr_workspace* ws, const void* d_q, int n_queries, int nq,
               unsigned flags, int k, float* d_all_scores, float* d_topk_scores,
               int64_t* d_topk_pids, cudaStream_t st) {
  if (!c || !ws || !d_q) return fail(FLMR_ERR_INVALID_ARG, "null corpus / workspace / query pointer");
  if (ws->corpus != c) return fail(FLMR_ERR_INVALID_ARG, "workspace belongs to a different corpus");
  if (n_queries < 0 || nq <= 0) return fail(FLMR_ERR_INVALID_ARG, "bad n_queries=%d nq=%d", n_queries, nq);
  if (k < 0 || k > kMaxK) return fail(FLMR_ERR_UNSUPPORTED, "k=%d outside [1, %d]", k, kMaxK);
  if (n_queries == 0) return FLMR_OK;
  if (const int code = *reinterpret_cast<volatile int*>(ws->h_status))
    return fail(FLMR_ERR_KERNEL,
                "an earlier scan on this workspace tripped the device watchdog (code %d: %s starved); "
                "the CUDA context is poisoned", code,
                code == kDevTimeoutProducer ? "TMA producer" : code == kDevTimeoutMma ? "MMA issuer" : "epilogue");
  DeviceGuard guard(c->device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);

  ScanParams p{};
  p.cta_row_begin = c->d_cta_row_begin;
  p.cta_tile_base = c->d_cta_tile_base;
  p.tile_end_mask = c->d_tile_end_mask;
  p.tile_first_pid = c->d_tile_first_pid;
  p.init_val = (flags & FLMR_FLAG_RELU) ? 0.f : -INFINITY;
  p.n_passages = c->n_passages;
  p.cand_keys = ws->d_cand_keys;
  p.q_pad = reinterpret_cast<const uint4*>(ws->d_qpad);
  p.status = ws->d_status;
  p.lane_mode_max_rbq = 4;   // measured (profiles/r01_debug_mode_probes.log): lane-per-query wins up to 4 row blocks per query
#ifdef FLMR_DEBUG   // timing experiments exist only in -DFLMR_DEBUG builds (tools/); the release library has no env hooks
  p.lane_mode_max_rbq = ws->dbg_lane_rbq;
  p.debug_mode = ws->dbg_mode;
  if (p.debug_mode == 6) {  // timestamps of CTA 0's accumulator hand-offs, dumped by the caller
    static long long* d_ts = nullptr;
    if (!d_ts) {
      FLMR_CUDA(cudaMallocManaged(reinterpret_cast<void**>(&d_ts), 64 * 8 * sizeof(long long)));
      memset(d_ts, 0, 64 * 8 * sizeof(long long));
    }
    p.dbg_ts = d_ts;
    if (const char* f = getenv("FLMR_DEBUG_TS_DUMP")) {   // dump what the PREVIOUS launch recorded
      cudaDeviceSynchronize();
      if (FILE* fp = fopen(f, "w")) {
        for (int a = 0; a < 64; ++a) {
          for (int i = 0; i < 8; ++i) fprintf(fp, "%lld ", d_ts[a * 8 + i]);
          fprintf(fp, "\n");
        }
        fclose(fp);
      }
    }
  }
#endif

  // CTA-pair passes (clusters of two CTAs stream one token range, each CTA with the residency of a normal pass, every
  // D tile fetched once and TMA-multicast into both: half the HBM / L2 traffic per query, ~6 % more sustained
  // throughput on this power-capped part, profiles/r02_scan_variant_probe.md) are planned for as many queries as fill
  // them when the shard spans every SM (variant 0 = product), always when forced (4), never under 2 / 3.
  const bool allow_pair = c->n_pairs > 0 && (g_scan_variant == 4 || (g_scan_variant == 0 && c->n_pairs * 2 == c->sm_count));
  // a call is processed in chunks of at most ws->max_queries queries (the candidate buffer's capacity);
  // within a chunk: every pass's scan, then the merge over the chunk's queries (one launch per kind of pass)
  std::vector<PassPlan> plan;
  std::vector<int> slot;
  int rc;
  for (int c0 = 0; c0 < n_queries; c0 += ws->max_queries) {
    const int nqc = std::min(ws->max_queries, n_queries - c0);
    const __nv_bfloat16* d_qc = static_cast<const __nv_bfloat16*>(d_q) + static_cast<int64_t>(c0) * nq * kDim;
    float* d_all_c = d_all_scores ? d_all_scores + static_cast<int64_t>(c0) * c->n_passages : nullptr;
    int group = 1, n_pair_q = 0;
    plan_passes(nqc, nq, allow_pair, &plan, &group, &n_pair_q);
    if (!d_all_c && nq > kRbMax * 32 && (rc = ensure_acc(ws, static_cast<int64_t>(group) * c->n_passages)))
      return rc;
    p.cand_q_stride = nqc;
    slot.assign(plan.size(), 0);
    size_t staged_until = 0;                    // passes [0, staged_until) have their queries staged
    for (size_t pi = 0; pi < plan.size(); ++pi) {
      if (pi == staged_until) {
        // the query blocks of as many of the next passes as fit the staging buffer (a pair pass takes two slots:
        // one block per CTA of a pair) are staged by ONE launch, ahead of their scans
        StageParams sp{};
        int used = 0;
        while (staged_until < plan.size()) {
          const PassPlan& q = plan[staged_until];
          const int need = (q.flags & kPassPair) ? 2 : 1;
          if (used + need > kStageMaxPasses) break;
          slot[staged_until] = used;
          for (int r = 0; r < need; ++r)
            sp.pass[used++] = {q.q_first + r * q.n_q, q.n_q, q.row0, q.rows, q.rbq, q.n_mtiles * kTileM};
          ++staged_until;
        }
        if ((rc = stage_queries(ws, d_qc, nq, sp, used, st))) return rc;
      }
      const PassPlan& pp = plan[pi];
      // partial / final scores of query (group_first + acc_slot + i) live in row i of `acc`
      float* acc = d_all_c
                       ? d_all_c + static_cast<int64_t>(pp.group_first + pp.acc_slot) * c->n_passages
                       : (ws->d_acc ? ws->d_acc + static_cast<int64_t>(pp.acc_slot) * c->n_passages : nullptr);
      p.q_pad = reinterpret_cast<const uint4*>(ws->d_qpad) + static_cast<int64_t>(slot[pi]) * (kMtMax * kTileM * 16);
      p.n_mtiles = pp.n_mtiles;
      p.nq_pass = pp.n_q;
      p.rbq = pp.rbq;
      p.acc_in = (pp.flags & kPassAccIn) ? acc : nullptr;
      p.acc_out = ((pp.flags & kPassAccOut) || ((pp.flags & kPassFinal) && d_all_c)) ? acc : nullptr;
      p.k = (pp.flags & kPassFinal) ? k : 0;
      p.cand_q_first = pp.q_first;
      if ((rc = launch_scan(c, ws, p, (pp.flags & kPassPair) != 0, st))) return rc;
    }
    if (k > 0) {
      float* os = d_topk_scores + static_cast<int64_t>(c0) * k;
      int64_t* op = d_topk_pids + static_cast<int64_t>(c0) * k;
      // queries of pair passes have one candidate list per CTA PAIR, the others one per CTA
      if ((rc = launch_merge_keys(c, ws, c->n_pairs, nqc, 0, n_pair_q, k, os, op, st))) return rc;
      if ((rc = launch_merge_keys(c, ws, c->n_ctas, nqc, n_pair_q, nqc - n_pair_q, k, os, op, st))) return rc;
    }
  }
  return FLMR_OK;
}

// Everything a corpus needs besides its token matrix: offsets / lengths, the CTA partition + per-tile metadata,
// the TMA descriptor, the kernel's shared-memory attribute.  Shared by flmr_corpus_create and the streaming builder.
int finish_corpus(flmr_corpus* c, const std::vector<int64_t>& poff, const int32_t* h_doclens, int sm_count) {
  const int64_t n_passages = c->n_passages;
  const int64_t n_rows = c->n_rows;
  int rc = FLMR_OK;
  auto bail = [](int code) { return code; };
  struct {
    int multiProcessorCount;
  } prop{sm_count};
  // --- offsets / lengths (SIMT cross-check kernel, info) ---
  {
    std::vector<int32_t> lens(h_doclens, h_doclens + n_passages);
    if ((rc = dev_upload(&c->d_poff, poff, &c->hbm_bytes))) return bail(rc);
    if ((rc = dev_upload(&c->d_doclen, lens, &c->hbm_bytes))) return bail(rc);
  }

  // --- partition + tile metadata ---
  int n_ctas = prop.multiProcessorCount;
#ifdef FLMR_DEBUG
  if (const char* e = getenv("FLMR_NUM_CTAS")) n_ctas = std::max(1, atoi(e));
#endif
  n_ctas = static_cast<int>(std::min<int64_t>(n_ctas, n_passages));
  c->n_ctas = n_ctas;
  {
    std::vector<int32_t> row_begin, first_pid;
    std::vector<int64_t> tile_base;
    std::vector<uint32_t> end_mask;
    build_partition(poff, n_ctas, kTileN, &row_begin, &tile_base, &end_mask, &first_pid);
    c->n_tiles = static_cast<int64_t>(end_mask.size());
    if ((rc = dev_upload(&c->d_cta_row_begin, row_begin, &c->hbm_bytes))) return bail(rc);
    if ((rc = dev_upload(&c->d_cta_tile_base, tile_base, &c->hbm_bytes))) return bail(rc);
    if ((rc = dev_upload(&c->d_tile_end_mask, end_mask, &c->hbm_bytes))) return bail(rc);
    if ((rc = dev_upload(&c->d_tile_first_pid, first_pid, &c->hbm_bytes))) return bail(rc);
  }
  if (c->nbits) {   // compressed: no tensor map, no CTA-pair partition; the decoding kernel's smem attribute
    cudaError_t e = cudaFuncSetAttribute(flmr_scan_plaid_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         PlaidSmem<1>::kBytes);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(flmr_scan_plaid_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               PlaidSmem<2>::kBytes);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(flmr_scan_plaid_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               PlaidSmem<4>::kBytes);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(flmr_scan_plaid_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               PlaidSmem<8>::kBytes);
    if (e != cudaSuccess)
      return bail(fail(FLMR_ERR_CUDA, "cannot raise the dynamic shared memory limit of the compressed scan: %s",
                       cudaGetErrorString(e)));
    return FLMR_OK;
  }
  if ((rc = encode_rows_map(&c->tmap_d, c->d_tokens, static_cast<uint64_t>(n_rows), kTileN)))
    return bail(rc);
  if (n_ctas >= 2 && n_passages >= n_ctas / 2) {   // CTA-pair experiment: its own partition + half-tile tensor map
    std::vector<int32_t> row_begin, first_pid;
    std::vector<int64_t> tile_base;
    std::vector<uint32_t> end_mask;
    c->n_pairs = n_ctas / 2;
    c->sm_count = sm_count;
    build_partition(poff, c->n_pairs, kTileN, &row_begin, &tile_base, &end_mask, &first_pid);
    c->n_tiles_pair = static_cast<int64_t>(end_mask.size());
    if ((rc = dev_upload(&c->d_pair_row_begin, row_begin, &c->hbm_bytes))) return bail(rc);
    if ((rc = dev_upload(&c->d_pair_tile_base, tile_base, &c->hbm_bytes))) return bail(rc);
    if ((rc = dev_upload(&c->d_pair_end_mask, end_mask, &c->hbm_bytes))) return bail(rc);
    if ((rc = dev_upload(&c->d_pair_first_pid, first_pid, &c->hbm_bytes))) return bail(rc);
    if ((rc = encode_rows_map(&c->tmap_half, c->d_tokens, static_cast<uint64_t>(n_rows), kTileN / 2))) return bail(rc);
    cudaError_t e3 = cudaFuncSetAttribute(flmr_scan_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          ScanSmem::kBytes);
    if (e3 != cudaSuccess) return bail(fail(FLMR_ERR_CUDA, "pair kernel attribute: %s", cudaGetErrorString(e3)));
  }
  {  // per-device function attribute, set here (idempotent) rather than at launch time
    cudaError_t e1 = cudaFuncSetAttribute(flmr_scan_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          ScanSmem::kBytes);
    if (e1 == cudaSuccess)
      e1 = cudaFuncSetAttribute(flmr_scan3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ScanSmem::kBytes);
#ifdef FLMR_DEBUG
    cudaError_t e2 = cudaFuncSetAttribute(flmr_scan_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          ScanSmem::kBytes);
#else
    cudaError_t e2 = cudaSuccess;
#endif
    if (e1 != cudaSuccess || e2 != cudaSuccess)
      return bail(fail(FLMR_ERR_CUDA, "cannot raise the dynamic shared memory limit to %d bytes: %s",
                       ScanSmem::kBytes, cudaGetErrorString(e1 != cudaSuccess ? e1 : e2)));
  }
  return FLMR_OK;
}

}  // namespace

// =================================== C ABI =============================================================
extern "C" {

const char* flmr_last_error(void) { return g_last_error.c_str(); }
int flmr_abi_version(void) { return FLMR_ABI_VERSION; }

int flmr_corpus_create(const void* tokens, const int32_t* h_doclens, int64_t n_passages, int dim,
                       int device, int64_t pid_base, unsigned flags, flmr_corpus_t** out) {
  if (!out) return fail(FLMR_ERR_INVALID_ARG, "out is null");
  *out = nullptr;
  if (dim != kDim) return fail(FLMR_ERR_UNSUPPORTED, "dim=%d (only %d is supported)", dim, kDim);
  if (n_passages <= 0 || !tokens || !h_doclens)
    return fail(FLMR_ERR_INVALID_ARG, "empty corpus or null tokens/doclens");
  std::vector<int64_t> soff(n_passages + 1), poff(n_passages + 1);
  soff[0] = poff[0] = 0;
  bool aligned = true;
  for (int64_t p = 0; p < n_passages; ++p) {
    const int32_t len = h_doclens[p];
    if (len < 1)
      return fail(FLMR_ERR_INVALID_ARG,
                  "passage %lld has length %d; zero-length passages have no defined MaxSim score",
                  (long long)p, len);
    soff[p + 1] = soff[p] + len;
    poff[p + 1] = poff[p] + (len + kGroup - 1) / kGroup * kGroup;
    aligned &= (len % kGroup == 0);
  }
  const int64_t n_rows = poff[n_passages];
  if (n_rows + kTileN >= (1ll << 31))
    return fail(FLMR_ERR_UNSUPPORTED, "%lld stored token rows exceed the 2^31 per-shard limit; shard the corpus",
                (long long)n_rows);

  DeviceGuard guard(device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  cudaDeviceProp prop;
  FLMR_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(FLMR_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is sm_100a only", device,
                prop.major, prop.minor);

  cudaPointerAttributes attr{};
  const bool is_device_ptr = (cudaPointerGetAttributes(&attr, tokens) == cudaSuccess) &&
                             (attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged);
  cudaGetLastError();
  if ((flags & FLMR_CORPUS_ADOPT) && !is_device_ptr)
    return fail(FLMR_ERR_INVALID_ARG, "FLMR_CORPUS_ADOPT requires a device pointer");
  if (is_device_ptr && attr.type == cudaMemoryTypeDevice && attr.device != device)
    return fail(FLMR_ERR_INVALID_ARG, "token matrix lives on device %d, corpus requested on %d",
                attr.device, device);

  flmr_corpus* c = new (std::nothrow) flmr_corpus();
  if (!c) return fail(FLMR_ERR_OOM, "host allocation failed");
  c->device = device;
  c->n_passages = n_passages;
  c->n_tokens = soff[n_passages];
  c->n_rows = n_rows;
  c->pid_base = pid_base;
  int rc = FLMR_OK;
  auto bail = [&](int code) {
    flmr_corpus_destroy(c);
    return code;
  };

  // --- token matrix residency ---
  if ((flags & FLMR_CORPUS_ADOPT) && aligned &&
      (reinterpret_cast<uintptr_t>(tokens) % 16 == 0)) {
    c->d_tokens = static_cast<__nv_bfloat16*>(const_cast<void*>(tokens));
    c->adopted = true;
  } else {
    const size_t bytes = static_cast<size_t>(n_rows) * kDim * 2;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&c->d_tokens), bytes);
    if (e != cudaSuccess)
      return bail(fail(FLMR_ERR_OOM, "cudaMalloc(%zu B) for the token matrix failed: %s", bytes,
                       cudaGetErrorString(e)));
    c->hbm_bytes += static_cast<int64_t>(bytes);
    int64_t *d_soff = nullptr, *d_poff_tmp = nullptr;
    if ((rc = dev_upload(&d_soff, soff, nullptr))) return bail(rc);
    if ((rc = dev_upload(&d_poff_tmp, poff, nullptr))) {
      cudaFree(d_soff);
      return bail(rc);
    }
    auto cleanup = [&]() {
      cudaFree(d_soff);
      cudaFree(d_poff_tmp);
    };
    if (is_device_ptr) {
      const int threads = 256;
      const int64_t blocks = (n_passages * 32 + threads - 1) / threads;
      flmr_repack_kernel<<<static_cast<unsigned>(blocks), threads>>>(
          static_cast<const uint4*>(tokens), d_soff, d_poff_tmp, reinterpret_cast<uint4*>(c->d_tokens),
          0, n_passages, 0);
      ++g_launches;
      e = cudaGetLastError();
      if (e == cudaSuccess) e = cudaDeviceSynchronize();
    } else {
      // host source: stage through a bounded device buffer, chunk by chunk of whole passages
      const int64_t chunk_rows = std::min<int64_t>(c->n_tokens, (256ll << 20) / (kDim * 2));
      int64_t max_len = 0;
      for (int64_t p = 0; p < n_passages; ++p) max_len = std::max<int64_t>(max_len, h_doclens[p]);
      const int64_t buf_rows = std::max(chunk_rows, max_len);
      uint4* d_stage = nullptr;
      e = cudaMalloc(reinterpret_cast<void**>(&d_stage), static_cast<size_t>(buf_rows) * kDim * 2);
      int64_t pa = 0;
      while (e == cudaSuccess && pa < n_passages) {
        int64_t pb = std::upper_bound(soff.begin() + pa, soff.end(), soff[pa] + buf_rows) - soff.begin() - 1;
        pb = std::max(pb, pa + 1);
        const int64_t rows = soff[pb] - soff[pa];
        e = cudaMemcpy(d_stage, static_cast<const char*>(tokens) + soff[pa] * kDim * 2,
                       static_cast<size_t>(rows) * kDim * 2, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) break;
        const int threads = 256;
        const int64_t cnt = pb - pa;
        const int64_t blocks = (cnt * 32 + threads - 1) / threads;
        flmr_repack_kernel<<<static_cast<unsigned>(blocks), threads>>>(
            d_stage, d_soff, d_poff_tmp, reinterpret_cast<uint4*>(c->d_tokens), pa, cnt, soff[pa]);
        ++g_launches;
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaDeviceSynchronize();
        pa = pb;
      }
      cudaFree(d_stage);
    }
    cleanup();
    if (e != cudaSuccess)
      return bail(fail(FLMR_ERR_CUDA, "corpus repack failed: %s", cudaGetErrorString(e)));
  }

  if ((rc = finish_corpus(c, poff, h_doclens, prop.multiProcessorCount))) return bail(rc);
  *out = c;
  return FLMR_OK;
}

int flmr_corpus_plaid_builder_create(const float* d_centroids, int64_t n_centroids, const float* d_bucket_weights,
                                     int nbits, const int32_t* h_doclens, int64_t n_passages, int dim, int device,
                                     int64_t pid_base, flmr_corpus_plaid_builder_t** out) {
  if (!out) return fail(FLMR_ERR_INVALID_ARG, "out is null");
  *out = nullptr;
  if (dim != kDim) return fail(FLMR_ERR_UNSUPPORTED, "dim=%d (only %d is supported)", dim, kDim);
  if (nbits != 1 && nbits != 2 && nbits != 4 && nbits != 8)
    return fail(FLMR_ERR_INVALID_ARG, "nbits=%d (the PLAID codec packs 1, 2, 4 or 8 bits per dim)", nbits);
  if (!d_centroids || !d_bucket_weights || !h_doclens) return fail(FLMR_ERR_INVALID_ARG, "null pointer");
  if (n_passages <= 0 || n_centroids < 1)
    return fail(FLMR_ERR_INVALID_ARG, "bad sizes n_passages=%lld n_centroids=%lld", (long long)n_passages,
                (long long)n_centroids);
  flmr_corpus_plaid_builder* b = new (std::nothrow) flmr_corpus_plaid_builder();
  if (!b) return fail(FLMR_ERR_OOM, "host allocation failed");
  auto bail = [&](int code) {
    flmr_corpus_plaid_builder_destroy(b);
    return code;
  };
  b->soff.resize(n_passages + 1);
  b->poff.resize(n_passages + 1);
  b->doclens.assign(h_doclens, h_doclens + n_passages);
  b->soff[0] = b->poff[0] = 0;
  for (int64_t p = 0; p < n_passages; ++p) {
    const int32_t len = h_doclens[p];
    if (len < 1)
      return bail(fail(FLMR_ERR_INVALID_ARG,
                       "passage %lld has length %d; zero-length passages have no defined MaxSim score",
                       (long long)p, len));
    b->soff[p + 1] = b->soff[p] + len;
    b->poff[p + 1] = b->poff[p] + (static_cast<int64_t>(len) + kGroup - 1) / kGroup * kGroup;
  }
  const int64_t n_rows = b->poff[n_passages];
  if (n_rows + kTileN >= (1ll << 31))
    return bail(fail(FLMR_ERR_UNSUPPORTED,
                     "%lld stored token rows exceed the 2^31 per-shard limit; shard the corpus", (long long)n_rows));
  DeviceGuard guard(device);
  if (!guard.ok) return bail(fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", device));
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return bail(fail(FLMR_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e)));
  if (prop.major != 10)
    return bail(fail(FLMR_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is sm_100a only", device, prop.major,
                     prop.minor));
  b->sm_count = prop.multiProcessorCount;
  if (int rc = check_device_ptrs({d_centroids, d_bucket_weights}, device)) return bail(rc);

  flmr_corpus* c = new (std::nothrow) flmr_corpus();
  if (!c) return bail(fail(FLMR_ERR_OOM, "host allocation failed"));
  b->corpus = c;
  c->device = device;
  c->n_passages = n_passages;
  c->n_tokens = b->soff[n_passages];
  c->n_rows = n_rows;
  c->pid_base = pid_base;
  c->nbits = nbits;
  c->n_centroids = n_centroids;
  const int packed = kDim * nbits / 8;
  const int64_t rows_alloc = n_rows + kTileN;   // + one tile of zero rows: the last tile never reads past the end
  auto alloc = [&](void** ptr, size_t bytes) -> int {
    cudaError_t err = cudaMalloc(ptr, bytes);
    if (err != cudaSuccess)
      return fail(FLMR_ERR_OOM, "cudaMalloc(%zu B) for the compressed corpus failed: %s", bytes,
                  cudaGetErrorString(err));
    c->hbm_bytes += static_cast<int64_t>(bytes);
    return FLMR_OK;
  };
  int rc;
  if ((rc = alloc(reinterpret_cast<void**>(&c->d_codes), static_cast<size_t>(rows_alloc) * 4)) ||
      (rc = alloc(reinterpret_cast<void**>(&c->d_residuals), static_cast<size_t>(rows_alloc) * packed)) ||
      (rc = alloc(reinterpret_cast<void**>(&c->d_inv_norm), static_cast<size_t>(rows_alloc) * 4)) ||
      (rc = alloc(reinterpret_cast<void**>(&c->d_centroids), static_cast<size_t>(n_centroids) * kDim * 4)) ||
      (rc = alloc(reinterpret_cast<void**>(&c->d_weights), static_cast<size_t>(4) << nbits)))
    return bail(rc);
  if ((rc = dev_upload(&b->d_soff, b->soff, nullptr)) || (rc = dev_upload(&b->d_poff, b->poff, nullptr)))
    return bail(rc);
  if ((e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaMalloc(reinterpret_cast<void**>(&b->d_bad), sizeof(int))) != cudaSuccess ||
      (e = cudaMemsetAsync(b->d_bad, 0, sizeof(int), b->stream)) != cudaSuccess ||
      (e = cudaMemcpyAsync(c->d_centroids, d_centroids, static_cast<size_t>(n_centroids) * kDim * 4,
                           cudaMemcpyDeviceToDevice, b->stream)) != cudaSuccess ||
      (e = cudaMemcpyAsync(c->d_weights, d_bucket_weights, static_cast<size_t>(4) << nbits, cudaMemcpyDeviceToDevice,
                           b->stream)) != cudaSuccess ||
      (e = cudaMemsetAsync(c->d_codes + n_rows, 0, kTileN * 4, b->stream)) != cudaSuccess ||
      (e = cudaMemsetAsync(c->d_residuals + n_rows * packed, 0, static_cast<size_t>(kTileN) * packed, b->stream)) !=
          cudaSuccess ||
      (e = cudaMemsetAsync(c->d_inv_norm + n_rows, 0, kTileN * 4, b->stream)) != cudaSuccess ||
      (e = cudaStreamSynchronize(b->stream)) != cudaSuccess)   // the caller may free the centroids on return
    return bail(fail(FLMR_ERR_CUDA, "compressed corpus setup: %s", cudaGetErrorString(e)));
  *out = b;
  return FLMR_OK;
}

int flmr_corpus_plaid_builder_append(flmr_corpus_plaid_builder_t* b, const int32_t* d_codes,
                                     const uint8_t* d_residuals, int64_t n_tokens) {
  if (!b || !d_codes || !d_residuals) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  flmr_corpus* c = b->corpus;
  const int64_t pa = b->passages_done;
  const int64_t want = b->soff[pa] + n_tokens;
  const int64_t pb = std::lower_bound(b->soff.begin() + pa, b->soff.end(), want) - b->soff.begin();
  if (n_tokens <= 0 || pb > c->n_passages || b->soff[pb] != want)
    return fail(FLMR_ERR_INVALID_ARG,
                "an append must hold whole passages: %lld tokens after passage %lld do not end on a passage boundary",
                (long long)n_tokens, (long long)pa);
  DeviceGuard guard(c->device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  if (int rc = check_device_ptrs({d_codes, d_residuals}, c->device)) return rc;
  const int threads = 256;
  const int64_t cnt = pb - pa;
  flmr_plaid_pack_kernel<<<static_cast<unsigned>((cnt * 32 + threads - 1) / threads), threads, 0, b->stream>>>(
      d_codes, d_residuals, b->d_soff, b->d_poff, pa, cnt, b->soff[pa], c->d_centroids, c->n_centroids, c->d_weights,
      c->nbits, c->d_codes, c->d_residuals, c->d_inv_norm, b->d_bad);
  ++g_launches;
  FLMR_CUDA(cudaGetLastError());
  FLMR_CUDA(cudaStreamSynchronize(b->stream));   // the caller may free or refill the chunk on return
  b->passages_done = pb;
  return FLMR_OK;
}

int flmr_corpus_plaid_builder_finish(flmr_corpus_plaid_builder_t* b, flmr_corpus_t** out) {
  if (!b || !out) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  flmr_corpus* c = b->corpus;
  if (b->passages_done != c->n_passages)
    return fail(FLMR_ERR_INVALID_ARG, "%lld of %lld passages appended", (long long)b->passages_done,
                (long long)c->n_passages);
  DeviceGuard guard(c->device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  int bad = 0;
  FLMR_CUDA(cudaMemcpyAsync(&bad, b->d_bad, sizeof(int), cudaMemcpyDeviceToHost, b->stream));
  FLMR_CUDA(cudaStreamSynchronize(b->stream));
  if (bad) return fail(FLMR_ERR_INVALID_ARG, "a centroid code is outside [0, %lld)", (long long)c->n_centroids);
  if (int rc = finish_corpus(c, b->poff, b->doclens.data(), b->sm_count)) return rc;
  b->corpus = nullptr;   // ownership passes to the caller
  flmr_corpus_plaid_builder_destroy(b);
  *out = c;
  return FLMR_OK;
}

int flmr_corpus_plaid_builder_destroy(flmr_corpus_plaid_builder_t* b) {
  if (!b) return FLMR_OK;
  if (b->stream) cudaStreamSynchronize(b->stream);
  cudaFree(b->d_soff);
  cudaFree(b->d_poff);
  cudaFree(b->d_bad);
  if (b->stream) cudaStreamDestroy(b->stream);
  if (b->corpus) flmr_corpus_destroy(b->corpus);
  delete b;
  return FLMR_OK;
}

int flmr_corpus_create_plaid(const int32_t* d_codes, const uint8_t* d_residuals, const float* d_centroids,
                             int64_t n_centroids, const float* d_bucket_weights, int nbits, const int32_t* h_doclens,
                             int64_t n_passages, int dim, int device, int64_t pid_base, flmr_corpus_t** out) {
  if (!out) return fail(FLMR_ERR_INVALID_ARG, "out is null");
  *out = nullptr;
  if (!d_codes || !d_residuals) return fail(FLMR_ERR_INVALID_ARG, "null pointer");
  flmr_corpus_plaid_builder_t* b = nullptr;
  int rc = flmr_corpus_plaid_builder_create(d_centroids, n_centroids, d_bucket_weights, nbits, h_doclens, n_passages,
                                            dim, device, pid_base, &b);
  if (rc) return rc;
  if ((rc = flmr_corpus_plaid_builder_append(b, d_codes, d_residuals, b->soff[n_passages])) ||
      (rc = flmr_corpus_plaid_builder_finish(b, out))) {
    const std::string msg = g_last_error;
    flmr_corpus_plaid_builder_destroy(b);
    g_last_error = msg;
    return rc;
  }
  return FLMR_OK;
}

int flmr_corpus_destroy(flmr_corpus_t* c) {
  if (!c) return FLMR_OK;
  DeviceGuard guard(c->device);
  if (!c->adopted && c->d_tokens) cudaFree(c->d_tokens);
  cudaFree(c->d_poff);
  cudaFree(c->d_doclen);
  cudaFree(c->d_cta_row_begin);
  cudaFree(c->d_cta_tile_base);
  cudaFree(c->d_tile_end_mask);
  cudaFree(c->d_tile_first_pid);
  cudaFree(c->d_pair_row_begin);
  cudaFree(c->d_pair_tile_base);
  cudaFree(c->d_pair_end_mask);
  cudaFree(c->d_pair_first_pid);
  cudaFree(c->d_codes);
  cudaFree(c->d_residuals);
  cudaFree(c->d_inv_norm);
  cudaFree(c->d_centroids);
  cudaFree(c->d_weights);
  delete c;
  return FLMR_OK;
}

int flmr_corpus_builder_create(const int32_t* h_doclens, int64_t n_passages, int dim, int device,
                               int64_t pid_base, flmr_corpus_builder_t** out) {
  if (!out) return fail(FLMR_ERR_INVALID_ARG, "out is null");
  *out = nullptr;
  if (dim != kDim) return fail(FLMR_ERR_UNSUPPORTED, "dim=%d (only %d is supported)", dim, kDim);
  if (n_passages <= 0 || !h_doclens) return fail(FLMR_ERR_INVALID_ARG, "empty corpus or null doclens");
  flmr_corpus_builder* b = new (std::nothrow) flmr_corpus_builder();
  if (!b) return fail(FLMR_ERR_OOM, "host allocation failed");
  auto bail = [&](int code) {
    flmr_corpus_builder_destroy(b);
    return code;
  };
  b->soff.resize(n_passages + 1);
  b->poff.resize(n_passages + 1);
  b->doclens.assign(h_doclens, h_doclens + n_passages);
  b->soff[0] = b->poff[0] = 0;
  for (int64_t p = 0; p < n_passages; ++p) {
    const int32_t len = h_doclens[p];
    if (len < 1)
      return bail(fail(FLMR_ERR_INVALID_ARG, "passage %lld has length %d; zero-length passages have no defined MaxSim score",
                       (long long)p, len));
    b->soff[p + 1] = b->soff[p] + len;
    b->poff[p + 1] = b->poff[p] + (len + kGroup - 1) / kGroup * kGroup;
    b->aligned &= (len % kGroup == 0);
  }
  const int64_t n_rows = b->poff[n_passages];
  if (n_rows + kTileN >= (1ll << 31))
    return bail(fail(FLMR_ERR_UNSUPPORTED, "%lld stored token rows exceed the 2^31 per-shard limit; shard the corpus",
                     (long long)n_rows));
  DeviceGuard guard(device);
  if (!guard.ok) return bail(fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", device));
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return bail(fail(FLMR_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e)));
  if (prop.major != 10)
    return bail(fail(FLMR_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is sm_100a only", device, prop.major,
                     prop.minor));
  b->sm_count = prop.multiProcessorCount;
  flmr_corpus* c = new (std::nothrow) flmr_corpus();
  if (!c) return bail(fail(FLMR_ERR_OOM, "host allocation failed"));
  b->corpus = c;
  c->device = device;
  c->n_passages = n_passages;
  c->n_tokens = b->soff[n_passages];
  c->n_rows = n_rows;
  c->pid_base = pid_base;
  const size_t bytes = static_cast<size_t>(n_rows) * kDim * 2;
  if ((e = cudaMalloc(reinterpret_cast<void**>(&c->d_tokens), bytes)) != cudaSuccess)
    return bail(fail(FLMR_ERR_OOM, "cudaMalloc(%zu B) for the token matrix failed: %s", bytes, cudaGetErrorString(e)));
  c->hbm_bytes += static_cast<int64_t>(bytes);
  const size_t buf_bytes = static_cast<size_t>(flmr_corpus_builder::kBufRows) * kDim * 2;
  if ((e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking)) != cudaSuccess)
    return bail(fail(FLMR_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)));
  for (int i = 0; i < flmr_corpus_builder::kBufs; ++i) {
    if ((e = cudaHostAlloc(&b->h_pin[i], buf_bytes, cudaHostAllocDefault)) != cudaSuccess ||
        (e = cudaEventCreateWithFlags(&b->free_ev[i], cudaEventDisableTiming)) != cudaSuccess ||
        (!b->aligned && (e = cudaMalloc(reinterpret_cast<void**>(&b->d_stage[i]), buf_bytes)) != cudaSuccess))
      return bail(fail(FLMR_ERR_OOM, "staging buffers: %s", cudaGetErrorString(e)));
  }
  if (!b->aligned) {
    int rc;
    if ((rc = dev_upload(&b->d_soff, b->soff, nullptr)) || (rc = dev_upload(&b->d_poff, b->poff, nullptr)))
      return bail(rc);
  }
  *out = b;
  return FLMR_OK;
}

extern "C++" {
namespace {
// Feed `n_rows` packed rows through the staging ring; `fill(dst, row0, rows)` writes rows [row0, row0 + rows) of
// this append into pinned memory (memcpy from a host buffer, or pread from a file).
template <typename Fill>
int builder_feed(flmr_corpus_builder* b, int64_t n_rows, Fill fill) {
  flmr_corpus* c = b->corpus;
  if (n_rows < 0 || b->rows_done + n_rows > c->n_tokens)
    return fail(FLMR_ERR_INVALID_ARG, "append of %lld rows overruns the %lld rows the doclens announce (%lld done)",
                (long long)n_rows, (long long)c->n_tokens, (long long)b->rows_done);
  DeviceGuard guard(c->device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  for (int64_t r0 = 0; r0 < n_rows; r0 += flmr_corpus_builder::kBufRows) {
    const int64_t rows = std::min<int64_t>(flmr_corpus_builder::kBufRows, n_rows - r0);
    const int i = b->next;
    b->next = (b->next + 1) % flmr_corpus_builder::kBufs;
    FLMR_CUDA(cudaEventSynchronize(b->free_ev[i]));          // the DMA that last read this buffer is done
    timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    if (int rc = fill(b->h_pin[i], r0, rows)) return rc;
    clock_gettime(CLOCK_MONOTONIC, &t1);
    b->fill_s += (t1.tv_sec - t0.tv_sec) + 1e-9 * (t1.tv_nsec - t0.tv_nsec);
    const size_t bytes = static_cast<size_t>(rows) * kDim * 2;
    const int64_t s0 = b->rows_done;
    if (b->aligned) {                                        // packed order == stored order: straight into place
      FLMR_CUDA(cudaMemcpyAsync(c->d_tokens + s0 * kDim, b->h_pin[i], bytes, cudaMemcpyHostToDevice, b->stream));
    } else {
      FLMR_CUDA(cudaMemcpyAsync(b->d_stage[i], b->h_pin[i], bytes, cudaMemcpyHostToDevice, b->stream));
      const int threads = 256;
      flmr_scatter_rows_kernel<<<static_cast<unsigned>((rows * 16 + threads - 1) / threads), threads, 0, b->stream>>>(
          b->d_stage[i], b->d_soff, b->d_poff, reinterpret_cast<uint4*>(c->d_tokens), s0, rows, c->n_passages);
      FLMR_CUDA(cudaGetLastError());
      ++g_launches;
    }
    FLMR_CUDA(cudaEventRecord(b->free_ev[i], b->stream));
    b->rows_done += rows;
  }
  return FLMR_OK;
}
}  // namespace
}  // extern "C++"

int flmr_corpus_builder_append(flmr_corpus_builder_t* b, const void* h_tokens_bf16, int64_t n_rows) {
  if (!b || !h_tokens_bf16) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  const char* src = static_cast<const char*>(h_tokens_bf16);
  return builder_feed(b, n_rows, [&](void* dst, int64_t r0, int64_t rows) {
    memcpy(dst, src + r0 * kDim * 2, static_cast<size_t>(rows) * kDim * 2);
    return FLMR_OK;
  });
}

int flmr_corpus_builder_append_file(flmr_corpus_builder_t* b, const char* path, int64_t byte_offset, int64_t n_rows) {
  if (!b || !path) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  const int fd = open(path, O_RDONLY);
  if (fd < 0) return fail(FLMR_ERR_INVALID_ARG, "cannot open %s: %s", path, strerror(errno));
  // the file is read straight into pinned memory by a few threads (pread is thread-safe): no intermediate copy
  const int rc = builder_feed(b, n_rows, [&](void* dst, int64_t r0, int64_t rows) {
    constexpr int kThreads = 8;
    const int64_t total = rows * kDim * 2, per = (total + kThreads - 1) / kThreads;
    int errs[kThreads] = {};
    std::thread th[kThreads];
    for (int t = 0; t < kThreads; ++t)
      th[t] = std::thread([&, t]() {
        int64_t a = t * per, e = std::min<int64_t>(total, a + per);
        while (a < e) {
          const ssize_t got = pread(fd, static_cast<char*>(dst) + a, static_cast<size_t>(e - a),
                                    byte_offset + r0 * kDim * 2 + a);
          if (got <= 0) {
            errs[t] = got == 0 ? -1 : errno;
            return;
          }
          a += got;
        }
      });
    for (auto& x : th) x.join();
    for (int e : errs)
      if (e) return fail(FLMR_ERR_INVALID_ARG, "short read from %s (%s)", path, e < 0 ? "end of file" : strerror(e));
    return static_cast<int>(FLMR_OK);
  });
  close(fd);
  return rc;
}

int flmr_corpus_builder_finish(flmr_corpus_builder_t* b, flmr_corpus_t** out, double* host_fill_seconds) {
  if (!b || !out) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  flmr_corpus* c = b->corpus;
  if (b->rows_done != c->n_tokens)
    return fail(FLMR_ERR_INVALID_ARG, "%lld rows appended, the doclens announce %lld", (long long)b->rows_done,
                (long long)c->n_tokens);
  DeviceGuard guard(c->device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  FLMR_CUDA(cudaStreamSynchronize(b->stream));
  if (int rc = finish_corpus(c, b->poff, b->doclens.data(), b->sm_count)) return rc;
  if (host_fill_seconds) *host_fill_seconds = b->fill_s;
  b->corpus = nullptr;     // ownership passes to the caller
  flmr_corpus_builder_destroy(b);
  *out = c;
  return FLMR_OK;
}

int flmr_corpus_builder_destroy(flmr_corpus_builder_t* b) {
  if (!b) return FLMR_OK;
  const int device = b->corpus ? b->corpus->device : -1;
  if (b->stream) cudaStreamSynchronize(b->stream);
  for (int i = 0; i < flmr_corpus_builder::kBufs; ++i) {
    if (b->h_pin[i]) cudaFreeHost(b->h_pin[i]);
    if (b->d_stage[i]) cudaFree(b->d_stage[i]);
    if (b->free_ev[i]) cudaEventDestroy(b->free_ev[i]);
  }
  cudaFree(b->d_soff);
  cudaFree(b->d_poff);
  if (b->stream) cudaStreamDestroy(b->stream);
  if (b->corpus) flmr_corpus_destroy(b->corpus);
  (void)device;
  delete b;
  return FLMR_OK;
}

int flmr_corpus_info(const flmr_corpus_t* c, flmr_corpus_info_t* out) {
  if (!c || !out) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  out->n_passages = c->n_passages;
  out->n_tokens = c->n_tokens;
  out->n_rows = c->n_rows;
  out->pid_base = c->pid_base;
  out->dim = kDim;
  out->device = c->device;
  out->n_ctas = c->n_ctas;
  out->adopted = c->adopted ? 1 : 0;
  out->n_tiles = c->n_tiles;
  out->hbm_bytes = c->hbm_bytes;
  return FLMR_OK;
}

int flmr_workspace_create(const flmr_corpus_t* c, int max_queries, int max_nq,
                          flmr_workspace_t** out) {
  if (!c || !out) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  if (max_queries < 1 || max_nq < 1)
    return fail(FLMR_ERR_INVALID_ARG, "max_queries=%d / max_nq=%d must be >= 1", max_queries, max_nq);
  DeviceGuard guard(c->device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  flmr_workspace* ws = new (std::nothrow) flmr_workspace();
  if (!ws) return fail(FLMR_ERR_OOM, "host allocation failed");
  ws->corpus = c;
  ws->device = c->device;
  ws->max_queries = max_queries;
  ws->max_nq = max_nq;
  auto bail = [&](int code) {
    flmr_workspace_destroy(ws);
    return code;
  };
  cudaError_t e;
  const size_t qbytes = static_cast<size_t>(kStageMaxPasses) * kMtMax * kTileM * kDim * 2;   // 10 MB
  if ((e = cudaMalloc(reinterpret_cast<void**>(&ws->d_qpad), qbytes)) != cudaSuccess ||
      (e = cudaMemset(ws->d_qpad, 0, qbytes)) != cudaSuccess ||
      (e = cudaMalloc(reinterpret_cast<void**>(&ws->d_cand_keys),
                      static_cast<size_t>(c->n_ctas) * max_queries * kMaxK * 8)) != cudaSuccess ||
      (e = cudaHostAlloc(reinterpret_cast<void**>(&ws->h_status), sizeof(int), cudaHostAllocMapped)) != cudaSuccess ||
      (e = cudaHostGetDevicePointer(reinterpret_cast<void**>(&ws->d_status), ws->h_status, 0)) != cudaSuccess)
    return bail(fail(FLMR_ERR_CUDA, "workspace allocation failed: %s", cudaGetErrorString(e)));
  *ws->h_status = 0;
  if (max_nq > kRbMax * 32) {   // row-sliced queries expected: size their partial-score rows now
    std::vector<PassPlan> plan;
    int group = 1;
    plan_passes(max_queries, max_nq, c->n_pairs > 0, &plan, &group, nullptr);
    if (int rc = ensure_acc(ws, static_cast<int64_t>(group) * c->n_passages)) return bail(rc);
  }
#ifdef FLMR_DEBUG
  if (const char* e = getenv("FLMR_DEBUG_MODE")) ws->dbg_mode = atoi(e);
  if (const char* e = getenv("FLMR_LANE_RBQ")) ws->dbg_lane_rbq = atoi(e);
#endif
  *out = ws;
  return FLMR_OK;
}

int flmr_workspace_destroy(flmr_workspace_t* ws) {
  if (!ws) return FLMR_OK;
  DeviceGuard guard(ws->device);
  cudaFree(ws->d_qpad);
  cudaFree(ws->d_cand_keys);
  cudaFree(ws->d_acc);
  if (ws->h_status) cudaFreeHost(ws->h_status);
  delete ws;
  return FLMR_OK;
}

int flmr_workspace_status(const flmr_workspace_t* ws, int* out) {
  if (!ws || !out) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  *out = ws->h_status ? *reinterpret_cast<volatile int*>(ws->h_status) : 0;
  return FLMR_OK;
}

int flmr_maxsim_scores(const flmr_corpus_t* corpus, flmr_workspace_t* ws, const void* d_q,
                       int n_queries, int nq, unsigned flags, float* d_out_scores, void* stream) {
  if (!d_out_scores) return fail(FLMR_ERR_INVALID_ARG, "d_out_scores is null");
  return run_search(corpus, ws, d_q, n_queries, nq, flags, 0, d_out_scores, nullptr, nullptr,
                    static_cast<cudaStream_t>(stream));
}

int flmr_maxsim_topk(const flmr_corpus_t* corpus, flmr_workspace_t* ws, const void* d_q,
                     int n_queries, int nq, int k, unsigned flags, float* d_out_scores,
                     int64_t* d_out_pids, void* stream) {
  if (!d_out_scores || !d_out_pids) return fail(FLMR_ERR_INVALID_ARG, "output pointer is null");
  if (k < 1) return fail(FLMR_ERR_INVALID_ARG, "k=%d must be >= 1", k);
  return run_search(corpus, ws, d_q, n_queries, nq, flags, k, nullptr, d_out_scores, d_out_pids,
                    static_cast<cudaStream_t>(stream));
}

int flmr_topk_merge(const float* d_in_scores, const int64_t* d_in_pids, int n_lists, int n_queries,
                    int k_in, int k_out, float* d_out_scores, int64_t* d_out_pids, int device,
                    void* stream) {
  if (!d_in_scores || !d_in_pids || !d_out_scores || !d_out_pids)
    return fail(FLMR_ERR_INVALID_ARG, "null pointer");
  if (n_lists < 1 || n_queries < 0 || k_in < 1 || k_out < 1 || k_out > kMaxK)
    return fail(FLMR_ERR_INVALID_ARG, "bad merge shape n_lists=%d n_queries=%d k_in=%d k_out=%d",
                n_lists, n_queries, k_in, k_out);
  if (static_cast<int64_t>(n_lists) * k_in > kMergeThreads * kMergePer)
    return fail(FLMR_ERR_UNSUPPORTED, "n_lists*k_in = %lld exceeds merge capacity %d",
                (long long)n_lists * k_in, kMergeThreads * kMergePer);
  if (n_queries == 0) return FLMR_OK;
  DeviceGuard guard(device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  flmr_merge_kernel<<<n_queries, kMergeThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      nullptr, d_in_scores, d_in_pids, n_lists, n_queries, k_in, k_out, 0, d_out_scores, d_out_pids, 0);
  FLMR_CUDA(cudaGetLastError());
  ++g_launches;
  return FLMR_OK;
}

int flmr_plaid_decode(const int32_t* d_codes, const uint8_t* d_residuals, int64_t n_tokens,
                      const float* d_centroids, int64_t n_centroids, const float* d_bucket_weights,
                      int nbits, int dim, int normalize, void* d_out_bf16, int device, void* stream) {
  if (!d_codes || !d_residuals || !d_centroids || !d_bucket_weights || !d_out_bf16)
    return fail(FLMR_ERR_INVALID_ARG, "null pointer");
  if (dim != kDim) return fail(FLMR_ERR_UNSUPPORTED, "dim=%d (only %d is supported)", dim, kDim);
  if (nbits != 1 && nbits != 2 && nbits != 4 && nbits != 8)
    return fail(FLMR_ERR_INVALID_ARG, "nbits=%d (the PLAID codec packs 1, 2, 4 or 8 bits per dim)", nbits);
  if (n_tokens < 0 || n_centroids < 1) return fail(FLMR_ERR_INVALID_ARG, "bad sizes");
  if (n_tokens == 0) return FLMR_OK;
  DeviceGuard guard(device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // "a code was out of range" flag: one pinned + mapped word per host thread, reused by every call
  thread_local int* h_bad = nullptr;
  if (!h_bad) FLMR_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&h_bad), sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
  int* d_bad = nullptr;
  FLMR_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void**>(&d_bad), h_bad, 0));
  *reinterpret_cast<volatile int*>(h_bad) = 0;
  cudaError_t e = cudaSuccess;
  const int threads = 256;
  const int64_t want = (n_tokens * 32 + threads - 1) / threads;
  const int blocks = static_cast<int>(std::min<int64_t>(want, 148 * 16));
  if (e == cudaSuccess) {
    flmr_plaid_decode_kernel<<<blocks, threads, 0, st>>>(d_codes, d_residuals, d_centroids,
                                                       d_bucket_weights, nbits, normalize, n_tokens,
                                                       n_centroids, static_cast<uint2*>(d_out_bf16), d_bad);
    ++g_launches;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  const int bad = *reinterpret_cast<volatile int*>(h_bad);
  if (e != cudaSuccess) return fail(FLMR_ERR_CUDA, "plaid decode failed: %s", cudaGetErrorString(e));
  if (bad) return fail(FLMR_ERR_INVALID_ARG, "a centroid code is outside [0, %lld)", (long long)n_centroids);
  return FLMR_OK;
}

int flmr_topk_select(const float* d_scores, int n_queries, int64_t n, int k, int64_t pid_base,
                     float* d_out_scores, int64_t* d_out_pids, int device, void* stream) {
  if (!d_scores || !d_out_scores || !d_out_pids) return fail(FLMR_ERR_INVALID_ARG, "null pointer");
  if (n_queries < 0 || n < 1 || k < 1) return fail(FLMR_ERR_INVALID_ARG, "bad shape n_queries=%d n=%lld k=%d", n_queries, (long long)n, k);
  if (k > kSelectMaxK) return fail(FLMR_ERR_UNSUPPORTED, "k=%d exceeds the selection capacity %d", k, kSelectMaxK);
  if (n >= (1ll << 32)) return fail(FLMR_ERR_UNSUPPORTED, "rows of 2^32 or more scores are not supported");
  if (n_queries == 0) return FLMR_OK;
  DeviceGuard guard(device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  flmr_select_kernel<<<n_queries, kSelectThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      d_scores, n, k, pid_base, d_out_scores, d_out_pids);
  FLMR_CUDA(cudaGetLastError());
  ++g_launches;
  return FLMR_OK;
}

int flmr_corpus_gather(const flmr_corpus_t* c, const int64_t* d_pids, int64_t n_pids, int nd_max,
                       void* d_out_bf16, uint8_t* d_mask, void* stream) {
  if (!c || !d_pids || !d_out_bf16) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  if (n_pids < 0 || nd_max < 1) return fail(FLMR_ERR_INVALID_ARG, "bad shape n_pids=%lld nd_max=%d", (long long)n_pids, nd_max);
  if (n_pids == 0) return FLMR_OK;
  DeviceGuard guard(c->device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  const int threads = 256;
  const int64_t blocks = (n_pids * nd_max * 32 + threads - 1) / threads;
  if (blocks > 0x7fffffffll) return fail(FLMR_ERR_UNSUPPORTED, "gather of %lld x %d rows is too large", (long long)n_pids, nd_max);
  if (c->nbits) {   // compressed corpus: decode the gathered rows
    flmr_gather_plaid_kernel<<<static_cast<unsigned>(blocks), threads, 0, static_cast<cudaStream_t>(stream)>>>(
        c->d_codes, c->d_residuals, c->d_inv_norm, c->d_centroids, c->d_weights, c->nbits, c->d_poff, c->d_doclen,
        d_pids, n_pids, nd_max, c->n_passages, c->pid_base, static_cast<uint2*>(d_out_bf16), d_mask);
    FLMR_CUDA(cudaGetLastError());
    ++g_launches;
    return FLMR_OK;
  }
  flmr_gather_kernel<<<static_cast<unsigned>(blocks), threads, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const uint2*>(c->d_tokens), c->d_poff, c->d_doclen, d_pids, n_pids, nd_max,
      c->n_passages, c->pid_base, static_cast<uint2*>(d_out_bf16), d_mask);
  FLMR_CUDA(cudaGetLastError());
  ++g_launches;
  return FLMR_OK;
}

// ---- the tcgen05 route of the arg-max forward (flmr_train_tc_kernel.cuh) --------------------------------------
thread_local int g_argmax_path = 0;   // 0 = by size, 1 = warp-MMA kernel, 2 = tcgen05 kernel (flmr_debug_set_argmax_path)

// The library's own stream-ordered memory pool (one per device) for per-call scratch: it keeps what it has
// been given (release threshold = max), so after the first call an allocation is a pointer bump in stream order —
// the default pool hands memory back to the driver at every synchronisation and re-maps it on the next call.
static int scratch_pool(cudaMemPool_t* out) {
  static cudaMemPool_t pools[64] = {};
  static std::mutex mu;
  int dev = 0;
  FLMR_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  if (!pools[dev & 63]) {
    cudaMemPoolProps props{};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = dev;
    cudaMemPool_t p = nullptr;
    FLMR_CUDA(cudaMemPoolCreate(&p, &props));
    uint64_t keep = ~0ull;
    FLMR_CUDA(cudaMemPoolSetAttribute(p, cudaMemPoolAttrReleaseThreshold, &keep));
    pools[dev & 63] = p;
  }
  *out = pools[dev & 63];
  return FLMR_OK;
}

static int argmax_tc(const void* d_q, int n_queries, int nq, const void* d_docs, const uint8_t* d_mask, int n_per,
                     int stride_b, int nd, int32_t* d_argmax, float* d_rowmax, cudaStream_t st) {
  const int64_t n_total = stride_b ? static_cast<int64_t>(n_queries) * n_per : n_per;
  const int nd_c = (nd + kTcTile - 1) / kTcTile * kTcTile;
  if (n_total * nd_c + kTcTile >= (1ll << 31) || static_cast<int64_t>(n_queries) * nq + kTcTile >= (1ll << 31))
    return fail(FLMR_ERR_UNSUPPORTED, "arg-max operands exceed 2^31 rows");
  // stream-ordered scratch: packed documents, their index maps and lengths (freed in stream order below)
  const size_t b_dc = static_cast<size_t>(n_total) * nd_c * kDim * 2;
  const size_t b_map = static_cast<size_t>(n_total) * nd_c * sizeof(int32_t);
  const size_t b_len = static_cast<size_t>(n_total) * sizeof(int32_t);
  char* scratch = nullptr;
  cudaMemPool_t pool = nullptr;
  if (int rc = scratch_pool(&pool)) return rc;
  FLMR_CUDA(cudaMallocFromPoolAsync(reinterpret_cast<void**>(&scratch), b_dc + b_map + b_len + 256, pool, st));
  uint4* dc = reinterpret_cast<uint4*>(scratch);
  int32_t* idx_map = reinterpret_cast<int32_t*>(scratch + b_dc);
  int32_t* doc_len = reinterpret_cast<int32_t*>(scratch + b_dc + b_map);
  auto done = [&](int code) {
    cudaFreeAsync(scratch, st);
    return code;
  };
  flmr_compact_docs_kernel<<<static_cast<unsigned>(n_total), 256, 0, st>>>(
      static_cast<const uint4*>(d_docs), d_mask, nd, nd_c, dc, idx_map, doc_len);
  ++g_launches;
  CUtensorMap tmap_q, tmap_d;
  int rc;
  if ((rc = encode_rows_map(&tmap_q, d_q, static_cast<uint64_t>(n_queries) * nq, kTcTile))) return done(rc);
  if ((rc = encode_rows_map(&tmap_d, dc, static_cast<uint64_t>(n_total) * nd_c, kTcTile))) return done(rc);
  static std::once_flag attr_once[64];
  int dev = 0;
  cudaGetDevice(&dev);
  cudaError_t attr_err = cudaSuccess;
  std::call_once(attr_once[dev & 63], [&]() {
    attr_err = cudaFuncSetAttribute(flmr_argmax_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kTcSmemBytes);
  });
  if (attr_err != cudaSuccess)
    return done(fail(FLMR_ERR_CUDA, "cannot raise the dynamic shared memory limit: %s", cudaGetErrorString(attr_err)));
  const int n_tiles = (nq + kTcTile - 1) / kTcTile;
  // documents per CTA: a CTA pays ~5 us of set-up (TMEM allocation, barriers, query tile, pipeline fill) before its
  // first MMA and ~0.3 us per 128-token chunk after it; pick the split with the shortest modelled makespan
  // (waves of 148 CTAs x per-CTA time): many documents per CTA unless that leaves SMs idle
  const int64_t pairs_q = static_cast<int64_t>(n_queries) * n_tiles;
  int dpc = 1;
  double best_t = 1e30;
  for (int d = 1; d <= 32 && d <= std::max(1, n_per); ++d) {
    const int64_t ctas = pairs_q * ((n_per + d - 1) / d);
    const double t = static_cast<double>((ctas + 147) / 148) * (5.0 + d * 0.3 * (nd_c / kTcTile));
    if (t < best_t) {
      best_t = t;
      dpc = d;
    }
  }
  ArgmaxTcParams prm{};
  prm.doc_len = doc_len;
  prm.idx_map = idx_map;
  prm.arg = d_argmax;
  prm.rowmax = d_rowmax;
  prm.nq = nq;
  prm.nd_c = nd_c;
  prm.n_per = n_per;
  prm.stride_b = stride_b;
  prm.docs_per_cta = dpc;
  prm.status = nullptr;
  dim3 grid(static_cast<unsigned>((n_per + dpc - 1) / dpc), static_cast<unsigned>(n_tiles),
            static_cast<unsigned>(n_queries));
  flmr_argmax_tc_kernel<<<grid, kTcThreads, kTcSmemBytes, st>>>(tmap_q, tmap_d, prm);
  cudaError_t e = cudaGetLastError();
  ++g_launches;
  if (e != cudaSuccess) return done(fail(FLMR_ERR_CUDA, "flmr_argmax_tc_kernel launch failed: %s", cudaGetErrorString(e)));
  return done(FLMR_OK);
}

// n_per documents per query; stride_b = 0: all queries meet documents [0, n_per) (all pairs),
// stride_b = n_per: query b meets documents [b * n_per, (b + 1) * n_per) (block diagonal).
static int argmax_impl(const void* d_q, int n_queries, int nq, const void* d_docs, const uint8_t* d_mask,
                       int n_per, int stride_b, int nd, int32_t* d_argmax, float* d_rowmax, int device,
                       void* stream) {
  if (!d_q || !d_docs || !d_mask || !d_argmax) return fail(FLMR_ERR_INVALID_ARG, "null pointer");
  if (n_queries < 0 || n_per < 0 || nq <= 0 || nd <= 0)
    return fail(FLMR_ERR_INVALID_ARG, "bad shape n_queries=%d nq=%d n_docs=%d nd=%d", n_queries, nq, n_per, nd);
  if (n_queries > 65535 || n_per > 65535)
    return fail(FLMR_ERR_UNSUPPORTED, "n_queries / n_docs above 65535 (training-sized batches only)");
  if (n_queries == 0 || n_per == 0) return FLMR_OK;
  DeviceGuard guard(device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  // tcgen05 route when the contraction is worth a TMA / TMEM pipeline (>= 16M query-row x token pairs and full
  // tiles), warp-MMA kernel below that: a RAG re-score of 5 passages stays on the small kernel
  const double pairs = static_cast<double>(n_queries) * n_per * nq * nd;
  const bool tc_ok = n_queries <= 65535 && (nq + kTcTile - 1) / kTcTile <= 65535;
  if (tc_ok && (g_argmax_path == 2 || (g_argmax_path == 0 && nq >= 64 && nd >= 128 && pairs >= 16e6)))
    return argmax_tc(d_q, n_queries, nq, d_docs, d_mask, n_per, stride_b, nd, d_argmax, d_rowmax,
                     static_cast<cudaStream_t>(stream));
  dim3 grid(static_cast<unsigned>((nq + kArgTile - 1) / kArgTile), static_cast<unsigned>(n_per),
            static_cast<unsigned>(n_queries));
#ifdef FLMR_DEBUG
  // debug builds: FLMR_ARGMAX_SIMT=1 selects the plain-FMA twin (cross-check / A-B timing)
  const char* simt = getenv("FLMR_ARGMAX_SIMT");
  if (simt && atoi(simt)) {
    flmr_argmax_kernel<<<grid, kArgThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        static_cast<const __nv_bfloat16*>(d_q), static_cast<const __nv_bfloat16*>(d_docs), d_mask, nq, nd,
        n_per, stride_b, d_argmax, d_rowmax);
    FLMR_CUDA(cudaGetLastError());
    ++g_launches;
    return FLMR_OK;
  }
#endif
  flmr_argmax_mma_kernel<<<grid, kMmaThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(d_q), static_cast<const __nv_bfloat16*>(d_docs), d_mask, nq, nd,
      n_per, stride_b, d_argmax, d_rowmax);
  FLMR_CUDA(cudaGetLastError());
  ++g_launches;
  return FLMR_OK;
}

static int backward_impl(const void* d_q, int n_queries, int nq, const void* d_docs, int n_per, int stride_b,
                         int nd, const int32_t* d_argmax, const float* d_grad, float* d_dq, float* d_dd,
                         int device, void* stream) {
  if (!d_q || !d_docs || !d_argmax || !d_grad) return fail(FLMR_ERR_INVALID_ARG, "null pointer");
  if (n_queries < 0 || n_per < 0 || nq <= 0 || nd <= 0)
    return fail(FLMR_ERR_INVALID_ARG, "bad shape n_queries=%d nq=%d n_docs=%d nd=%d", n_queries, nq, n_per, nd);
  DeviceGuard guard(device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int threads = 256;
  const int64_t n_docs_total = stride_b ? static_cast<int64_t>(n_queries) * n_per : n_per;
  if (d_dq && n_queries > 0) {
    const int64_t warps = static_cast<int64_t>(n_queries) * nq;
    if (n_per == 0) {
      FLMR_CUDA(cudaMemsetAsync(d_dq, 0, static_cast<size_t>(warps) * kDim * sizeof(float), st));
    } else {
      flmr_bwd_dq_kernel<<<static_cast<unsigned>((warps * 32 + threads - 1) / threads), threads, 0, st>>>(
          static_cast<const __nv_bfloat16*>(d_docs), d_argmax, d_grad, n_queries, nq, n_per, nd, stride_b, d_dq);
      FLMR_CUDA(cudaGetLastError());
      ++g_launches;
    }
  }
  if (d_dd && n_docs_total > 0) {
    FLMR_CUDA(cudaMemsetAsync(d_dd, 0, static_cast<size_t>(n_docs_total) * nd * kDim * sizeof(float), st));
    const int64_t warps = static_cast<int64_t>(n_queries) * n_per * nq;
    if (warps > 0) {
      if ((warps * 32 + threads - 1) / threads > 0x7fffffffll)
        return fail(FLMR_ERR_UNSUPPORTED, "backward grid too large (%lld warps)", (long long)warps);
      flmr_bwd_dd_kernel<<<static_cast<unsigned>((warps * 32 + threads - 1) / threads), threads, 0, st>>>(
          static_cast<const __nv_bfloat16*>(d_q), d_argmax, d_grad, n_queries, nq, n_per, nd, stride_b, d_dd);
      FLMR_CUDA(cudaGetLastError());
      ++g_launches;
    }
  }
  return FLMR_OK;
}

int flmr_maxsim_argmax(const void* d_q, int n_queries, int nq, const void* d_docs,
                       const uint8_t* d_mask, int n_docs, int nd, int32_t* d_argmax, float* d_rowmax,
                       int device, void* stream) {
  return argmax_impl(d_q, n_queries, nq, d_docs, d_mask, n_docs, 0, nd, d_argmax, d_rowmax, device, stream);
}

int flmr_maxsim_backward(const void* d_q, int n_queries, int nq, const void* d_docs, int n_docs, int nd,
                         const int32_t* d_argmax, const float* d_grad, float* d_dq, float* d_dd,
                         int device, void* stream) {
  return backward_impl(d_q, n_queries, nq, d_docs, n_docs, 0, nd, d_argmax, d_grad, d_dq, d_dd, device, stream);
}

int flmr_ib_loss(const float* d_rowmax, int n_queries, int n_docs, int nq, int nway, int label0,
                 float* d_scores, float* d_loss_per_query, float* d_dscores, int device, void* stream) {
  if (!d_rowmax || !d_scores || !d_loss_per_query || !d_dscores) return fail(FLMR_ERR_INVALID_ARG, "null pointer");
  if (n_queries < 1 || n_docs < 1 || nq < 1 || nway < 1 || label0 < 0 ||
      static_cast<int64_t>(label0) + static_cast<int64_t>(n_queries - 1) * nway >= n_docs)
    return fail(FLMR_ERR_INVALID_ARG, "bad shape n_queries=%d n_docs=%d nq=%d nway=%d label0=%d", n_queries, n_docs,
                nq, nway, label0);
  if (static_cast<size_t>(n_docs) * sizeof(float) > 200 * 1024)
    return fail(FLMR_ERR_UNSUPPORTED, "%d documents per query exceed the loss kernel's shared memory", n_docs);
  DeviceGuard guard(device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  const size_t smem = static_cast<size_t>(n_docs) * sizeof(float);
  if (smem > 48 * 1024)
    FLMR_CUDA(cudaFuncSetAttribute(flmr_ib_loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  flmr_ib_loss_kernel<<<n_queries, kIbThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      d_rowmax, n_queries, n_docs, nq, nway, label0, d_scores, d_loss_per_query, d_dscores);
  FLMR_CUDA(cudaGetLastError());
  ++g_launches;
  return FLMR_OK;
}

int flmr_maxsim_argmax_grouped(const void* d_q, int n_queries, int nq, const void* d_docs,
                               const uint8_t* d_mask, int docs_per_query, int nd, int32_t* d_argmax,
                               float* d_rowmax, int device, void* stream) {
  if (docs_per_query < 1) return fail(FLMR_ERR_INVALID_ARG, "docs_per_query=%d must be >= 1", docs_per_query);
  return argmax_impl(d_q, n_queries, nq, d_docs, d_mask, docs_per_query, docs_per_query, nd, d_argmax, d_rowmax,
                     device, stream);
}

int flmr_maxsim_backward_grouped(const void* d_q, int n_queries, int nq, const void* d_docs,
                                 int docs_per_query, int nd, const int32_t* d_argmax, const float* d_grad,
                                 float* d_dq, float* d_dd, int device, void* stream) {
  if (docs_per_query < 1) return fail(FLMR_ERR_INVALID_ARG, "docs_per_query=%d must be >= 1", docs_per_query);
  return backward_impl(d_q, n_queries, nq, d_docs, docs_per_query, docs_per_query, nd, d_argmax, d_grad, d_dq,
                       d_dd, device, stream);
}

int flmr_debug_maxsim_scores_simt(const flmr_corpus_t* c, const void* d_q, int n_queries, int nq,
                                  unsigned flags, float* d_out_scores, void* stream) {
  if (!c || !d_q || !d_out_scores) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  if (n_queries <= 0 || nq <= 0) return fail(FLMR_ERR_INVALID_ARG, "bad shape");
  if (c->n_passages > 0x7fffffffll || n_queries > 65535)
    return fail(FLMR_ERR_UNSUPPORTED, "SIMT cross-check grid too large");
  if (c->nbits) return fail(FLMR_ERR_UNSUPPORTED, "the SIMT cross-check reads bf16 tokens; this corpus is compressed");
  DeviceGuard guard(c->device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  const int threads = nq >= 256 ? 256 : (nq > 128 ? 256 : 128);
  dim3 grid(static_cast<unsigned>(c->n_passages), static_cast<unsigned>(n_queries));
  flmr_simt_maxsim_kernel<<<grid, threads, 0, static_cast<cudaStream_t>(stream)>>>(
      c->d_tokens, c->d_poff, c->d_doclen, static_cast<const __nv_bfloat16*>(d_q), nq,
      (flags & FLMR_FLAG_RELU) ? 0.f : -INFINITY, d_out_scores, c->n_passages);
  FLMR_CUDA(cudaGetLastError());
  ++g_launches;
  return FLMR_OK;
}

int flmr_debug_set_scan_variant(int variant) {
  if (variant != 0 && variant != 2 && variant != 3 && variant != 4)
    return fail(FLMR_ERR_INVALID_ARG, "variant must be 0 (default), 2 or 3 (epilogue warpgroups) or 4 (CTA-pair experiment)");
  g_scan_variant = variant;
  return FLMR_OK;
}

int flmr_debug_set_argmax_path(int path) {
  if (path < 0 || path > 2) return fail(FLMR_ERR_INVALID_ARG, "path must be 0 (by size), 1 (warp-MMA) or 2 (tcgen05)");
  g_argmax_path = path;
  return FLMR_OK;
}

int flmr_debug_build_partition(const int32_t* h_doclens, int64_t n_passages, int n_ctas,
                               int32_t* cta_row_begin, int64_t* cta_tile_base,
                               uint32_t* tile_end_mask, int32_t* tile_first_pid,
                               int64_t tile_capacity, int64_t* n_tiles_out) {
  if (!h_doclens || n_passages <= 0 || n_ctas < 1 || !cta_row_begin || !cta_tile_base || !n_tiles_out)
    return fail(FLMR_ERR_INVALID_ARG, "bad argument");
  std::vector<int64_t> poff(n_passages + 1);
  poff[0] = 0;
  for (int64_t p = 0; p < n_passages; ++p) {
    if (h_doclens[p] < 1) return fail(FLMR_ERR_INVALID_ARG, "passage %lld has length %d", (long long)p, h_doclens[p]);
    poff[p + 1] = poff[p] + (h_doclens[p] + kGroup - 1) / kGroup * kGroup;
  }
  n_ctas = static_cast<int>(std::min<int64_t>(n_ctas, n_passages));
  std::vector<int32_t> rb, fp;
  std::vector<int64_t> tb;
  std::vector<uint32_t> em;
  build_partition(poff, n_ctas, kTileN, &rb, &tb, &em, &fp);
  *n_tiles_out = static_cast<int64_t>(em.size());
  std::copy(rb.begin(), rb.end(), cta_row_begin);
  std::copy(tb.begin(), tb.end(), cta_tile_base);
  if (tile_end_mask && tile_first_pid) {
    if (static_cast<int64_t>(em.size()) > tile_capacity)
      return fail(FLMR_ERR_INVALID_ARG, "tile_capacity %lld < %zu tiles", (long long)tile_capacity, em.size());
    std::copy(em.begin(), em.end(), tile_end_mask);
    std::copy(fp.begin(), fp.end(), tile_first_pid);
  }
  return FLMR_OK;
}

int flmr_debug_plan_passes(int n_queries, int nq, int allow_pair, int32_t* out_plan, int capacity, int* n_passes_out) {
  if (n_queries < 0 || nq <= 0 || !n_passes_out) return fail(FLMR_ERR_INVALID_ARG, "bad argument");
  std::vector<PassPlan> plan;
  int group = 1;
  plan_passes(n_queries, nq, allow_pair != 0, &plan, &group, nullptr);
  *n_passes_out = static_cast<int>(plan.size());
  if (out_plan) {
    if (static_cast<int>(plan.size()) > capacity)
      return fail(FLMR_ERR_INVALID_ARG, "capacity %d < %zu passes", capacity, plan.size());
    for (size_t i = 0; i < plan.size(); ++i) {
      const PassPlan& q = plan[i];
      const int32_t row[8] = {q.q_first, q.n_q, q.row0, q.rows, q.rbq, q.n_mtiles, q.flags, q.group_first + q.acc_slot};
      std::copy(row, row + 8, out_plan + i * 8);
    }
  }
  return FLMR_OK;
}

int flmr_comm_unique_id(void* out_id_128_bytes) {
  if (!out_id_128_bytes) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  const NcclApi* api = nullptr;
  if (int rc = load_nccl(&api)) return rc;
  FLMR_NCCL(api, api->GetUniqueId(out_id_128_bytes));
  return FLMR_OK;
}

int flmr_comm_create(const void* id_128_bytes, int rank, int world_size, int device, flmr_comm_t** out) {
  if (!id_128_bytes || !out) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  if (world_size < 1 || rank < 0 || rank >= world_size)
    return fail(FLMR_ERR_INVALID_ARG, "bad rank %d / world size %d", rank, world_size);
  const NcclApi* api = nullptr;
  if (int rc = load_nccl(&api)) return rc;
  DeviceGuard guard(device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", device);
  flmr_comm* c = new (std::nothrow) flmr_comm();
  if (!c) return fail(FLMR_ERR_OOM, "host allocation failed");
  NcclId id;
  memcpy(id.internal, id_128_bytes, sizeof id.internal);
  const int r = api->CommInitRank(&c->nccl, world_size, id, rank);
  if (r != 0) {
    delete c;
    return fail(FLMR_ERR_CUDA, "ncclCommInitRank failed: %s", api->GetErrorString(r));
  }
  c->rank = rank;
  c->world = world_size;
  c->device = device;
  c->owned = true;
  *out = c;
  return FLMR_OK;
}

int flmr_comm_adopt(void* nccl_comm, int device, flmr_comm_t** out) {
  if (!nccl_comm || !out) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  *out = nullptr;
  const NcclApi* api = nullptr;
  if (int rc = load_nccl(&api)) return rc;
  flmr_comm* c = new (std::nothrow) flmr_comm();
  if (!c) return fail(FLMR_ERR_OOM, "host allocation failed");
  c->nccl = nccl_comm;
  c->device = device;
  int r = api->CommCount(nccl_comm, &c->world);
  if (r == 0) r = api->CommUserRank(nccl_comm, &c->rank);
  if (r != 0) {
    delete c;
    return fail(FLMR_ERR_CUDA, "ncclCommCount / ncclCommUserRank failed: %s", api->GetErrorString(r));
  }
  *out = c;
  return FLMR_OK;
}

int flmr_comm_destroy(flmr_comm_t* c) {
  if (!c) return FLMR_OK;
  DeviceGuard guard(c->device);
  cudaFree(c->d_send_s);
  cudaFree(c->d_send_p);
  cudaFree(c->d_recv_s);
  cudaFree(c->d_recv_p);
  if (c->owned && c->nccl) {
    const NcclApi* api = nullptr;
    if (load_nccl(&api) == FLMR_OK) api->CommDestroy(c->nccl);
  }
  delete c;
  return FLMR_OK;
}

int flmr_comm_info(const flmr_comm_t* c, int* rank, int* world_size) {
  if (!c) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  if (rank) *rank = c->rank;
  if (world_size) *world_size = c->world;
  return FLMR_OK;
}

int flmr_topk_exchange(flmr_comm_t* c, const float* d_scores, const int64_t* d_pids, int n_queries, int k_in,
                       int k_out, float* d_out_scores, int64_t* d_out_pids, void* stream) {
  if (!c || !d_scores || !d_pids || !d_out_scores || !d_out_pids) return fail(FLMR_ERR_INVALID_ARG, "null argument");
  if (n_queries < 0 || k_in < 1 || k_out < 1 || k_out > kMaxK)
    return fail(FLMR_ERR_INVALID_ARG, "bad shape n_queries=%d k_in=%d k_out=%d", n_queries, k_in, k_out);
  if (static_cast<int64_t>(c->world) * k_in > kMergeThreads * kMergePer)
    return fail(FLMR_ERR_UNSUPPORTED, "world*k_in = %lld exceeds merge capacity %d", (long long)c->world * k_in,
                kMergeThreads * kMergePer);
  if (n_queries == 0) return FLMR_OK;
  const NcclApi* api = nullptr;
  if (int rc = load_nccl(&api)) return rc;
  DeviceGuard guard(c->device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", c->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n = static_cast<int64_t>(n_queries) * k_in;
  if (c->capacity < n) {   // (grown only when a call brings more entries than any before: not on the steady path)
    cudaFree(c->d_recv_s);
    cudaFree(c->d_recv_p);
    c->d_recv_s = nullptr;
    c->d_recv_p = nullptr;
    c->capacity = 0;
    FLMR_CUDA(cudaMalloc(reinterpret_cast<void**>(&c->d_recv_s), static_cast<size_t>(n) * c->world * sizeof(float)));
    FLMR_CUDA(cudaMalloc(reinterpret_cast<void**>(&c->d_recv_p), static_cast<size_t>(n) * c->world * sizeof(int64_t)));
    c->capacity = n;
  }
  // one exchange step: both all-gathers in ONE NCCL group (a single fused launch on the wire), then the merge
  FLMR_NCCL(api, api->GroupStart());
  int r1 = api->AllGather(d_scores, c->d_recv_s, static_cast<size_t>(n), kNcclFloat32, c->nccl, st);
  int r2 = api->AllGather(d_pids, c->d_recv_p, static_cast<size_t>(n), kNcclInt64, c->nccl, st);
  FLMR_NCCL(api, api->GroupEnd());
  if (r1 != 0 || r2 != 0)
    return fail(FLMR_ERR_CUDA, "ncclAllGather failed: %s", api->GetErrorString(r1 ? r1 : r2));
  flmr_merge_kernel<<<n_queries, kMergeThreads, 0, st>>>(nullptr, c->d_recv_s, c->d_recv_p, c->world, n_queries,
                                                        k_in, k_out, 0, d_out_scores, d_out_pids, 0);
  FLMR_CUDA(cudaGetLastError());
  ++g_launches;
  return FLMR_OK;
}

int flmr_maxsim_topk_sharded(const flmr_corpus_t* corpus, flmr_workspace_t* ws, flmr_comm_t* comm, const void* d_q,
                             int n_queries, int nq, int k, unsigned flags, float* d_out_scores,
                             int64_t* d_out_pids, void* stream) {
  if (!comm) return fail(FLMR_ERR_INVALID_ARG, "comm is null");
  if (!d_out_scores || !d_out_pids) return fail(FLMR_ERR_INVALID_ARG, "output pointer is null");
  if (k < 1 || k > kMaxK) return fail(FLMR_ERR_INVALID_ARG, "k=%d outside [1, %d]", k, kMaxK);
  if (corpus && corpus->device != comm->device)
    return fail(FLMR_ERR_INVALID_ARG, "corpus on device %d, communicator on device %d", corpus->device, comm->device);
  if (n_queries <= 0) return n_queries == 0 ? FLMR_OK : fail(FLMR_ERR_INVALID_ARG, "bad n_queries=%d", n_queries);
  DeviceGuard guard(comm->device);
  if (!guard.ok) return fail(FLMR_ERR_CUDA, "cudaSetDevice(%d) failed", comm->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t n = static_cast<int64_t>(n_queries) * k;
  if (comm->capacity < n || !comm->d_send_s) {
    cudaFree(comm->d_send_s);
    cudaFree(comm->d_send_p);
    comm->d_send_s = nullptr;
    comm->d_send_p = nullptr;
    FLMR_CUDA(cudaMalloc(reinterpret_cast<void**>(&comm->d_send_s), static_cast<size_t>(n) * sizeof(float)));
    FLMR_CUDA(cudaMalloc(reinterpret_cast<void**>(&comm->d_send_p), static_cast<size_t>(n) * sizeof(int64_t)));
  }
  // this rank's shard (the fused scan fills short lists with (-inf, -1), which the merge ignores)
  if (int rc = run_search(corpus, ws, d_q, n_queries, nq, flags, k, nullptr, comm->d_send_s, comm->d_send_p, st))
    return rc;
  return flmr_topk_exchange(comm, comm->d_send_s, comm->d_send_p, n_queries, k, k, d_out_scores, d_out_pids, stream);
}

int64_t flmr_launch_count(int reset) {
  const int64_t v = g_launches;
  if (reset) g_launches = 0;
  return v;
}

int flmr_set_profiling(int enable) {
  g_profiling = enable != 0;
  return FLMR_OK;
}

int flmr_scan_kernel_stats(double* total_ms, int64_t* launches, int reset) {
  double tot = 0.0;
  int64_t n = 0;
  for (auto& ev : g_scan_events) {
    float ms = 0.f;
    if (cudaEventSynchronize(ev.b) == cudaSuccess && cudaEventElapsedTime(&ms, ev.a, ev.b) == cudaSuccess) {
      tot += ms;
      ++n;
    }
  }
  if (total_ms) *total_ms = tot;
  if (launches) *launches = n;
  if (reset) {
    for (auto& ev : g_scan_events) {
      cudaEventDestroy(ev.a);
      cudaEventDestroy(ev.b);
    }
    g_scan_events.clear();
  }
  return FLMR_OK;
}

}  // extern "C"
