// Similarity + top-k over one row shard of the descriptor database.
//
// Replaces the reference's dense  scores = matmul(q, db)  (dirtorch/utils/common.py:30-38, test_dir.py:145) +
// per-query sort (datasets/generic.py:207,221) for the first k ranks, without materialising the Q x N matrix:
//
//   1. queries -> fp16, counters / retry gates / status cleared                    (search_prep_kernel)
//   2. seed:   tcgen05 GEMM of the queries against the first S rows.  The epilogue keeps the maximum of every group
//              of 32 consecutive rows (PERS_EPI_SIM_GMAX; 1/32 of the dense score traffic); per query the k-th largest
//              group maximum t_S has >= k rows at or above it, so it is a lower bound on the final k-th score.
//              (fewer than k groups: dense scores, PERS_EPI_SIM_DENSE)                 (kth_dense_kernel)
//   3. filter: tcgen05 GEMM against all N rows; the epilogue appends (score,row) to the query's candidate list
//              only when score >= t_S - 2*eps16                                     (PERS_EPI_SIM_FILTER)
//      (for N <= S step 3 is a scan of the dense scores instead: dense_compact_kernel)
//   4. select: exact k-th largest candidate score t (radix select, cand_kth_kernel).  A query whose list overflowed
//              gets a tighter threshold from what was captured and raises a device-side gate; the (always enqueued)
//              retry passes of steps 3-4 return at once unless their gate is up - no host round trip.
//   5. finish: survivors = candidates with score >= t - 2*eps16, exact re-scoring (fp64 accumulation of the fp32
//              rows) and sort (score desc, index asc), one launch, one block per query      (search_finish_kernel)
// The only host synchronisation is the status check at the very end (overflow that the retries could not resolve);
// with option deferred_check it moves to dirb200_index_check / the start of the next search.
//
// eps16 bounds |fp16-path score - exact score| (unit-norm rows: 2 * 2^-11 from the operand roundings + fp32
// accumulation, default 1.2e-3); any row of the true top-k then satisfies the step-3 and step-4 conditions, so the
// result is the exact top-k (same argument twice).  Candidate-buffer overflow raises the threshold from what was
// captured and re-runs the filter pass.  With several shards the phases are split (search_begin / search_finish)
// so that the caller can MIN-reduce the per-shard selection thresholds in between (see cand_kth_kernel).
// The GEMMs run on the persistent warp-specialised kernel of conv_pers.cuh (128 x 256 tiles, K = D).
#include <math.h>

#include <limits.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "conv.h"
#include "conv_pers.cuh"

namespace dirb {
namespace {

constexpr int SEL_THREADS = 512;

// Exact score of one (query, row) pair by one warp: fp64 accumulation of the fp32 products, fixed summation order
// (lane-strided float4 loads, xor-shuffle tree).  Every exact score of the library comes from this function, so two
// evaluations of the same pair - or of two identical rows - are bit-identical wherever they are computed.
__device__ __forceinline__ double exact_dot_warp(const float* __restrict__ qrow, const float* __restrict__ dbrow, int D,
                                                 int lane) {
  const float4* a = reinterpret_cast<const float4*>(qrow);
  const float4* b = reinterpret_cast<const float4*>(dbrow);
  double acc = 0.0;
  for (int i = lane; i < D / 4; i += 32) {
    const float4 x = __ldg(a + i), y = __ldg(b + i);
    acc += static_cast<double>(x.x) * y.x;
    acc += static_cast<double>(x.y) * y.y;
    acc += static_cast<double>(x.z) * y.z;
    acc += static_cast<double>(x.w) * y.w;
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  return acc;
}

__device__ __forceinline__ uint32_t f2key(float f) {  // monotone increasing map float -> uint32
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

struct DenseAcc {
  const float* p;
  __device__ float operator()(int i) const { return p[i]; }
};
struct CandAcc {
  const unsigned long long* p;
  __device__ float operator()(int i) const { return __uint_as_float(static_cast<uint32_t>(p[i] >> 32)); }
};

// k-th largest of n values (block-wide MSB-first radix select, 4 passes of 8 bits). n < k -> -inf.
template <class Acc>
__device__ float block_kth_largest(Acc acc, int n, int k, uint32_t* hist /*[256]*/, uint32_t* bc /*[2]*/) {
  if (n < k) return -INFINITY;
  uint32_t prefix = 0, mask = 0;
  int kk = k;
  for (int pass = 3; pass >= 0; --pass) {
    const int shift = pass * 8;
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    // similarity scores share their high bits, so most keys of a pass land in one or two bins: aggregate the
    // lanes of a warp that hit the same bin and let one of them add the whole group
    const int n_round = (n + 31) & ~31;
    for (int i = threadIdx.x; i < n_round; i += blockDim.x) {
      uint32_t bin = 0xffffffffu;
      if (i < n) {
        const uint32_t key = f2key(acc(i));
        if ((key & mask) == prefix) bin = (key >> shift) & 255u;
      }
      const uint32_t peers = __match_any_sync(0xffffffffu, bin);
      if (bin != 0xffffffffu && (threadIdx.x & 31) == (__ffs(peers) - 1)) atomicAdd(&hist[bin], static_cast<uint32_t>(__popc(peers)));
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      // Find the bin holding the kk-th largest key: lane l owns bins [8l, 8l+8); a suffix scan over the lanes gives
      // the number of keys in higher bins, the owning lane walks its 8 bins.  (A single thread walking 256 bins
      // serially cost ~10 us per pass.)
      const int lane = threadIdx.x;
      uint32_t loc[8], sum = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        loc[j] = hist[8 * lane + j];
        sum += loc[j];
      }
      uint32_t suf = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_down_sync(0xffffffffu, suf, o);
        if (lane + o < 32) suf += v;
      }
      const uint32_t above = suf - sum;
      const uint32_t want = static_cast<uint32_t>(kk);
      if (above < want && want <= above + sum) {
        uint32_t cum = above;
#pragma unroll
        for (int j = 7; j >= 0; --j) {
          if (cum + loc[j] >= want) {
            bc[0] = 8 * lane + j;
            bc[1] = want - cum;
            break;
          }
          cum += loc[j];
        }
      }
    }
    __syncthreads();
    prefix |= bc[0] << shift;
    mask |= 255u << shift;
    kk = bc[1];
    __syncthreads();
  }
  return key2f(prefix);
}

// thr[q] = (k-th largest of dense[q][0..S)) - band; k2 > 0: also thr2[q] = (k2-th largest) - band (the seed bound a shard
// contributes to the MIN over the shards, see dirb200_index_search_sharded).
__global__ void __launch_bounds__(SEL_THREADS) kth_dense_kernel(const float* __restrict__ dense, int64_t ld, int S,
                                                                int k, float band, float* __restrict__ thr, int k2,
                                                                float* __restrict__ thr2) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t bc[2];
  const int q = blockIdx.x;
  const float t = block_kth_largest(DenseAcc{dense + q * ld}, S, k, hist, bc);
  if (threadIdx.x == 0) thr[q] = t - band;
  if (k2 > 0) {
    __syncthreads();
    const float t2 = (k2 == k) ? t : block_kth_largest(DenseAcc{dense + q * ld}, S, k2, hist, bc);
    if (threadIdx.x == 0) thr2[q] = t2 - band;
  }
}

// N <= S: candidates straight from the dense scores.
__global__ void dense_compact_kernel(const float* __restrict__ dense, int64_t ld, int N, const float* __restrict__ thr,
                                     unsigned long long* __restrict__ cand, int* __restrict__ cnt, int cap,
                                     const int* __restrict__ gate) {
  if (gate != nullptr && *reinterpret_cast<const volatile int*>(gate) == 0) return;
  const int q = blockIdx.y;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const float v = dense[q * ld + n];
  if (v >= thr[q]) {
    const int pos = atomicAdd(cnt + q, 1);
    if (pos < cap)
      cand[static_cast<int64_t>(q) * cap + pos] = (static_cast<unsigned long long>(__float_as_uint(v)) << 32) | static_cast<unsigned>(n);
  }
}

// Status block of a search (device, 8 x u64; copied to pinned host memory at the end of phase 2):
//   [0] error bits: 1 = candidate overflow left after the last retry pass, 2 = more than cap2 survivors for some query
//   [1] candidates captured (sum over queries)   [2] survivors re-scored   [3] retry passes that actually ran
enum { ST_ERR = 0, ST_CAND = 1, ST_SURV = 2, ST_RETRIES = 3, ST_WORDS = 8 };

// Per query: exact k-th and k_shard-th largest candidate scores (fp16-path scores).
//   kth_k[q]  : local k-th best - always a valid lower bound on the global k-th best
//   sel[q]    : local min(k_shard, N)-th best; the MINIMUM of this value over all shards is a valid and much tighter
//               lower bound on the global k-th best as long as the shards certify k rows between them,
//               sum_g min(k_shard, N_g) >= min(k, N_total) (shard g holds min(k_shard, N_g) rows at or above its own
//               value) - the caller picks k_shard accordingly (ceil(k / shards) for evenly filled shards, see
//               dist.py: shard_quota) and min-reduces sel.
// Overflow (cnt > cap) is resolved on the device: the query's list is emptied, the tighter threshold
// kth(captured) - band goes to thr[q] and gate_out[0] is raised, which arms the next (gated) filter pass + selection;
// finished queries get thr[q] = +inf so that a re-run leaves them alone.  `gate_in` != nullptr: this launch is itself
// such a retry pass and returns at once unless *gate_in != 0.  `last` = no further retry follows: a remaining
// overflow becomes error bit 1.
__global__ void __launch_bounds__(SEL_THREADS) cand_kth_kernel(const unsigned long long* __restrict__ cand,
                                                               int* __restrict__ cnt, int cap, int k, int k_shard,
                                                               float band, float* __restrict__ kth_k,
                                                               float* __restrict__ sel, float* __restrict__ thr,
                                                               int64_t n_rows, const int* __restrict__ gate_in,
                                                               int* __restrict__ gate_out, int last,
                                                               unsigned long long* __restrict__ status) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t bc[2];
  if (gate_in != nullptr && *reinterpret_cast<const volatile int*>(gate_in) == 0) return;
  const int q = blockIdx.x;
  if (gate_in != nullptr && q == 0 && threadIdx.x == 0) atomicAdd(status + ST_RETRIES, 1ull);
  const int total = cnt[q];
  const int n = min(total, cap);
  const float thr_in = thr[q];                 // what the filter pass used: (a lower bound on the global k-th best) - band
  const unsigned long long* c = cand + static_cast<int64_t>(q) * cap;
  const int kk = (n_rows < static_cast<int64_t>(k)) ? static_cast<int>(n_rows) : k;
  const float t = block_kth_largest(CandAcc{c}, n, kk, hist, bc);
  if (total > cap) {
    if (threadIdx.x == 0) {
      if (last) {
        atomicOr(status + ST_ERR, 1ull);
        kth_k[q] = INFINITY;      // no survivors for this query; the error is reported by the status check
        sel[q] = INFINITY;
        thr[q] = INFINITY;
      } else {
        thr[q] = t - band;
        cnt[q] = 0;               // the retry pass refills the list from scratch
        *gate_out = 1;
      }
    }
    return;
  }
  float ts = t;
  if (k_shard < kk) {
    __syncthreads();
    ts = block_kth_largest(CandAcc{c}, n, k_shard, hist, bc);
  }
  // Fewer than k_shard rows above a filter threshold that came from the other shards: this shard's k_shard-th best lies
  // below that bound, which is itself a valid lower bound on the global k-th best - report the bound instead of -inf
  // (the MIN over the shards must stay selective).  Shards with fewer than k_shard ROWS report their worst row.
  if (ts == -INFINITY && n_rows >= static_cast<int64_t>(k_shard) && thr_in != -INFINITY) ts = thr_in + band;
  if (threadIdx.x == 0) {
    kth_k[q] = t;
    sel[q] = ts;
    thr[q] = INFINITY;
  }
}

// Start of a search: queries -> fp16 (the A operand of the tensor-core passes), candidate counters, retry gates and
// the status block cleared.  One launch instead of a conversion kernel + memsets.
__global__ void search_prep_kernel(const float* __restrict__ q32, __half* __restrict__ q16, int64_t n, int* __restrict__ cnt,
                                   int Q, int* __restrict__ gates, int n_gates, unsigned long long* __restrict__ status) {
  const int64_t gtid = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  const int64_t i = gtid * 4;
  if (i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(q32 + i);
    uint2 o;
    o.x = pack_h2(v.x, v.y);
    o.y = pack_h2(v.z, v.w);
    *reinterpret_cast<uint2*>(q16 + i) = o;
  } else {
    for (int64_t j = i; j < n; ++j) q16[j] = __float2half_rn(q32[j]);
  }
  if (gtid < Q) cnt[gtid] = 0;
  if (gtid < n_gates) gates[gtid] = 0;
  if (gtid < ST_WORDS) status[gtid] = 0ull;
}

// Empty shard: nothing can be selected (+inf never lowers the MIN over the shards) / nothing to return.
__global__ void fill_f32_kernel(float* __restrict__ p, int n, float v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
__global__ void fill_empty_result_kernel(double* __restrict__ sc, int64_t* __restrict__ ix, int64_t n) {
  const int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x;
  if (i < n) {
    sc[i] = -INFINITY;
    ix[i] = -1;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Peer exchange of the sharded search (dirb200_index_search_sharded): the two collectives of the protocol - MIN of the
// per-shard selection thresholds, gather of the per-shard lists - are done by the producing kernels themselves with
// stores into the peers' memory over NVLink (P2P mappings, CUDA IPC between the one-process-per-GPU ranks), and the
// consuming kernels wait on flags in their OWN memory.  Every rank owns one exchange buffer of identical layout:
//   [0]   epoch (u32; the current search, bumped by the last block of the merge)      [16..] block-completion counters
//   [64]  flag_sel[2][8]   [128] flag_list[2][8]   [192] flag_seed[2][8]
//                                                    written by rank g into slot g of EVERY rank (release, system scope)
//   [256] sel[2][G][max_q], seed[2][G][max_q] fp32 | score[2][G][max_q*max_k] fp64 | idx[2][G][max_q*max_k] int64
// Slots are double-buffered by epoch parity: rank r overwrites parity p two searches later, after it has seen every peer's
// lists of the search in between - which a peer publishes only after its own merge of the earlier search has read them.
constexpr int X_MAXW = 8;
constexpr int X_OFF_EPOCH = 0, X_OFF_CNT = 16, X_OFF_FSEL = 64, X_OFF_FLIST = 128, X_OFF_FSEED = 192, X_OFF_SEL = 256;
constexpr int X_TAB_SEL = 0, X_TAB_SEED = 1;              // float tables [2][G][max_q]: selection thresholds, seed bounds
struct PeerX {
  int world, rank, max_q, max_k;      // world == 0: no exchange (plain single-shard kernels)
  uint8_t* peer[X_MAXW];              // every rank's exchange buffer as mapped in THIS process (peer[rank] = own)
};
__host__ __device__ inline size_t x_tab_bytes(int world, int max_q) { return (static_cast<size_t>(2) * world * max_q * 4 + 255) / 256 * 256; }
__host__ __device__ inline size_t x_sel_bytes(int world, int max_q) { return 2 * x_tab_bytes(world, max_q); }
__host__ __device__ inline size_t x_off_tab(int tab, int world, int max_q) { return X_OFF_SEL + tab * x_tab_bytes(world, max_q); }
__host__ __device__ inline size_t x_list_elems(int max_q, int max_k) { return static_cast<size_t>(max_q) * max_k; }
__host__ __device__ inline size_t x_off_score(int world, int max_q) { return X_OFF_SEL + x_sel_bytes(world, max_q); }
__host__ __device__ inline size_t x_off_idx(int world, int max_q, int max_k) {
  return x_off_score(world, max_q) + static_cast<size_t>(2) * world * x_list_elems(max_q, max_k) * 8;
}
__host__ __device__ inline size_t x_total_bytes(int world, int max_q, int max_k) {
  return x_off_idx(world, max_q, max_k) + static_cast<size_t>(2) * world * x_list_elems(max_q, max_k) * 8;
}

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t x_epoch(const PeerX& x) {
  return *reinterpret_cast<const volatile uint32_t*>(x.peer[x.rank] + X_OFF_EPOCH);
}
// One thread: wait until every rank has published epoch e in this rank's flag row.  Bounded (~10 s): a peer that never
// arrives becomes error bit 4 of the status block instead of a hung GPU.
__device__ __forceinline__ void x_wait_flags(const PeerX& x, int flag_off, uint32_t e, unsigned long long* status) {
  const uint32_t* f = reinterpret_cast<const uint32_t*>(x.peer[x.rank] + flag_off) + (e & 1u) * X_MAXW;
  for (int g = 0; g < x.world; ++g) {
    uint32_t spins = 0;
    while (static_cast<int32_t>(ld_acquire_sys(f + g) - e) < 0) {
      __nanosleep(100);
      if (++spins > (1u << 26)) {
        if (status) atomicOr(status + ST_ERR, 4ull);
        break;
      }
    }
  }
}
// End of a producing kernel: the LAST block to get here publishes epoch e in slot `rank` of every rank's flag row.
__device__ __forceinline__ void x_signal_when_all_blocks_done(const PeerX& x, int cnt_slot, int flag_off, uint32_t e) {
  __threadfence_system();                                   // this thread's stores to the peers before its block's arrival
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int* cnt = reinterpret_cast<unsigned int*>(x.peer[x.rank] + X_OFF_CNT) + cnt_slot;
    if (atomicAdd(cnt, 1u) == gridDim.x * gridDim.y - 1u) {
      *cnt = 0u;
      __threadfence_system();
      for (int g = 0; g < x.world; ++g)
        st_release_sys(reinterpret_cast<uint32_t*>(x.peer[g] + flag_off) + (e & 1u) * X_MAXW + x.rank, e);
    }
  }
}

// This shard's per-query values (seed bounds / selection thresholds) into slot `rank` of every rank's float table.
__global__ void tab_push_kernel(PeerX x, const float* __restrict__ local, int Q, int tab, int flag_off, int cnt_slot) {
  const uint32_t e = x_epoch(x);
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < Q) {
    const float v = local[q];
    const size_t o = x_off_tab(tab, x.world, x.max_q) + ((static_cast<size_t>(e & 1u) * x.world + x.rank) * x.max_q + q) * 4;
    for (int g = 0; g < x.world; ++g) *reinterpret_cast<float*>(x.peer[g] + o) = v;
  }
  x_signal_when_all_blocks_done(x, cnt_slot, flag_off, e);
}

// MIN over the shards of one float table, per query (waits for every rank's flag).
__device__ __forceinline__ float x_tab_min(const PeerX& x, int tab, uint32_t epoch, int q) {
  const float* t = reinterpret_cast<const float*>(x.peer[x.rank] + x_off_tab(tab, x.world, x.max_q)) +
                   static_cast<size_t>(epoch & 1u) * x.world * x.max_q;
  float m = INFINITY;
  for (int g = 0; g < x.world; ++g) m = fminf(m, __ldcg(t + static_cast<size_t>(g) * x.max_q + q));
  return m;
}

// Filter threshold of the sharded search: thr[q] = max(local k-th seed bound, MIN over the shards of their c-th seed
// bounds).  Both are lower bounds on the global k-th best score (the second by the shard-quota argument: every shard
// certifies c rows at or above its own value, G * c >= k), and the second is ~10x more selective on a G = 8 split:
// the local one keeps ~k / S of the rows as candidates, the global one ~c / S.
__global__ void thr_min_kernel(PeerX x, float* __restrict__ thr, int Q, unsigned long long* status) {
  const uint32_t e = x_epoch(x);
  if (threadIdx.x == 0) x_wait_flags(x, X_OFF_FSEED, e, status);
  __syncthreads();
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < Q) thr[q] = fmaxf(thr[q], x_tab_min(x, X_TAB_SEED, e, q));
}

// Phase 2 of a search in ONE launch, one block per query:
//   survivors = candidates with fp16-path score >= max(sel[q], kth_k[q]) - band   (compacted into shared memory)
//   exact score of each survivor = fp64-accumulated dot product of the fp32 rows  (one warp per survivor)
//   bitonic sort by (score desc, row asc), first k written as (fp64 score, int64 global index).
// Replaces three launches whose grids were sized for the worst case (cap2 survivors per query) although a shard of a
// G-way split keeps only ~1.4 k / G rows per query.
constexpr int FIN_THREADS = 512;
__global__ void __launch_bounds__(FIN_THREADS) search_finish_kernel(
    const unsigned long long* __restrict__ cand, const int* __restrict__ cnt, int cap, const float* __restrict__ kth_k,
    const float* __restrict__ sel, float band, const float* __restrict__ q32, const float* __restrict__ db32, int D,
    int cap2, int64_t offset, int k, double* __restrict__ out_score, int64_t* __restrict__ out_idx,
    unsigned long long* __restrict__ status, const PeerX x) {
  // x.world > 0 (sharded search over peer memory): the selection threshold is the MINIMUM over the shards of the values the
  // peers stored into this rank's sel table (waits for their flags), and the ordered list goes to slot `rank` of EVERY
  // rank's list table instead of out_score / out_idx - MIN all-reduce and all-gather fused into this kernel.
  extern __shared__ uint8_t sm[];
  __shared__ int s_n;
  __shared__ float s_sel;
  double* sc = reinterpret_cast<double*>(sm);          // [cap2]
  int* ix = reinterpret_cast<int*>(sc + cap2);         // [cap2]
  const int q = blockIdx.x;
  const int n = cnt ? min(cnt[q], cap) : 0;            // (empty shard: no candidate buffers at all)
  const unsigned long long* c = cand + static_cast<int64_t>(q) * cap;
  const uint32_t epoch = x.world > 0 ? x_epoch(x) : 0u;
  if (threadIdx.x == 0) {
    s_n = 0;
    if (x.world > 0) {
      x_wait_flags(x, X_OFF_FSEL, epoch, status);
      s_sel = x_tab_min(x, X_TAB_SEL, epoch, q);
    } else {
      s_sel = sel[q];
    }
  }
  __syncthreads();
  const float t2 = fmaxf(s_sel, kth_k ? kth_k[q] : INFINITY) - band;
  for (int i = threadIdx.x; i < n; i += FIN_THREADS) {
    const unsigned long long e = c[i];
    if (__uint_as_float(static_cast<uint32_t>(e >> 32)) >= t2) {
      const int pos = atomicAdd(&s_n, 1);
      if (pos < cap2) ix[pos] = static_cast<int>(e & 0xffffffffu);
    }
  }
  __syncthreads();
  const int found = s_n;
  const int ns = min(found, cap2);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int w = warp; w < ns; w += FIN_THREADS / 32) {
    const double acc = exact_dot_warp(q32 + static_cast<int64_t>(q) * D, db32 + static_cast<int64_t>(ix[w]) * D, D, lane);
    if (lane == 0) sc[w] = acc;
  }
  int P = 2;
  while (P < ns) P <<= 1;
  for (int i = ns + threadIdx.x; i < P; i += FIN_THREADS) {
    sc[i] = -INFINITY;
    ix[i] = INT_MAX;
  }
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1) {
    for (int st = size >> 1; st > 0; st >>= 1) {
      for (int i = threadIdx.x; i < P / 2; i += FIN_THREADS) {
        const int lo = 2 * i - (i & (st - 1));
        const int hi = lo + st;
        const bool up = ((lo & size) == 0);  // "up" = this block sorted best-first
        const double va = sc[lo], vb = sc[hi];
        const int ia = ix[lo], ib = ix[hi];
        const bool a_first = (va > vb) || (va == vb && ia < ib);
        if (a_first != up) {
          sc[lo] = vb; sc[hi] = va;
          ix[lo] = ib; ix[hi] = ia;
        }
      }
      __syncthreads();
    }
  }
  if (x.world > 0) {
    const size_t slot = (static_cast<size_t>(epoch & 1u) * x.world + x.rank) * x_list_elems(x.max_q, x.max_k) + static_cast<size_t>(q) * k;
    const size_t o_sc = x_off_score(x.world, x.max_q) + slot * 8, o_ix = x_off_idx(x.world, x.max_q, x.max_k) + slot * 8;
    for (int i = threadIdx.x; i < k; i += FIN_THREADS) {
      const bool ok = i < ns;
      const double vs = ok ? sc[i] : -INFINITY;
      const int64_t vi = ok ? static_cast<int64_t>(ix[i]) + offset : -1;
      for (int g = 0; g < x.world; ++g) {
        reinterpret_cast<double*>(x.peer[g] + o_sc)[i] = vs;
        reinterpret_cast<int64_t*>(x.peer[g] + o_ix)[i] = vi;
      }
    }
  } else {
    for (int i = threadIdx.x; i < k; i += FIN_THREADS) {
      const bool ok = i < ns;
      out_score[static_cast<int64_t>(q) * k + i] = ok ? sc[i] : -INFINITY;
      out_idx[static_cast<int64_t>(q) * k + i] = ok ? static_cast<int64_t>(ix[i]) + offset : -1;
    }
  }
  if (threadIdx.x == 0) {
    if (found > cap2) atomicOr(status + ST_ERR, 2ull);
    atomicAdd(status + ST_CAND, static_cast<unsigned long long>(n));
    atomicAdd(status + ST_SURV, static_cast<unsigned long long>(ns));
  }
  if (x.world > 0) x_signal_when_all_blocks_done(x, 1, X_OFF_FLIST, epoch);
}

// Exact dense scores for small evaluation sets: grid (ceil(N/8), ceil(Q/4)), warp = one db row x 4 queries.
__global__ void scores_exact_kernel(const float* __restrict__ q, int Q, const float* __restrict__ db, int64_t N, int D,
                                    float* __restrict__ out) {
  const int64_t n = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  const int q0 = blockIdx.y * 4;
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  double acc[4] = {0, 0, 0, 0};
  const float4* b = reinterpret_cast<const float4*>(db + n * D);
  for (int i = lane; i < D / 4; i += 32) {
    const float4 y = __ldg(b + i);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (q0 + j < Q) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(q + static_cast<int64_t>(q0 + j) * D) + i);
        acc[j] += static_cast<double>(x.x) * y.x + static_cast<double>(x.y) * y.y + static_cast<double>(x.z) * y.z +
                  static_cast<double>(x.w) * y.w;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    double v = acc[j];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0 && q0 + j < Q) out[static_cast<int64_t>(q0 + j) * N + n] = static_cast<float>(v);
  }
}

// alpha query expansion: out_i = normalize(q_i + sum_j db[idx_ij] * s_ij^alpha)   (test_dir.py:38-42; the mean's
// 1/(k+1) cancels in the normalisation).  partial: un-normalised neighbour sum only.
__global__ void aqe_kernel(const float* __restrict__ q, int D, const float* __restrict__ db, const int64_t* __restrict__ nn,
                           const double* __restrict__ ns, int k, double alpha, int partial, int64_t row_offset,
                           int64_t n_rows, float* __restrict__ out) {
  extern __shared__ float wts[];  // [k] weights, then [k] local rows (as int64 pairs of floats)
  __shared__ float sh[32];
  int64_t* rows = reinterpret_cast<int64_t*>(wts + ((k + 1) & ~1));
  const int i = blockIdx.x;
  for (int j = threadIdx.x; j < k; j += blockDim.x) {
    int64_t r = nn[static_cast<int64_t>(i) * k + j];
    if (r >= 0 && (partial || n_rows > 0)) {         // sharded: global index -> local row of this shard, or "not mine"
                                                     // (partial sums are per shard by definition, also for an EMPTY shard)
      r -= row_offset;
      if (r < 0 || r >= n_rows) r = -1;
    }
    rows[j] = r;
    wts[j] = (r >= 0) ? static_cast<float>(pow(ns[static_cast<int64_t>(i) * k + j], alpha)) : 0.f;
  }
  __syncthreads();
  float ss = 0.f;
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float acc = partial ? 0.f : q[static_cast<int64_t>(i) * D + c];
    for (int j = 0; j < k; ++j) {
      const int64_t r = rows[j];
      if (r >= 0) acc += db[r * D + c] * wts[j];
    }
    out[static_cast<int64_t>(i) * D + c] = acc;
    ss += acc * acc;
  }
  if (!partial) {
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) sh[w] = ss;
    __syncthreads();
    float t = (l < (blockDim.x >> 5)) ? sh[l] : 0.f;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    const float inv = 1.0f / sqrtf(t);
    for (int c = threadIdx.x; c < D; c += blockDim.x) out[static_cast<int64_t>(i) * D + c] *= inv;
  }
}


// ------------------------------------------------------------------------------------------------ rank counting
// AP needs, per query, only the RANKS of the labelled rows (generic.py:196-224: full argsort, junk dropped, positions
// of the positives) - not the Q x N score matrix.  For each (query, target row) the kernels below return the exact
// score s_t and above_t = the number of database rows that rank before the target under the library's order (exact
// score descending, ties -> lower index first):
//   1. exact scores of the targets                                                          (target_scores_kernel)
//   2. per query thr = min over the counted targets of s_t - eps16                          (count_thr_kernel)
//   3. tcgen05 filter pass: rows with fp16-path score >= thr go to the query's candidate list (PERS_EPI_SIM_FILTER);
//      every row NOT captured has exact score < s_t for every counted target
//   4. per (query, target): candidates with fp16-path score > s_t + eps16 rank before it for certain, those within
//      +-eps16 are re-scored exactly and compared (score, index)                            (rank_count_kernel)
// A query whose list overflows (a positive buried in the bulk of the score distribution) or whose band overflows is
// flagged and counted exactly from the fp32 rows instead                                    (rank_count_exact_kernel)

// one warp per target: score[t] = <q[t_q[t]], db[row - offset]> if this shard owns the row, else 0 (summed over shards)
__global__ void target_scores_kernel(const float* __restrict__ q32, const float* __restrict__ db32, int D,
                                     const int* __restrict__ t_q, const int64_t* __restrict__ t_rows, int T,
                                     int64_t offset, int64_t n_rows, double* __restrict__ t_score) {
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (t >= T) return;
  const int64_t r = t_rows[t] - offset;
  double v = 0.0;
  if (r >= 0 && r < n_rows) v = exact_dot_warp(q32 + static_cast<int64_t>(t_q[t]) * D, db32 + r * D, D, lane);
  if (lane == 0) t_score[t] = v;
}

// thr[q] = (float, rounded down) min over counted targets of s_t - eps; +inf when the query counts nothing
__global__ void count_thr_kernel(const int* __restrict__ t_off, const unsigned char* __restrict__ t_flags,
                                 const double* __restrict__ t_score, int Q, double eps, float* __restrict__ thr) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  double m = INFINITY;
  for (int t = t_off[q]; t < t_off[q + 1]; ++t)
    if (t_flags[t]) m = fmin(m, t_score[t]);
  thr[q] = (m == INFINITY) ? INFINITY : __double2float_rd(m - eps);
}

constexpr int RC_THREADS = 512;
constexpr int RC_BAND = 2048;
__global__ void __launch_bounds__(RC_THREADS) rank_count_kernel(
    const unsigned long long* __restrict__ cand, const int* __restrict__ cnt, int cap, const float* __restrict__ q32,
    const float* __restrict__ db32, int D, int64_t offset, double eps, const int* __restrict__ t_off,
    const int64_t* __restrict__ t_rows, const unsigned char* __restrict__ t_flags, const double* __restrict__ t_score,
    long long* __restrict__ above, int* __restrict__ q_over) {
  __shared__ int band[RC_BAND];
  __shared__ int s_band;
  __shared__ unsigned long long s_count;
  const int q = blockIdx.x;
  const int total = cnt[q];
  if (total > cap) {                      // uniform over the block
    if (threadIdx.x == 0) q_over[q] = 1;
    return;
  }
  const unsigned long long* c = cand + static_cast<int64_t>(q) * cap;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = t_off[q]; t < t_off[q + 1]; ++t) {
    if (!t_flags[t]) continue;            // uniform
    const double s = t_score[t];
    const int64_t trow = t_rows[t];
    const double hi = s + eps, lo = s - eps;
    if (threadIdx.x == 0) {
      s_band = 0;
      s_count = 0ull;
    }
    __syncthreads();
    unsigned int mine = 0;
    for (int i = threadIdx.x; i < total; i += RC_THREADS) {
      const unsigned long long e = c[i];
      const double sh = static_cast<double>(__uint_as_float(static_cast<uint32_t>(e >> 32)));
      if (sh > hi) {
        ++mine;
      } else if (sh >= lo) {
        const int pos = atomicAdd(&s_band, 1);
        if (pos < RC_BAND) band[pos] = static_cast<int>(e & 0xffffffffu);
      }
    }
    __syncthreads();
    const int nb = s_band;
    if (nb > RC_BAND) {                   // uniform: too many near-ties for the shared-memory band
      if (threadIdx.x == 0) q_over[q] = 1;
      return;
    }
    for (int w = warp; w < nb; w += RC_THREADS / 32) {
      const int row = band[w];
      const double sc = exact_dot_warp(q32 + static_cast<int64_t>(q) * D, db32 + static_cast<int64_t>(row) * D, D, lane);
      const int64_t g = static_cast<int64_t>(row) + offset;
      if (lane == 0 && g != trow && (sc > s || (sc == s && g < trow))) ++mine;
    }
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if (lane == 0 && mine) atomicAdd(&s_count, static_cast<unsigned long long>(mine));
    __syncthreads();
    if (threadIdx.x == 0) above[t] = static_cast<long long>(s_count);
    __syncthreads();
  }
}

// Exact fallback, one query per blockIdx.y: every database row is scored exactly (warp per row, fp64) and compared
// with the query's counted targets.  Reads the whole fp32 shard once per query.
constexpr int RCE_THREADS = 256;
__global__ void __launch_bounds__(RCE_THREADS) rank_count_exact_kernel(
    const float* __restrict__ q32, const float* __restrict__ db32, int D, int64_t n_rows, int64_t offset,
    const int* __restrict__ q_list, const int* __restrict__ t_off, const int64_t* __restrict__ t_rows,
    const unsigned char* __restrict__ t_flags, const double* __restrict__ t_score, unsigned long long* __restrict__ above) {
  extern __shared__ unsigned int cnts[];                   // [max targets per query of this launch]
  const int q = q_list[blockIdx.y];
  const int t0 = t_off[q], nt = t_off[q + 1] - t0;
  for (int i = threadIdx.x; i < nt; i += RCE_THREADS) cnts[i] = 0u;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t wstride = static_cast<int64_t>(gridDim.x) * (RCE_THREADS / 32);
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * (RCE_THREADS / 32) + warp; r < n_rows; r += wstride) {
    const double sc = exact_dot_warp(q32 + static_cast<int64_t>(q) * D, db32 + r * D, D, lane);
    const int64_t g = r + offset;
    for (int i = lane; i < nt; i += 32) {
      if (!t_flags[t0 + i]) continue;
      const double s = t_score[t0 + i];
      const int64_t trow = t_rows[t0 + i];
      if (g != trow && (sc > s || (sc == s && g < trow))) atomicAdd(&cnts[i], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nt; i += RCE_THREADS)
    if (cnts[i]) atomicAdd(above + t0 + i, static_cast<unsigned long long>(cnts[i]));
}


// Merge G per-shard lists that are each already ordered (score desc, index asc; empty slots = index -1 at the tail):
// the final position of an entry = its position in its own list + the number of entries of every other list that come
// before it (binary search) - no sorting network, no barriers after the load.  One block per query.
// x.world > 0: the lists are the ones the peers stored into this rank's list table (waits for their flags); the last block
// then opens the next epoch of the exchange.
__global__ void __launch_bounds__(1024) merge_lists_kernel(const double* in_score, const int64_t* in_idx,
                                                          int G, int k, int64_t shard_stride, double* __restrict__ out_score,
                                                          int64_t* __restrict__ out_idx, const PeerX x,
                                                          unsigned long long* status) {
  extern __shared__ uint8_t sm[];
  __shared__ int s_valid;
  const int q = blockIdx.x;
  const int n = G * k;
  double* sc = reinterpret_cast<double*>(sm);
  int64_t* ix = reinterpret_cast<int64_t*>(sc + n);
  if (x.world > 0) {
    const uint32_t epoch = x_epoch(x);
    if (threadIdx.x == 0) x_wait_flags(x, X_OFF_FLIST, epoch, status);
    const size_t base = static_cast<size_t>(epoch & 1u) * x.world * x_list_elems(x.max_q, x.max_k);
    in_score = reinterpret_cast<const double*>(x.peer[x.rank] + x_off_score(x.world, x.max_q)) + base;
    in_idx = reinterpret_cast<const int64_t*>(x.peer[x.rank] + x_off_idx(x.world, x.max_q, x.max_k)) + base;
    shard_stride = static_cast<int64_t>(x_list_elems(x.max_q, x.max_k));
  }
  if (threadIdx.x == 0) s_valid = 0;
  __syncthreads();                                        // (peer mode: the flags were acquired by thread 0)
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const int64_t src = static_cast<int64_t>(e / k) * shard_stride + static_cast<int64_t>(q) * k + e % k;
    sc[e] = __ldcg(in_score + src);
    ix[e] = __ldcg(in_idx + src);
  }
  __syncthreads();
  int my_valid = 0;
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const int g = e / k, j = e - g * k;
    const double se = sc[e];
    const int64_t ie = ix[e];
    if (ie < 0) continue;
    ++my_valid;
    int rank = j;
    for (int h = 0; h < G; ++h) {
      if (h == g) continue;
      const double* hs = sc + h * k;
      const int64_t* hi = ix + h * k;
      int lo = 0, hi_ = k;                      // first position of list h that does NOT come before (se, ie)
      while (lo < hi_) {
        const int mid = (lo + hi_) >> 1;
        const bool before = hi[mid] >= 0 && (hs[mid] > se || (hs[mid] == se && hi[mid] < ie));
        if (before) lo = mid + 1; else hi_ = mid;
      }
      rank += lo;
    }
    if (rank < k) {
      out_score[static_cast<int64_t>(q) * k + rank] = se;
      out_idx[static_cast<int64_t>(q) * k + rank] = ie;
    }
  }
  if (my_valid) atomicAdd(&s_valid, my_valid);
  __syncthreads();
  for (int r = s_valid + threadIdx.x; r < k; r += blockDim.x) {      // fewer than k rows in the whole database
    out_score[static_cast<int64_t>(q) * k + r] = -INFINITY;
    out_idx[static_cast<int64_t>(q) * k + r] = -1;
  }
  if (x.world > 0) {                                      // last block: this search is over, open the next epoch
    __syncthreads();
    if (threadIdx.x == 0) {
      unsigned int* cnt = reinterpret_cast<unsigned int*>(x.peer[x.rank] + X_OFF_CNT) + 2;
      if (atomicAdd(cnt, 1u) == gridDim.x - 1u) {
        *cnt = 0u;
        uint32_t* ep = reinterpret_cast<uint32_t*>(x.peer[x.rank] + X_OFF_EPOCH);
        *ep = *ep + 1u;
      }
    }
  }
}

}  // namespace
}  // namespace dirb

using namespace dirb;

// Encoded 2-D tensor maps, kept per (base, rows, box): a search re-uses the same three maps every call.
struct TmapCache {
  struct E { const void* base; uint64_t inner, outer; uint32_t box; CUtensorMap m; };
  std::vector<E> es;
  int get(const void* base, uint64_t inner, uint64_t outer, uint32_t box, const CUtensorMap** out) {
    for (auto& e : es)
      if (e.base == base && e.inner == inner && e.outer == outer && e.box == box) { *out = &e.m; return 0; }
    if (es.size() >= 16) es.erase(es.begin());
    E e{base, inner, outer, box, {}};
    DIRB_TRY(encode_tmap_2d(&e.m, base, inner, outer, inner * 2, 64, box));
    es.push_back(e);
    *out = &es.back().m;
    return 0;
  }
};

struct dirb200_index {
  int device = 0, dim = 0;
  const float* db32 = nullptr;
  const __half* db16 = nullptr;
  int64_t N = 0, offset = 0;
  bool has_db = false;
  double eps16 = 1.2e-3;
  int64_t sample_rows = 0;
  int cand_cap = 0;          // 0 = auto
  int count_cap = 0;         // candidate capacity per query of dirb200_index_rank_count (0 = 32768)
  int retries = 1;           // gated retry passes enqueued after the first filter pass (device-side predicate)
  int deferred = 0;          // 1 = search calls never synchronise; the caller collects the status (dirb200_index_check)
  // workspaces (grown on demand)
  void* ws = nullptr;
  size_t ws_bytes = 0;
  unsigned long long* h_status = nullptr;   // pinned copy of the device status block
  cudaEvent_t status_ev = nullptr;
  bool status_pending = false;
  int status_cap2 = 0;
  double status_band = 0;
  int64_t stats[5] = {0, 0, 0, 0, 0};
  float* sel_own = nullptr;        // selection thresholds of the single-shard entry point
  size_t sel_bytes = 0;
  // state of a search between dirb200_index_search_begin and _finish
  struct Pending {
    bool active = false;
    int Q = 0, k = 0, cap = 0, cap2 = 0, mark_i = 0;
    int64_t S = 0, launches0 = 0;
    float band = 0;
    int* cnt = nullptr;
    unsigned long long* cand = nullptr;
    unsigned long long* status = nullptr;
    float* kth_k = nullptr;
    // between the seed half and the filter half of phase 1 (the sharded search exchanges seed bounds in between)
    float* thr = nullptr;
    float* dense = nullptr;
    float* sel_dev = nullptr;
    __half* q16 = nullptr;
    int* gates = nullptr;
    int64_t S_ld = 0;
    bool small = false;
    int ks = 0;
  } pend;
  TmapCache tmaps;
  int profile = 0;                 // option "profile": time the phases of a search with CUDA events
  cudaEvent_t ev[10] = {};
  double phase_ms[9] = {};
};

// Similarity GEMM on the persistent tcgen05 kernel (conv_pers.cuh): A = queries [Q][D], B = database rows [rows][D],
// 128 x 256 tiles, K = D.  Tiles are ordered query-tile-fastest, so CTAs running at the same time share the streamed
// database tile (L2) and the database is read from HBM once.  Encoded tensor maps are kept per (base, rows) in the
// handle: a search re-uses the same three maps every call.
struct SimArgs {
  float* dense = nullptr; int64_t dense_ld = 0;
  const float* thr = nullptr; unsigned long long* cand = nullptr; int* cand_cnt = nullptr; int cand_cap = 0;
  const int* gate = nullptr;
};
static int sim_gemm(dirb200_index* h, int epi, const __half* q16, int Q, const __half* db16, int64_t rows, int D,
                    const SimArgs& a, cudaStream_t stream) {
  constexpr int BN = 256;
  const CUtensorMap *tmA, *tmB;
  {
    TmapCache& c = h->tmaps;
    DIRB_TRY(c.get(q16, D, Q, 128, &tmA));
    CUtensorMap a_copy = *tmA;                    // `get` may reallocate the vector: copy before the second lookup
    DIRB_TRY(c.get(db16, D, rows, BN, &tmB));
    CUtensorMap b_copy = *tmB;
    ConvPersParams p{};
    p.a_spatial = 0;
    p.taps = 1; p.kw_taps = 1; p.cin_blocks = D / 64; p.stride = 1; p.pad = 0;
    p.tw = 128; p.th = 1; p.nb = 1; p.tiles_w = 1; p.tiles_h = 1;
    p.M = Q;
    p.N = static_cast<int>(rows);
    p.n_tiles = static_cast<int>(ceil_div(rows, BN));
    p.m_tiles = static_cast<int>(ceil_div(Q, 128));
    p.m_fastest = 1;
    const int64_t total = static_cast<int64_t>(p.m_tiles) * p.n_tiles;
    DIRB_REQUIRE(total < (int64_t(1) << 31), DIRB200_ENOTSUP, "too many tiles");
    p.total_tiles = static_cast<int>(total);
    p.dense = a.dense; p.dense_ld = a.dense_ld;
    p.thr = a.thr; p.cand = a.cand; p.cand_cnt = a.cand_cnt; p.cand_cap = a.cand_cap;
    p.gate = a.gate;
    if (epi == PERS_EPI_SIM_DENSE)
      return conv_pers_launch<BN, 4, PERS_EPI_SIM_DENSE>(a_copy, b_copy, a_copy, a_copy, p, num_sms(), stream);
    if (epi == PERS_EPI_SIM_GMAX)
      return conv_pers_launch<BN, 4, PERS_EPI_SIM_GMAX>(a_copy, b_copy, a_copy, a_copy, p, num_sms(), stream);
    return conv_pers_launch<BN, 4, PERS_EPI_SIM_FILTER>(a_copy, b_copy, a_copy, a_copy, p, num_sms(), stream);
  }
}

extern "C" {

int dirb200_index_create(int device, int dim, dirb200_index** out) {
  DIRB_REQUIRE(out != nullptr, DIRB200_EINVAL, "null out");
  DIRB_TRY(dirb200_device_check(device));
  DIRB_REQUIRE(dim > 0 && dim % 64 == 0, DIRB200_ENOTSUP, "descriptor dim must be a multiple of 64 (got %d)", dim);
  auto* h = new dirb200_index();
  h->device = device;
  h->dim = dim;
  *out = h;
  return 0;
}

int dirb200_index_set_db(dirb200_index* h, const float* db32_dev, const void* db16_dev, int64_t N,
                         int64_t index_offset) {
  DIRB_REQUIRE(h && N >= 0 && (N == 0 || (db32_dev && db16_dev)), DIRB200_EINVAL, "bad db arguments");   // an empty shard has no buffers
  DIRB_REQUIRE(N < (int64_t(1) << 31) - 256, DIRB200_ENOTSUP, "shard too large (%lld rows)", (long long)N);
  h->db32 = db32_dev;
  h->db16 = static_cast<const __half*>(db16_dev);
  h->N = N;
  h->offset = index_offset;
  h->has_db = true;
  h->tmaps.es.clear();
  return 0;
}

int dirb200_index_set_option(dirb200_index* h, const char* key, double value) {
  DIRB_REQUIRE(h && key, DIRB200_EINVAL, "null");
  const std::string k(key);
  if (k == "eps16") h->eps16 = value;
  else if (k == "sample_rows") h->sample_rows = static_cast<int64_t>(value);
  else if (k == "cand_cap") h->cand_cap = static_cast<int>(value);
  else if (k == "profile") h->profile = value != 0;
  else if (k == "count_cap") h->count_cap = static_cast<int>(value);
  else if (k == "retries") h->retries = std::max(0, std::min(4, static_cast<int>(value)));
  else if (k == "deferred_check") h->deferred = value != 0;
  else DIRB_REQUIRE(false, DIRB200_EKEY, "unknown index option '%s'", key);
  return 0;
}

// Collect the status of the last search (waits for it to finish): overflow errors + counters.
int dirb200_index_check(dirb200_index* h) {
  DIRB_REQUIRE(h, DIRB200_EINVAL, "null");
  if (!h->status_pending) return 0;
  DIRB_CUDA(cudaSetDevice(h->device));
  DIRB_CUDA(cudaEventSynchronize(h->status_ev));
  h->status_pending = false;
  const unsigned long long err = h->h_status[ST_ERR];
  h->stats[1] = static_cast<int64_t>(h->h_status[ST_CAND]);
  h->stats[2] = static_cast<int64_t>(h->h_status[ST_SURV]);
  h->stats[3] = static_cast<int64_t>(h->h_status[ST_RETRIES]);
  if (h->profile && h->pend.mark_i >= 2) {
    for (int i = 0; i + 1 < h->pend.mark_i && i < 8; ++i) {
      float ms = 0;
      cudaEventElapsedTime(&ms, h->ev[i], h->ev[i + 1]);
      h->phase_ms[i] = ms;
    }
  }
  DIRB_REQUIRE((err & 1ull) == 0, DIRB200_EOVERFLOW,
               "candidate buffer overflow not resolved after %d retry passes (raise option cand_cap)", h->retries);
  DIRB_REQUIRE((err & 4ull) == 0, DIRB200_EOVERFLOW,
               "sharded search: a peer rank did not publish its thresholds / lists in time (ranks out of step?)");
  DIRB_REQUIRE((err & 2ull) == 0, DIRB200_EOVERFLOW,
               "more than %d rows within 2*eps16=%g of the k-th score for some query (near-duplicate rows?)",
               h->status_cap2, h->status_band);
  return 0;
}

int dirb200_index_last_stats(dirb200_index* h, int64_t stats[5]) {
  DIRB_REQUIRE(h && stats, DIRB200_EINVAL, "null");
  if (h->status_pending) {                      // counters of a deferred search: wait for it, keep its error for _check
    DIRB_CUDA(cudaSetDevice(h->device));
    DIRB_CUDA(cudaEventSynchronize(h->status_ev));
    h->stats[1] = static_cast<int64_t>(h->h_status[ST_CAND]);
    h->stats[2] = static_cast<int64_t>(h->h_status[ST_SURV]);
    h->stats[3] = static_cast<int64_t>(h->h_status[ST_RETRIES]);
  }
  for (int i = 0; i < 5; ++i) stats[i] = h->stats[i];
  return 0;
}

int dirb200_index_last_profile(dirb200_index* h, double out9[9]) {
  DIRB_REQUIRE(h && out9, DIRB200_EINVAL, "null");
  for (int i = 0; i < 9; ++i) out9[i] = h->phase_ms[i];
  return 0;
}

int dirb200_index_destroy(dirb200_index* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  for (auto e : h->ev) if (e) cudaEventDestroy(e);
  if (h->status_ev) cudaEventDestroy(h->status_ev);
  if (h->ws) cudaFree(h->ws);
  if (h->sel_own) cudaFree(h->sel_own);
  if (h->h_status) cudaFreeHost(h->h_status);
  delete h;
  return 0;
}

static void mark_phase(dirb200_index* h, cudaStream_t stream) {
  if (!h->profile || h->pend.mark_i >= 10) return;
  if (!h->ev[h->pend.mark_i]) cudaEventCreate(&h->ev[h->pend.mark_i]);
  cudaEventRecord(h->ev[h->pend.mark_i++], stream);
}

// Phase 1: fp16 queries, seed pass, filter pass (+ device-gated retry passes), local k-th / k_shard-th candidate
// scores.  sel_dev[Q] receives the local k_shard-th best fp16-path score per query; with several shards the caller
// MIN-reduces it over the shards before phase 2 (k_shard = ceil(k / shards)); with one shard k_shard = k.
// Nothing here waits for the GPU: everything is enqueued on `stream`.
// Split in two halves: search_begin_seed (queries -> fp16, seed pass, seed bounds) and search_begin_filter (filter pass,
// candidate selection, gated retries).  seed2 != nullptr: the seed half also writes the k_shard-th seed bound of every
// query there - what a shard contributes to the MIN over the shards that tightens the filter threshold of the sharded
// search (thr_min_kernel, issued between the halves by dirb200_index_search_sharded_phase).
static int search_begin_seed(dirb200_index* h, const float* q32, int Q, int k, int k_shard, float* sel_dev, cudaStream_t stream,
                             float* seed2) {
  DIRB_REQUIRE(h && q32 && sel_dev, DIRB200_EINVAL, "null argument");
  DIRB_REQUIRE(h->has_db, DIRB200_ESTATE, "index has no database attached");
  DIRB_REQUIRE(Q > 0 && k > 0 && k <= 1024, DIRB200_ENOTSUP, "need 0 < Q and 0 < k <= 1024 (got Q=%d k=%d)", Q, k);
  DIRB_REQUIRE(k_shard >= 1 && k_shard <= k, DIRB200_EINVAL, "k_shard must be in [1, k]");
  DIRB_CUDA(cudaSetDevice(h->device));
  DIRB_TRY(dirb200_index_check(h));          // an uncollected error of the previous search must not get lost
  const int D = h->dim;
  const int64_t N = h->N;
  auto& P = h->pend;
  P = dirb200_index::Pending();
  P.active = true;
  P.Q = Q;
  P.k = k;
  P.launches0 = launches_total();
  P.cap2 = (k > 256) ? 2048 : 1024;
  P.sel_dev = sel_dev;
  if (N == 0) {   // empty shard: nothing can be selected; +inf never lowers the MIN over the shards
    fill_f32_kernel<<<static_cast<unsigned>(ceil_div(Q, 256)), 256, 0, stream>>>(sel_dev, Q, INFINITY);
    count_launch();
    if (seed2) {
      fill_f32_kernel<<<static_cast<unsigned>(ceil_div(Q, 256)), 256, 0, stream>>>(seed2, Q, INFINITY);
      count_launch();
    }
    DIRB_CUDA(cudaGetLastError());
    return 0;
  }
  // ---- sizes
  int64_t S = h->sample_rows > 0 ? h->sample_rows : std::max<int64_t>(8192, ceil_div(N, 16));
  S = std::min<int64_t>(std::min<int64_t>(S, 65536), N);
  S = std::max<int64_t>(S, std::min<int64_t>(N, 4 * k));
  const bool small = (N <= S);
  if (small) S = N;
  if (!small && S / 32 < k) S = std::min<int64_t>(N, std::max<int64_t>(S, 32 * static_cast<int64_t>(k)));
  // seed threshold from group maxima (1/32 of the dense traffic) whenever there are at least k groups
  const bool use_gmax = !small && (S / 32 >= k);
  const int64_t S_ld = ceil_div(S, 128) * 128;   // dense row stride (16-byte aligned rows)
  const double expect = small ? (2.0 * k + 64) : (1.5 * k * static_cast<double>(N) / S);
  int cap = static_cast<int>(std::min<double>(std::max<double>(4096, 4 * expect), 1 << 18));
  if (h->cand_cap > 0) cap = std::max(h->cand_cap, 2 * k);
  cap = (cap + 255) / 256 * 256;
  const float band = static_cast<float>(2.0 * h->eps16);
  P.S = S;
  P.cap = cap;
  P.band = band;

  // ---- workspace carve-up
  size_t off = 0;
  auto carve = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  const size_t o_q16 = carve(static_cast<size_t>(Q) * D * 2);
  const size_t o_dense = carve(static_cast<size_t>(Q) * S_ld * 4);
  const size_t o_thr = carve(static_cast<size_t>(Q) * 4);
  const size_t o_cnt = carve(static_cast<size_t>(Q) * 4);
  const size_t o_cand = carve(static_cast<size_t>(Q) * cap * 8);
  const size_t o_kthk = carve(static_cast<size_t>(Q) * 4);
  const size_t o_gates = carve(8 * 4);
  const size_t o_status = carve(ST_WORDS * 8);
  if (off > h->ws_bytes) {
    if (h->ws) DIRB_CUDA(cudaFree(h->ws));
    h->ws = nullptr;
    h->ws_bytes = 0;
    DIRB_CUDA(cudaMalloc(&h->ws, off));
    h->ws_bytes = off;
    h->tmaps.es.clear();                    // the cached query map pointed into the old workspace
  }
  uint8_t* w = static_cast<uint8_t*>(h->ws);
  __half* q16 = reinterpret_cast<__half*>(w + o_q16);
  float* dense = reinterpret_cast<float*>(w + o_dense);
  float* thr = reinterpret_cast<float*>(w + o_thr);
  int* gates = reinterpret_cast<int*>(w + o_gates);
  P.cnt = reinterpret_cast<int*>(w + o_cnt);
  P.cand = reinterpret_cast<unsigned long long*>(w + o_cand);
  P.kth_k = reinterpret_cast<float*>(w + o_kthk);
  P.status = reinterpret_cast<unsigned long long*>(w + o_status);
  int* cnt = P.cnt;

  mark_phase(h, stream);  // 0
  // ---- 1. queries to fp16, counters / gates / status cleared
  {
    const int64_t n = static_cast<int64_t>(Q) * D;
    const int64_t threads = std::max<int64_t>(ceil_div(n, 4), std::max<int64_t>(Q, 8));
    search_prep_kernel<<<static_cast<unsigned>(ceil_div(threads, 256)), 256, 0, stream>>>(q32, q16, n, cnt, Q, gates, 8, P.status);
    count_launch();
  }
  mark_phase(h, stream);  // 1: convert
  // ---- 2. seed pass over the first S rows
  {
    SimArgs a;
    a.dense = dense;
    a.dense_ld = S_ld;
    DIRB_TRY(sim_gemm(h, use_gmax ? PERS_EPI_SIM_GMAX : PERS_EPI_SIM_DENSE, q16, Q, h->db16, S, D, a, stream));
    mark_phase(h, stream);  // 2: seed GEMM
    const int n_vals = use_gmax ? static_cast<int>(ceil_div(S, 32)) : static_cast<int>(S);
    const int kk = static_cast<int>(std::min<int64_t>(k, n_vals));
    const int kk2 = seed2 ? static_cast<int>(std::min<int64_t>(k_shard, n_vals)) : 0;
    kth_dense_kernel<<<Q, SEL_THREADS, 0, stream>>>(dense, S_ld, n_vals, kk, band, thr, kk2, seed2);
    count_launch();
    mark_phase(h, stream);  // 3: k-th of the seed scores
  }
  P.thr = thr;
  P.dense = dense;
  P.q16 = q16;
  P.gates = gates;
  P.S_ld = S_ld;
  P.small = small;
  P.ks = std::min<int>(k_shard, static_cast<int>(std::min<int64_t>(k, N)));
  DIRB_CUDA(cudaGetLastError());
  return 0;
}

static int search_begin_filter(dirb200_index* h, cudaStream_t stream) {
  auto& P = h->pend;
  DIRB_REQUIRE(P.active, DIRB200_ESTATE, "filter half of a search without its seed half");
  const int64_t N = h->N;
  if (N == 0) return 0;
  DIRB_CUDA(cudaSetDevice(h->device));
  const int Q = P.Q, k = P.k, D = h->dim, cap = P.cap, ks = P.ks;
  const bool small = P.small;
  const int64_t S_ld = P.S_ld;
  const float band = P.band;
  float* thr = P.thr;
  float* dense = P.dense;
  float* sel_dev = P.sel_dev;
  __half* q16 = P.q16;
  int* gates = P.gates;
  int* cnt = P.cnt;
  unsigned long long* cand = P.cand;
  // ---- 3./4. candidates + local k-th / k_shard-th candidate scores; pass r > 0 is armed by gate[r-1], which the
  //            selection of pass r-1 raises when some query overflowed its candidate list
  for (int r = 0; r <= h->retries; ++r) {
    const int* gate_in = r > 0 ? gates + (r - 1) : nullptr;
    if (small) {
      dim3 g(static_cast<unsigned>(ceil_div(N, 256)), static_cast<unsigned>(Q));
      dense_compact_kernel<<<g, 256, 0, stream>>>(dense, S_ld, static_cast<int>(N), thr, cand, cnt, cap, gate_in);
      count_launch();
    } else {
      SimArgs a;
      a.thr = thr;
      a.cand = cand;
      a.cand_cnt = cnt;
      a.cand_cap = cap;
      a.gate = gate_in;
      DIRB_TRY(sim_gemm(h, PERS_EPI_SIM_FILTER, q16, Q, h->db16, N, D, a, stream));
    }
    if (r == 0) mark_phase(h, stream);  // 4: filter pass
    cand_kth_kernel<<<Q, SEL_THREADS, 0, stream>>>(cand, cnt, cap, k, ks, band, P.kth_k, sel_dev, thr, N, gate_in, gates + r,
                                                   r == h->retries ? 1 : 0, P.status);
    count_launch();
    if (r == 0) mark_phase(h, stream);  // 5: candidate selection
  }
  mark_phase(h, stream);  // 6: gated retry passes (empty launches unless a list overflowed)
  DIRB_CUDA(cudaGetLastError());
  return 0;
}

int dirb200_index_search_begin(dirb200_index* h, const float* q32, int Q, int k, int k_shard, float* sel_dev,
                               void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DIRB_TRY(search_begin_seed(h, q32, Q, k, k_shard, sel_dev, stream, nullptr));
  return search_begin_filter(h, stream);
}

// Phase 2: survivors (candidates within the band of max(sel, local k-th)), exact re-scoring, ordered output - one
// launch (search_finish_kernel) + an asynchronous copy of the status block.  Unless option deferred_check is set the
// call ends with dirb200_index_check (the only host synchronisation of a search).
// Asynchronous copy of the status block of the search in flight + the event dirb200_index_check waits for.
static int post_status_copy(dirb200_index* h, cudaStream_t stream) {
  if (!h->h_status) DIRB_CUDA(cudaMallocHost(reinterpret_cast<void**>(&h->h_status), ST_WORDS * 8));
  if (!h->status_ev) DIRB_CUDA(cudaEventCreateWithFlags(&h->status_ev, cudaEventDisableTiming));
  DIRB_CUDA(cudaMemcpyAsync(h->h_status, h->pend.status, ST_WORDS * 8, cudaMemcpyDeviceToHost, stream));
  DIRB_CUDA(cudaEventRecord(h->status_ev, stream));
  h->status_pending = true;
  return 0;
}

static int search_finish_impl(dirb200_index* h, const float* q32, const float* sel_dev, double* scores_dev, int64_t* idx_dev,
                              cudaStream_t stream, const PeerX& px, unsigned long long* x_status) {
  auto& P = h->pend;
  DIRB_REQUIRE(P.active, DIRB200_ESTATE, "dirb200_index_search_finish without a matching _begin");
  DIRB_CUDA(cudaSetDevice(h->device));
  const int Q = P.Q, k = P.k, cap2 = P.cap2;
  P.active = false;
  if (h->N == 0) {
    if (px.world > 0) {   // an empty shard still publishes its (empty) lists: the peers wait for every rank's flag
      search_finish_kernel<<<Q, FIN_THREADS, static_cast<size_t>(cap2) * 12, stream>>>(nullptr, nullptr, 0, nullptr, sel_dev, 0.f, q32, nullptr,
                                                                                     h->dim, cap2, h->offset, k, nullptr, nullptr, x_status, px);
    } else {
      const int64_t n = static_cast<int64_t>(Q) * k;
      fill_empty_result_kernel<<<static_cast<unsigned>(ceil_div(n, 256)), 256, 0, stream>>>(scores_dev, idx_dev, n);
    }
    count_launch();
    DIRB_CUDA(cudaGetLastError());
    h->stats[0] = h->stats[1] = h->stats[2] = h->stats[3] = 0;
    h->stats[4] = launches_total() - P.launches0;
    return 0;
  }
  const size_t smem = static_cast<size_t>(cap2) * 12;
  search_finish_kernel<<<Q, FIN_THREADS, smem, stream>>>(P.cand, P.cnt, P.cap, P.kth_k, sel_dev, P.band, q32, h->db32, h->dim,
                                                         cap2, h->offset, k, scores_dev, idx_dev, P.status, px);
  count_launch();
  DIRB_CUDA(cudaGetLastError());
  mark_phase(h, stream);  // 7: survivors + exact re-scoring + sort
  h->status_cap2 = cap2;
  h->status_band = P.band;
  h->stats[0] = P.S;
  h->stats[4] = launches_total() - P.launches0;
  if (px.world > 0) return 0;               // sharded search over peer memory: the merge (phase 3) can still raise error bits
  DIRB_TRY(post_status_copy(h, stream));
  if (!h->deferred) return dirb200_index_check(h);
  return 0;
}

int dirb200_index_search_finish(dirb200_index* h, const float* q32, const float* sel_dev, double* scores_dev,
                                int64_t* idx_dev, void* stream_) {
  DIRB_REQUIRE(h && q32 && sel_dev && scores_dev && idx_dev, DIRB200_EINVAL, "null argument");
  return search_finish_impl(h, q32, sel_dev, scores_dev, idx_dev, static_cast<cudaStream_t>(stream_), PeerX{}, nullptr);
}

// Single-shard search = phase 1 with k_shard = k followed directly by phase 2.
int dirb200_index_search(dirb200_index* h, const float* q32, int Q, int k, double* scores_dev, int64_t* idx_dev,
                         void* stream_) {
  DIRB_REQUIRE(h && q32 && scores_dev && idx_dev, DIRB200_EINVAL, "null argument");
  DIRB_REQUIRE(Q > 0, DIRB200_ENOTSUP, "need Q > 0");
  if (static_cast<size_t>(Q) * 4 > h->sel_bytes) {
    if (h->sel_own) cudaFree(h->sel_own);
    h->sel_own = nullptr;
    DIRB_CUDA(cudaMalloc(reinterpret_cast<void**>(&h->sel_own), static_cast<size_t>(Q) * 4));
    h->sel_bytes = static_cast<size_t>(Q) * 4;
  }
  DIRB_TRY(dirb200_index_search_begin(h, q32, Q, k, k, h->sel_own, stream_));
  return dirb200_index_search_finish(h, q32, h->sel_own, scores_dev, idx_dev, stream_);
}

// ---- rank counting (see the kernels above): exact scores of the labelled rows + number of rows ranking before them
int dirb200_index_target_scores(dirb200_index* h, const float* q32, int Q, const int* t_q_dev, const int64_t* t_rows_dev,
                                int T, double* t_score_dev, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DIRB_REQUIRE(h && q32 && Q > 0 && T >= 0, DIRB200_EINVAL, "bad arguments");
  DIRB_REQUIRE(h->has_db, DIRB200_ESTATE, "index has no database attached");
  if (T == 0) return 0;
  DIRB_REQUIRE(t_q_dev && t_rows_dev && t_score_dev, DIRB200_EINVAL, "null argument");
  DIRB_CUDA(cudaSetDevice(h->device));
  target_scores_kernel<<<static_cast<unsigned>(ceil_div(T, 8)), 256, 0, stream>>>(q32, h->db32, h->dim, t_q_dev, t_rows_dev, T,
                                                                                  h->offset, h->N, t_score_dev);
  count_launch();
  DIRB_CUDA(cudaGetLastError());
  return 0;
}

int dirb200_index_rank_count(dirb200_index* h, const float* q32, int Q, const int* t_off_host, const int* t_off_dev,
                             const int64_t* t_rows_dev, const unsigned char* t_flags_dev, const double* t_score_dev,
                             int T, int64_t* above_dev, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DIRB_REQUIRE(h && q32 && Q > 0 && T >= 0 && t_off_host, DIRB200_EINVAL, "bad arguments");
  DIRB_REQUIRE(h->has_db, DIRB200_ESTATE, "index has no database attached");
  if (T == 0) return 0;
  DIRB_REQUIRE(t_off_dev && t_rows_dev && t_flags_dev && t_score_dev && above_dev, DIRB200_EINVAL, "null argument");
  DIRB_REQUIRE(t_off_host[0] == 0 && t_off_host[Q] == T, DIRB200_EINVAL, "target offsets must run from 0 to T");
  DIRB_CUDA(cudaSetDevice(h->device));
  DIRB_TRY(dirb200_index_check(h));
  h->pend.active = false;                        // shares the search workspace
  const int64_t launches0 = launches_total();
  DIRB_CUDA(cudaMemsetAsync(above_dev, 0, static_cast<size_t>(T) * 8, stream));
  h->stats[0] = h->stats[1] = h->stats[2] = h->stats[3] = 0;
  if (h->N == 0) {
    h->stats[4] = launches_total() - launches0;
    return 0;
  }
  const int D = h->dim;
  const int64_t N = h->N;
  int cap = h->count_cap > 0 ? h->count_cap : 32768;
  cap = std::max(1024, (cap + 255) / 256 * 256);
  size_t off = 0;
  auto carve = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
  const size_t o_q16 = carve(static_cast<size_t>(Q) * D * 2);
  const size_t o_thr = carve(static_cast<size_t>(Q) * 4);
  const size_t o_cnt = carve(static_cast<size_t>(Q) * 4);
  const size_t o_cand = carve(static_cast<size_t>(Q) * cap * 8);
  const size_t o_gates = carve(8 * 4);
  const size_t o_status = carve(ST_WORDS * 8);
  const size_t o_over = carve(static_cast<size_t>(Q) * 4);
  const size_t o_qlist = carve(static_cast<size_t>(Q) * 4);
  if (off > h->ws_bytes) {
    if (h->ws) DIRB_CUDA(cudaFree(h->ws));
    h->ws = nullptr;
    h->ws_bytes = 0;
    DIRB_CUDA(cudaMalloc(&h->ws, off));
    h->ws_bytes = off;
    h->tmaps.es.clear();
  }
  uint8_t* w = static_cast<uint8_t*>(h->ws);
  __half* q16 = reinterpret_cast<__half*>(w + o_q16);
  float* thr = reinterpret_cast<float*>(w + o_thr);
  int* cnt = reinterpret_cast<int*>(w + o_cnt);
  unsigned long long* cand = reinterpret_cast<unsigned long long*>(w + o_cand);
  int* gates = reinterpret_cast<int*>(w + o_gates);
  unsigned long long* status = reinterpret_cast<unsigned long long*>(w + o_status);
  int* q_over = reinterpret_cast<int*>(w + o_over);
  int* q_list = reinterpret_cast<int*>(w + o_qlist);
  {
    const int64_t n = static_cast<int64_t>(Q) * D;
    const int64_t threads = std::max<int64_t>(ceil_div(n, 4), std::max<int64_t>(Q, 8));
    search_prep_kernel<<<static_cast<unsigned>(ceil_div(threads, 256)), 256, 0, stream>>>(q32, q16, n, cnt, Q, gates, 8, status);
    count_launch();
  }
  DIRB_CUDA(cudaMemsetAsync(q_over, 0, static_cast<size_t>(Q) * 4, stream));
  count_thr_kernel<<<static_cast<unsigned>(ceil_div(Q, 128)), 128, 0, stream>>>(t_off_dev, t_flags_dev, t_score_dev, Q, h->eps16, thr);
  count_launch();
  {
    SimArgs a;
    a.thr = thr;
    a.cand = cand;
    a.cand_cnt = cnt;
    a.cand_cap = cap;
    DIRB_TRY(sim_gemm(h, PERS_EPI_SIM_FILTER, q16, Q, h->db16, N, D, a, stream));
  }
  rank_count_kernel<<<Q, RC_THREADS, 0, stream>>>(cand, cnt, cap, q32, h->db32, D, h->offset, h->eps16, t_off_dev, t_rows_dev,
                                                  t_flags_dev, t_score_dev, reinterpret_cast<long long*>(above_dev), q_over);
  count_launch();
  DIRB_CUDA(cudaGetLastError());
  std::vector<int> over(Q), hcnt(Q);
  DIRB_CUDA(cudaMemcpyAsync(over.data(), q_over, static_cast<size_t>(Q) * 4, cudaMemcpyDeviceToHost, stream));
  DIRB_CUDA(cudaMemcpyAsync(hcnt.data(), cnt, static_cast<size_t>(Q) * 4, cudaMemcpyDeviceToHost, stream));
  DIRB_CUDA(cudaStreamSynchronize(stream));
  std::vector<int> list;
  int max_nt = 0;
  int64_t cand_total = 0;
  for (int q = 0; q < Q; ++q) {
    cand_total += std::min(hcnt[q], cap);
    if (!over[q]) continue;
    list.push_back(q);
    max_nt = std::max(max_nt, t_off_host[q + 1] - t_off_host[q]);
    // a band overflow may have left partial counts behind
    DIRB_CUDA(cudaMemsetAsync(above_dev + t_off_host[q], 0, static_cast<size_t>(t_off_host[q + 1] - t_off_host[q]) * 8, stream));
  }
  if (!list.empty()) {
    DIRB_REQUIRE(static_cast<size_t>(max_nt) * 4 <= 200 * 1024, DIRB200_ENOTSUP, "more than 51200 labelled rows for one query");
    DIRB_CUDA(cudaMemcpyAsync(q_list, list.data(), list.size() * 4, cudaMemcpyHostToDevice, stream));
    const size_t smem = static_cast<size_t>(std::max(max_nt, 1)) * 4;
    DIRB_CUDA(cudaFuncSetAttribute(rank_count_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    const int gx = static_cast<int>(std::min<int64_t>(ceil_div(N, RCE_THREADS / 32), 4 * static_cast<int64_t>(num_sms())));
    // a few queries per launch: each grid row re-reads the whole fp32 shard
    for (size_t i0 = 0; i0 < list.size(); i0 += 4096) {
      const unsigned ny = static_cast<unsigned>(std::min<size_t>(4096, list.size() - i0));
      rank_count_exact_kernel<<<dim3(gx, ny), RCE_THREADS, smem, stream>>>(
          q32, h->db32, D, N, h->offset, q_list + i0, t_off_dev, t_rows_dev, t_flags_dev, t_score_dev,
          reinterpret_cast<unsigned long long*>(above_dev));
      count_launch();
    }
    DIRB_CUDA(cudaGetLastError());
    DIRB_CUDA(cudaStreamSynchronize(stream));    // `list` is read by the async copy above
  }
  h->stats[1] = cand_total;
  h->stats[3] = static_cast<int64_t>(list.size());
  h->stats[4] = launches_total() - launches0;
  return 0;
}

// merge_lists_kernel holds all G*k (fp64 score, int64 index) entries of a query in dynamic shared memory: up to
// MERGE_MAX_ENTRIES * 16 = 64 KiB.  Without opting in a launch gets 48 KiB including the kernel's static shared memory,
// so G*k >= 3072 would fail to launch.
constexpr int MERGE_MAX_ENTRIES = 4096;
static int merge_smem_opt_in() {
  static std::atomic<uint64_t> attr_done{0};
  if (first_launch_on_device(attr_done))
    DIRB_CUDA(cudaFuncSetAttribute(merge_lists_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, MERGE_MAX_ENTRIES * 16));
  return 0;
}

int dirb200_topk_merge(const double* scores_dev, const int64_t* idx_dev, int G, int Q, int k, int64_t shard_stride,
                       double* out_scores_dev, int64_t* out_idx_dev, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DIRB_REQUIRE(scores_dev && idx_dev && out_scores_dev && out_idx_dev, DIRB200_EINVAL, "null argument");
  DIRB_REQUIRE(G >= 1 && Q >= 1 && k >= 1 && static_cast<int64_t>(G) * k <= MERGE_MAX_ENTRIES, DIRB200_ENOTSUP,
               "merge supports G*k <= %d (got G=%d k=%d)", MERGE_MAX_ENTRIES, G, k);
  // shard g holds [Q][k] at element offset g*shard_stride, each list already ordered: rank-based merge, read in place
  if (shard_stride <= 0) shard_stride = static_cast<int64_t>(Q) * k;
  const int n = G * k;
  const int threads = std::min(1024, (n + 31) / 32 * 32);
  DIRB_TRY(merge_smem_opt_in());
  merge_lists_kernel<<<Q, threads, static_cast<size_t>(n) * 16, stream>>>(scores_dev, idx_dev, G, k, shard_stride, out_scores_dev,
                                                                        out_idx_dev, PeerX{}, nullptr);
  count_launch();
  DIRB_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Peer-memory exchange of the sharded search (device side: PeerX, sel_push_kernel, search_finish_kernel, merge_lists_kernel)
struct dirb200_exchange {
  int device = 0, world = 1, rank = 0, max_q = 0, max_k = 0;
  uint8_t* base = nullptr;           // this rank's window (cudaMalloc: exportable through CUDA IPC)
  size_t bytes = 0;
  uint8_t* peer[X_MAXW] = {};        // every rank's window as mapped in this process
  bool ipc_opened[X_MAXW] = {};
  bool open = false;
  float* sel_local = nullptr;        // [max_q] this shard's selection thresholds before they are pushed
  float* seed_local = nullptr;       // [max_q] this shard's k_shard-th seed bounds before they are pushed
  unsigned long long* status = nullptr;   // status words for kernels of an empty shard (no index workspace)
};

static PeerX peer_view(const dirb200_exchange* x) {
  PeerX v{};
  v.world = x->world; v.rank = x->rank; v.max_q = x->max_q; v.max_k = x->max_k;
  for (int g = 0; g < x->world; ++g) v.peer[g] = x->peer[g];
  return v;
}

int dirb200_exchange_create(int device, int world, int rank, int max_q, int max_k, dirb200_exchange** out) {
  DIRB_REQUIRE(out, DIRB200_EINVAL, "null argument");
  DIRB_REQUIRE(world >= 1 && world <= X_MAXW && rank >= 0 && rank < world, DIRB200_ENOTSUP,
               "peer exchange supports 1..%d ranks of one box (got world=%d rank=%d)", X_MAXW, world, rank);
  DIRB_REQUIRE(max_q >= 1 && max_k >= 1 && max_k <= 1024 && static_cast<int64_t>(world) * max_k <= MERGE_MAX_ENTRIES,
               DIRB200_ENOTSUP, "need max_q >= 1, 1 <= max_k <= 1024 and world * max_k <= %d", MERGE_MAX_ENTRIES);
  DIRB_TRY(dirb200_device_check(device));
  DIRB_CUDA(cudaSetDevice(device));
  auto* x = new dirb200_exchange();
  x->device = device; x->world = world; x->rank = rank; x->max_q = max_q; x->max_k = max_k;
  x->bytes = x_total_bytes(world, max_q, max_k);
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&x->base), x->bytes);
  if (e == cudaSuccess) e = cudaMemset(x->base, 0, x->bytes);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&x->sel_local), static_cast<size_t>(max_q) * 4);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&x->seed_local), static_cast<size_t>(max_q) * 4);
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&x->status), ST_WORDS * 8);
  if (e == cudaSuccess) e = cudaMemset(x->status, 0, ST_WORDS * 8);
  if (e == cudaSuccess) {
    const uint32_t one = 1;          // epochs start at 1: the zero-initialised flags read as "not yet published"
    e = cudaMemcpy(x->base + X_OFF_EPOCH, &one, 4, cudaMemcpyHostToDevice);
  }
  if (e != cudaSuccess) {
    set_error("exchange window of %zu bytes: %s", x->bytes, cudaGetErrorString(e));
    dirb200_exchange_destroy(x);
    return static_cast<int>(e);
  }
  x->peer[rank] = x->base;
  *out = x;
  return 0;
}

int dirb200_exchange_ipc_handle(dirb200_exchange* x, void* handle64_out) {
  DIRB_REQUIRE(x && handle64_out, DIRB200_EINVAL, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
  DIRB_CUDA(cudaSetDevice(x->device));
  cudaIpcMemHandle_t hd;
  DIRB_CUDA(cudaIpcGetMemHandle(&hd, x->base));
  memcpy(handle64_out, &hd, 64);
  return 0;
}

int dirb200_exchange_open(dirb200_exchange* x, const void* handles) {
  DIRB_REQUIRE(x && handles, DIRB200_EINVAL, "null argument");
  DIRB_REQUIRE(!x->open, DIRB200_ESTATE, "exchange already opened");
  DIRB_CUDA(cudaSetDevice(x->device));
  for (int g = 0; g < x->world; ++g) {
    if (g == x->rank) continue;
    cudaIpcMemHandle_t hd;
    memcpy(&hd, static_cast<const uint8_t*>(handles) + static_cast<size_t>(g) * 64, 64);
    void* ptr = nullptr;
    DIRB_CUDA(cudaIpcOpenMemHandle(&ptr, hd, cudaIpcMemLazyEnablePeerAccess));
    x->peer[g] = static_cast<uint8_t*>(ptr);
    x->ipc_opened[g] = true;
  }
  x->open = true;
  return 0;
}

int dirb200_exchange_open_local(dirb200_exchange* x, dirb200_exchange* const* all) {
  DIRB_REQUIRE(x && all, DIRB200_EINVAL, "null argument");
  DIRB_REQUIRE(!x->open, DIRB200_ESTATE, "exchange already opened");
  for (int g = 0; g < x->world; ++g) {
    DIRB_REQUIRE(all[g] && all[g]->world == x->world && all[g]->rank == g && all[g]->max_q == x->max_q && all[g]->max_k == x->max_k,
                 DIRB200_EINVAL, "exchange %d of the group does not match (world / rank / sizes)", g);
    if (all[g]->device != x->device) {
      int can = 0;
      DIRB_CUDA(cudaDeviceCanAccessPeer(&can, x->device, all[g]->device));
      DIRB_REQUIRE(can, DIRB200_ENOTSUP, "device %d cannot access device %d", x->device, all[g]->device);
      DIRB_CUDA(cudaSetDevice(x->device));
      cudaError_t e = cudaDeviceEnablePeerAccess(all[g]->device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) DIRB_CUDA(e);
      cudaGetLastError();
    }
    x->peer[g] = all[g]->base;
  }
  x->open = true;
  return 0;
}

// Unmap the other ranks' windows (CUDA IPC).  An exporting process must not free its window while an importer still has
// it mapped: ranks call this, synchronise among themselves (a barrier), and only then destroy their own window.
int dirb200_exchange_close_peers(dirb200_exchange* x) {
  DIRB_REQUIRE(x, DIRB200_EINVAL, "null argument");
  DIRB_CUDA(cudaSetDevice(x->device));
  DIRB_CUDA(cudaDeviceSynchronize());                       // no kernel of this rank may still be writing to a peer
  for (int g = 0; g < x->world; ++g) {
    if (x->ipc_opened[g] && x->peer[g]) {
      DIRB_CUDA(cudaIpcCloseMemHandle(x->peer[g]));
      x->ipc_opened[g] = false;
    }
    if (g != x->rank) x->peer[g] = nullptr;
  }
  x->open = false;
  return 0;
}

int dirb200_exchange_destroy(dirb200_exchange* x) {
  if (!x) return 0;
  cudaSetDevice(x->device);
  for (int g = 0; g < x->world; ++g)
    if (x->ipc_opened[g] && x->peer[g]) cudaIpcCloseMemHandle(x->peer[g]);
  if (x->base) cudaFree(x->base);
  if (x->sel_local) cudaFree(x->sel_local);
  if (x->seed_local) cudaFree(x->seed_local);
  if (x->status) cudaFree(x->status);
  delete x;
  return 0;
}

int dirb200_index_search_sharded_phase(dirb200_index* h, dirb200_exchange* x, int phase, const float* q32, int Q, int k, int k_shard,
                                       double* scores_dev, int64_t* idx_dev, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DIRB_REQUIRE(h && x && q32, DIRB200_EINVAL, "null argument");
  DIRB_REQUIRE(x->open, DIRB200_ESTATE, "exchange not opened (dirb200_exchange_open / _open_local)");
  DIRB_REQUIRE(x->device == h->device, DIRB200_EINVAL, "index and exchange live on different devices");
  DIRB_REQUIRE(Q >= 1 && Q <= x->max_q && k >= 1 && k <= x->max_k, DIRB200_ENOTSUP,
               "exchange window holds %d queries x %d results (got Q=%d k=%d)", x->max_q, x->max_k, Q, k);
  const PeerX px = peer_view(x);
  const unsigned tb = static_cast<unsigned>(ceil_div(Q, 256));
  if (phase == 1) {          // queries -> fp16, seed pass; this shard's k_shard-th seed bound -> every peer's window
    DIRB_REQUIRE(k_shard >= 1 && k_shard <= k, DIRB200_EINVAL, "k_shard must be in [1, k]");
    DIRB_TRY(search_begin_seed(h, q32, Q, k, k_shard, x->sel_local, stream, x->seed_local));
    tab_push_kernel<<<tb, 256, 0, stream>>>(px, x->seed_local, Q, X_TAB_SEED, X_OFF_FSEED, 3);
    count_launch();
    DIRB_CUDA(cudaGetLastError());
    return 0;
  }
  if (phase == 2) {          // filter threshold = max(local bound, MIN of the shards' seed bounds); filter pass + selection;
                             // this shard's selection thresholds -> every peer's window
    if (h->N > 0) {
      thr_min_kernel<<<tb, 256, 0, stream>>>(px, h->pend.thr, Q, h->pend.status);
      count_launch();
    }
    DIRB_TRY(search_begin_filter(h, stream));
    tab_push_kernel<<<tb, 256, 0, stream>>>(px, x->sel_local, Q, X_TAB_SEL, X_OFF_FSEL, 0);
    count_launch();
    DIRB_CUDA(cudaGetLastError());
    return 0;
  }
  if (phase == 3)            // MIN over the shards + survivors + exact re-scoring -> ordered list into every peer's window
    return search_finish_impl(h, q32, x->sel_local, nullptr, nullptr, stream, px, x->status);
  DIRB_REQUIRE(phase == 4 && scores_dev && idx_dev, DIRB200_EINVAL, "phase is 1 .. 4 (4 needs the output buffers)");
  const int n = x->world * k;
  const int threads = std::min(1024, (n + 31) / 32 * 32);
  DIRB_TRY(merge_smem_opt_in());
  merge_lists_kernel<<<Q, threads, static_cast<size_t>(n) * 16, stream>>>(nullptr, nullptr, x->world, k, 0, scores_dev, idx_dev, px,
                                                                        h->pend.status ? h->pend.status : x->status);
  count_launch();
  DIRB_CUDA(cudaGetLastError());
  if (h->pend.status) DIRB_TRY(post_status_copy(h, stream));   // (an empty shard has no status block of its own)
  return 0;
}

int dirb200_index_search_sharded(dirb200_index* h, dirb200_exchange* x, const float* q32, int Q, int k, int k_shard,
                                 double* scores_dev, int64_t* idx_dev, void* stream_) {
  DIRB_REQUIRE(scores_dev && idx_dev, DIRB200_EINVAL, "null argument");
  for (int phase = 1; phase <= 4; ++phase)
    DIRB_TRY(dirb200_index_search_sharded_phase(h, x, phase, q32, Q, k, k_shard, scores_dev, idx_dev, stream_));
  return 0;
}

int dirb200_scores_exact(const float* q_dev, int Q, const float* db_dev, int64_t N, int D, float* out_dev,
                         void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DIRB_REQUIRE(q_dev && db_dev && out_dev && D % 4 == 0, DIRB200_EINVAL, "bad arguments");
  if (Q == 0 || N == 0) return 0;
  dim3 g(static_cast<unsigned>(ceil_div(N, 8)), static_cast<unsigned>(ceil_div(Q, 4)));
  scores_exact_kernel<<<g, 256, 0, stream>>>(q_dev, Q, db_dev, N, D, out_dev);
  count_launch();
  DIRB_CUDA(cudaGetLastError());
  return 0;
}

int dirb200_aqe_expand(const float* q_dev, int Q, int D, const float* db32_dev, const int64_t* nn_idx_dev,
                       const double* nn_scores_dev, int k, double alpha, int partial, int64_t row_offset, int64_t n_rows,
                       float* out_dev, void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DIRB_REQUIRE(q_dev && nn_idx_dev && nn_scores_dev && out_dev && (db32_dev || (partial && n_rows == 0)), DIRB200_EINVAL,
               "null argument");
  DIRB_REQUIRE(k >= 1 && alpha >= 0, DIRB200_EINVAL, "k and alpha must be non-negative (test_dir.py:25)");
  DIRB_REQUIRE(k <= 2048, DIRB200_ENOTSUP, "at most 2048 neighbours per query (got %d)", k);
  if (Q == 0) return 0;
  const size_t smem = static_cast<size_t>((k + 1) & ~1) * 4 + static_cast<size_t>(k) * 8;
  aqe_kernel<<<Q, 256, smem, stream>>>(q_dev, D, db32_dev, nn_idx_dev, nn_scores_dev, k, alpha, partial, row_offset,
                                       n_rows, out_dev);
  count_launch();
  DIRB_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
