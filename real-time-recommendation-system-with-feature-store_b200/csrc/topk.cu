// Exact inner-product top-K (K4): catalogue-scoring GEMM on tcgen05 fused with a threshold-filtered select.
// Replaces faiss.IndexFlatIP.search (reference src/serving/retrieval.py:171) and the np.dot+argsort eval twin
// (scripts/evaluate_model.py:217-232, src/evaluation/metrics.py:381-396).
//
// Every query owns ONE running top-k list T in global memory (L2 resident) shared by all CTAs that scan a slice of
// the catalogue for it, guarded by a spin lock, plus a published threshold tau = score of T's k-th entry.
//   * epilogue threads (one TMEM lane = one query) only FILTER (score >= tau) and APPEND 64-bit keys
//     (ordered score << 32 | ~row) to a private double-buffered candidate list;
//   * when a list fills, its owner posts a request in a shared-memory mailbox and flips lists; four helper warps
//     take the lock, merge list and T with a warp radix select staged in shared memory, raise tau, release;
//   * helper warps also refresh the per-slot thresholds in shared memory from the global tau, so every feeder
//     benefits from what the other feeders of the same query have already seen (single-stream insertion count).
// Ties: keys order by (score desc, row asc) and the filter is >=, so the result is the exact faiss order even when a
// later-merged feeder holds a lower row id at the threshold score.  Scores are never written to HBM.
#include <cfloat>
#include <cstdlib>
#include <mutex>
#include "stream_scores.cuh"
#include "stream_scores2.cuh"
#include "../../include/b200rec.h"

namespace b200 {

// ---------------------------------------------------------------------------------------------------------------
// warp-level radix select helpers
// ---------------------------------------------------------------------------------------------------------------
// hist[256] holds digit counts; find digit d with  count(digits > d) < need <= count(digits >= d).
// Returns d; need is reduced by count(digits > d); bucket = hist[d].  Called by a full warp.
__device__ __forceinline__ int warp_pick_digit(const uint32_t* hist, int& need, int& bucket, int lane) {
  uint32_t c[8];
  uint32_t lane_total = 0;
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    c[b] = hist[lane * 8 + b];
    lane_total += c[b];
  }
  uint32_t incl = lane_total;  // sum over lanes >= lane
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_down_sync(FULL_MASK, incl, o);
    if (lane + o < 32) incl += t;
  }
  const uint32_t above = incl - lane_total;
  const bool mine = (above < (uint32_t)need) && ((uint32_t)need <= incl);
  int d = 0, nn = 0, bk = 0;
  if (mine) {
    uint32_t acc = above;
#pragma unroll
    for (int b = 7; b >= 0; --b) {
      if (acc + c[b] >= (uint32_t)need) {
        d = lane * 8 + b;
        nn = need - (int)acc;
        bk = (int)c[b];
        break;
      }
      acc += c[b];
    }
  }
  const uint32_t who = __ballot_sync(FULL_MASK, mine);
  const int src = __ffs(who) - 1;  // exactly one lane when need <= total
  d = __shfl_sync(FULL_MASK, d, src);
  need = __shfl_sync(FULL_MASK, nn, src);
  bucket = __shfl_sync(FULL_MASK, bk, src);
  return d;
}

// Exact k-th-largest threshold of `n` distinct 64-bit keys produced by `load(i)` (n > k): returns (prefix, shift) such
// that exactly k keys satisfy (key >> shift) >= prefix.  MSB-first radix select, 8-bit digits, one warp.
template <class Loader>
__device__ __forceinline__ void warp_select_threshold(const Loader& load, int n, int k, uint32_t* hist, int lane,
                                                      uint64_t& prefix_out, int& shift_out) {
  uint64_t prefix = 0;
  int need = k, shift = 56;
  for (int pass = 0; pass < 8; ++pass, shift -= 8) {
    for (int i = lane; i < 256; i += 32) hist[i] = 0;
    __syncwarp();
    for (int i0 = 0; i0 < n; i0 += 128) {  // 4 independent loads in flight per lane
      uint64_t key[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * 32 + lane;
        key[u] = (i < n) ? load(i) : 0ull;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * 32 + lane;
        const bool match = (i < n) && ((pass == 0) || ((key[u] >> (shift + 8)) == prefix));
        if (match) atomicAdd(&hist[(uint32_t)(key[u] >> shift) & 255u], 1u);
      }
    }
    __syncwarp();
    int bucket;
    const int d = warp_pick_digit(hist, need, bucket, lane);
    prefix = (prefix << 8) | (uint64_t)d;
    __syncwarp();
    if (bucket == need) break;
  }
  if (shift < 0) shift = 0;
  prefix_out = prefix;
  shift_out = shift;
}

// row filter: bit r of the bitmap (LSB first, faiss IDSelectorBitmap layout); rows past allow_n are not allowed
__device__ __forceinline__ bool row_allowed(const uint32_t* bits, uint32_t n, uint32_t row) {
  return row < n && ((__ldg(bits + (row >> 5)) >> (row & 31u)) & 1u) != 0u;
}

__device__ __noinline__ bool row_excluded(const int32_t* rows, int n, uint32_t row) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if ((uint32_t)__ldg(rows + mid) < row)
      lo = mid + 1;
    else
      hi = mid;
  }
  return lo < n && (uint32_t)__ldg(rows + lo) == row;
}

// development counters (B200REC_TOPK_DEBUG=2): appends, requests, epilogue wait cycles, helper busy cycles, lock misses
__device__ unsigned long long g_cta_end[512];  // development: globaltimer at which each CTA's helper warp 0 finished
__device__ unsigned long long g_topk_stats[16];  // [8] slow-path cycles, [9] slow-path entries, [10] group re-reads (per warp)

struct QMeta {        // one per query, global memory
  uint32_t lock;      // 0 free, 1 held by a helper warp
  uint32_t tcount;    // valid keys in the current T list
  uint32_t tsel;      // which of the two T buffers is current
  float tau;          // score of T's k-th key once T is full, else the initial threshold
};

// ---------------------------------------------------------------------------------------------------------------
// top-K epilogue policy for stream_scores_kernel
// scratch words: [0,1024) helper histograms | [1024,1536) tau_pub (u64: q<<32 | tau bits) | [1536,1792) req
//                | [1792,2048) qidx (query a slot scans now) | [2048] done | [2112,2368) reqq (query of the posted request)
//                | [2368, ...) helper staging (4 x TOPK_STG keys)
// ---------------------------------------------------------------------------------------------------------------
constexpr uint32_t REQ_VALID = 1u << 31, REQ_FINAL = 1u << 30, REQ_BUF = 1u << 29, REQ_CNT = (1u << 29) - 1u;
constexpr int TOPK_STG = 704;  // keys a helper warp can stage in shared memory (5.5 KB)
constexpr uint32_t NO_QUERY = 0xFFFFFFFFu;

struct TopkArgs {
  uint64_t* lists;                // [grid][128*NQ][2*cap]   private candidate lists A/B
  uint64_t* tlists;               // [Q][2*k]                shared running top-k lists T0/T1
  QMeta* meta;                    // [Q]
  uint32_t* left;                 // [grid][128*NQ]  leftover (list id << 31 | count) of each CTA's last segment
  const int64_t* excl_indptr;     // [Q+1] or null
  const int32_t* excl_rows;       // sorted per query
  const uint32_t* allow;          // row filter bitmap (bit r = bit r&31 of word r>>5) or null; rows >= allow_n are out
  uint32_t allow_n;
  int k;
  int cap;
  int flush;  // hand a list to the helper warps once it holds this many candidates (keeps tau fresh)
  int debug;  // development knob (DBG instantiation only): 1 = reject everything, 2 = count events, 3/5/6/8 = partial pipelines
  int hsleep; // nanoseconds an idle helper warp sleeps between mailbox polls
};

// DBG = false is the release instantiation: every development knob, counter and clock stamp below is compiled out
// (dbgv() folds to 0).  DBG = true is launched only when B200REC_TOPK_DEBUG / B200REC_STREAM_STATS is set (tools/).
template <bool DBG>
struct TopkEpiT {
  static constexpr bool kDbg = DBG;
  static constexpr int SCRATCH_BYTES = 2368 * 4 + 4 * TOPK_STG * 8;
  using Args = TopkArgs;
  static __device__ __forceinline__ int dbgv(const Args& ea) { return DBG ? dbgv(ea) : 0; }
  float tau[2];
  int cnt[2];
  uint32_t active[2] = {0u, 0u};  // which of the slot's two lists is being filled (kept across segments)
  uint32_t qid[2];
  uint64_t* buf[2];
  const int32_t* ex_lo[2];
  int ex_n[2];
  long long sp_cyc = 0;      // development counters (debug == 2), accumulated in registers, one atomic per warp at the end
  int sp_ent = 0, sp_grp = 0, n_app = 0, dbg_seg = 0;
  long long sp_a = 0, sp_b = 0, sp_c = 0;  // entry -> pending known, TMEM re-read, tests + appends

  static __device__ __forceinline__ void init_scratch(uint32_t* scratch, int lane) {
    for (int i = lane; i < 256; i += 32) {
      reinterpret_cast<uint64_t*>(scratch + 1024)[i] = ~0ull;  // tag NO_QUERY
      scratch[1536 + i] = 0u;
      scratch[1792 + i] = NO_QUERY;
    }
    if (lane == 0) scratch[2048] = 0u;
  }
  static __device__ __forceinline__ void epilogue_exit(uint32_t* scratch, int lane) {
    __syncwarp();
    if (lane == 0) atomicAdd(&scratch[2048], 1u);
  }
  static __device__ __forceinline__ void wait_idle(volatile uint32_t* req) {
    while (*req != 0u) __nanosleep(40);
  }

  template <int SLOTS, int QPT>
  __device__ __forceinline__ void begin_segment(const Args& ea, const StreamGeom& g, int s, int part,
                                                const long long (&qrow)[QPT], const int (&qslot)[QPT], int lane,
                                                uint32_t* scratch) {
    if (dbgv(ea) == 2 && blockIdx.x == 144 && threadIdx.x == 128 && dbg_seg < 60) {
      unsigned long long ns;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
      g_cta_end[256 + 2 * dbg_seg] = ns;
    }
#pragma unroll
    for (int a = 0; a < QPT; ++a) {
      const long long q = qrow[a];
      const bool valid = (q >= 0) && dbgv(ea) != 1 && dbgv(ea) != 3 && dbgv(ea) != 5;
      qid[a] = valid ? (uint32_t)q : NO_QUERY;
      tau[a] = valid ? __ldcg(&ea.meta[q].tau) : INFINITY;
      cnt[a] = 0;
      buf[a] = ea.lists + ((size_t)blockIdx.x * SLOTS + qslot[a]) * (2 * (size_t)ea.cap);
      ex_lo[a] = nullptr;
      ex_n[a] = 0;
      if (ea.excl_indptr != nullptr && valid) {
        const int64_t lo = ea.excl_indptr[q], hi = ea.excl_indptr[q + 1];
        ex_lo[a] = ea.excl_rows + lo;
        ex_n[a] = (int)(hi - lo);
      }
      // a hand-over request of the previous segment may still be in the mailbox: it names its own query (reqq) and
      // list, and this segment fills the other list
      *reinterpret_cast<volatile uint32_t*>(scratch + 1792 + qslot[a]) = qid[a];
    }
  }

  // pick up thresholds raised by any feeder of this query; hand over a list that could overflow during the next tile
  template <int BN, int QPT>
  __device__ __forceinline__ void pre_tile(const Args& ea, const StreamGeom& g, const int (&qslot)[QPT], int lane,
                                           uint32_t* scratch) {
#pragma unroll
    for (int a = 0; a < QPT; ++a) {
      const uint64_t pub = *reinterpret_cast<volatile uint64_t*>(scratch + 1024 + 2 * qslot[a]);
      if ((uint32_t)(pub >> 32) == qid[a] && qid[a] != NO_QUERY) tau[a] = fmaxf(tau[a], __uint_as_float((uint32_t)pub));
      const bool must = cnt[a] + BN > ea.cap;   // the list could overflow during the next tile
      volatile uint32_t* reqp = scratch + 1536 + qslot[a];
      if (dbgv(ea) == 6) {  // development knob: candidates are found and appended but never merged
        if (must || cnt[a] >= ea.flush) cnt[a] = 0;
      } else if (must || (cnt[a] >= ea.flush && *reqp == 0u)) {
        volatile uint32_t* req = reqp;
        if (dbgv(ea) == 2) {
          const long long t0 = clock64();
          wait_idle(req);
          atomicAdd(&g_topk_stats[2], (unsigned long long)(clock64() - t0));
          atomicAdd(&g_topk_stats[1], 1ull);
        } else {
          wait_idle(req);
        }
        *reinterpret_cast<volatile uint32_t*>(scratch + 2112 + qslot[a]) = qid[a];
        __threadfence_block();
        *req = REQ_VALID | (active[a] ? REQ_BUF : 0u) | (uint32_t)cnt[a];
        active[a] ^= 1u;
        cnt[a] = 0;
      }
    }
  }

  // Append one candidate (rare).  Kept out of the scan on purpose: the whole epilogue loop must stay inside the
  // instruction cache and free of branches (a fully unrolled 64-column scan with an inlined exclusion search was
  // 70 KB of SASS and spent 80% of its issue slots waiting for instruction fetch).
  __device__ __forceinline__ void append(const Args& ea, int a, float x, uint32_t row) {
    if ((ex_n[a] == 0 || !row_excluded(ex_lo[a], ex_n[a], row)) && (ea.allow == nullptr || row_allowed(ea.allow, ea.allow_n, row))) {
      __stcg(buf[a] + (active[a] ? ea.cap : 0) + cnt[a], make_key(x, row));
      ++cnt[a];
      if (dbgv(ea) == 2) ++n_app;
    }
  }

  // One accumulator buffer: BN columns of this thread's TMEM lane (= one query), 64 at a time.
  //   common case  : eight 8-column group maxima folded into one maximum (35 max ops), one compare, one vote
  //   rare case    : some lane saw a score >= tau.  The flagged groups come from the group maxima already in registers
  //                  (one REDUX.OR over the warp); each flagged group is re-read from TMEM (warp-uniform loop, tcgen05.ld
  //                  is warp-collective) and its eight scores are tested.  This path gates the MMA pipe: an accumulator
  //                  is only released when every epilogue warp that reads it is done.
  template <int BN>
  __device__ __forceinline__ void tile(const Args& ea, const StreamGeom& g, int a, uint32_t taddr,
                                       unsigned long long row0_ll) {
    const uint32_t row0 = (uint32_t)row0_ll;
    if (dbgv(ea) == 3) return;  // development knob: MMA + TMA pipeline only (TMEM never read)
#pragma unroll 1
    for (int c = 0; c < BN; c += 64) {
      uint32_t v0[32], v1[32];
      tmem_ld_32x32(taddr + c, v0);
      tmem_ld_32x32(taddr + c + 32, v1);
      tmem_ld_wait();
      if (dbgv(ea) == 5) {  // development knob: TMEM read cost only
        asm volatile("" ::"r"(v0[0]), "r"(v1[31]));
        continue;
      }
      // fast path: eight 8-column group maxima (4 max ops each) folded into one maximum, one compare, one vote
      float gm[8];
      group_max(v0, gm);
      group_max(v1, gm + 4);
      const float m64 = fmax3(fmax3(gm[0], gm[1], gm[2]), fmax3(gm[3], gm[4], gm[5]), fmaxf(gm[6], gm[7]));
      if (!__any_sync(FULL_MASK, m64 >= tau[a])) continue;
      long long sp0 = 0;
      if (dbgv(ea) == 2) sp0 = clock64();
      uint32_t gbits = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) gbits |= (gm[j] >= tau[a]) ? (1u << j) : 0u;
      uint32_t pending = __reduce_or_sync(FULL_MASK, gbits);
      if (dbgv(ea) == 2) {
        const long long t1 = clock64();
        sp_a += t1 - sp0;
      }
      const uint32_t base = row0 + c;
      const bool edge = base + 64u > (uint32_t)g.N;  // only the last tile of a shard can hold rows past its end
#pragma unroll 1
      while (pending) {
        const int j = __ffs(pending) - 1;
        pending &= pending - 1;
        uint32_t w[8];
        long long t2 = 0;
        if (dbgv(ea) == 2) t2 = clock64();
        tmem_ld_32x8(taddr + c + 8 * j, w);
        tmem_ld_wait();
        if (dbgv(ea) == 2) {
          asm volatile("" ::"r"(w[0]), "r"(w[7]) : "memory");
          const long long t3 = clock64();
          sp_b += t3 - t2;
          t2 = t3;
        }
        const uint32_t rb = base + 8u * (uint32_t)j;
        test_group(ea, g, a, w, rb, edge);
        if (dbgv(ea) == 2) {
          ++sp_grp;
          sp_c += clock64() - t2;
        }
      }
      if (dbgv(ea) == 2) {
        sp_cyc += clock64() - sp0;
        ++sp_ent;
      }
    }
  }

  // Tests the eight scores of one flagged group and appends the candidates.  Branch-free hit mask first (every lane
  // runs it; each instruction of a cold, serial path costs ~10 cycles), then only lanes that hold a candidate
  // (typically one lane, one score) diverge.
  __device__ __forceinline__ void test_group(const Args& ea, const StreamGeom& g, int a, const uint32_t (&w)[8],
                                             uint32_t rb, bool edge) {
    uint32_t hits = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) hits |= (__uint_as_float(w[i]) >= tau[a]) ? (1u << i) : 0u;
    if (edge) hits &= rb < (uint32_t)g.N ? (((uint32_t)g.N - rb) >= 8u ? 0xFFu : (1u << ((uint32_t)g.N - rb)) - 1u) : 0u;
    if (hits) {
      if ((hits & (hits - 1u)) == 0u) {  // one hit: it is the group maximum
        const float m0 = fmax3(__uint_as_float(w[0]), __uint_as_float(w[1]), __uint_as_float(w[2]));
        const float m1 = fmax3(__uint_as_float(w[3]), __uint_as_float(w[4]), __uint_as_float(w[5]));
        const float x = fmax3(m0, m1, fmaxf(__uint_as_float(w[6]), __uint_as_float(w[7])));
        if (!edge) {
          append(ea, a, x, rb + (uint32_t)(__ffs(hits) - 1));
          hits = 0;
        }
      }
#pragma unroll 1
      while (hits) {
        const int i = __ffs(hits) - 1;
        hits &= hits - 1;
        uint32_t xb = w[0];
#pragma unroll
        for (int u = 1; u < 8; ++u) xb = (i == u) ? w[u] : xb;
        append(ea, a, __uint_as_float(xb), rb + (uint32_t)i);
      }
    }
  }

  // maxima of the four 8-column groups of a 32-column register block
  static __device__ __forceinline__ void group_max(const uint32_t (&v)[32], float* gm) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float m0 = fmax3(__uint_as_float(v[8 * j + 0]), __uint_as_float(v[8 * j + 1]), __uint_as_float(v[8 * j + 2]));
      const float m1 = fmax3(__uint_as_float(v[8 * j + 3]), __uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5]));
      gm[j] = fmax3(m0, m1, fmaxf(__uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7])));
    }
  }

  // End of a segment.  A CTA's LAST segment does not merge: it waits for its in-flight merges and publishes what is
  // left in the active list (id << 31 | count); the final per-query kernel selects over T u leftovers with one CTA per
  // query, which replaces a serialised tail of ~38 K locked merges.  Earlier segments (CTAs spanning a supertile
  // boundary) hand the list to the helper warps as usual because their buffers are reused by the next segment.
  template <int SLOTS, int QPT>
  __device__ __forceinline__ void end_segment(const Args& ea, const StreamGeom& g, int s, int part,
                                              const int (&qslot)[QPT], int lane, uint32_t* scratch, bool last) {
    if (dbgv(ea) == 2 && blockIdx.x == 144 && threadIdx.x == 128 && dbg_seg < 60) {
      unsigned long long ns;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
      g_cta_end[256 + 2 * dbg_seg + 1] = ns;
      g_cta_end[400 + 4 * dbg_seg] = (unsigned long long)sp_ent;
      g_cta_end[401 + 4 * dbg_seg] = (unsigned long long)n_app;
      g_cta_end[402 + 4 * dbg_seg] = (unsigned long long)__float_as_uint(tau[0]);
      g_cta_end[403 + 4 * dbg_seg] = (unsigned long long)sp_cyc;
      ++dbg_seg;
    }
    if (last) {
      if (dbgv(ea) == 2) {
        const int apps = __reduce_add_sync(FULL_MASK, n_app);
        if (lane == 0 && (blockIdx.x == 144 || blockIdx.x == 145 || blockIdx.x == 0)) {
          const int w = (blockIdx.x == 0 ? 16 : (blockIdx.x - 144) * 8) + (threadIdx.x >> 5) - 4;
          g_cta_end[300 + 3 * w] = (unsigned long long)sp_ent;
          g_cta_end[301 + 3 * w] = (unsigned long long)apps;
          g_cta_end[302 + 3 * w] = (unsigned long long)sp_cyc;
        }
        if (lane == 0) {
          atomicAdd(&g_topk_stats[0], (unsigned long long)apps);
          atomicAdd(&g_topk_stats[8], (unsigned long long)sp_cyc);
          atomicAdd(&g_topk_stats[9], (unsigned long long)sp_ent);
          atomicAdd(&g_topk_stats[10], (unsigned long long)sp_grp);
          atomicAdd(&g_topk_stats[11], (unsigned long long)sp_a);
          atomicAdd(&g_topk_stats[12], (unsigned long long)sp_b);
          atomicAdd(&g_topk_stats[13], (unsigned long long)sp_c);
        }
      }
#pragma unroll
      for (int a = 0; a < QPT; ++a) {
        wait_idle(scratch + 1536 + qslot[a]);
        ea.left[(size_t)blockIdx.x * SLOTS + qslot[a]] =
            (qid[a] != NO_QUERY) ? ((active[a] << 31) | (uint32_t)cnt[a]) : 0u;
      }
      return;
    }
#pragma unroll
    for (int a = 0; a < QPT; ++a) {
      // hand the list over and move on: the next segment fills the other list, and its first flush waits for this
      // request like for any other (waiting here for up to 256 merges per CTA made every supertile switch ~175 us)
      volatile uint32_t* req = scratch + 1536 + qslot[a];
      wait_idle(req);
      *reinterpret_cast<volatile uint32_t*>(scratch + 2112 + qslot[a]) = qid[a];
      __threadfence_block();
      *req = REQ_VALID | REQ_FINAL | (active[a] ? REQ_BUF : 0u) | (uint32_t)cnt[a];
      active[a] ^= 1u;
      cnt[a] = 0;
    }
  }

  // ------------------------------------------------------------------ helper warps: asynchronous merge into T
  struct SmemLoader {
    const uint64_t* keys;
    __device__ __forceinline__ uint64_t operator()(int i) const { return keys[i]; }
  };
  struct UnionLoader {
    const uint64_t* t;
    const uint64_t* src;
    int tc;
    __device__ __forceinline__ uint64_t operator()(int i) const { return i < tc ? __ldcg(t + i) : __ldcg(src + (i - tc)); }
  };

  template <class Loader>
  static __device__ __forceinline__ float merge_select(const Loader& ld, int total, int k, uint64_t* tnext,
                                                       uint32_t* hist, int lane) {
    uint64_t prefix;
    int shift;
    warp_select_threshold(ld, total, k, hist, lane, prefix, shift);
    const uint32_t lt_mask = (1u << lane) - 1u;
    int outp = 0;
    uint64_t minkey = ~0ull;
    for (int i0 = 0; i0 < total; i0 += 32) {
      const int i = i0 + lane;
      const uint64_t key = (i < total) ? ld(i) : 0ull;
      const bool keep = (i < total) && ((key >> shift) >= prefix);
      const uint32_t b = __ballot_sync(FULL_MASK, keep);
      if (keep) {
        const int pos = outp + __popc(b & lt_mask);
        if (pos < k) __stcg(tnext + pos, key);
        minkey = key < minkey ? key : minkey;
      }
      outp += __popc(b);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const uint64_t t = __shfl_xor_sync(FULL_MASK, minkey, o);
      minkey = t < minkey ? t : minkey;
    }
    return ord_f32((uint32_t)(minkey >> 32));
  }

  // Small merge (tc + n <= 256 keys, the common case for k <= ~200): every lane keeps 8 keys in registers and the warp
  // finds the k-th largest by a bit-wise descent from the highest bit in which the keys differ — per bit 8 compares,
  // one REDUX.SUM — stopping as soon as exactly k keys lie above the probe (about log2(total) + 4 steps on distinct
  // scores).  ~5x fewer cycles than the shared-memory histogram select below, which matters because the number of
  // merges per query is independent of the catalogue size: on a 1.25 M-row shard they were half of the kernel time.
  static __device__ __forceinline__ float merge_select_regs(const uint64_t* tcur, int tc, const uint64_t* src, int n,
                                                             int k, uint64_t* tnext, int lane) {
    const int total = tc + n;
    uint64_t key[8];
    uint64_t orv = 0ull, andv = ~0ull;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int i = j * 32 + lane;
      key[j] = 0ull;
      if (i < total) {
        key[j] = i < tc ? __ldcg(tcur + i) : __ldcg(src + (i - tc));
        orv |= key[j];
        andv &= key[j];
      }
    }
    const uint32_t or_hi = __reduce_or_sync(FULL_MASK, (uint32_t)(orv >> 32)), or_lo = __reduce_or_sync(FULL_MASK, (uint32_t)orv);
    const uint32_t and_hi = __reduce_and_sync(FULL_MASK, (uint32_t)(andv >> 32)), and_lo = __reduce_and_sync(FULL_MASK, (uint32_t)andv);
    const uint64_t diff = (((uint64_t)(or_hi ^ and_hi)) << 32) | (uint64_t)(or_lo ^ and_lo);
    uint64_t P = ((uint64_t)and_hi << 32) | and_lo;
    if (diff != 0ull) {
      const int hb = 63 - __clzll((long long)diff);
      P = hb == 63 ? 0ull : (P & ~((2ull << hb) - 1ull));
      for (int b = hb; b >= 0; --b) {
        const uint64_t cand = P | (1ull << b);
        int c = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) c += key[j] >= cand ? 1 : 0;
        c = __reduce_add_sync(FULL_MASK, c);
        if (c >= k) P = cand;
        if (c == k) break;
      }
    }
    // exactly k keys are >= P (keys are distinct: one per catalogue row)
    const uint32_t lt_mask = (1u << lane) - 1u;
    int outp = 0;
    uint64_t minkey = ~0ull;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const bool keep = key[j] >= P && key[j] != 0ull;
      const uint32_t bal = __ballot_sync(FULL_MASK, keep);
      if (keep) {
        const int pos = outp + __popc(bal & lt_mask);
        if (pos < k) __stcg(tnext + pos, key[j]);
        minkey = key[j] < minkey ? key[j] : minkey;
      }
      outp += __popc(bal);
    }
    const uint32_t mh = __reduce_min_sync(FULL_MASK, (uint32_t)(minkey >> 32));  // tau only needs the score half
    return ord_f32(mh);
  }

  template <int SLOTS, int EPI_WARPS>
  static __device__ void helper(const Args& ea, const StreamGeom& g, int hw, int lane, uint32_t* scratch) {
    constexpr int QS = SLOTS;
    constexpr int PER_LANE = SLOTS / 128;  // SLOTS / (4 warps * 32 lanes)
    uint32_t* hist = scratch + hw * 256;
    volatile uint64_t* tau_pub = reinterpret_cast<volatile uint64_t*>(scratch + 1024);
    volatile uint32_t* reqs = scratch + 1536;
    volatile uint32_t* qidx = scratch + 1792;
    volatile uint32_t* done = scratch + 2048;
    volatile uint32_t* reqq = scratch + 2112;
    uint64_t* stage = reinterpret_cast<uint64_t*>(scratch + 2368) + hw * TOPK_STG;
    const int k = ea.k;
    // SM cycles and wall nanoseconds of this launch as seen by CTA 0 (=> the SM clock the kernel really ran at)
    const bool stamp = DBG && hw == 0 && lane == 0;
    long long c_begin = 0;
    unsigned long long ns_begin = 0;
    if (stamp) {
      c_begin = clock64();
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns_begin));
    }
    for (;;) {
      const bool finished = (*done == (uint32_t)EPI_WARPS);
      bool any = false;
#pragma unroll
      for (int j = 0; j < PER_LANE; ++j) {
        const int my_slot = hw * 32 * PER_LANE + j * 32 + lane;
        const uint32_t r = reqs[my_slot];
        const uint32_t rq = reqq[my_slot];  // query of the posted request (the slot may already scan another one)
        const uint32_t myq = qidx[my_slot];
        // refresh this slot's published threshold from the query's global tau (tagged with the query id, so a slot that
        // has meanwhile moved on to another query ignores it)
        if (myq != NO_QUERY) {
          const float t = __ldcg(&ea.meta[myq].tau);
          tau_pub[my_slot] = ((uint64_t)myq << 32) | (uint64_t)__float_as_uint(t);
        }
        uint32_t todo = __ballot_sync(FULL_MASK, (r & REQ_VALID) != 0u);
        while (todo) {
          any = true;
          const long long hb0 = DBG ? clock64() : 0;
          const int owner = __ffs(todo) - 1;
          todo &= todo - 1;
          const uint32_t ro = __shfl_sync(FULL_MASK, r, owner);
          const uint32_t q = __shfl_sync(FULL_MASK, rq, owner);
          const int slot = hw * 32 * PER_LANE + j * 32 + owner;
          const int n = (int)(ro & REQ_CNT);
          if (q == NO_QUERY || n == 0) {  // nothing to merge: acknowledge
            __syncwarp();
            if (lane == 0) reqs[slot] = 0u;
            continue;
          }
          QMeta* m = ea.meta + q;
          uint32_t got = 0;
          if (lane == 0) got = (atomicCAS(&m->lock, 0u, 1u) == 0u) ? 1u : 0u;
          got = __shfl_sync(FULL_MASK, got, 0);
          if (!got) {  // another CTA is merging into this query's T: retry on the next poll
            if (dbgv(ea) == 2 && lane == 0) atomicAdd(&g_topk_stats[4], 1ull);
            continue;
          }
          __threadfence();
          const uint64_t* src = ea.lists + ((size_t)blockIdx.x * QS + slot) * (2 * (size_t)ea.cap) + ((ro & REQ_BUF) ? ea.cap : 0);
          int tc = (int)__ldcg(&m->tcount);
          int ts = (int)__ldcg(&m->tsel);
          uint64_t* tcur = ea.tlists + (size_t)q * 2 * k + (size_t)ts * k;
          uint64_t* tnext = ea.tlists + (size_t)q * 2 * k + (size_t)(ts ^ 1) * k;
          if (tc + n <= k) {
            for (int i = lane; i < n; i += 32) __stcg(tcur + tc + i, __ldcg(src + i));
            tc += n;
            __threadfence();
            if (lane == 0) m->tcount = (uint32_t)tc;
          } else {
            const int total = tc + n;
            float newtau;
            if (total <= 256 && dbgv(ea) != 8) {
              newtau = merge_select_regs(tcur, tc, src, n, k, tnext, lane);
            } else if (total <= TOPK_STG) {
              for (int i = lane; i < total; i += 32) stage[i] = (i < tc) ? __ldcg(tcur + i) : __ldcg(src + (i - tc));
              __syncwarp();
              newtau = merge_select(SmemLoader{stage}, total, k, tnext, hist, lane);
            } else {
              newtau = merge_select(UnionLoader{tcur, src, tc}, total, k, tnext, hist, lane);
            }
            __threadfence();
            if (lane == 0) {
              m->tsel = (uint32_t)(ts ^ 1);
              m->tcount = (uint32_t)k;
              *reinterpret_cast<volatile float*>(&m->tau) = newtau;
            }
          }
          __syncwarp();
          if (lane == 0) {
            __threadfence();
            atomicExch(&m->lock, 0u);
            reqs[slot] = 0u;
          }
          __syncwarp();
          if (dbgv(ea) == 2 && lane == 0) atomicAdd(&g_topk_stats[3], (unsigned long long)(clock64() - hb0));
        }
      }
      if (!any) {
        if (finished) break;
        __nanosleep(ea.hsleep);  // idle helper warps must not burn issue slots (the kernel is power-limited)
      }
    }
    if (stamp) {
      unsigned long long ns_end;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns_end));
      if (blockIdx.x == 0) g_topk_stats[6] = (unsigned long long)(clock64() - c_begin) * 1000ull / (ns_end - ns_begin + 1);  // MHz
      atomicMax(&g_topk_stats[5], ~ns_begin);  // ~(earliest CTA start)
      atomicMax(&g_topk_stats[7], ns_end);     // latest CTA end
      if (blockIdx.x < 512) g_cta_end[blockIdx.x] = ns_end;
    }
  }
};

using TopkEpi = TopkEpiT<false>;
using TopkEpiDbg = TopkEpiT<true>;

// ---------------------------------------------------------------------------------------------------------------
// Sampling pass policy: the same streaming kernel over a strided sample of the catalogue (m = N/32 rows), fast path
// only — each epilogue thread writes the MAXIMUM score of every group of `gw` sampled rows for its query.  Group
// maxima belong to distinct rows, so the k-th largest of them is a valid lower bound of the final k-th score; with
// thousands of groups per query it is nearly as tight as the exact k-th of the whole sample, and it costs no
// selection at all.  It removes the cold-start phase in which almost every score is a candidate.
// MASK = true (filtered search): sampled rows outside the row filter count as -inf, so the group maxima stay a lower
// bound of the k-th ALLOWED score; a threshold taken from disallowed rows could exceed it and drop results.
// ---------------------------------------------------------------------------------------------------------------
struct SampleArgs {
  float* out;              // [Q][ngroups]
  int ngroups;             // m / gw
  int gw;                  // 32, 64 or 128 sampled rows per group
  const uint32_t* allow;   // MASK only: row filter bitmap and its length in rows
  uint32_t allow_n;
  uint32_t stride;         // MASK only: sampled row j is catalogue row j * stride
};

template <bool MASK>
struct SampleMaxEpiT {
  static constexpr bool kDbg = false;
  static constexpr int SCRATCH_BYTES = 64;
  using Args = SampleArgs;
  long long qrow[2];

  static __device__ __forceinline__ void init_scratch(uint32_t*, int) {}
  static __device__ __forceinline__ void epilogue_exit(uint32_t*, int) {}
  template <int SLOTS, int EPI_WARPS>
  static __device__ __forceinline__ void helper(const Args&, const StreamGeom&, int, int, uint32_t*) {}

  template <int SLOTS, int QPT>
  __device__ __forceinline__ void begin_segment(const Args&, const StreamGeom&, int, int, const long long (&q)[QPT],
                                                const int (&)[QPT], int, uint32_t*) {
#pragma unroll
    for (int a = 0; a < QPT; ++a) qrow[a] = q[a];
  }
  template <int BN, int QPT>
  __device__ __forceinline__ void pre_tile(const Args&, const StreamGeom&, const int (&)[QPT], int, uint32_t*) {}

  template <int BN>
  __device__ __forceinline__ void tile(const Args& ea, const StreamGeom&, int a, uint32_t taddr,
                                       unsigned long long row0) {
    float run = -INFINITY;
#pragma unroll 1
    for (int c = 0; c < BN; c += 32) {
      uint32_t v[32];
      tmem_ld_32x32(taddr + c, v);
      tmem_ld_wait();
      if (MASK) {  // column c + i of the tile is sampled row row0 + c + i: one bitmap probe per lane, one vote
        const unsigned long long row = (row0 + c + (threadIdx.x & 31u)) * (unsigned long long)ea.stride;
        const uint32_t ok = __ballot_sync(FULL_MASK, row < ea.allow_n && row_allowed(ea.allow, ea.allow_n, (uint32_t)row));
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = ((ok >> i) & 1u) ? v[i] : __float_as_uint(-INFINITY);
      }
      float m4[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float m0 = fmax3(__uint_as_float(v[8 * j + 0]), __uint_as_float(v[8 * j + 1]), __uint_as_float(v[8 * j + 2]));
        const float m1 = fmax3(__uint_as_float(v[8 * j + 3]), __uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5]));
        m4[j] = fmax3(m0, m1, fmaxf(__uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7])));
      }
      run = fmaxf(run, fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])));
      if (((c + 32) % ea.gw) == 0) {
        if (qrow[a] >= 0) ea.out[(size_t)qrow[a] * ea.ngroups + (row0 + c) / ea.gw] = run;
        run = -INFINITY;
      }
    }
  }

  template <int SLOTS, int QPT>
  __device__ __forceinline__ void end_segment(const Args&, const StreamGeom&, int, int, const int (&)[QPT], int,
                                              uint32_t*, bool) {}
};
using SampleMaxEpi = SampleMaxEpiT<false>;

// ---------------------------------------------------------------------------------------------------------------
// block-level exact select + sort of `n` keys produced by a loader; one CTA (256 threads) per query
// ---------------------------------------------------------------------------------------------------------------
constexpr int FIN_THREADS = 256;

template <class Loader>
__device__ void block_select_sort_core(const Loader& load, int n, int k_out, uint64_t* skeys /*[pow2 >= k_out]*/, int P,
                                       uint32_t* hist /*[256]*/, int* s_misc /*[8]*/) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // count valid keys
  if (tid == 0) s_misc[0] = 0;
  __syncthreads();
  int local = 0;
  for (int i = tid; i < n; i += FIN_THREADS) local += load(i) != 0ull;
  for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(FULL_MASK, local, o);
  if (lane == 0 && local) atomicAdd(&s_misc[0], local);
  __syncthreads();
  const int n_valid = s_misc[0];
  uint64_t prefix = 1;
  int shift = 0;
  if (n_valid > k_out) {
    prefix = 0;
    shift = 56;
    int need = k_out;
    for (int pass = 0; pass < 8; ++pass, shift -= 8) {
      hist[tid] = 0;
      __syncthreads();
      for (int i = tid; i < n; i += FIN_THREADS) {
        const uint64_t key = load(i);
        const bool match = (pass == 0) || ((key >> (shift + 8)) == prefix);
        if (match && key != 0ull) atomicAdd(&hist[(uint32_t)(key >> shift) & 255u], 1u);
      }
      __syncthreads();
      if (warp == 0) {
        int bucket;
        const int d = warp_pick_digit(hist, need, bucket, lane);
        if (lane == 0) {
          s_misc[1] = d;
          s_misc[2] = need;
          s_misc[3] = bucket;
        }
      }
      __syncthreads();
      prefix = (prefix << 8) | (uint64_t)s_misc[1];
      need = s_misc[2];
      const int bucket = s_misc[3];
      __syncthreads();
      if (bucket == need) break;
    }
    if (shift < 0) shift = 0;
  }
  // gather survivors, pad, bitonic sort descending
  if (tid == 0) s_misc[4] = 0;
  for (int i = tid; i < P; i += FIN_THREADS) skeys[i] = 0ull;
  __syncthreads();
  for (int i = tid; i < n; i += FIN_THREADS) {
    const uint64_t key = load(i);
    if (key != 0ull && (key >> shift) >= prefix) {
      const int pos = atomicAdd(&s_misc[4], 1);
      if (pos < P) skeys[pos] = key;
    }
  }
  __syncthreads();
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < P / 2; i += FIN_THREADS) {
        const int lo = 2 * i - (i & (stride - 1));  // index with bit `stride` cleared
        const int hi = lo + stride;
        const bool desc = ((lo & size) == 0);
        const uint64_t a = skeys[lo], b = skeys[hi];
        if ((a < b) == desc) {
          skeys[lo] = b;
          skeys[hi] = a;
        }
      }
      __syncthreads();
    }
  }
}

struct StagedKeys {
  const uint64_t* keys;
  __device__ __forceinline__ uint64_t operator()(int i) const { return keys[i]; }
};
// The select makes up to ten passes over the candidates: stage them in shared memory once when they fit (the loaders
// read global memory through index arithmetic or a binary search over source lists).
template <class Loader>
__device__ __forceinline__ void block_select_sort(const Loader& load, int n, int k_out, uint64_t* skeys, int P,
                                                  uint32_t* hist, int* s_misc, uint64_t* stage, int stage_cap) {
  if (n <= stage_cap) {
    for (int i = threadIdx.x; i < n; i += FIN_THREADS) stage[i] = load(i);
    __syncthreads();
    block_select_sort_core(StagedKeys{stage}, n, k_out, skeys, P, hist, s_misc);
  } else {
    block_select_sort_core(load, n, k_out, skeys, P, hist, s_misc);
  }
}

// Result fan-out: the per-query result rows are stored to `n` destinations — the caller's own buffer and, in row-sharded
// search, the slot of this shard in every peer GPU's gather buffer (peer-mapped NVLink addresses).  The select kernel
// then IS the all-gather: no separate collective launch, the stores ride NVLink while other queries are still selected.
constexpr int FAN_MAX = 16;
struct OutFan {
  int n;
  float* s[FAN_MAX];
  int64_t* i[FAN_MAX];
};

// remap (nullable): the select ran over a compacted catalogue whose row j is local row remap[j] (compact filtered search
// of a row shard); the id leaves the kernel already mapped, because on the peer path it is stored straight to the peers
__device__ __forceinline__ void write_result(const uint64_t* skeys, int k_out, int64_t row_offset, const int64_t* remap,
                                             float* out_s, int64_t* out_i) {
  for (int i = threadIdx.x; i < k_out; i += FIN_THREADS) {
    const uint64_t key = skeys[i];
    if (key == 0ull) {
      out_s[i] = -FLT_MAX;
      out_i[i] = -1;
    } else {
      out_s[i] = ord_f32((uint32_t)(key >> 32));
      const uint32_t row = ~(uint32_t)key;
      out_i[i] = (remap != nullptr ? __ldg(remap + row) : (int64_t)row) + row_offset;
    }
  }
}

// Final per-query kernel: candidates = the query's shared list T  u  the leftovers published by every CTA whose last
// segment scanned this query's supertile; exact select of the k best + bitonic sort (score desc, row asc).
constexpr int FIN_MAX_SRC = 160;
struct MultiLoader {
  const uint64_t* const* ptr;  // shared memory
  const int* off;              // shared memory, nsrc + 1 prefix offsets
  int nsrc;
  __device__ __forceinline__ uint64_t operator()(int i) const {
    int lo = 0, hi = nsrc - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (off[mid] <= i)
        lo = mid;
      else
        hi = mid - 1;
    }
    return __ldcg(ptr[lo] + (i - off[lo]));
  }
};

__global__ void __launch_bounds__(FIN_THREADS)
topk_final_kernel(const StreamGeom g, int v2, int qs /*queries per supertile*/, int slots /*per CTA*/,
                  const uint64_t* __restrict__ tlists, const QMeta* __restrict__ meta,
                  const uint64_t* __restrict__ lists, const uint32_t* __restrict__ left, int cap, int k, int P,
                  int stage_cap, int64_t row_offset, const int64_t* __restrict__ remap, const OutFan fan) {
  extern __shared__ uint64_t fin_smem[];
  __shared__ uint32_t hist[256];
  __shared__ int s_misc[8];
  __shared__ const uint64_t* s_ptr[FIN_MAX_SRC];
  __shared__ int s_off[FIN_MAX_SRC + 1];
  __shared__ int s_last[FIN_MAX_SRC];  // 2-CTA kernel: supertile of every unit's last segment (64-bit divisions: in parallel)
  const int q = blockIdx.x;
  const int s = q / qs, inq = q - s * qs;
  if (v2) {
    for (int u = threadIdx.x; u < g.grid / 2 && u < FIN_MAX_SRC; u += FIN_THREADS) s_last[u] = geom2_last_super(g, u);
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    int n = 0, ns = 0;
    s_ptr[ns] = tlists + (size_t)q * 2 * k + (size_t)meta[q].tsel * k;
    s_off[ns++] = n;
    n += (int)meta[q].tcount;
    // work units (CTAs, or CTA pairs when v2) whose LAST segment scanned this query's supertile left a list behind
    const int u0 = v2 ? 0 : geom_first_cta(g, s), u1 = v2 ? g.grid / 2 - 1 : geom_last_cta(g, s);
    for (int u = u0; u <= u1; ++u) {
      if (v2) {
        if (u >= FIN_MAX_SRC || s_last[u] != s) continue;
      } else {
        long long wend = (long long)(u + 1) * g.W;
        if (wend > g.total) wend = g.total;
        if ((int)((wend - 1) / g.T) != s) continue;  // that unit's last segment belongs to another supertile
      }
      const int cta = v2 ? 2 * u + ((inq >> 7) & 1) : u;
      const int nslot = v2 == 1 ? 2 : 1;
      for (int h = 0; h < nslot && ns < FIN_MAX_SRC; ++h) {
        const int slot = v2 == 1 ? h * 128 + (inq & 127) : (v2 == 2 ? (inq >> 8) * 128 + (inq & 127) : inq);
        const uint32_t l = left[(size_t)cta * slots + slot];
        const int cnt = (int)(l & 0x7FFFFFFFu);
        if (cnt == 0) continue;
        s_ptr[ns] = lists + ((size_t)cta * slots + slot) * (2 * (size_t)cap) + ((l >> 31) ? cap : 0);
        s_off[ns++] = n;
        n += cnt;
      }
    }
    s_off[ns] = n;
    s_misc[5] = ns;
    s_misc[6] = n;
  }
  __syncthreads();
  MultiLoader ld{s_ptr, s_off, s_misc[5]};
  const int n = s_misc[6];
  __syncthreads();
  block_select_sort(ld, n, k, fin_smem, P, hist, s_misc, fin_smem + P, stage_cap);
  for (int d = 0; d < fan.n; ++d)
    write_result(fin_smem, k, row_offset, remap, fan.s[d] + (size_t)q * k, fan.i[d] + (size_t)q * k);
}

// per-query k largest group maxima of the sampling pass (descending; -FLT_MAX padding): what shards exchange so that
// every GPU starts from the k-th best of the UNION of all samples
struct FloatRowLoader {
  const float* row;
  __device__ __forceinline__ uint64_t operator()(int i) const {
    return (static_cast<uint64_t>(f32_ord(__ldcg(row + i))) << 32) | static_cast<uint64_t>(~(uint32_t)i);
  }
};
__global__ void __launch_bounds__(FIN_THREADS)
sample_topk_kernel(const float* __restrict__ S, int m, int k, int P, int stage_cap, const OutFan fan) {
  extern __shared__ uint64_t fin_smem[];
  __shared__ uint32_t hist[256];
  __shared__ int s_misc[8];
  const int q = blockIdx.x;
  FloatRowLoader ld{S + (size_t)q * m};
  block_select_sort(ld, m, k, fin_smem, P, hist, s_misc, fin_smem + P, stage_cap);
  for (int i = threadIdx.x; i < k; i += FIN_THREADS) {
    const uint64_t key = fin_smem[i];
    const float v = key == 0ull ? -FLT_MAX : ord_f32((uint32_t)(key >> 32));
    for (int d = 0; d < fan.n; ++d) fan.s[d][(size_t)q * k + i] = v;
  }
}

// n values `s` (and ids `id` where the destination has an id array) stored to every fan-out destination: the padding rows
// a row shard with nothing to sample or search still owes every peer's gather buffer
__global__ void __launch_bounds__(256) fan_fill_kernel(const OutFan fan, int64_t n, float s, int64_t id) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    for (int d = 0; d < fan.n; ++d) {
      fan.s[d][i] = s;
      if (fan.i[d] != nullptr) fan.i[d][i] = id;
    }
}

// k-th largest of the `parts` x k_in pooled sample maxima of every query (parts-major layout [parts][Q][k_in], as the
// shards' fan-out stores leave it): the shared threshold of row-sharded search in one launch (no ids, no sort output)
struct PooledLoader {
  const float* vals;
  size_t part_stride;
  int k_in;
  __device__ __forceinline__ uint64_t operator()(int i) const {
    const int p = i / k_in, j = i - p * k_in;
    return (static_cast<uint64_t>(f32_ord(__ldcg(vals + (size_t)p * part_stride + j))) << 32) | static_cast<uint64_t>(~(uint32_t)i);
  }
};
__global__ void __launch_bounds__(FIN_THREADS)
pooled_kth_kernel(const float* __restrict__ vals, int parts, long long Q, int k_in, int k, int P, int stage_cap,
                  float* __restrict__ out_kth) {
  extern __shared__ uint64_t fin_smem[];
  __shared__ uint32_t hist[256];
  __shared__ int s_misc[8];
  const long long q = blockIdx.x;
  PooledLoader ld{vals + (size_t)q * k_in, (size_t)Q * k_in, k_in};
  block_select_sort(ld, parts * k_in, k, fin_smem, P, hist, s_misc, fin_smem + P, stage_cap);
  if (threadIdx.x == 0) {
    const uint64_t key = fin_smem[k - 1];
    out_kth[q] = key == 0ull ? -FLT_MAX : ord_f32((uint32_t)(key >> 32));
  }
}

// thresholds supplied by the caller (a valid lower bound of each query's final k-th score), with the same 64-ulp slack
__global__ void topk_init_from_kernel(QMeta* meta, int Q, const float* __restrict__ tau_init) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < Q) {
    uint32_t key = f32_ord(tau_init[q]);
    key = key > 64u ? key - 64u : 0u;
    QMeta m;
    m.lock = 0u;
    m.tcount = 0u;
    m.tsel = 0u;
    m.tau = fmaxf(ord_f32(key), nextafterf(-FLT_MAX, 0.f));
    meta[q] = m;
  }
}

__global__ void topk_init_kernel(QMeta* meta, int Q, float tau0) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q < Q) {
    QMeta m;
    m.lock = 0u;
    m.tcount = 0u;
    m.tsel = 0u;
    m.tau = tau0;
    meta[q] = m;
  }
}

struct ListLoader {
  const float* scores;
  const int64_t* ids;
  size_t s_stride, i_stride;  // element distance between consecutive parts (Q * k_in when the arrays are dense)
  int k_in;
  __device__ __forceinline__ uint64_t operator()(int i) const {
    const int p = i / k_in, j = i - p * k_in;
    const int64_t id = ids[(size_t)p * i_stride + j];
    return id < 0 ? 0ull : make_key(scores[(size_t)p * s_stride + j], (uint32_t)id);
  }
};

__global__ void __launch_bounds__(FIN_THREADS)
topk_merge_kernel(const float* __restrict__ scores, const int64_t* __restrict__ ids, int parts, long long Q, int k_in,
                  int k_out, int P, int stage_cap, long long s_stride, long long i_stride,
                  float* __restrict__ out_scores, int64_t* __restrict__ out_ids) {
  extern __shared__ uint64_t fin_smem[];
  __shared__ uint32_t hist[256];
  __shared__ int s_misc[8];
  const long long q = blockIdx.x;
  ListLoader ld;
  ld.scores = scores + (size_t)q * k_in;
  ld.ids = ids + (size_t)q * k_in;
  ld.s_stride = (size_t)s_stride;
  ld.i_stride = (size_t)i_stride;
  ld.k_in = k_in;
  block_select_sort(ld, parts * k_in, k_out, fin_smem, P, hist, s_misc, fin_smem + P, stage_cap);
  write_result(fin_smem, k_out, 0, nullptr, out_scores + (size_t)q * k_out, out_ids + (size_t)q * k_out);
}

// Initial thresholds from a strided catalogue sample: tau0[q] = (a lower bound of) the k-th largest of the m sampled
// scores S[q, :].  The sampled rows are scanned again by the main pass, so tau0 only has to be a valid lower bound
// of the final k-th score: it removes the cold-start phase in which every score is a candidate.
__global__ void __launch_bounds__(FIN_THREADS)
sample_kth_kernel(const float* __restrict__ S, int m, int k, QMeta* __restrict__ meta) {
  __shared__ uint32_t hist[256];
  __shared__ int s_misc[4];
  const int q = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* row = S + (size_t)q * m;
  uint32_t prefix = 0;
  int need = k, shift = 24;
  for (int pass = 0; pass < 4; ++pass, shift -= 8) {
    hist[tid] = 0;
    __syncthreads();
    for (int i = tid; i < m; i += FIN_THREADS) {
      const uint32_t key = f32_ord(__ldcg(row + i));
      const bool match = (pass == 0) || ((key >> (shift + 8)) == prefix);
      if (match) atomicAdd(&hist[(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (warp == 0) {
      int bucket, nd = need;
      const int d = warp_pick_digit(hist, nd, bucket, lane);
      if (lane == 0) {
        s_misc[0] = d;
        s_misc[1] = nd;
        s_misc[2] = bucket;
      }
    }
    __syncthreads();
    prefix = (prefix << 8) | (uint32_t)s_misc[0];
    need = s_misc[1];
    const int bucket = s_misc[2];
    __syncthreads();
    if (bucket == need) break;
  }
  if (shift < 0) shift = 0;
  if (tid == 0) {
    uint32_t key = prefix << shift;         // smallest key carrying the selected prefix: <= the true k-th key
    key = key > 64u ? key - 64u : 0u;        // 64 ulps of slack against accumulation-order differences
    const float floor0 = nextafterf(-FLT_MAX, 0.f);
    QMeta mm;
    mm.lock = 0u;
    mm.tcount = 0u;
    mm.tsel = 0u;
    mm.tau = fmaxf(ord_f32(key), floor0);
    meta[q] = mm;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
static int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// optional CUDA-event bracket around the dominant kernel (bench.py's roofline line), on the launching stream
static int g_time_kernel = 0;
static cudaEvent_t g_ev0 = nullptr, g_ev1 = nullptr;

struct TopkPlan {
  int v2;      // 1: CTA-pair kernel (stream_scores2.cuh), 0: single-CTA kernel
  int nq, bn;
  StreamGeom g;
  int cap;
  size_t lists_bytes, tlists_bytes, meta_bytes, left_bytes, sample_bytes;
  int64_t sample_m, sample_stride;  // 0 = no sampling pass
  int sample_gw;
  int sample_k_out;                 // b200rec_topk_sample: group maxima returned per query (<= k)
  StreamGeom gs;                    // geometry of the sampling pass
  size_t total() const { return lists_bytes + tlists_bytes + meta_bytes + left_bytes + sample_bytes; }
};

// Development knobs come from the environment ONCE (first call) — not ~10 getenv() per search; tools that change them
// inside one process call b200rec_debug_reload_env().
struct TopkKnobs {
  int capmult = 2, v2 = -1, force_nq = 0, nosample = 0, sample_frac = 0, flush = -1, debug = 0, hsleep = 400,
      stream_stats = 0, stats_unit = -1;
};
static int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}
static TopkKnobs read_knobs() {
  TopkKnobs k;
  k.capmult = env_int("B200REC_TOPK_CAPMULT", 2);
  k.v2 = env_int("B200REC_TOPK_V2", -1);
  k.force_nq = env_int("B200REC_TOPK_NQ", 0);
  k.nosample = env_int("B200REC_TOPK_NOSAMPLE", 0);
  k.sample_frac = env_int("B200REC_TOPK_SAMPLE_FRAC", 0);
  k.flush = env_int("B200REC_TOPK_FLUSH", -1);
  k.debug = env_int("B200REC_TOPK_DEBUG", 0);
  k.hsleep = env_int("B200REC_TOPK_HSLEEP", 400);
  k.stream_stats = getenv("B200REC_STREAM_STATS") != nullptr ? 1 : 0;
  k.stats_unit = env_int("B200REC_STATS_UNIT", -1);
  return k;
}
static TopkKnobs& knobs() {
  static TopkKnobs k = read_knobs();
  return k;
}

static int cap_for(int k, int bn) { return ((knobs().capmult * k + bn + 31) / 32) * 32; }

// Encoded tensor maps are pure functions of (base, rows, ld, pitch, box): the catalogue's and — with a caching
// allocator behind the caller — the query operand's recur call after call, so a search re-encodes nothing.
struct TmapKey {
  const void* base;
  uint64_t rows, cols, ld;
  uint32_t box;
  bool operator==(const TmapKey& o) const { return base == o.base && rows == o.rows && cols == o.cols && ld == o.ld && box == o.box; }
};
static std::mutex g_cache_mu;
static int cached_tmap(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box) {
  constexpr int SLOTS = 32;
  static TmapKey keys[SLOTS];
  static CUtensorMap maps[SLOTS];
  static int used = 0, next = 0;
  const TmapKey key{base, rows, cols, ld, box};
  std::lock_guard<std::mutex> lock(g_cache_mu);
  for (int i = 0; i < used; ++i)
    if (keys[i] == key) {
      *out = maps[i];
      return 0;
    }
  if (make_tmap_bf16_2d(out, base, rows, cols, ld, box)) return 1;
  const int slot = used < SLOTS ? used++ : (next = (next + 1) % SLOTS);
  keys[slot] = key;
  maps[slot] = *out;
  return 0;
}

static int plan_topk_uncached(TopkPlan& p, int64_t N, int64_t ld, int64_t Q, int k, int shards) {
  const TopkKnobs& kn = knobs();
  if (N <= 0 || Q <= 0) return fail("topk: empty catalogue or query set");
  if (N >= (1ll << 32) - 1) return fail("topk: a shard holds at most 2^32-2 rows");
  if (Q > INT32_MAX / 2) return fail("topk: too many queries");
  if (k < 1 || k > 2048) return fail("topk: k must be in [1, 2048] (got %d)", k);
  if (ld <= 0 || (ld % 64)) return fail("topk: leading dimension must be a positive multiple of 64 (got %lld)", (long long)ld);
  const int KB = (int)(ld / 64);
  const int sms = num_sms();
  const int q128 = (int)((Q + 127) / 128);
  bool ok = false;
  p.v2 = 0;
  const bool want_v2 = kn.v2 != 0;
  const int v2shape = kn.v2 >= 0 ? kn.v2 : (q128 >= 3 ? 2 : 1);
  if (want_v2 && q128 >= 2 && (sms % 2) == 0) {
    // (the final kernel tabulates every unit's last supertile in FIN_MAX_SRC shared-memory slots)
    if (v2shape == 2 && stream_geom2<2>(p.g, N, (int)Q, KB, sms, TopkEpi::SCRATCH_BYTES) && p.g.max_parts + 1 <= FIN_MAX_SRC &&
        p.g.grid / 2 <= FIN_MAX_SRC) {
      p.v2 = 2, p.nq = 2, p.bn = 128, ok = true;  // nq/bn describe one CTA's share: 256 slots, 128 columns per thread
    } else if (stream_geom2<1>(p.g, N, (int)Q, KB, sms, TopkEpi::SCRATCH_BYTES) && 2 * p.g.max_parts + 1 <= FIN_MAX_SRC &&
               p.g.grid / 2 <= FIN_MAX_SRC) {
      p.v2 = 1, p.nq = 2, p.bn = 128, ok = true;
    }
  }
  const int fnq = kn.force_nq;
  if (ok) {
  } else if (fnq == 2 && stream_geom<2, 128>(p.g, N, (int)Q, KB, sms, TopkEpi::SCRATCH_BYTES)) {
    p.nq = 2, p.bn = 128, ok = true;
  } else if (fnq == 1 && stream_geom<1, 256>(p.g, N, (int)Q, KB, sms, TopkEpi::SCRATCH_BYTES)) {
    p.nq = 1, p.bn = 256, ok = true;
  } else if (q128 >= 2 && stream_geom<2, 128>(p.g, N, (int)Q, KB, sms, TopkEpi::SCRATCH_BYTES) && p.g.stages >= 3) {
    p.nq = 2, p.bn = 128, ok = true;
  } else if (stream_geom<1, 256>(p.g, N, (int)Q, KB, sms, TopkEpi::SCRATCH_BYTES) && p.g.stages >= 3) {
    p.nq = 1, p.bn = 256, ok = true;
  } else if (stream_geom<1, 64>(p.g, N, (int)Q, KB, sms, TopkEpi::SCRATCH_BYTES)) {
    p.nq = 1, p.bn = 64, ok = true;
  }
  if (!ok) return fail("topk: dimension too large for the resident query tile (ld=%lld)", (long long)ld);
  p.cap = cap_for(k, p.bn);
  p.lists_bytes = (size_t)p.g.grid * 128 * p.nq * 2 * (size_t)p.cap * sizeof(uint64_t);
  p.tlists_bytes = (size_t)Q * 2 * (size_t)k * sizeof(uint64_t);
  p.meta_bytes = (((size_t)Q * sizeof(QMeta)) + 255) / 256 * 256;
  p.left_bytes = (((size_t)p.g.grid * 128 * p.nq * sizeof(uint32_t)) + 255) / 256 * 256;
  if (!p.v2 && p.g.max_parts + 1 > FIN_MAX_SRC) return fail("topk: too many catalogue slices per query (%d)", p.g.max_parts);
  // sampling pass: group maxima over m = N/32 strided rows (fast path only; see SampleMaxEpi)
  p.sample_m = p.sample_stride = 0;
  p.sample_bytes = 0;
  p.sample_gw = 32;
  // `shards` row shards pool their samples (b200rec_topk_sample): the density is chosen for the pooled catalogue
  const int64_t n_pool = N * (shards > 1 ? shards : 1);
  int64_t frac = n_pool >= (4ll << 20) ? 32 : (n_pool >= (256ll << 10) ? 16 : 8);
  // A shard cannot see the other shards' running thresholds, so its own threshold only climbs to the LOCAL k-th score:
  // a tighter pooled start pays for a denser sample (8 x 1.25 M rows: 1/16 -> 1.58 ms per batch, 1/32 -> 1.69, 1/8 -> 1.64)
  if (shards > 1 && frac > 8) frac /= 2;
  if (kn.sample_frac > 0) frac = kn.sample_frac;
  int64_t m = (N / frac) / 256 * 256;
  if (!kn.nosample && m >= 2048) {
    int gw = 32;
    while (gw < 128 && gw < p.bn && m / gw > 8192) gw *= 2;
    if (m / gw >= 2 * (int64_t)k) {
      p.sample_m = m;
      p.sample_stride = N / m;
      p.sample_gw = gw;
      p.sample_bytes = (size_t)Q * (m / gw) * sizeof(float);
      bool sok;
      if (p.v2 == 2) sok = stream_geom2<2>(p.gs, m, (int)Q, KB, sms, SampleMaxEpi::SCRATCH_BYTES);
      else if (p.v2 == 1) sok = stream_geom2<1>(p.gs, m, (int)Q, KB, sms, SampleMaxEpi::SCRATCH_BYTES);
      else if (p.nq == 2) sok = stream_geom<2, 128>(p.gs, m, (int)Q, KB, sms, SampleMaxEpi::SCRATCH_BYTES);
      else if (p.bn == 256) sok = stream_geom<1, 256>(p.gs, m, (int)Q, KB, sms, SampleMaxEpi::SCRATCH_BYTES);
      else sok = stream_geom<1, 64>(p.gs, m, (int)Q, KB, sms, SampleMaxEpi::SCRATCH_BYTES);
      if (!sok) p.sample_m = 0, p.sample_bytes = 0;
    }
  }
  return 0;
}

// plans are pure functions of (N, ld, Q, k, shards) and the knobs: computed once per shape
struct PlanKey {
  int64_t N, ld, Q;
  int k, shards;
  bool operator==(const PlanKey& o) const { return N == o.N && ld == o.ld && Q == o.Q && k == o.k && shards == o.shards; }
};
static PlanKey g_plan_keys[64];
static TopkPlan g_plans[64];
static int g_plan_used = 0, g_plan_next = 0;

static int plan_topk(TopkPlan& p, int64_t N, int64_t ld, int64_t Q, int k, int shards = 1) {
  const PlanKey key{N, ld, Q, k, shards};
  {
    std::lock_guard<std::mutex> lock(g_cache_mu);
    for (int i = 0; i < g_plan_used; ++i)
      if (g_plan_keys[i] == key) {
        p = g_plans[i];
        return 0;
      }
  }
  if (plan_topk_uncached(p, N, ld, Q, k, shards)) return 1;   // argument errors are not cached
  std::lock_guard<std::mutex> lock(g_cache_mu);
  const int slot = g_plan_used < 64 ? g_plan_used++ : (g_plan_next = (g_plan_next + 1) % 64);
  g_plan_keys[slot] = key;
  g_plans[slot] = p;
  return 0;
}

// the plan a search of one of `shards` pooled row shards runs with
static int search_plan(TopkPlan& p, int64_t N, int64_t ld, int64_t Q, int k, int shards) {
  if (plan_topk(p, N, ld, Q, k, shards)) return 1;
  if (shards > 1 && p.sample_m == 0 && plan_topk(p, N, ld, Q, k)) return 1;  // pooled density too thin for this shard
  return 0;
}

// hand a list over every ~k/4 candidates: each merge selects over k + list keys, so the threshold scales with k
// (k = 1000: 7.6 ms per 1024-query batch at 32, 5.3 ms at 256).  Few queries and a large k (the serving loop's
// top-1000 for <= 256 users): every unit feeds the same few queries, the merges serialise on those queries' locks and
// a fresher threshold saves little, so lists are only handed over when full and the final select does the merging
// (50 M x 64, k = 1000: Q = 1 4.44 -> 1.55 ms, Q = 128 5.07 -> 3.37 ms; at Q >= 512 the k/4 rule wins: 6.6 vs 8.2 ms).
static int flush_for(const TopkPlan& p, int64_t Q, int k) {
  const TopkKnobs& kn = knobs();
  return kn.flush >= 0 ? kn.flush : ((k > 128 && Q <= 256) ? p.cap : (k / 4 > 32 ? (k / 4) / 32 * 32 : 32));
}

template <int NQ, int BN, int V2, bool DBG>
static int launch_topk(const TopkPlan& p, const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q,
                       int k, int64_t row_offset, const int64_t* excl_indptr, const int32_t* excl_rows,
                       const uint32_t* allow, int64_t allow_n, float* out_scores, int64_t* out_ids, void* workspace,
                       cudaStream_t st, const float* tau_init, float* sample_vals_out, const OutFan* fan_in,
                       const int64_t* remap) {
  OutFan fan;
  if (fan_in != nullptr) {
    fan = *fan_in;
  } else {
    fan.n = 1;
    fan.s[0] = sample_vals_out != nullptr ? sample_vals_out : out_scores;
    fan.i[0] = out_ids;
  }
  using Epi = TopkEpiT<DBG>;
  const TopkKnobs& kn = knobs();
  CUtensorMap tq, tx;
  if (cached_tmap(&tq, queries, (uint64_t)Q, (uint64_t)ld, (uint64_t)ld, 128)) return 1;
  constexpr int XBOX = V2 == 1 ? 128 : (V2 == 2 ? 64 : BN);  // rows per TMA box (a CTA of a pair loads its half)
  if (cached_tmap(&tx, catalogue, (uint64_t)N, (uint64_t)ld, (uint64_t)ld, XBOX)) return 1;
  TopkArgs ea;
  ea.lists = reinterpret_cast<uint64_t*>(workspace);
  ea.tlists = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(workspace) + p.lists_bytes);
  ea.meta = reinterpret_cast<QMeta*>(reinterpret_cast<uint8_t*>(workspace) + p.lists_bytes + p.tlists_bytes);
  ea.left = reinterpret_cast<uint32_t*>(reinterpret_cast<uint8_t*>(workspace) + p.lists_bytes + p.tlists_bytes + p.meta_bytes);
  B200_CUDA_OK(cudaMemsetAsync(ea.left, 0, p.left_bytes, st));
  ea.excl_indptr = excl_indptr;
  ea.excl_rows = excl_rows;
  ea.allow = allow;
  ea.allow_n = (uint32_t)allow_n;
  ea.k = k;
  ea.cap = p.cap;
  ea.flush = flush_for(p, Q, k);
  ea.debug = kn.debug;
  ea.hsleep = kn.hsleep;
  void (*kern)(const CUtensorMap, const CUtensorMap, const StreamGeom, const TopkArgs);
  if constexpr (V2 != 0) kern = stream_scores2_kernel<(V2 == 2 ? 2 : 1), Epi>;
  else kern = stream_scores_kernel<NQ, BN, Epi>;
  static int smem_set = 0;
  if (smem_set < p.g.smem_bytes) {
    B200_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, ST_SMEM_LIMIT));
    smem_set = ST_SMEM_LIMIT;
  }
  if (tau_init != nullptr) {
    topk_init_from_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, st>>>(ea.meta, (int)Q, tau_init);
    B200_LAUNCH_OK("topk_init_from_kernel");
  } else if (p.sample_m > 0 && excl_indptr == nullptr) {
    float* S = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + p.lists_bytes + p.tlists_bytes + p.meta_bytes + p.left_bytes);
    CUtensorMap ts;  // row i of this map is catalogue row i * stride
    if (cached_tmap(&ts, catalogue, (uint64_t)p.sample_m, (uint64_t)ld, (uint64_t)(ld * p.sample_stride), XBOX)) return 1;
    SampleArgs sa;
    sa.out = S;
    sa.ngroups = (int)(p.sample_m / p.sample_gw);
    sa.gw = p.sample_gw;
    sa.allow = allow;
    sa.allow_n = (uint32_t)allow_n;
    sa.stride = (uint32_t)p.sample_stride;
    void (*skern)(const CUtensorMap, const CUtensorMap, const StreamGeom, const SampleArgs);
    if constexpr (V2 != 0) {
      skern = allow ? stream_scores2_kernel<(V2 == 2 ? 2 : 1), SampleMaxEpiT<true>> : stream_scores2_kernel<(V2 == 2 ? 2 : 1), SampleMaxEpi>;
    } else {
      skern = allow ? stream_scores_kernel<NQ, BN, SampleMaxEpiT<true>> : stream_scores_kernel<NQ, BN, SampleMaxEpi>;
    }
    static bool sattr[2] = {false, false};
    if (!sattr[allow ? 1 : 0]) {
      B200_CUDA_OK(cudaFuncSetAttribute(skern, cudaFuncAttributeMaxDynamicSharedMemorySize, ST_SMEM_LIMIT));
      sattr[allow ? 1 : 0] = true;
    }
    skern<<<p.gs.grid, ST_THREADS, p.gs.smem_bytes, st>>>(tq, ts, p.gs, sa);
    B200_LAUNCH_OK("stream_scores_kernel<sample>");
    if (sample_vals_out != nullptr) {  // sampling only: hand the k best group maxima per query to the caller
      const int P = next_pow2(k);
      const int sc = sa.ngroups <= 4096 ? sa.ngroups : 0;
      sample_topk_kernel<<<(unsigned)Q, FIN_THREADS, (P + sc) * sizeof(uint64_t), st>>>(S, sa.ngroups, p.sample_k_out, P, sc, fan);
      B200_LAUNCH_OK("sample_topk_kernel");
      return 0;
    }
    sample_kth_kernel<<<(unsigned)Q, FIN_THREADS, 0, st>>>(S, sa.ngroups, k, ea.meta);
    B200_LAUNCH_OK("sample_kth_kernel");
  } else if (sample_vals_out != nullptr) {
    return fail("topk_sample: no sampling pass for this shape (catalogue too small or exclusion lists given)");
  } else {
    // every finite score must be able to enter: start just above -FLT_MAX (faiss' heap neutral, never returned)
    topk_init_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, st>>>(ea.meta, (int)Q, nextafterf(-FLT_MAX, 0.f));
    B200_LAUNCH_OK("topk_init_kernel");
  }
  if (g_time_kernel) {
    if (!g_ev0) {
      B200_CUDA_OK(cudaEventCreate(&g_ev0));
      B200_CUDA_OK(cudaEventCreate(&g_ev1));
    }
    B200_CUDA_OK(cudaEventRecord(g_ev0, st));
  }
  StreamGeom gl = p.g;
  gl.dbg_nofeed = (ea.debug == 4) ? 1 : 0;
  gl.dbg_stats = (ea.debug == 2 || kn.stream_stats) ? 1 : 0;
  if (kn.stats_unit >= 0) gl.dbg_stats = 2 + kn.stats_unit;
  if (ea.debug == 4) ea.debug = 3;
  kern<<<gl.grid, ST_THREADS, gl.smem_bytes, st>>>(tq, tx, gl, ea);
  B200_LAUNCH_OK("stream_scores_kernel<topk>");
  if (g_time_kernel) B200_CUDA_OK(cudaEventRecord(g_ev1, st));
  const int P = next_pow2(k);
  const int fin_stage = P <= 1024 ? 1024 : 0;  // T + leftovers of a query usually are a few hundred keys
  topk_final_kernel<<<(unsigned)Q, FIN_THREADS, (P + fin_stage) * sizeof(uint64_t), st>>>(
      p.g, V2, V2 == 2 ? 512 : (V2 == 1 ? 256 : 128 * NQ), V2 ? S2_SLOTS : 128 * NQ, ea.tlists, ea.meta, ea.lists, ea.left, p.cap,
      k, P, fin_stage, row_offset, remap, fan);
  B200_LAUNCH_OK("topk_final_kernel");
  return 0;
}

}  // namespace b200

extern "C" int b200rec_debug_reload_env(void) {
  using namespace b200;
  std::lock_guard<std::mutex> lock(g_cache_mu);
  knobs() = read_knobs();
  stream_knobs() = read_stream_knobs();
  g_plan_used = g_plan_next = 0;
  return 0;
}

// The plan a search of (N, ld, Q, k) on one of `shards` row shards runs with, without launching anything (no GPU
// needed): out[0..n_out) = sms, v2, nq, bn, stages, ks, grid, max_parts, S, T, W, R, n_main, Tmain, Tt, sample_m,
// sample_gw, cap, flush (R, n_main, Tmain and Tt are 0 for the single-CTA kernel, which has no such decomposition).
// Tests use it to prove which kernel instantiation and work decomposition a shape reaches.
extern "C" int b200rec_debug_topk_plan(int64_t N, int64_t ld, int64_t Q, int k, int shards, long long* out, int n_out) {
  using namespace b200;
  if (out == nullptr || n_out < 0) return fail("topk_plan: null output");
  TopkPlan p;
  if (search_plan(p, N, ld, Q, k, shards)) return 1;
  const bool v2 = p.v2 != 0;
  const long long v[] = {num_sms(), p.v2, p.nq, p.bn, p.g.stages, p.g.ks, p.g.grid, p.g.max_parts, p.g.S, p.g.T, p.g.W,
                         v2 ? p.g.R : 0, v2 ? p.g.n_main : 0, v2 ? p.g.Tmain : 0, v2 ? p.g.Tt : 0, p.sample_m,
                         p.sample_gw, p.cap, flush_for(p, Q, k)};
  for (int i = 0; i < n_out && i < (int)(sizeof(v) / sizeof(v[0])); ++i) out[i] = v[i];
  return 0;
}

extern "C" int b200rec_debug_topk_stats(unsigned long long* out8_host, int reset) {
  using namespace b200;
  B200_CUDA_OK(cudaMemcpyFromSymbol(out8_host, g_topk_stats, sizeof(unsigned long long) * 8));
  if (reset) {
    unsigned long long z[8] = {0};
    B200_CUDA_OK(cudaMemcpyToSymbol(g_topk_stats, z, sizeof(z)));
  }
  return 0;
}

extern "C" int b200rec_debug_topk_stats16(unsigned long long* out24_host, int reset) {
  using namespace b200;
  B200_CUDA_OK(cudaMemcpyFromSymbol(out24_host, g_topk_stats, sizeof(unsigned long long) * 16));
  B200_CUDA_OK(cudaMemcpyFromSymbol(out24_host + 16, g_stream_stats, sizeof(unsigned long long) * 8));
  if (reset) {
    unsigned long long z[16] = {0};
    B200_CUDA_OK(cudaMemcpyToSymbol(g_topk_stats, z, sizeof(z)));
    B200_CUDA_OK(cudaMemcpyToSymbol(g_stream_stats, z, sizeof(unsigned long long) * 8));
  }
  return 0;
}

extern "C" int b200rec_debug_topk_cta_end(unsigned long long* out512_host) {
  using namespace b200;
  B200_CUDA_OK(cudaMemcpyFromSymbol(out512_host, g_cta_end, sizeof(unsigned long long) * 512));
  return 0;
}

extern "C" int b200rec_debug_topk_kernel_timing(int enable, float* last_ms_host) {
  using namespace b200;
  if (last_ms_host) {
    *last_ms_host = 0.f;
    if (g_ev0 && g_ev1) {
      B200_CUDA_OK(cudaEventSynchronize(g_ev1));
      B200_CUDA_OK(cudaEventElapsedTime(last_ms_host, g_ev0, g_ev1));
    }
  }
  g_time_kernel = enable;
  return 0;
}

extern "C" size_t b200rec_topk_workspace_bytes(int64_t N, int64_t ld, int64_t Q, int k) {
  // one workspace serves the search and the pooled sampling pass of row shards, whose densest sample (two shards) is
  // twice as dense as the local one
  b200::TopkPlan p, p2;
  if (b200::plan_topk(p, N, ld, Q, k)) return 0;
  size_t need = p.total();
  if (b200::plan_topk(p2, N, ld, Q, k, 2) == 0 && p2.total() > need) need = p2.total();
  return need;
}

static int topk_dispatch(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q, int k,
                         int64_t row_offset, const int64_t* exclude_indptr, const int32_t* exclude_rows,
                         const uint32_t* allow, int64_t allow_n, const float* tau_init, float* out_scores,
                         int64_t* out_ids, float* sample_vals_out,
                         int sample_k_out, int shards, const b200::OutFan* fan, const int64_t* remap,
                         void* workspace, size_t workspace_bytes, void* stream) {
  using namespace b200;
  TopkPlan p;
  if (search_plan(p, N, ld, Q, k, shards)) return 1;
  p.sample_k_out = sample_k_out;
  if (workspace_bytes < p.total()) return fail("topk: workspace too small (%zu < %zu)", workspace_bytes, p.total());
  if ((exclude_indptr == nullptr) != (exclude_rows == nullptr)) return fail("topk: exclusion CSR needs both arrays");
  if (sample_vals_out != nullptr && p.sample_m == 0) return fail("topk_sample: catalogue too small for a sampling pass");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
#define B200_TOPK_ARGS p, catalogue, N, ld, queries, Q, k, row_offset, exclude_indptr, exclude_rows, allow, allow_n, out_scores, out_ids, workspace, st, tau_init, sample_vals_out, fan, remap
  if (knobs().debug != 0 || knobs().stream_stats || knobs().stats_unit >= 0) {  // development instantiation
    if (p.v2 == 2) return launch_topk<2, 128, 2, true>(B200_TOPK_ARGS);
    if (p.v2 == 1) return launch_topk<2, 128, 1, true>(B200_TOPK_ARGS);
    if (p.nq == 2) return launch_topk<2, 128, 0, true>(B200_TOPK_ARGS);
    if (p.bn == 256) return launch_topk<1, 256, 0, true>(B200_TOPK_ARGS);
    return launch_topk<1, 64, 0, true>(B200_TOPK_ARGS);
  }
  if (p.v2 == 2) return launch_topk<2, 128, 2, false>(B200_TOPK_ARGS);
  if (p.v2 == 1) return launch_topk<2, 128, 1, false>(B200_TOPK_ARGS);
  if (p.nq == 2) return launch_topk<2, 128, 0, false>(B200_TOPK_ARGS);
  if (p.bn == 256) return launch_topk<1, 256, 0, false>(B200_TOPK_ARGS);
  return launch_topk<1, 64, 0, false>(B200_TOPK_ARGS);
#undef B200_TOPK_ARGS
}

extern "C" int b200rec_flat_ip_topk(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q, int k,
                                    int64_t row_offset, const int64_t* exclude_indptr, const int32_t* exclude_rows,
                                    const float* tau_init, float* out_scores, int64_t* out_ids, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  if (!catalogue || !queries || !out_scores || !out_ids || !workspace) return b200::fail("topk: null pointer");
  return topk_dispatch(catalogue, N, ld, queries, Q, k, row_offset, exclude_indptr, exclude_rows, nullptr, 0, tau_init,
                       out_scores, out_ids, nullptr, k, 1, nullptr, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int b200rec_flat_ip_topk_filtered(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q,
                                             int k, int64_t row_offset, const uint32_t* allow_bits, int64_t allow_n,
                                             float* out_scores, int64_t* out_ids, void* workspace,
                                             size_t workspace_bytes, void* stream) {
  if (!catalogue || !queries || !allow_bits || !out_scores || !out_ids || !workspace)
    return b200::fail("topk_filtered: null pointer");
  if (allow_n < 0) return b200::fail("topk_filtered: allow_n must be >= 0");
  return topk_dispatch(catalogue, N, ld, queries, Q, k, row_offset, nullptr, nullptr, allow_bits, allow_n < N ? allow_n : N,
                       nullptr, out_scores, out_ids, nullptr, k, 1, nullptr, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int b200rec_topk_sample(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q, int k,
                                   int k_out, int shards, float* out_vals, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  if (!catalogue || !queries || !out_vals || !workspace) return b200::fail("topk_sample: null pointer");
  if (k_out < 1 || k_out > k) return b200::fail("topk_sample: k_out must be in [1, k]");
  return topk_dispatch(catalogue, N, ld, queries, Q, k, 0, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, out_vals, k_out,
                       shards < 1 ? 1 : shards, nullptr, nullptr, workspace, workspace_bytes, stream);
}

static int make_fan(b200::OutFan& fan, int n_dst, void* const* dst_scores, void* const* dst_ids, bool want_ids) {
  if (n_dst < 1 || n_dst > b200::FAN_MAX) return b200::fail("topk fan-out: n_dst must be in [1, %d]", b200::FAN_MAX);
  if (!dst_scores || (want_ids && !dst_ids)) return b200::fail("topk fan-out: null destination table");
  fan.n = n_dst;
  for (int d = 0; d < n_dst; ++d) {
    fan.s[d] = reinterpret_cast<float*>(dst_scores[d]);
    fan.i[d] = want_ids ? reinterpret_cast<int64_t*>(dst_ids[d]) : nullptr;
    if (!fan.s[d] || (want_ids && !fan.i[d])) return b200::fail("topk fan-out: null destination %d", d);
  }
  return 0;
}

extern "C" int b200rec_flat_ip_topk_fanout(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q,
                                           int k, int64_t row_offset, const float* tau_init, int n_dst,
                                           void* const* dst_scores, void* const* dst_ids, void* workspace,
                                           size_t workspace_bytes, void* stream) {
  if (!catalogue || !queries || !workspace) return b200::fail("topk: null pointer");
  b200::OutFan fan;
  if (make_fan(fan, n_dst, dst_scores, dst_ids, true)) return 1;
  return topk_dispatch(catalogue, N, ld, queries, Q, k, row_offset, nullptr, nullptr, nullptr, 0, tau_init, fan.s[0], fan.i[0], nullptr, k,
                       1, &fan, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int b200rec_topk_sample_fanout(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q,
                                          int k, int k_out, int shards, int n_dst, void* const* dst_vals, void* workspace,
                                          size_t workspace_bytes, void* stream) {
  if (!catalogue || !queries || !workspace) return b200::fail("topk_sample: null pointer");
  if (k_out < 1 || k_out > k) return b200::fail("topk_sample: k_out must be in [1, k]");
  b200::OutFan fan;
  if (make_fan(fan, n_dst, dst_vals, nullptr, false)) return 1;
  return topk_dispatch(catalogue, N, ld, queries, Q, k, 0, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, fan.s[0], k_out,
                       shards < 1 ? 1 : shards, &fan, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int b200rec_topk_has_sample(int64_t N, int64_t ld, int64_t Q, int k) {
  b200::TopkPlan p;
  if (b200::plan_topk(p, N, ld, Q, k)) return 0;
  return p.sample_m > 0 ? 1 : 0;
}

extern "C" int b200rec_topk_pooled_kth(const float* vals, int parts, int64_t Q, int k_in, int k, float* out_kth,
                                       void* stream) {
  using namespace b200;
  if (!vals || !out_kth) return fail("topk_pooled_kth: null pointer");
  if (parts < 1 || Q < 1 || k_in < 1 || k < 1 || k > 2048) return fail("topk_pooled_kth: bad sizes");
  if ((int64_t)parts * k_in < k) return fail("topk_pooled_kth: the pool holds fewer than k values");
  const int P = next_pow2(k);
  const int64_t n_in = (int64_t)parts * k_in;
  const int sc = (n_in + P) * 8 <= 40960 ? (int)n_in : 0;
  pooled_kth_kernel<<<(unsigned)Q, FIN_THREADS, (P + sc) * sizeof(uint64_t), reinterpret_cast<cudaStream_t>(stream)>>>(
      vals, parts, (long long)Q, k_in, k, P, sc, out_kth);
  B200_LAUNCH_OK("pooled_kth_kernel");
  return 0;
}

extern "C" int b200rec_topk_merge(const float* scores, const int64_t* ids, int parts, int64_t Q, int k_in, int k_out,
                                  int64_t scores_part_stride, int64_t ids_part_stride, float* out_scores,
                                  int64_t* out_ids, void* stream) {
  using namespace b200;
  if (!scores || !ids || !out_scores || !out_ids) return fail("topk_merge: null pointer");
  if (parts < 1 || Q < 1 || k_in < 1) return fail("topk_merge: empty input");
  if (k_out < 1 || k_out > 2048) return fail("topk_merge: k_out must be in [1, 2048]");
  if ((int64_t)parts * k_in > INT32_MAX) return fail("topk_merge: too many candidates per query");
  const int P = next_pow2(k_out);
  const int64_t n_in = (int64_t)parts * k_in;
  const int sc = (n_in + P) * 8 <= 40960 ? (int)n_in : 0;
  topk_merge_kernel<<<(unsigned)Q, FIN_THREADS, (P + sc) * sizeof(uint64_t), reinterpret_cast<cudaStream_t>(stream)>>>(
      scores, ids, parts, (long long)Q, k_in, k_out, P, sc,
      (long long)(scores_part_stride > 0 ? scores_part_stride : Q * k_in),
      (long long)(ids_part_stride > 0 ? ids_part_stride : Q * k_in), out_scores, out_ids);
  B200_LAUNCH_OK("topk_merge_kernel");
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// filtered row-shard steps: every shard takes part in every exchange, so a shard that has nothing to sample or search
// (no allowed rows, or a shape without a sampling pass) stores padding rows instead of failing
// ---------------------------------------------------------------------------------------------------------------
static int fan_fill(const b200::OutFan& fan, int64_t n, float s, int64_t id, void* stream) {
  using namespace b200;
  const int64_t blocks = (n + 255) / 256;
  const int grid = (int)(blocks < 4 * (int64_t)num_sms() ? (blocks > 0 ? blocks : 1) : 4 * (int64_t)num_sms());
  fan_fill_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(fan, n, s, id);
  B200_LAUNCH_OK("fan_fill_kernel");
  return 0;
}

static int sample_filtered(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q, int k, int k_out,
                           int shards, const uint32_t* allow_bits, int64_t allow_n, const b200::OutFan& fan,
                           void* workspace, size_t workspace_bytes, void* stream) {
  using namespace b200;
  if (Q < 1) return fail("topk_sample_filtered: Q must be >= 1");
  if (k < 1 || k > 2048) return fail("topk_sample_filtered: k must be in [1, 2048] (got %d)", k);
  if (k_out < 1 || k_out > k) return fail("topk_sample_filtered: k_out must be in [1, k]");
  if (N < 0 || allow_n < 0) return fail("topk_sample_filtered: N and allow_n must be >= 0");
  shards = shards < 1 ? 1 : shards;
  const int64_t an = allow_bits != nullptr ? (allow_n < N ? allow_n : N) : N;
  bool pad = N == 0 || an == 0;
  if (!pad) {
    TopkPlan p;
    if (plan_topk(p, N, ld, Q, k, shards)) return 1;
    if (p.sample_m == 0 && plan_topk(p, N, ld, Q, k)) return 1;
    pad = p.sample_m == 0;
  }
  if (pad) return fan_fill(fan, Q * k_out, -FLT_MAX, 0, stream);
  if (!catalogue || !workspace) return fail("topk_sample_filtered: null catalogue or workspace");
  return topk_dispatch(catalogue, N, ld, queries, Q, k, 0, nullptr, nullptr, allow_bits, an, nullptr, nullptr, nullptr,
                       fan.s[0], k_out, shards, &fan, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int b200rec_topk_sample_filtered(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q,
                                            int k, int k_out, int shards, const uint32_t* allow_bits, int64_t allow_n,
                                            float* out_vals, void* workspace, size_t workspace_bytes, void* stream) {
  if (!queries || !out_vals) return b200::fail("topk_sample_filtered: null pointer");
  b200::OutFan fan;
  fan.n = 1;
  fan.s[0] = out_vals;
  fan.i[0] = nullptr;
  return sample_filtered(catalogue, N, ld, queries, Q, k, k_out, shards, allow_bits, allow_n, fan, workspace,
                         workspace_bytes, stream);
}

extern "C" int b200rec_topk_sample_filtered_fanout(const void* catalogue, int64_t N, int64_t ld, const void* queries,
                                                   int64_t Q, int k, int k_out, int shards, const uint32_t* allow_bits,
                                                   int64_t allow_n, int n_dst, void* const* dst_vals, void* workspace,
                                                   size_t workspace_bytes, void* stream) {
  if (!queries) return b200::fail("topk_sample_filtered: null pointer");
  b200::OutFan fan;
  if (make_fan(fan, n_dst, dst_vals, nullptr, false)) return 1;
  return sample_filtered(catalogue, N, ld, queries, Q, k, k_out, shards, allow_bits, allow_n, fan, workspace,
                         workspace_bytes, stream);
}

extern "C" int b200rec_flat_ip_topk_filtered_fanout(const void* catalogue, int64_t N, int64_t ld, const void* queries,
                                                    int64_t Q, int k, int64_t row_offset, const uint32_t* allow_bits,
                                                    int64_t allow_n, const int64_t* remap_rows, int64_t n_remap,
                                                    const float* tau_init, int n_dst, void* const* dst_scores,
                                                    void* const* dst_ids, void* workspace, size_t workspace_bytes,
                                                    void* stream) {
  using namespace b200;
  if (!queries) return fail("topk_filtered_fanout: null pointer");
  if ((allow_bits == nullptr) == (remap_rows == nullptr))
    return fail("topk_filtered_fanout: exactly one of allow_bits and remap_rows must be given");
  OutFan fan;
  if (make_fan(fan, n_dst, dst_scores, dst_ids, true)) return 1;
  if (Q < 1) return fail("topk_filtered_fanout: Q must be >= 1");
  if (k < 1 || k > 2048) return fail("topk_filtered_fanout: k must be in [1, 2048] (got %d)", k);
  if (N < 0 || allow_n < 0) return fail("topk_filtered_fanout: N and allow_n must be >= 0");
  if (remap_rows != nullptr && n_remap != N) return fail("topk_filtered_fanout: n_remap must equal N (one row per compacted row)");
  const int64_t an = allow_bits != nullptr ? (allow_n < N ? allow_n : N) : N;
  if (N == 0 || an == 0) return fan_fill(fan, Q * k, -FLT_MAX, -1, stream);
  if (!catalogue || !workspace) return fail("topk_filtered_fanout: null catalogue or workspace");
  return topk_dispatch(catalogue, N, ld, queries, Q, k, row_offset, nullptr, nullptr, allow_bits, an, tau_init, fan.s[0],
                       fan.i[0], nullptr, k, 1, &fan, remap_rows, workspace, workspace_bytes, stream);
}
