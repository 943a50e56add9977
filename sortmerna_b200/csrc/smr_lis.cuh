// Candidate voting, LIS, region selection, Smith-Waterman and the accept / replace / stop state
// machine: one warp per read, executing the reference's SEQUENTIAL decision order for that read.
//
// Stands in for the pass loop of traverse() (src/sortmerna/paralleltraversal.cpp:114-297),
// compute_lis_alignment() + find_lis() (src/sortmerna/alignment.cpp:58-509) and the per-read body of
// align2() (src/sortmerna/processor.cpp:104-162) for one (index, part).
//
// The seed kernel has already produced, per read, the id hits of every window of every pass; this
// kernel replays pass 1 / 2 / 3 on them.  Differences in mechanism (not in results):
//   * votes per reference are counted in a warp-private histogram in HBM (epoch-tagged, so it is never
//     cleared) instead of a std::map (alignment.cpp:118-130); the candidate list is sorted by
//     (count desc, ref asc) with a warp bitonic sort (:143-148);
//   * a candidate's (refpos, readpos) pairs are gathered by binary search in the per-id position
//     lists, which the flattener keeps sorted by (seq,pos), instead of rescanning every list (:181-194);
//   * the deque `match_set` is a [front, next) index range over the sorted pairs (:205-238, 486-506);
//   * ssw_align's reverse pass and CIGAR are deferred to the finalize kernel: accept / replace / stop
//     decisions only need score1 (:388-469).
//
// Warp specialisation.  One persistent CTA of 32 warps per SM; its warps have three roles (16 scorers, 1 fetcher, 15 planners):
//   * PLANNER warps own reads.  For each compute_lis_alignment call they vote, order and group as above, then walk the
//     candidates in the reference's order WITHOUT scoring: every (candidate, sliding-window step) that would reach
//     ssw_align becomes a task record (window, query segment).  Which steps reach it is score-independent -- the
//     (it, f) trajectory of the deque only depends on the pairs (:231-238, 486-506) -- except for heuristic 1 (:243-246),
//     the `best` countdown (:165-169) and the stop rules (:462-469), which the REPLAY applies afterwards to the table of
//     scores, in order, exactly as the reference would have.  Batches are sized so that little is scored in vain: a batch
//     never reaches the level drop at which the countdown could stop the call, tasks behind a successful alignment of
//     the same candidate (skipped by heuristic 1) are only submitted when their lead task failed, and batches grow
//     geometrically so that a perfect-score stop wastes at most what was useful.
//   * SCORER warps drain a global multi-producer/multi-consumer queue of task PAIRS and score two tasks per pass with
//     the packed 16-bit DPX kernel (smr_sw.cuh), whoever the read belongs to: a read with thousands of candidates is
//     scored by the whole GPU instead of by its one warp (round 1: the heaviest read occupied one warp for 310 of the
//     376 ms), and the integer-pipe loop never waits on the memory-latency phases of voting and grouping.
//   * The FETCHER warp (one lane per scorer input slot) pops the queue and stages the scorers' inputs -- reference window and query
//     segment -- with TMA bulk copies (cp.async.bulk + mbarrier), two slots per scorer: one fills while the other is scored.
// Hand-over without fences: __threadfence() is MEMBAR.SC.GPU + CCTL.IVALL on sm_100a -- it also invalidates the SM's whole L1.  A
// planner publishes a queue entry with a release store (MEMBAR.ALL.GPU + ST) after marking the score words of its tasks pending;
// the fetcher reads entry and task records past L1; a scorer stores its scores and adds to the planner's counter with no fence in
// between; the planner takes the counter as a hint and then looks at every score word itself.
#pragma once
#include "smr_seed.cuh"
#include "smr_sw.cuh"

namespace smr {

// One CTA of 32 warps per SM: 16 scorers + 1 fetcher (one lane per scorer slot) + 15 planners.  (Two CTAs of 8 + 1 + 7 need two
// fetcher warps per SM: one planner fewer -- 213.1 vs 207.1 ms per 500 k reads; 14 + 1 + 17: 209.6.)
#ifndef SMR_SCORER_WARPS
#define SMR_SCORER_WARPS 16
#endif
#ifndef SMR_PLANNER_WARPS
#define SMR_PLANNER_WARPS 15
#endif
#ifndef SMR_LIS_MIN_CTAS
#define SMR_LIS_MIN_CTAS 1
#endif
// Phase accounting with clock64 (the cycle shares bench.py reports) is a template parameter of the kernel: the product runs the
// instantiation without it (smr_set_instrumentation; 199.6 vs 204.9 ms per 500 k reads with it).
template <bool kInstr> __device__ __forceinline__ long long lis_clock() { return kInstr ? clock64() : 0ll; }
// Timeline of the instrumented instantiation (SMR_TIMELINE=1 prints it): nanoseconds per role and state in 1 ms buckets since the
// start of the kernel -- g.dbg + kTlBase + row * kTlBuckets; rows: 0 scorers waiting for a staged pair, 1 scorers busy, 2 planners
// waiting for scores, 3 planners voting / ordering / grouping, 4 reads finished (count), 5 planner warps alive (ns).
constexpr int kTlBuckets = 512, kTlRows = 6, kTlBase = 16;
constexpr unsigned long long kTlBucketNs = 1000000ull;
__device__ __forceinline__ unsigned long long tl_now() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
__device__ __noinline__ void tl_add(unsigned long long* row, const unsigned long long t_start, unsigned long long a, const unsigned long long b) {
  if (lane_id() != 0 || b <= a) return;
#pragma unroll 1
  while (a < b) {
    const unsigned long long k = (a - t_start) / kTlBucketNs, edge = t_start + (k + 1) * kTlBucketNs, e = b < edge ? b : edge;
    if (k < (unsigned long long)kTlBuckets) atomicAdd(row + k, e - a);
    a = e;
  }
}
constexpr int kScorerWarps = SMR_SCORER_WARPS;     // the first warps of a CTA score
constexpr int kFetcherWarps = 1;                   // then one warp that pops the task queue and stages the scorers' inputs (TMA bulk copies)
constexpr int kPlannerWarps = SMR_PLANNER_WARPS;   // the others plan
constexpr int kLisMinCtas = SMR_LIS_MIN_CTAS;      // CTAs per SM the register budget is set for
constexpr int kLisWarpsPerCta = kScorerWarps + kFetcherWarps + kPlannerWarps;
static_assert(2 * kScorerWarps <= 32, "one fetcher lane per (scorer, slot)");

// A scorer's input slot (two per scorer: one is filled while the other is scored).  The fetcher lane writes the header, arms
// the mbarrier with the byte count and issues the bulk copies; the scorer waits on the mbarrier's phase.
constexpr int kWinOff = 48;                         // bulk destination inside win[]: 32 sentinel columns + 15 bytes of alignment slack fit in front
constexpr int kWinBuf = kWinOff + kRefStage + 64;   // 560: 16-byte aligned copy of <= 448 + 30 bytes, then sentinels up to column nmax + 32
constexpr int kQBuf = 288;                          // 16-byte aligned copy of <= 256 + 30 query bytes
struct __align__(16) ScSlot {
  uint8_t win[2][kWinBuf];
  uint8_t q[2][kQBuf];
  uint32_t planner, ta, tb, slow;     // slow: outside the packed kernel's range -> nothing staged, s32 fallback from global memory
  uint32_t mA, nA, woffA, qoffA;      // rows, columns, index of column 0 in win[0], index of query element 0 in q[0]
  uint32_t mB, nB, woffB, qoffB;
  uint32_t metaA, metaB, qabsA, qabsB;
  uint32_t refA, refB, pad0, pad1;
  unsigned long long bar;             // "full" mbarrier: 1 arrival (the fetcher lane) + the bulk copies' bytes
  unsigned long long ebar;            // "empty" mbarrier: 1 arrival (the scorer, when it has finished with the slot)
};
constexpr int kScorerSmem = 2 * kPairProfWords * 4 + 2 * (int)sizeof(ScSlot);   // two query profiles + two input slots
constexpr int kPlannerSmem = 128 * 16;                                          // kPairsShared pairs + LIS arrays
constexpr int kLisSmemBytes = kScorerWarps * kScorerSmem + kPlannerWarps * kPlannerSmem;
constexpr int kPairsShared = 128;  // pairs / LIS arrays kept in shared memory up to this many
constexpr uint32_t kQueueCap = 1u << 20;         // task-pair ring (slots), per queue
constexpr uint32_t kSmallRound = 32;              // rounds of up to this many pairs go to the express queue
constexpr uint32_t kNoTask = 0xFFFFFFu;
constexpr uint32_t kPoison = 0xFFFFu;             // planner id of the shutdown entries
constexpr uint32_t kBatchCandCap = 4096;          // candidates per batch
#ifndef SMR_PLANNER_POLL_NS
#define SMR_PLANNER_POLL_NS 1024                    // sleep between two looks of a planner at its score counter (256: 215.1 ms, 512: 214.2, 1024: 213.4)
#endif
constexpr uint32_t kScorePending = 0xFFFFFFFFu;     // score word of a task that has been handed to the scorers and not been scored yet
// Sensitivity experiments (tools/ab_round.sh; never set in the shipped build): stretch a role's own work by N per cent with sleeps
// (no issue slots taken) -- how much the kernel slows tells which role bounds it.
// Schedule of the reads over the planner warps.  The seed kernel bins the reads of a chunk by log2 of their voting work; index 0 of the
// schedule is the heaviest read.  With ONE heaviest-first cursor (round 2a) every planner starts on a read whose votes take
// milliseconds: the scorers wait for 20 ms of 205 (the kernel's role timeline, SMR_TIMELINE / tools/timeline_summary.py).  So two
// cursors: SMR_SCHED_A planners in 8 take the heaviest nwork >> SMR_SPLIT_SHIFT reads in order, the others start right behind them,
// on reads whose few candidates reach the scorers within microseconds -- the scorers are busy 12 ms after the launch -- and go on
// towards the light end; a planner whose region is exhausted helps in the other.  SMR_SCHED_A = 0: the single cursor.
// Measured (ms per 500 k reads, candidate kernel): single cursor 201.8; 4 in 8 planners on the heaviest 1/64: 198.1, 1/16: 195.3,
// 1/8: 191.5 - 194.8; 2 in 8 on 1/32: 195.5; variants that also start planners at the light end (the reads without Smith-Waterman
// work, which otherwise end the kernel with idle scorers) lost what they gained there at the start: 197 - 206.
#ifndef SMR_SCHED_A
#define SMR_SCHED_A 4
#endif
#ifndef SMR_SPLIT_SHIFT
#define SMR_SPLIT_SHIFT 3
#endif
#ifndef SMR_EXP_PLANNER_DELAY
#define SMR_EXP_PLANNER_DELAY 0
#endif
#ifndef SMR_EXP_SCORER_DELAY
#define SMR_EXP_SCORER_DELAY 0
#endif
__device__ __forceinline__ void exp_delay(const long long t0, const int pct) {
  const long long now = clock64(), until = now + (now - t0) * pct / 100;
  while (clock64() < until) __nanosleep(256);
}
#ifndef SMR_BATCH_CAP0
#define SMR_BATCH_CAP0 32                         // candidates in the first batch of a call (8: 219.5 ms, 32: 216.8, 128: 216.8 per 500 k reads)
#endif

// one Smith-Waterman call the reference would make (alignment.cpp:365-381), as the scorers see it
struct SwTask {
  uint32_t ref_abs;     // first window column in parts[part].refseq
  uint32_t q_abs;       // query element 0 in seq04 (reverse strand: last base of the segment, walked backwards, complemented)
  uint32_t alen, qlen;  // window columns, query rows
  uint32_t meta;        // part slot | reversed << 16
  uint32_t score;       // OUT (scorer): ssw score
  uint32_t pad0, pad1;
};
// ... and as the replay sees it
struct PlanTask {
  uint32_t max_ref, win_start, aqs;
  uint32_t cf;          // candidate (relative to the batch) | flags << 24
  uint32_t lead;        // index of the unconditional task that decides whether this (conditional) one is needed
};
constexpr uint32_t kTfPush = 1u;     // the step pushed new pairs into the window (alignment.cpp:231-238)
constexpr uint32_t kTfUncond = 2u;   // not skippable by heuristic 1 whatever the earlier scores are
constexpr uint32_t kTfReset = 4u;    // a step without a task but with a push lies between the previous task and this one

struct QSlot { uint32_t seq, planner, ta, tb; };   // one queue entry = up to two tasks of one planner (tb == kNoTask: one)

struct LisArena {            // per-warp scratch in HBM
  uint32_t* hist;            // [hist_cap] epoch<<20 | count, indexed by reference number
  unsigned long long* cand;  // [cand_cap] candidate keys in ascending reference order
  unsigned long long* grp;   // [cand_cap] the group of candidates being processed (one count level, or all when <= 32)
  unsigned long long* pall;  // [pall_cap] (refpos<<32 | readpos) of ALL candidates of a call, grouped per reference
  uint32_t pall_cap;
  uint32_t* bitmap;          // [ceil(hist_cap/32)] references that reached num_seeds votes
  uint32_t* summary;         // [ceil(hist_cap/1024)] non-zero words of bitmap
  unsigned long long* pairs; // [pair_cap] (power of two) refpos<<32 | readpos
  uint32_t* lis_b; uint32_t* lis_p;  // [pair_cap]
  SwTask* tasks; PlanTask* ptasks;   // [task_cap]
  uint32_t* sel;                     // [task_cap] task indices of the round being submitted
  uint32_t* cfirst;                  // [3][kBatchCandCap] per candidate of the batch: first task; count | big << 30 | ends-on-reset << 31; uncond mask
  uint32_t hist_cap, cand_cap, pair_cap, task_cap;
};

struct LisGlobals {
  uint8_t* arena_base; size_t arena_stride;   // per-planner arena
  uint32_t hist_cap, cand_cap, pair_cap, row_cap, pall_cap, task_cap;
  uint32_t* epochs;                            // [planners]
  QSlot* ring;                                 // [2][kQueueCap]: queue 0 = small rounds (latency matters), queue 1 = bulk
  uint32_t* q_head; uint32_t* q_tail;          // consumer / producer cursors; queue q uses [q * 16] (64 bytes apart)
  uint32_t* planners_done;                     // planners that ran out of reads
  uint32_t* done;                              // [planners] tasks scored so far for each planner
  int32_t* score_rows;                         // [scorers][2 * row_cap] scratch of the s32 row-block fallback
  unsigned long long* dbg;                     // [16] phase cycles of the read that took longest (SMR_VERBOSE); [kTlBase ..) the timeline rows
  AlnWork* aln_work;                           // [nreads * slots]
  uint32_t slots;
  uint32_t* work_next;                         // [1] persistent-loop cursor (SMR_SCHED_A: over the heaviest reads)
  uint32_t* work_next_b;                       // [1] second cursor (SMR_SCHED_A: over the rest of the schedule)
  const DevIndex* parts; uint32_t nparts;      // every loaded (index,part) in --ref order
};

__device__ __forceinline__ LisArena carve_arena(const LisGlobals& g, uint32_t warp) {
  LisArena a;
  uint8_t* p = g.arena_base + (size_t)warp * g.arena_stride;
  a.hist_cap = g.hist_cap; a.cand_cap = g.cand_cap; a.pair_cap = g.pair_cap; a.task_cap = g.task_cap;
  // the part that must start zeroed comes first (lis_arena_zero_bytes): epoch-tagged votes, candidate bitmap and its summary
  a.hist = (uint32_t*)p; p += (size_t)g.hist_cap * 4;
  a.bitmap = (uint32_t*)p; p += (size_t)((g.hist_cap + 31) / 32) * 4;
  a.summary = (uint32_t*)p; p += (size_t)((g.hist_cap + 1023) / 1024) * 4;
  p = (uint8_t*)(((uintptr_t)p + 15) & ~(uintptr_t)15);
  a.cand = (unsigned long long*)p; p += (size_t)g.cand_cap * 8;
  a.grp = (unsigned long long*)p; p += (size_t)g.cand_cap * 8;
  a.pairs = (unsigned long long*)p; p += (size_t)g.pair_cap * 8;
  a.lis_b = (uint32_t*)p; p += (size_t)g.pair_cap * 4;
  a.lis_p = (uint32_t*)p; p += (size_t)g.pair_cap * 4;
  a.sel = (uint32_t*)p; p += (size_t)g.task_cap * 4;
  a.cfirst = (uint32_t*)p; p += (size_t)kBatchCandCap * 3 * 4;
  p = (uint8_t*)(((uintptr_t)p + 31) & ~(uintptr_t)31);
  a.pall = (unsigned long long*)p; a.pall_cap = g.pall_cap; p += (size_t)g.pall_cap * 8;
  a.tasks = (SwTask*)p; p += (size_t)g.task_cap * sizeof(SwTask);
  a.ptasks = (PlanTask*)p;
  return a;
}
__host__ __device__ inline size_t lis_arena_zero_bytes(uint32_t hist_cap) { return (size_t)hist_cap * 4 + (size_t)((hist_cap + 31) / 32) * 4 + (size_t)((hist_cap + 1023) / 1024) * 4; }
__host__ __device__ inline size_t lis_arena_bytes(uint32_t hist_cap, uint32_t cand_cap, uint32_t pair_cap, uint32_t task_cap, uint32_t pall_cap) {
  size_t b = (size_t)cand_cap * 16 + (size_t)pair_cap * 8 + (size_t)hist_cap * 4 + (size_t)pair_cap * 8 + (size_t)task_cap * 4 +
             (size_t)kBatchCandCap * 3 * 4 + (size_t)((hist_cap + 31) / 32) * 4 + (size_t)((hist_cap + 1023) / 1024) * 4 + 64 +
             (size_t)pall_cap * 8 + (size_t)task_cap * (sizeof(SwTask) + sizeof(PlanTask));
  return (b + 255) & ~(size_t)255;
}

// ---- warp bitonic sort of 64-bit keys, ascending; n_pow2 = power of two >= n, tail padded by the caller ----
__device__ __noinline__ void warp_sort_u64(unsigned long long* a, uint32_t n_pow2) {
  const unsigned lane = lane_id();
  for (uint32_t k = 2; k <= n_pow2; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t i = lane; i < n_pow2; i += 32) {
        const uint32_t l = i ^ j;
        if (l > i) {
          const unsigned long long x = a[i], y = a[l];
          const bool up = (i & k) == 0;
          if ((x > y) == up) { a[i] = y; a[l] = x; }
        }
      }
      __syncwarp();
    }
  }
}
// ascending sort of one 64-bit key per lane (pad with ~0ull), entirely in registers
// `n` (warp-uniform) = number of real keys: only the first next_pow2(n) lanes need to end up sorted, which takes the
// merge stages up to that block size only (3 of the 15 stages for n <= 4)
__device__ __noinline__ unsigned long long warp_sort32_u64(unsigned long long key, const unsigned n = 32) {
  const unsigned lane = lane_id();
#pragma unroll
  for (unsigned k = 2; k <= 32; k <<= 1) {
    if ((k >> 1) >= n) break;
#pragma unroll
    for (unsigned j = k >> 1; j > 0; j >>= 1) {
      const unsigned long long other = __shfl_xor_sync(kFull, key, j);
      const bool up = (lane & k) == 0, lower = (lane & j) == 0;
      const unsigned long long mn = key < other ? key : other, mx = key < other ? other : key;
      key = (lower == up) ? mn : mx;
    }
  }
  return key;
}
__device__ __forceinline__ uint32_t next_pow2(uint32_t v) { uint32_t p = 1; while (p < v) p <<= 1; return p; }

struct ReadCtx {           // per-read working state (uniform across the warp)
  uint32_t r, len, seq_base;
  bool reversed, hasn;
  uint32_t vcls[3];        // variant in effect when pass class c was searched on the current strand
  uint32_t pass_n;         // passes with class <= pass_n are in id_win_hits
  // Read fields
  uint32_t hit_seeds, min_index, max_index, n_align;
  int32_t best;
  uint32_t max_SW_count;
  bool is_done, is_hit, is_new_hit;
  bool form04;             // read currently in the 0-4 alphabet (read.is04); only meaningful when hasn
  bool ovf_slots;          // an accepted alignment did not fit the per-read stride (all-alignments mode)
  uint32_t flags;
};

__device__ __forceinline__ bool hit_selected(const uint2 h, const ReadCtx& rc, uint32_t s0, uint32_t s1, uint32_t s2) {
  const uint32_t var = (h.y >> 24) & 15u, c = h.y >> 28;   // class computed once, by the seed kernel (paralleltraversal.cpp:118-131)
  if (c > rc.pass_n) return false;
  return var == rc.vcls[c];
}

// find_lis (alignment.cpp:58-98) over pairs[f .. f+n): returns |LIS| and the index (relative to f) of its first element
template <class IdxT>
__device__ uint32_t find_lis_dev(const unsigned long long* __restrict__ P, uint32_t n, IdxT* b, IdxT* p, uint32_t& first) {
  if (n == 0) { first = 0; return 0; }
  uint32_t nb = 1; b[0] = 0;
#pragma unroll 1
  for (uint32_t i = 1; i < n; ++i) {
    const uint32_t ai = (uint32_t)P[i];
    if ((uint32_t)P[b[nb - 1]] < ai) { p[i] = b[nb - 1]; b[nb++] = (IdxT)i; continue; }
    uint32_t u = 0, v = nb - 1;
#pragma unroll 1
    while (u < v) { const uint32_t c = (u + v) >> 1; if ((uint32_t)P[b[c]] < ai) u = c + 1; else v = c; }
    if (ai < (uint32_t)P[b[u]]) { if (u > 0) p[i] = b[u - 1]; b[u] = (IdxT)i; }
  }
  uint32_t v = b[nb - 1];
#pragma unroll 1
  for (uint32_t u = nb; u-- > 1;) v = p[v];
  first = v;
  return nb;
}

struct PassEnv {
  const DevIndex* ix; const DevBatch* b; const DevParams* prm; const LisGlobals* g;
  LisArena ar; uint32_t* epoch_ptr; uint32_t epoch;
  unsigned long long* s_pairs; uint32_t* s_b; uint32_t* s_p;   // shared-memory fast buffers (kPairsShared)
  const uint2* hits; uint32_t nh;                               // hit region of (current part, current read)
  uint32_t planner;                                             // ordinal of this planner warp
  unsigned long long tl0;                                       // %globaltimer at the start of the kernel (instrumented instantiation)
  uint32_t submitted;                                           // tasks handed to the scorers so far (g.done[planner] catches up)
  unsigned long long n_sw_calls, n_sw_cells, n_pos_entries, n_lis_calls, n_spec_calls, n_spec_cells /* rounds A */, n_rounds_b, w1_cyc, w1_cnt;
  unsigned long long cyc[8];                                    // warp cycles per phase: vote, order, group, plan, wait, replay
};

// ---- the task queue (bounded MPMC ring, per-slot sequence numbers) ----
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) { return *(const volatile uint32_t*)p; }
__device__ __forceinline__ void st_volatile_u32(uint32_t* p, uint32_t v) { *(volatile uint32_t*)p = v; }
__device__ __forceinline__ void st_release_gpu_u32(uint32_t* p, uint32_t v) { asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }

// hands the tasks sel[0 .. nsel) of this planner to the scorers, two per queue entry, and waits for their scores
template <bool kInstr>
__device__ __noinline__ void submit_and_wait(PassEnv& E, const uint32_t nsel) {
  if (nsel == 0) return;
  const LisGlobals& g = *E.g;
  const unsigned lane = lane_id();
  const uint32_t npairs = (nsel + 1) >> 1;
  // two queues: a planner with a handful of tasks must not wait behind the thousands of pairs of a read from a conserved region
  // (each scorer keeps one input slot for either queue, so the express queue is served within about one alignment time)
  const uint32_t qi = npairs <= kSmallRound ? 0u : 1u;
  QSlot* ring = g.ring + (size_t)qi * kQueueCap;
  uint32_t base = 0;
  if (lane == 0) base = atomicAdd(g.q_tail + qi * 16, npairs);
  base = __shfl_sync(kFull, base, 0);
  // One pass: entry, then its sequence number with a RELEASE store (MEMBAR.ALL.GPU + ST: the task records -- written by any lane
  // before the __syncwarp -- and the entry are visible before the number that publishes them).  __threadfence() would also
  // invalidate the SM's whole L1 (CCTL.IVALL: its acquire half), every time, for every warp of the SM.
  __syncwarp();
#pragma unroll 1
  for (uint32_t i = lane; i < npairs; i += 32) {
    const uint32_t idx = base + i;
    QSlot* sl = ring + (idx & (kQueueCap - 1));
#pragma unroll 1
    while (ld_volatile_u32(&sl->seq) != idx) __nanosleep(64);        // the consumer of the previous lap has left the slot
    const uint32_t ta = E.ar.sel[2 * i], tb = (2 * i + 1 < nsel) ? E.ar.sel[2 * i + 1] : kNoTask;
    E.ar.tasks[ta].score = kScorePending; if (tb != kNoTask) E.ar.tasks[tb].score = kScorePending;
    sl->planner = E.planner; sl->ta = ta; sl->tb = tb;
    st_release_gpu_u32(&sl->seq, idx + 1);
  }
  E.submitted += nsel;
  const long long tw0 = lis_clock<kInstr>();
  const unsigned long long tlw = kInstr ? tl_now() : 0ull;
  if (lane == 0) {
    // (pointer and target in registers: the poll is four instructions -- the waiting planners share their schedulers with the scorers)
    const uint32_t* const dp = g.done + E.planner;
    const uint32_t want = E.submitted;
    while (ld_volatile_u32(dp) != want) __nanosleep(SMR_PLANNER_POLL_NS);
  }
  __syncwarp();
  // The counter is only a hint: a scorer adds to it after a plain store of the score, with no fence in between (a MEMBAR per pair
  // cost the scorers 5 % of their time).  What is relied on is each score word itself: it held kScorePending at submission.
#pragma unroll 1
  for (uint32_t i = lane; i < nsel; i += 32) {
    const uint32_t* const sp = &E.ar.tasks[E.ar.sel[i]].score;
#pragma unroll 1
    while (ld_volatile_u32(sp) == kScorePending) __nanosleep(64);
  }
  __syncwarp();
  if (npairs == 1) { E.w1_cyc += (unsigned long long)(lis_clock<kInstr>() - tw0); E.w1_cnt++; }
  if (kInstr && g.dbg) tl_add(g.dbg + kTlBase + 2 * kTlBuckets, E.tl0, tlw, tl_now());

}

template <bool kInstr>
__device__ void run_candidates(PassEnv& E, ReadCtx& rc, bool& search, const uint32_t max_SW_score, const uint32_t ncand, const bool by_level,
                               uint32_t level, const bool grouped);

// compute_lis_alignment (alignment.cpp:100-509).  Uniform control flow; warp-parallel inner scans.
// (not inlined: the compiler otherwise clones this function -- and run_candidates inside it -- for both strands and both sides of the
//  pass loop, four copies = 150 KB of kernel text that the planner warps walk through: a fifth of the kernel's stall samples were
//  instruction fetches)
template <bool kInstr>
__device__ __noinline__ void compute_lis_dev(PassEnv& E, ReadCtx& rc, bool& search, const uint32_t max_SW_score) {
  const DevIndex& ix = *E.ix; const DevBatch& B = *E.b; const DevParams& o = *E.prm;
  const unsigned lane = lane_id();
  const uint32_t s0 = ix.skip[0], s1 = ix.skip[1], s2 = ix.skip[2];
  const uint2* hits = E.hits;
  const uint32_t nh = E.nh;
  const uint32_t ns = (uint32_t)max(o.num_seeds, 1);
  E.n_lis_calls++;
  long long tph = lis_clock<kInstr>();
  const unsigned long long tlv = kInstr ? tl_now() : 0ull;
  const long long t_call0 = SMR_EXP_PLANNER_DELAY ? clock64() : 0ll;

  // ---- 1. votes per reference (alignment.cpp:118-138) ----
  if (++E.epoch >= 2048u) {   // epoch tag wrapped (11 bits: bit 31 of a histogram word marks a pair cursor): clear once
#pragma unroll 1
    for (uint32_t i = lane; i < E.ar.hist_cap; i += 32) E.ar.hist[i] = 0;
    E.epoch = 1; __syncwarp();
  }
  const uint32_t ep = E.epoch;
  uint32_t ncand = 0;
#pragma unroll 1
  for (uint32_t h0 = 0; h0 < nh; h0 += 32) {
    const uint32_t h = h0 + lane;
    uint32_t o_l = 0, s_l = 0;
    if (h < nh) {
      const uint2 hv = hits[h];
      if (hit_selected(hv, rc, s0, s1, s2)) { o_l = __ldg(ix.pos_off + hv.x); s_l = __ldg(ix.pos_off + hv.x + 1) - o_l; }
    }
    const uint32_t incl = warp_incl_scan_u32(s_l), tot = __shfl_sync(kFull, incl, 31), excl = incl - s_l;
    E.n_pos_entries += tot;
    // entry e of the concatenated position lists of these 32 hits -> its reference number (0xFFFFFFFF past the end)
    auto fetch_seq = [&](const uint32_t e0) -> uint32_t {
      const uint32_t e = e0 + lane;
      uint32_t lo = 0;                       // owner = first lane whose inclusive sum exceeds e
#pragma unroll
      for (int stp = 16; stp > 0; stp >>= 1) { const uint32_t v = __shfl_sync(kFull, incl, lo + stp - 1); if (v <= e) lo += stp; }
      lo = min(lo, 31u);
      const uint32_t o_own = __shfl_sync(kFull, o_l, lo), ex_own = __shfl_sync(kFull, excl, lo);
      return e < tot ? __ldg(&ix.pos[o_own + (e - ex_own)]).y : 0xFFFFFFFFu;
    };
    uint32_t seq_next = tot ? fetch_seq(0) : 0xFFFFFFFFu;
    // one leader lane per distinct reference of the step reads the epoch-tagged word and writes it back
#pragma unroll 1
    for (uint32_t e0 = 0; e0 < tot; e0 += 32) {
      const uint32_t seq = seq_next;
      if (e0 + 32 < tot) seq_next = fetch_seq(e0 + 32);   // in flight while this round's histogram words are read
      const bool act = seq != 0xFFFFFFFFu;
      const unsigned grp = __match_any_sync(kFull, seq);
      bool trans = false;
      if (act && (unsigned)(__ffs(grp) - 1) == lane && seq < E.ar.hist_cap) {
        const uint32_t old = E.ar.hist[seq];
        const uint32_t c = (old >> 20) == ep ? (old & 0xFFFFFu) : 0u;
        const uint32_t nn = min(c + (uint32_t)__popc(grp), 0xFFFFFu);
        E.ar.hist[seq] = (ep << 20) | nn;
        trans = c < ns && nn >= ns;
      }
      const unsigned tb = __ballot_sync(kFull, trans);
      if (trans) {
        const uint32_t slot = ncand + __popc(tb & ((1u << lane) - 1));
        if (slot < 32u) E.ar.cand[slot] = seq;      // the first 32 in discovery order serve the small-list path
        atomicOr(&E.ar.bitmap[seq >> 5], 1u << (seq & 31u));
        atomicOr(&E.ar.summary[seq >> 10], 1u << ((seq >> 5) & 31u));
      }
      ncand += __popc(tb);
      __syncwarp();
    }
  }
  { const long long t2 = lis_clock<kInstr>(); E.cyc[0] += (unsigned long long)(t2 - tph); tph = t2; }
  if (ncand == 0) return;
  if (ncand > E.ar.cand_cap) { rc.flags |= kOvfPairs; return; }
  __syncwarp();
  // ---- 2. order candidates: count desc, reference number asc (alignment.cpp:143-148) ----
  // Small lists (the common case) are sorted in registers.  Large ones -- reads from conserved regions vote for
  // thousands of references -- are never sorted: the bitmap yields them in ascending reference order and they
  // are then taken one count level at a time, which is the same order.
  const bool by_level = ncand > 32u;
  uint32_t level = 0;
  if (!by_level) {
    unsigned long long key = ~0ull;
    if (lane < ncand) {
      const uint32_t seq = (uint32_t)E.ar.cand[lane]; const uint32_t c = __ldcg(&E.ar.hist[seq]) & 0xFFFFFu;   // (read at L2, where the pair cursors of the grouping pass -- atomics -- live as well)
      key = ((unsigned long long)(0xFFFFFu - c) << 32) | seq;
      E.ar.bitmap[seq >> 5] = 0; E.ar.summary[seq >> 10] = 0;
    }
    key = warp_sort32_u64(key, ncand);
    E.ar.grp[lane] = key;
    E.ar.cand[lane] = key;   // (kept for the cursor clean-up; grp is the working group buffer)
  } else {
    const uint32_t n_sum = (E.ar.hist_cap + 1023u) / 1024u;
    uint32_t out = 0;
#pragma unroll 1
    for (uint32_t s0w = 0; s0w < n_sum; s0w += 32) {
      uint32_t sw = 0;
      if (s0w + lane < n_sum) { sw = E.ar.summary[s0w + lane]; if (sw) E.ar.summary[s0w + lane] = 0; }
      unsigned lanes = __ballot_sync(kFull, sw != 0);
#pragma unroll 1
      while (lanes) {
        const int L = __ffs(lanes) - 1; lanes &= lanes - 1;
        const uint32_t w = __shfl_sync(kFull, sw, L), base_word = (s0w + L) * 32u;
        uint32_t bw = 0;
        if ((w >> lane) & 1u) { bw = E.ar.bitmap[base_word + lane]; E.ar.bitmap[base_word + lane] = 0; }
        const uint32_t pc = __popc(bw), incl = warp_incl_scan_u32(pc), tot = __shfl_sync(kFull, incl, 31);
        uint32_t pos = out + incl - pc;
#pragma unroll 1
        while (bw) {
          const uint32_t bit = __ffs(bw) - 1; bw &= bw - 1;
          const uint32_t seq = (base_word + lane) * 32u + bit, c = __ldcg(&E.ar.hist[seq]) & 0xFFFFFu;
          if (pos < E.ar.cand_cap) E.ar.cand[pos] = ((unsigned long long)(0xFFFFFu - c) << 32) | seq;
          ++pos; level = max(level, c);
        }
        out += tot;
      }
    }
    if (out != ncand) { rc.flags |= kErrTrace; return; }   // internal consistency
#pragma unroll
    for (int o2 = 16; o2 > 0; o2 >>= 1) level = max(level, __shfl_xor_sync(kFull, level, o2));
  }
  __syncwarp();

  { const long long t2 = lis_clock<kInstr>(); E.cyc[1] += (unsigned long long)(t2 - tph); tph = t2; }
  // ---- 2b. group the (refpos, readpos) pairs of ALL candidates in one pass over the position lists ----
  // (the reference rescans every list once per candidate, alignment.cpp:181-194; with thousands of candidates a
  //  per-candidate gather -- even by binary search -- dominates, so the pairs are scattered into per-reference
  //  segments with one atomic cursor per reference, kept in the vote histogram word, bit 31 = "cursor")
  bool grouped = false;
  {
    uint32_t running = 0;
    const unsigned long long* list = E.ar.cand;
    uint32_t tc = 0;
#pragma unroll 1
    for (uint32_t i0 = 0; i0 < ncand; i0 += 32) { const uint32_t i = i0 + lane; if (i < ncand) tc += 0xFFFFFu - (uint32_t)(list[i] >> 32); }
    tc = warp_sum_u32(tc);
    if (tc <= E.ar.pall_cap && ncand > 1) {
#pragma unroll 1
      for (uint32_t i0 = 0; i0 < ncand; i0 += 32) {
        const uint32_t i = i0 + lane;
        uint32_t c = 0, seq = 0;
        if (i < ncand) { const unsigned long long key = list[i]; c = 0xFFFFFu - (uint32_t)(key >> 32); seq = (uint32_t)key; }
        const uint32_t incl = warp_incl_scan_u32(c), tot = __shfl_sync(kFull, incl, 31);
        if (i < ncand) E.ar.hist[seq] = 0x80000000u | (running + incl - c);
        running += tot;
      }
      __syncwarp();
#pragma unroll 1
      for (uint32_t h0 = 0; h0 < nh; h0 += 32) {
        const uint32_t h = h0 + lane;
        uint32_t o_l = 0, s_l = 0, w_l = 0;
        if (h < nh) {
          const uint2 hv = hits[h];
          if (hit_selected(hv, rc, s0, s1, s2)) { o_l = __ldg(ix.pos_off + hv.x); s_l = __ldg(ix.pos_off + hv.x + 1) - o_l; w_l = hv.y & kWinMask; }
        }
        const uint32_t incl = warp_incl_scan_u32(s_l), tot = __shfl_sync(kFull, incl, 31), excl = incl - s_l;
        uint32_t w_cur = 0, w_nxt = 0;
        auto fetch_pos = [&](const uint32_t e0, uint32_t& w_own) -> uint2 {
          const uint32_t e = e0 + lane;
          uint32_t lo = 0;
#pragma unroll
          for (int stp = 16; stp > 0; stp >>= 1) { const uint32_t v = __shfl_sync(kFull, incl, lo + stp - 1); if (v <= e) lo += stp; }
          lo = min(lo, 31u);
          const uint32_t o_own = __shfl_sync(kFull, o_l, lo), ex_own = __shfl_sync(kFull, excl, lo);
          w_own = __shfl_sync(kFull, w_l, lo);
          return e < tot ? __ldg(&ix.pos[o_own + (e - ex_own)]) : make_uint2(0u, 0xFFFFFFFFu);
        };
        uint2 ps_next = tot ? fetch_pos(0, w_nxt) : make_uint2(0u, 0xFFFFFFFFu);
        // ONE round trip per entry: the add returns the cursor when bit 31 is set; on the word of a non-candidate (an epoch-tagged
        // count below num_seeds that nothing reads again in this epoch) the extra count is harmless.
#pragma unroll 1
        for (uint32_t e0 = 0; e0 < tot; e0 += 32) {
          const uint2 ps = ps_next; w_cur = w_nxt;
          if (e0 + 32 < tot) ps_next = fetch_pos(e0 + 32, w_nxt);
          if (ps.y < E.ar.hist_cap) {
            const uint32_t old = atomicAdd(&E.ar.hist[ps.y], 1u);
            if (old & 0x80000000u) E.ar.pall[old & 0x7FFFFFFFu] = ((unsigned long long)ps.x << 32) | w_cur;
          }
        }
      }
      __syncwarp();
      grouped = true;
    }
  }
  { const long long t2 = lis_clock<kInstr>(); E.cyc[2] += (unsigned long long)(t2 - tph); tph = t2; }
  if (kInstr && E.g->dbg) tl_add(E.g->dbg + kTlBase + 3 * kTlBuckets, E.tl0, tlv, tl_now());
  if (SMR_EXP_PLANNER_DELAY) exp_delay(t_call0, SMR_EXP_PLANNER_DELAY);
  run_candidates<kInstr>(E, rc, search, max_SW_score, ncand, by_level, level, grouped);
  __syncwarp();
  if (grouped) {   // the cursors must not survive the call: histogram words are epoch-tagged votes otherwise
    const unsigned long long* list = E.ar.cand;
#pragma unroll 1
    for (uint32_t i = lane; i < ncand; i += 32) E.ar.hist[(uint32_t)list[i]] = 0;
    __syncwarp();
  }
}

constexpr int kLanePairs = 16;    // candidates with up to this many pairs are planned by ONE lane (32 candidates per warp step); thread-local arrays:
                                  // 16 pairs + two byte-sized LIS arrays = 160 B of local memory per lane (32 pairs with u32 arrays cost 3x the DRAM write-back)

struct CandPlan { uint32_t cnt, umask, nuncond; bool reset; };   // tasks of a candidate; umask: bit j = task j is unconditional (j < 32)

// The sliding window of one candidate over its SORTED pairs (alignment.cpp:205-507 without the ssw_align call), by ONE thread:
// one task per step that would reach ssw_align, written to tasks[toff ..].  The trajectory of (it, f) does not depend on any score.
template <class IdxT>
__device__ __noinline__ void plan_slide_thread(const PassEnv& E, const ReadCtx& rc, const unsigned long long* __restrict__ P, const uint32_t np, IdxT* lb, IdxT* lp,
                                  const uint32_t max_ref, const uint64_t ref_base, const uint64_t reflen, const uint32_t cand_rel, const uint32_t toff,
                                  CandPlan& out) {
  const DevIndex& ix = *E.ix; const DevParams& o = *E.prm;
  const uint64_t rlen = rc.len, lnwin = ix.lnwin;
  const uint32_t edges = o.edges_is_percent ? (uint32_t)((o.edges / 100.0) * (double)rlen) : (uint32_t)o.edges;  // :278-282
  const uint64_t em1 = (uint64_t)(uint32_t)(edges - 1u);
  uint32_t it = 0, f = 0, cnt = 0, umask = 0, nunc = 0;
  uint32_t begin_ref = (uint32_t)(P[0] >> 32), begin_read = (uint32_t)P[0];
  bool reset = false;            // a push step without a task since the previous task of this candidate
  uint32_t lead = kNoTask;       // the last unconditional task of this candidate
#pragma unroll 1
  while (it != np) {
    const uint64_t end_ref_max = (uint64_t)begin_ref + rlen - begin_read - lnwin + 1;     // :231
    bool push = false;
#pragma unroll 1
    while (it != np && (uint64_t)(uint32_t)(P[it] >> 32) <= end_ref_max) { ++it; push = true; }
    bool task = false;
    if ((it - f) >= (uint32_t)o.num_seeds) {
      uint32_t lis_first = 0;
      const uint32_t lis_len = find_lis_dev(P + f, it - f, lb, lp, lis_first);
      if (lis_len >= (uint32_t)o.min_lis) {                                               // :261
        const uint32_t lcs_ref_start = (uint32_t)(P[f + lis_first] >> 32), lcs_que_start = (uint32_t)P[f + lis_first];
        uint64_t head = 0, tail = 0, ars = 0, aqs = 0, alen = 0;
        if (lcs_ref_start < lcs_que_start) {                                              // :288-330
          aqs = lcs_que_start - lcs_ref_start;
          if (reflen < rlen) {
            if (aqs > (rlen - reflen)) alen = reflen - (aqs - (rlen - reflen)); else alen = reflen;
          } else {
            tail = reflen - ars - rlen; if (tail > em1) tail = edges;
            alen = rlen + head + tail - aqs;
          }
        } else {                                                                          // :331-357
          ars = lcs_ref_start - lcs_que_start;
          if (ars > em1) head = edges;
          if (ars + rlen > reflen) { tail = 0; alen = reflen - ars - head; }
          else { tail = reflen - ars - rlen; if (tail > em1) tail = edges; alen = rlen + head + tail; }
        }
        const int32_t qlen = (int32_t)(alen - head - tail);
        const uint32_t win_start = (uint32_t)(ars - head);
        const bool unc = push || reset;
        const uint32_t fl = (push ? kTfPush : 0u) | (unc ? kTfUncond : 0u) | (reset ? kTfReset : 0u);
        const uint32_t ti = toff + cnt;
        SwTask t;
        t.ref_abs = (uint32_t)ref_base + win_start;
        t.q_abs = rc.reversed ? rc.seq_base + (rc.len - 1u - (uint32_t)aqs) : rc.seq_base + (uint32_t)aqs;   // query = current strand, 0-4 alphabet (:360-366)
        t.alen = (uint32_t)alen; t.qlen = qlen > 0 ? (uint32_t)qlen : 0u;
        t.meta = ix.slot | (rc.reversed ? 0x10000u : 0u);
        t.score = 0; t.pad0 = 0; t.pad1 = 0;
        E.ar.tasks[ti] = t;
        PlanTask pt;
        pt.max_ref = max_ref; pt.win_start = win_start; pt.aqs = (uint32_t)aqs; pt.cf = cand_rel | (fl << 24);
        pt.lead = unc ? ti : lead;
        E.ar.ptasks[ti] = pt;
        if (unc) { lead = ti; ++nunc; if (cnt < 32u) umask |= 1u << cnt; }
        ++cnt;
        task = true; reset = false;
      }
    }
    if (!task && push) reset = true;
    // pop (:486-506)
    if (it > f) ++f;
    if (it == f) {
      if (it != np) { begin_ref = (uint32_t)(P[it] >> 32); begin_read = (uint32_t)P[it]; } else break;
    } else { begin_ref = (uint32_t)(P[f] >> 32); begin_read = (uint32_t)P[f]; }
  }
  out.cnt = cnt; out.umask = umask; out.nuncond = nunc; out.reset = reset;
}

// A candidate with more than kLanePairs pairs (or whose pairs were not grouped by the scatter): the warp gathers and sorts the
// pairs (alignment.cpp:181-201), lane 0 slides.  Returns false on scratch overflow (rc.flags set).
__device__ __noinline__ bool plan_candidate_warp(PassEnv& E, ReadCtx& rc, const unsigned long long ck, const uint32_t cand_rel, const uint32_t toff, const bool grouped,
                                    CandPlan& out) {
  const DevIndex& ix = *E.ix;
  const unsigned lane = lane_id();
  const uint32_t s0 = ix.skip[0], s1 = ix.skip[1], s2 = ix.skip[2];
  const uint2* hits = E.hits;
  const uint32_t nh = E.nh;
  const uint32_t max_ref = (uint32_t)ck, max_occur = 0xFFFFFu - (uint32_t)(ck >> 32);
  const uint64_t ref_base = __ldg(ix.ref_off + max_ref), ref_next = __ldg(ix.ref_off + max_ref + 1);
  const uint32_t np = max_occur;
  unsigned long long* P; uint32_t* lb; uint32_t* lp;
  if (np <= (uint32_t)kPairsShared) { P = E.s_pairs; lb = E.s_b; lp = E.s_p; }
  else if (np <= E.ar.pair_cap) { P = E.ar.pairs; lb = E.ar.lis_b; lp = E.ar.lis_p; }
  else { rc.flags |= kOvfPairs; return false; }
  uint32_t filled = 0;
  if (grouped) {   // the pairs of this reference were grouped by the one-pass scatter
    const uint32_t seg_end = __ldcg(&E.ar.hist[max_ref]) & 0x7FFFFFFFu, seg = seg_end - np;
#pragma unroll 1
    for (uint32_t i = lane; i < np; i += 32) P[i] = E.ar.pall[seg + i];
    filled = np;
  } else
#pragma unroll 1
  for (uint32_t h0 = 0; h0 < nh; h0 += 32) {
    const uint32_t h = h0 + lane;
    uint32_t first = 0, cnt = 0, win = 0;
    if (h < nh) {
      const uint2 hv = hits[h];
      if (hit_selected(hv, rc, s0, s1, s2)) {
        win = hv.y & kWinMask;
        uint32_t lo = __ldg(ix.pos_off + hv.x), hi = __ldg(ix.pos_off + hv.x + 1);
        const uint32_t end = hi;
#pragma unroll 1
        while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (__ldg(&ix.pos[mid]).y < max_ref) lo = mid + 1; else hi = mid; }
        first = lo;
#pragma unroll 1
        while (first + cnt < end && __ldg(&ix.pos[first + cnt]).y == max_ref) ++cnt;
      }
    }
    const uint32_t incl = warp_incl_scan_u32(cnt), tot = __shfl_sync(kFull, incl, 31);
    uint32_t w = filled + incl - cnt;
#pragma unroll 1
    for (uint32_t c = 0; c < cnt; ++c, ++w) if (w < np) P[w] = ((unsigned long long)__ldg(&ix.pos[first + c]).x << 32) | win;
    filled += tot;
  }
  __syncwarp();
  if (filled != np) { rc.flags |= kErrTrace; return false; }   // internal consistency: votes == gathered pairs
  if (np <= 32u) {
    unsigned long long key = lane < np ? P[lane] : ~0ull;
    __syncwarp();
    key = warp_sort32_u64(key, np);
    if (lane < np) P[lane] = key;
    __syncwarp();
  } else {
    const uint32_t np2 = next_pow2(np);
#pragma unroll 1
    for (uint32_t i = np + lane; i < np2; i += 32) P[i] = ~0ull;
    __syncwarp();
    warp_sort_u64(P, np2);
  }
  CandPlan cp{0, 0, 0, false};
  if (lane == 0) plan_slide_thread(E, rc, P, np, lb, lp, max_ref, ref_base, ref_next - ref_base, cand_rel, toff, cp);
  out.cnt = __shfl_sync(kFull, cp.cnt, 0); out.umask = __shfl_sync(kFull, cp.umask, 0); out.nuncond = __shfl_sync(kFull, cp.nuncond, 0);
  out.reset = __shfl_sync(kFull, cp.reset ? 1u : 0u, 0) != 0;
  __syncwarp();
  return true;
}

// candidates in order (alignment.cpp:150-508), in batches: plan -> score (by the scorer warps) -> replay.
// Returns through rc.flags on scratch overflow.
template <bool kInstr>
__device__ void run_candidates(PassEnv& E, ReadCtx& rc, bool& search, const uint32_t max_SW_score, const uint32_t ncand, const bool by_level,
                               uint32_t level, const bool grouped) {
  const DevIndex& ix = *E.ix; const DevBatch& B = *E.b; const DevParams& o = *E.prm;
  const unsigned lane = lane_id();
  const unsigned lt = (1u << lane) - 1u;
  bool is_aligned = false, first_cand = true, stop_all = false, searching = true;
  uint32_t prev_occur = 0;
  const uint32_t N = (uint32_t)o.num_alignments;
  AlnWork* slots = E.g->aln_work + (size_t)rc.r * E.g->slots;
  uint32_t cap = SMR_BATCH_CAP0;   // candidates per batch; doubles per batch (a perfect-score stop wastes at most what was useful)
  uint32_t* cfirst = E.ar.cfirst; uint32_t* ccnt = cfirst + kBatchCandCap; uint32_t* cumask = ccnt + kBatchCandCap;

#pragma unroll 1
  for (;;) {
    // the next group: everything (sorted) for small lists, else the members of the current count level
    uint32_t ngrp = ncand, next_level = 0;
    if (by_level) {
      if (level == 0) break;
      ngrp = 0;
#pragma unroll 1
      for (uint32_t i0 = 0; i0 < ncand; i0 += 32) {
        const uint32_t i = i0 + lane;
        unsigned long long key = 0; uint32_t c = 0;
        if (i < ncand) { key = E.ar.cand[i]; c = 0xFFFFFu - (uint32_t)(key >> 32); }
        const bool pick = i < ncand && c == level;
        const unsigned pm = __ballot_sync(kFull, pick);
        if (pick) E.ar.grp[ngrp + __popc(pm & lt)] = key;
        ngrp += __popc(pm);
        if (i < ncand && c < level) next_level = max(next_level, c);
      }
#pragma unroll
      for (int o2 = 16; o2 > 0; o2 >>= 1) next_level = max(next_level, __shfl_xor_sync(kFull, next_level, o2));
      __syncwarp();
    }
    uint32_t k = 0;
#pragma unroll 1
    while (k < ngrp && searching) {
      long long tc0 = lis_clock<kInstr>();
      // ---- entry of the batch's first candidate (:158-169): decided now, with the scores known so far ----
      {
        const uint32_t occ = 0xFFFFFu - (uint32_t)(E.ar.grp[k] >> 32);
        if (occ < (uint32_t)o.num_seeds) { stop_all = true; break; }                                                                    // :158
        if (is_aligned && o.min_lis > 0 && !first_cand && occ < prev_occur) { --rc.best; if (rc.best < 1) { stop_all = true; break; } }   // :165-169
        prev_occur = occ; first_cand = false;
      }
      // ---- extent of the batch: candidates k .. k + nb.  It ends before the level drop at which the countdown of `best` could
      //      end the call (so nothing behind a possible stop is scored), at `cap` candidates, or when the task array is full ----
      const uint32_t budget = o.min_lis > 0 ? (uint32_t)max(rc.best, 1) : 0xFFFFFFFFu;
      // without `best`, the call ends at the N-th accepted alignment (:466-468): speculate on no more than are still wanted
      const uint32_t cap_now = min((N > 0 && !o.is_best) ? min(cap, 2u * (N > rc.n_align ? N - rc.n_align : 1u)) : cap, (uint32_t)kBatchCandCap);
      uint32_t nb = 0;
      {
        uint32_t drops = 0, tsum = 0, prev = prev_occur; bool ended = false;
#pragma unroll 1
        for (uint32_t c0 = 0; !ended; c0 += 32) {
          const uint32_t c = c0 + lane;
          const bool in = k + c < ngrp && c < cap_now;
          const uint32_t occ = in ? 0xFFFFFu - (uint32_t)(E.ar.grp[k + c] >> 32) : 0u;
          uint32_t up = __shfl_up_sync(kFull, occ, 1); if (lane == 0) up = prev;
          const uint32_t d = (in && occ < up) ? 1u : 0u;
          const uint32_t dincl = drops + warp_incl_scan_u32(d), tincl = tsum + warp_incl_scan_u32(occ);
          // candidate c belongs to the batch unless: out of range, a drop that exhausts the budget, the call's end (:158), or no room
          const bool stop = !in || (c > 0 && (dincl >= budget || occ < (uint32_t)o.num_seeds || tincl > E.ar.task_cap));
          const unsigned sm = __ballot_sync(kFull, stop);
          if (sm) { nb = c0 + (uint32_t)(__ffs(sm) - 1); ended = true; }
          else { drops = __shfl_sync(kFull, dincl, 31); tsum = __shfl_sync(kFull, tincl, 31); prev = __shfl_sync(kFull, occ, 31); }
        }
      }
      if (nb == 0) { rc.flags |= kErrTrace; return; }   // (the first candidate always belongs: its pairs fit, np <= pair_cap is checked below)
      // ---- plan: one candidate per lane (its few pairs in thread-local arrays); candidates with many pairs by the whole warp ----
      uint32_t tbase = 0, nselA = 0, ncond = 0;
#pragma unroll 1
      for (uint32_t c0 = 0; c0 < nb; c0 += 32) {
        const uint32_t c = c0 + lane;
        const bool valid = c < nb;
        const unsigned long long ck = valid ? E.ar.grp[k + c] : 0ull;
        const uint32_t max_ref = (uint32_t)ck, np = valid ? 0xFFFFFu - (uint32_t)(ck >> 32) : 0u;
        const uint32_t incl = warp_incl_scan_u32(np), toff = tbase + incl - np;
        const bool small = valid && grouped && np <= (uint32_t)kLanePairs;
        CandPlan cp{0, 0, 0, false};
        if (small) {
          const uint64_t ref_base = __ldg(ix.ref_off + max_ref), ref_next = __ldg(ix.ref_off + max_ref + 1);
          const uint32_t seg = (__ldcg(&E.ar.hist[max_ref]) & 0x7FFFFFFFu) - np;
          unsigned long long P[kLanePairs]; uint8_t lb[kLanePairs], lp[kLanePairs];
#pragma unroll 1
          for (uint32_t i = 0; i < np; ++i) {    // insertion sort while loading (refpos asc, readpos asc: alignment.cpp:197-201)
            const unsigned long long v = E.ar.pall[seg + i];
            uint32_t j = i;
#pragma unroll 1
            while (j > 0 && P[j - 1] > v) { P[j] = P[j - 1]; --j; }
            P[j] = v;
          }
          plan_slide_thread(E, rc, P, np, lb, lp, max_ref, ref_base, ref_next - ref_base, c, toff, cp);
        }
        unsigned big = __ballot_sync(kFull, valid && !small);
#pragma unroll 1
        while (big) {
          const int L = __ffs(big) - 1; big &= big - 1;
          const unsigned long long ckL = __shfl_sync(kFull, ck, L);
          const uint32_t toffL = __shfl_sync(kFull, toff, L);
          CandPlan cb{0, 0, 0, false};
          if (!plan_candidate_warp(E, rc, ckL, c0 + (uint32_t)L, toffL, grouped, cb)) return;
          if ((int)lane == L) { cp = cb; cp.umask = 0; }
          // its unconditional tasks go to round A now (they may be more than 32: no mask)
#pragma unroll 1
          for (uint32_t t0 = 0; t0 < cb.cnt; t0 += 32) {
            const uint32_t t = t0 + lane;
            const bool pick = t < cb.cnt && ((E.ar.ptasks[toffL + t].cf >> 24) & kTfUncond);
            const unsigned pm = __ballot_sync(kFull, pick);
            if (pick) E.ar.sel[nselA + __popc(pm & lt)] = toffL + t;
            nselA += __popc(pm);
          }
        }
        if (valid) { cfirst[c] = toff; ccnt[c] = cp.cnt | (cp.reset ? 0x80000000u : 0u) | (small ? 0u : 0x40000000u); cumask[c] = cp.umask; }
        // round A entries of the lane-planned candidates
        {
          const uint32_t nu = small ? (uint32_t)__popc(cp.umask) : 0u;
          const uint32_t ui = warp_incl_scan_u32(nu);
          uint32_t w = nselA + ui - nu, m = small ? cp.umask : 0u;
#pragma unroll 1
          while (m) { const uint32_t j = (uint32_t)__ffs(m) - 1u; m &= m - 1u; E.ar.sel[w++] = toff + j; }
          nselA += __shfl_sync(kFull, ui, 31);
        }
        ncond += warp_sum_u32(valid ? cp.cnt - cp.nuncond : 0u);
        tbase += __shfl_sync(kFull, incl, 31);
      }
      __syncwarp();
      { const long long t2 = lis_clock<kInstr>(); E.cyc[3] += (unsigned long long)(t2 - tc0); tc0 = t2; }
      // ---- score, round A: the unconditional tasks ----
      submit_and_wait<kInstr>(E, nselA);
      E.n_spec_calls += nselA; E.n_spec_cells += nselA ? 1 : 0;
      // ---- round B: tasks heuristic 1 would skip after a successful lead (:243-246) are needed when the lead failed ----
      if (ncond) {
        uint32_t nselB = 0;
#pragma unroll 1
        for (uint32_t c0 = 0; c0 < nb; c0 += 32) {
          const uint32_t c = c0 + lane;
          const bool valid = c < nb;
          const uint32_t toff = valid ? cfirst[c] : 0u, cw = valid ? ccnt[c] : 0u, cnt = cw & 0x3FFFFFFFu;
          const bool bigc = (cw & 0x40000000u) != 0;
          uint32_t bmask = 0;
          if (valid && !bigc && cnt) {
            uint32_t m = cumask[c];
#pragma unroll 1
            while (m) {
              const uint32_t j = (uint32_t)__ffs(m) - 1u; m &= m - 1u;
              const uint32_t jn = m ? (uint32_t)__ffs(m) - 1u : cnt;        // next unconditional task (or the end)
              if (jn > j + 1 && (__ldcg(&E.ar.tasks[toff + j].score) & 0xFFFFu) <= ix.minimal_score) bmask |= ((jn < 32u ? (1u << jn) : 0u) - 1u) & ~((2u << j) - 1u);
            }
          }
          const uint32_t nbm = (uint32_t)__popc(bmask), bi = warp_incl_scan_u32(nbm);
          uint32_t w = nselB + bi - nbm;
#pragma unroll 1
          while (bmask) { const uint32_t j = (uint32_t)__ffs(bmask) - 1u; bmask &= bmask - 1u; E.ar.sel[w++] = toff + j; }
          nselB += __shfl_sync(kFull, bi, 31);
          unsigned big = __ballot_sync(kFull, valid && bigc && cnt);
#pragma unroll 1
          while (big) {
            const int L = __ffs(big) - 1; big &= big - 1;
            const uint32_t toffL = __shfl_sync(kFull, toff, L), cntL = __shfl_sync(kFull, cnt, L);
#pragma unroll 1
            for (uint32_t t0 = 0; t0 < cntL; t0 += 32) {
              const uint32_t t = t0 + lane;
              bool pick = false;
              if (t < cntL) {
                const PlanTask pt = E.ar.ptasks[toffL + t];
                if (!((pt.cf >> 24) & kTfUncond)) pick = (__ldcg(&E.ar.tasks[pt.lead].score) & 0xFFFFu) <= ix.minimal_score;
              }
              const unsigned pm = __ballot_sync(kFull, pick);
              if (pick) E.ar.sel[nselB + __popc(pm & lt)] = toffL + t;
              nselB += __popc(pm);
            }
          }
        }
        __syncwarp();
        submit_and_wait<kInstr>(E, nselB);
        E.n_spec_calls += nselB; E.n_rounds_b += nselB ? 1 : 0;
      }
      { const long long t2 = lis_clock<kInstr>(); E.cyc[4] += (unsigned long long)(t2 - tc0); tc0 = t2; }
      // ---- replay: the reference's decisions over the scores, in order ----
#pragma unroll 1
      for (uint32_t c0 = 0; c0 < nb && searching; c0 += 32) {
        // this chunk's candidates: (first task, count, flags, votes), one per lane
        const uint32_t cl = c0 + lane;
        const uint32_t v_toff = cl < nb ? cfirst[cl] : 0u, v_cw = cl < nb ? ccnt[cl] : 0u;
        const uint32_t v_occ = cl < nb ? 0xFFFFFu - (uint32_t)(E.ar.grp[k + cl] >> 32) : 0u;
        const uint32_t cend = min(32u, nb - c0);
        // fast path: candidates none of whose tasks aligned change nothing but the call counters (every task of such a candidate was
        // scored and consumed: heuristic 1 only skips behind a success) -- one candidate per lane; the sequential replay starts at
        // the first candidate of the chunk that holds a success
        uint32_t ci0 = 0;
        {
          const uint32_t cntl = v_cw & 0x3FFFFFFFu;
          bool succ = cl < nb && (v_cw & 0x40000000u) != 0 && cntl > 0;   // (many-pair candidates take the sequential path)
          unsigned long long cells = 0;
          if (cl < nb && !(v_cw & 0x40000000u)) {
#pragma unroll 1
            for (uint32_t j = 0; j < cntl; ++j) {
              const uint4 w0 = __ldcg((const uint4*)&E.ar.tasks[v_toff + j]);
              if ((__ldcg(&E.ar.tasks[v_toff + j].score) & 0xFFFFu) > ix.minimal_score) { succ = true; break; }
              cells += (unsigned long long)w0.z * (unsigned long long)w0.w;
            }
          }
          const unsigned sm = __ballot_sync(kFull, succ);
          ci0 = sm ? (uint32_t)(__ffs(sm) - 1) : cend;
          const bool mine = lane < ci0 && cl < nb;
          const uint32_t ncons = warp_sum_u32(mine ? cntl : 0u);
          E.n_sw_calls += ncons; E.n_sw_cells += warp_sum_u64(mine ? cells : 0ull);
          if (ncons && rc.hasn) rc.form04 = true;                                               // flip34 before SSW (:360-361)
          if (ci0 > 0) {
            // entry of the chunk's first candidate (:165-169) with the state the previous chunk left; behind it nothing is aligned
            if (c0 > 0 && is_aligned && o.min_lis > 0 && __shfl_sync(kFull, v_occ, 0) < prev_occur) --rc.best;   // (cannot reach 0 inside a batch)
            is_aligned = false; prev_occur = __shfl_sync(kFull, v_occ, ci0 - 1);
          }
        }
#pragma unroll 1
        for (uint32_t ci = ci0; ci < cend && searching; ++ci) {
          const uint32_t c = c0 + ci;
          const uint32_t toff = __shfl_sync(kFull, v_toff, ci), cw = __shfl_sync(kFull, v_cw, ci), occ = __shfl_sync(kFull, v_occ, ci);
          const uint32_t cnt = cw & 0x3FFFFFFFu;
          if (c > 0) {   // entry of a later candidate of the batch (:158-169); the countdown cannot reach 0 inside a batch
            if (is_aligned && o.min_lis > 0 && occ < prev_occur) { --rc.best; if (rc.best < 1) { stop_all = true; searching = false; break; } }
            prev_occur = occ;
          }
          is_aligned = false;   // the first step of a candidate always pushes: `else is_aligned = false` (:245)
#pragma unroll 1
          for (uint32_t t0 = 0; t0 < cnt && searching; t0 += 32) {
            // this chunk's tasks: flags, score, cells, one per lane
            const uint32_t tl = toff + t0 + lane;
            uint32_t v_fl = 0, v_sc = 0, v_alen = 0, v_qlen = 0;
            if (t0 + lane < cnt) {
              v_fl = E.ar.ptasks[tl].cf >> 24;
              const uint4 w0 = __ldcg((const uint4*)&E.ar.tasks[tl]);
              v_alen = w0.z; v_qlen = w0.w; v_sc = __ldcg(&E.ar.tasks[tl].score);
            }
            const uint32_t tend = min(32u, cnt - t0);
#pragma unroll 1
            for (uint32_t ti = 0; ti < tend && searching; ++ti) {
              const uint32_t fl = __shfl_sync(kFull, v_fl, ti);
              if (fl & kTfReset) is_aligned = false;
              if (!(fl & kTfPush) && is_aligned) continue;                                      // heuristic 1 (:244-245)
              is_aligned = false;
              const uint32_t sw = __shfl_sync(kFull, v_sc, ti), alen = __shfl_sync(kFull, v_alen, ti), qlen = __shfl_sync(kFull, v_qlen, ti);
              const uint32_t t = toff + t0 + ti;
              if (rc.hasn) rc.form04 = true;                                                    // flip34 before SSW (:360-361)
              E.n_sw_calls++; E.n_sw_cells += (unsigned long long)alen * (unsigned long long)qlen;
              const uint32_t score1 = sw & 0xFFFFu;                                             // s_align.score1 is uint16
              is_aligned = score1 > ix.minimal_score;                                           // :388
              if (is_aligned) {
                const PlanTask pt = E.ar.ptasks[t];
                if (!(fl & kTfUncond) && (__ldcg(&E.ar.tasks[pt.lead].score) & 0xFFFFu) > ix.minimal_score) { rc.flags |= kErrTrace; return; }   // consistency: it was scored
                if (score1 == max_SW_score) ++rc.max_SW_count;                                  // :391
                AlnWork a;
                a.ref_num = pt.max_ref; a.win_ref_start = pt.win_start; a.win_len = alen; a.q_start = pt.aqs; a.q_len = qlen;
                a.score1 = (uint16_t)score1; a.part = (uint16_t)ix.part; a.index_num = (uint16_t)ix.index_num;
                a.strand = rc.reversed ? 0 : 1; a.idx_slot = (uint16_t)ix.slot; a.pad0 = 0;
                if (!rc.is_hit) {                                                               // :411-416
                  rc.is_hit = true;   // readstats.num_aligned / reads_matched_per_db are summed from hit_db at download time
                  if (lane == 0) B.hit_db[rc.r] = (uint16_t)ix.index_num;
                }
                if (N == 0 || !o.is_best || (o.is_best && rc.n_align < N)) {                    // :420-424
                  // (N == 0, "all alignments": the count runs on past the caller's stride so that the host can name the stride needed)
                  if (rc.n_align < E.g->slots) { if (lane == 0) slots[rc.n_align] = a; } else rc.ovf_slots = true;
                  rc.n_align++; rc.is_new_hit = true;
                } else if (o.is_best && rc.n_align == N && slots[rc.min_index].score1 < score1) {  // :425-459
                  if (N > 1 && rc.max_index == 0 && rc.min_index == 0) {
                    uint32_t mn = 0, mx = 0, mns = slots[0].score1, mxs = slots[0].score1;      // findMinIndex / findMaxIndex (:533-561)
#pragma unroll 1
                    for (uint32_t i2 = 0; i2 < rc.n_align; ++i2) { const uint32_t s = slots[i2].score1; if (s < mns) { mns = s; mn = i2; } if (s > mxs) { mxs = s; mx = i2; } }
                    rc.min_index = mn; rc.max_index = mx;
                  }
                  const uint32_t mn = rc.min_index, mx = rc.max_index;
                  __syncwarp();
                  if (lane == 0) slots[mn] = a;
                  __syncwarp();
                  rc.is_new_hit = true;
                  if (score1 > slots[mx].score1 && rc.n_align > 1) {
                    rc.max_index = mn;
                    uint32_t m2 = 0, ms = slots[0].score1;
#pragma unroll 1
                    for (uint32_t i2 = 0; i2 < rc.n_align; ++i2) { const uint32_t s = slots[i2].score1; if (s < ms) { ms = s; m2 = i2; } }
                    rc.min_index = m2;
                  }
                }
                __syncwarp();
                if (N > 0) {                                                                    // :462-469
                  if (o.is_best) { if (N == rc.max_SW_count) searching = false; }
                  else if (N == rc.n_align) searching = false;
                }
                search = false;                                                                 // :472
              }
            }
          }
          if (searching && (cw & 0x80000000u)) is_aligned = false;
        }
      }
      { const long long t2 = lis_clock<kInstr>(); E.cyc[5] += (unsigned long long)(t2 - tc0); }
      k += nb;
      cap = min(cap * 2u, (uint32_t)kBatchCandCap);
      __syncwarp();
    }
    if (!by_level || stop_all || !searching) break;
    level = next_level;
  }
}

// traverse() pass loop for one strand (paralleltraversal.cpp:92-297)
template <bool kInstr>
__device__ void traverse_dev(PassEnv& E, ReadCtx& rc, const bool is_last_strand) {
  const DevIndex& ix = *E.ix; const DevBatch& B = *E.b; const DevParams& o = *E.prm;
  const unsigned lane = lane_id();
  const uint32_t s0 = ix.skip[0], s1 = ix.skip[1], s2 = ix.skip[2];
  const uint2* hits = E.hits;
  const uint32_t nh = E.nh;
  const uint32_t max_SW_score = rc.len * (uint32_t)o.match;                                 // :101
  // which seed variant the windows of this strand see (SURVEY A.10)
  uint32_t var = rc.reversed ? kVarRevT : kVarFwd;
  uint32_t pass_n = 0;
  bool search = true;
#pragma unroll 1
  while (search) {
    // first window of the pass: `if (read.is04) read.flip34()` (:126) -> back to 0-3 with N positions = 0 (A)
    if (rc.hasn && rc.form04) { rc.form04 = false; if (rc.reversed) var = kVarRevA; }
    rc.vcls[pass_n] = var;
    rc.pass_n = pass_n;
    // windows searched for the first time in this pass that produced hits (:242-249)
    uint32_t newly = 0;
#pragma unroll 1
    for (uint32_t h0 = 0; h0 < nh; h0 += 32) {
      const uint32_t h = h0 + lane;
      bool cnt = false;
      if (h < nh) {
        const uint2 hv = hits[h];
        if (((hv.y >> 24) & 15u) == var && (hv.y >> 28) == pass_n) cnt = (h == 0) || (hits[h - 1].y != hv.y);
      }
      newly += __popc(__ballot_sync(kFull, cnt));
    }
    rc.hit_seeds += newly;
    if (rc.hit_seeds >= (uint32_t)o.num_seeds) compute_lis_dev<kInstr>(E, rc, search, max_SW_score);  // :256-258
    if (rc.flags) return;
    if (search) {                                                                              // :262-277
      if (pass_n == 2) search = false;
      else {
#pragma unroll 1
        while (pass_n < 2 && ix.skip[pass_n] == ix.skip[pass_n + 1]) { ++pass_n; rc.vcls[pass_n] = var; }
        if (++pass_n > 2) search = false;
      }
    }
  }
  const uint32_t N = (uint32_t)o.num_alignments;                                              // :286-297
  if (N > 0) {
    if ((o.is_best && N == rc.max_SW_count) || (!o.is_best && rc.n_align == N)) rc.is_done = true;
  } else if (ix.is_last && is_last_strand && rc.n_align > 0) rc.is_done = true;
}

// Stages one task pair into slot `sl` and arrives on its "full" mbarrier (ONE lane).  da / db: the first four words of the two
// SwTask records (ref_abs, q_abs, alen, qlen), ma / mb their meta words; two = false: no task B.  Pairs the packed kernel cannot
// score (sw_pair_ok) are marked slow and nothing is copied; an empty B task (no rows or no columns) rides along as a dead problem.
// ref_of(meta) gives the reference buffer a task's window lies in; seq04: the reads.  Both must extend at least 15 bytes past the
// last byte a task names (the copies are 16-byte aligned supersets).  The candidate kernel's fetcher and smr_debug_sw_tasks share it.
template <class RefOf>
__device__ __forceinline__ void stage_pair(ScSlot* sl, const uint4 da, const uint32_t ma, const bool two, const uint4 db, const uint32_t mb,
                                           const uint8_t* const& seq04, const SwScore sc, const RefOf ref_of) {
  const bool oka = da.w > 0 && da.z > 0 && sw_pair_ok((int32_t)da.w, (int32_t)da.z, sc);
  const bool okb = !two || db.w == 0 || db.z == 0 || sw_pair_ok((int32_t)db.w, (int32_t)db.z, sc);
  const bool fast = oka && okb;
  const bool liveb = two && db.w > 0 && db.z > 0;
  sl->slow = fast ? 0u : 1u;
  sl->mA = da.w; sl->nA = da.z; sl->metaA = ma; sl->qabsA = da.y; sl->refA = da.x;
  sl->mB = two ? db.w : 0u; sl->nB = two ? db.z : 0u; sl->metaB = mb; sl->qabsB = db.y; sl->refB = db.x;
  if (!fast) mbar_arrive(&sl->bar);
  else {
    // 16-byte aligned supersets of [ref_abs, ref_abs + n) and of the query segment (minus strand: it ends at q_abs)
    const uint8_t* ra = ref_of(ma);
    const uint32_t wa0 = da.x & ~15u, wab = ((da.x & 15u) + da.z + 15u) & ~15u;
    const uint32_t qsa = (ma & 0x10000u) ? da.y - (da.w - 1u) : da.y, qa0 = qsa & ~15u, qab = ((qsa & 15u) + da.w + 15u) & ~15u;
    sl->woffA = kWinOff + (da.x & 15u); sl->qoffA = (ma & 0x10000u) ? (qsa & 15u) + da.w - 1u : (qsa & 15u);
    uint32_t wb0 = 0, wbb = 0, qb0 = 0, qbb = 0; const uint8_t* rb = ra;
    if (liveb) {
      rb = ref_of(mb);
      wb0 = db.x & ~15u; wbb = ((db.x & 15u) + db.z + 15u) & ~15u;
      const uint32_t qsb = (mb & 0x10000u) ? db.y - (db.w - 1u) : db.y;
      qb0 = qsb & ~15u; qbb = ((qsb & 15u) + db.w + 15u) & ~15u;
      sl->woffB = kWinOff + (db.x & 15u); sl->qoffB = (mb & 0x10000u) ? (qsb & 15u) + db.w - 1u : (qsb & 15u);
    } else { sl->woffB = kWinOff; sl->qoffB = 0; sl->mB = 0; sl->nB = 0; }
    mbar_arrive_expect_tx(&sl->bar, wab + qab + wbb + qbb);
    bulk_g2s(sl->win[0] + kWinOff, ra + wa0, wab, &sl->bar);
    bulk_g2s(sl->q[0], seq04 + qa0, qab, &sl->bar);
    if (liveb) { bulk_g2s(sl->win[1] + kWinOff, rb + wb0, wbb, &sl->bar); bulk_g2s(sl->q[1], seq04 + qb0, qbb, &sl->bar); }
  }
}

// Scores the task pair staged in slot S (whole warp, after the slot's "full" mbarrier completed) into sa / sb; returns true when the
// packed 16-bit pass ran, false for the s32 fallback.  s_prof: the two query profiles (kPairProfWords each), reused while keyq / keym
// / keyR (the identity of the profile in each half: q_abs, qlen | rev << 31, and the R both were built for) say they still hold the
// right query.  The fallback reads the inputs from global memory (ref_of, seq04) and scores a problem only if its window fits the row
// scratch (rowH / rowF, row_cap ints each).  loaded(): called between profile set-up and the score pass; slow(): called when the
// fallback ran (the instrumented kernel's phase clock and counters).  The candidate kernel's scorers and smr_debug_sw_tasks share it.
// (Lazy arguments -- references, callbacks -- keep each global load inside the branch that needs it, as in the loop this came from.)
template <class RefOf, class Loaded, class Slow>
__device__ __forceinline__ bool score_slot(ScSlot& S, const bool two, uint32_t* s_prof, uint32_t (&keyq)[2], uint32_t (&keym)[2], int& keyR, const SwScore sc, const uint8_t* const& seq04,
                                           const RefOf ref_of, int32_t* rowH, int32_t* rowF, const uint32_t& row_cap, const Loaded loaded,
                                           const Slow slow, uint32_t& sa, uint32_t& sb) {
  const int32_t mA = (int32_t)S.mA, nA = (int32_t)S.nA, mB = (int32_t)S.mB, nB = (int32_t)S.nB;
  sa = 0; sb = 0;
  if (!S.slow) {
    const int R = pair_rows(max(mA, mB));
    const int32_t nmax = max(nA, nB);
    uint8_t* wa = S.win[0] + S.woffA; uint8_t* wb = S.win[1] + S.woffB;
    pair_sentinels(wa, nA, nmax);
    pair_sentinels(wb, nB, nmax);
    const uint32_t kqa = S.qabsA, kma = (uint32_t)mA | ((S.metaA & 0x10000u) << 15), kqb = mB ? S.qabsB : 0xFFFFFFFEu, kmb = mB ? ((uint32_t)mB | ((S.metaB & 0x10000u) << 15)) : 0u;
    // the two tasks of a pair are usually steps of one read on one strand with the same query segment: one profile serves both
    if (R != keyR) { keyq[0] = keyq[1] = 0xFFFFFFFFu; keyR = R; }
    if (!(keyq[0] == kqa && keym[0] == kma)) { const bool rev = (S.metaA & 0x10000u) != 0; pair_profile(S.q[0] + S.qoffA, rev ? -1 : 1, rev, mA, R, sc, s_prof); keyq[0] = kqa; keym[0] = kma; }
    const uint32_t* profB = s_prof;
    if (!(kqb == kqa && kmb == kma)) {
      if (!(keyq[1] == kqb && keym[1] == kmb)) { const bool rev = (S.metaB & 0x10000u) != 0; pair_profile(S.q[1] + S.qoffB, rev ? -1 : 1, rev, mB, R, sc, s_prof + kPairProfWords); keyq[1] = kqb; keym[1] = kmb; }
      profB = s_prof + kPairProfWords;
    }
    __syncwarp();
    loaded();
    const uint32_t r2 = sw_pair_dispatch(R, s_prof, profB, wa, wb, nmax, sc);
    sa = r2 & 0xFFFFu; sb = r2 >> 16;
    return true;
  }
  // shapes or scoring schemes outside the 16-bit kernel: the s32 wavefront (row blocks for long queries), from global memory
  keyR = 0;
  const bool reva = (S.metaA & 0x10000u) != 0, revb = (S.metaB & 0x10000u) != 0;
  if (mA > 0 && nA > 0 && (uint32_t)nA <= row_cap)
    sa = (uint32_t)sw_forward_any(SeqView{seq04, (int32_t)S.qabsA, reva ? -1 : 1, reva}, mA, SeqView{ref_of(S.metaA), (int32_t)S.refA, 1, false}, nA, sc, rowH, rowF).score;
  if (two && mB > 0 && nB > 0 && (uint32_t)nB <= row_cap)
    sb = (uint32_t)sw_forward_any(SeqView{seq04, (int32_t)S.qabsB, revb ? -1 : 1, revb}, mB, SeqView{ref_of(S.metaB), (int32_t)S.refB, 1, false}, nB, sc, rowH, rowF).score;
  slow();
  return false;
}

// ---- fetcher role: one lane per (scorer, slot) pops task pairs from the queue and stages their inputs ----
__device__ void fetcher_loop(const DevBatch& b, const DevParams& prm, const LisGlobals& g, uint8_t* scorer_smem) {
  const unsigned lane = lane_id();
  const SwScore sc{prm.match, prm.mismatch, prm.score_N, prm.gap_open, prm.gap_ext, prm.one};
  const bool mine = lane < 2u * kScorerWarps;
  ScSlot* sl = (ScSlot*)(scorer_smem + (size_t)(lane >> 1) * kScorerSmem + 2 * kPairProfWords * 4) + (lane & 1u);
  uint32_t eph = 1, h = 0;                       // parity of the "empty" phase to wait for: a fresh mbarrier counts as released
  bool have = false, done = !mine;
  const uint32_t qi = lane & 1u;                 // slot 0 of every scorer is fed from the express queue, slot 1 from the bulk queue
  QSlot* ring = g.ring + (size_t)qi * kQueueCap;
  uint32_t* q_head = g.q_head + qi * 16;
  for (;;) {
    bool progress = false;
    if (!done) {
      if (!have && mbar_try_wait(&sl->ebar, eph)) { eph ^= 1u; h = atomicAdd(q_head, 1u); have = true; }   // the scorer has released the slot
      if (have) {
        QSlot* qs = ring + (h & (kQueueCap - 1));
        if (ld_volatile_u32(&qs->seq) == h + 1u) {
          // (the entry and the task records are read past L1 -- ld.cg -- after the number has been seen: no L1 invalidation needed)
          const uint32_t planner = __ldcg(&qs->planner), ta = __ldcg(&qs->ta), tb = __ldcg(&qs->tb);
          st_volatile_u32(&qs->seq, h + kQueueCap);   // slot free for the next lap (after the payload was read)
          have = false; progress = true;
          sl->planner = planner; sl->ta = ta; sl->tb = tb;
          if (planner == kPoison) { mbar_arrive(&sl->bar); done = true; }
          else {
            const SwTask* tasks = carve_arena(g, planner).tasks;
            const uint4 da = __ldcg((const uint4*)(tasks + ta));
            const uint32_t ma = __ldcg(&tasks[ta].meta);
            const bool two = tb != kNoTask;
            uint4 db = make_uint4(0, 0, 0, 0); uint32_t mb = 0;
            if (two) { db = __ldcg((const uint4*)(tasks + tb)); mb = __ldcg(&tasks[tb].meta); }
            stage_pair(sl, da, ma, two, db, mb, b.seq04, sc, [&](const uint32_t& meta) { return g.parts[meta & 0xFFFFu].refseq; });
          }
        }
      }
    }
    if (__all_sync(kFull, done)) break;
    if (!__any_sync(kFull, progress)) __nanosleep(256);   // polling costs issue slots the scorers want; a quarter of a microsecond is 1 % of one alignment
  }
}

// ---- scorer role: take a staged task pair, score it with the packed kernel, report ----
template <bool kInstr>
__device__ void scorer_loop(const DevBatch& b, const DevParams& prm, const LisGlobals& g, uint8_t* sm, const uint32_t scorer) {
  const unsigned lane = lane_id();
  const SwScore sc{prm.match, prm.mismatch, prm.score_N, prm.gap_open, prm.gap_ext, prm.one};
  uint32_t* s_prof = (uint32_t*)sm;
  ScSlot* slots = (ScSlot*)(sm + 2 * kPairProfWords * 4);
  int32_t* rowH = g.score_rows + (size_t)scorer * 2 * g.row_cap; int32_t* rowF = rowH + g.row_cap;
  // identity of the query profile resident in each half: (q_abs, qlen | rev << 31, R)
  uint32_t keyq[2] = {0xFFFFFFFFu, 0xFFFFFFFFu}, keym[2] = {0xFFFFFFFFu, 0xFFFFFFFFu}; int keyR = 0;
  uint32_t par[2] = {0, 0}, exited = 0;
  unsigned long long n_pairs = 0, n_cells = 0, n_slow = 0, cy_wait = 0, cy_load = 0, cy_sw = 0, cy_pub = 0;
  const unsigned long long tl0 = kInstr ? tl_now() : 0ull;
  for (;;) {
    long long tq = lis_clock<kInstr>();
    const unsigned long long tla = kInstr ? tl_now() : 0ull;
    int k = -1;
    for (;;) {
      if (!(exited & 1u) && mbar_try_wait(&slots[0].bar, par[0])) { k = 0; break; }
      if (!(exited & 2u) && mbar_try_wait(&slots[1].bar, par[1])) { k = 1; break; }
      __nanosleep(128);
    }
    par[k] ^= 1u;
    ScSlot& S = slots[k];
    { const long long t2 = lis_clock<kInstr>(); cy_wait += (unsigned long long)(t2 - tq); tq = t2; }
    const unsigned long long tlb = kInstr ? tl_now() : 0ull;
    if (kInstr && g.dbg) tl_add(g.dbg + kTlBase + 0 * kTlBuckets, tl0, tla, tlb);
    const uint32_t planner = S.planner;
    if (planner == kPoison) { exited |= 1u << k; if (exited == 3u) break; continue; }
    const uint32_t ta = S.ta, tb = S.tb;
    const bool two = tb != kNoTask;
    const int32_t mA = (int32_t)S.mA, nA = (int32_t)S.nA, mB = (int32_t)S.mB, nB = (int32_t)S.nB;
    uint32_t sa, sb;
    score_slot(S, two, s_prof, keyq, keym, keyR, sc, b.seq04, [&](const uint32_t& meta) { return g.parts[meta & 0xFFFFu].refseq; }, rowH, rowF, g.row_cap,
               [&] { const long long t2 = lis_clock<kInstr>(); cy_load += (unsigned long long)(t2 - tq); tq = t2; }, [&] { ++n_slow; }, sa, sb);
    ++n_pairs; n_cells += (unsigned long long)nA * mA + (unsigned long long)nB * mB;
    if (SMR_EXP_SCORER_DELAY) exp_delay(tq, SMR_EXP_SCORER_DELAY);
    { const long long t2 = lis_clock<kInstr>(); cy_sw += (unsigned long long)(t2 - tq); tq = t2; }
    __syncwarp();
    if (lane == 0) {
      mbar_arrive(&S.ebar);                        // the fetcher may refill this slot
      SwTask* tasks = carve_arena(g, planner).tasks;
      st_volatile_u32(&tasks[ta].score, sa);
      if (two) st_volatile_u32(&tasks[tb].score, sb);
      atomicAdd(g.done + planner, two ? 2u : 1u);
    }
    __syncwarp();
    { const long long t2 = lis_clock<kInstr>(); cy_pub += (unsigned long long)(t2 - tq); }
    if (kInstr && g.dbg) tl_add(g.dbg + kTlBase + 1 * kTlBuckets, tl0, tlb, tl_now());
  }
  if (lane == 0) {
    atomicAdd(&b.counters[dcSpecCells], n_cells); atomicAdd(&b.counters[dcSpecPairs], n_pairs); atomicAdd(&b.counters[dcSlowPairs], n_slow);
    atomicAdd(&b.counters[dcScWait], cy_wait); atomicAdd(&b.counters[dcScLoad], cy_load); atomicAdd(&b.counters[dcScSw], cy_sw); atomicAdd(&b.counters[dcScPub], cy_pub);
  }
}

// The candidate kernel.  Planner warps drain the chunk's reads heaviest-first; each read is taken
// through every loaded (index, part) in --ref order -- the reference's index-major loop
// (processor.cpp:219-277) run read-major, with the KVDB carry-over of read.cpp:429-539 kept in
// DevBatch::state between parts (equivalent because reads are independent, SURVEY 8(b)).  Scorer warps
// run scorer_loop until the last planner has published the shutdown entries.
template <bool kInstr>
__global__ void __launch_bounds__(kLisWarpsPerCta * 32, kLisMinCtas)
lis_kernel(DevBatch b, DevParams prm, LisGlobals g) {
  extern __shared__ __align__(16) uint8_t lis_smem[];     // kLisSmemBytes: scorer warps first, then planner warps
  __shared__ uint32_t s_bin_start[kCostBins + 1];
  const unsigned lane = lane_id();
  const uint32_t wic = threadIdx.x >> 5;
  if (threadIdx.x == 0) {   // bins are drained from the heaviest (highest log2 cost) down
    uint32_t acc = 0;
    for (int k = 0; k < kCostBins; ++k) { s_bin_start[k] = acc; acc += b.bin_count[kCostBins - 1 - k]; }
    s_bin_start[kCostBins] = acc;
  }
  if (threadIdx.x < 2u * kScorerWarps) {   // the input slots' mbarriers and hand-back counters
    ScSlot* sl = (ScSlot*)(lis_smem + (size_t)(threadIdx.x >> 1) * kScorerSmem + 2 * kPairProfWords * 4) + (threadIdx.x & 1u);
    mbar_init(&sl->bar, 1); mbar_init(&sl->ebar, 1);
  }
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncthreads();
  if (wic < (uint32_t)kScorerWarps) { scorer_loop<kInstr>(b, prm, g, lis_smem + (size_t)wic * kScorerSmem, blockIdx.x * kScorerWarps + wic); return; }
  if (wic == (uint32_t)kScorerWarps) { fetcher_loop(b, prm, g, lis_smem); return; }
  const uint32_t pw = wic - kScorerWarps - kFetcherWarps, planner = blockIdx.x * kPlannerWarps + pw;
  PassEnv E;
  E.b = &b; E.prm = &prm; E.g = &g;
  E.ar = carve_arena(g, planner);
  E.planner = planner; E.submitted = 0; E.tl0 = kInstr ? tl_now() : 0ull;
  E.epoch_ptr = g.epochs + planner; E.epoch = *E.epoch_ptr;
  {
    uint8_t* sm = lis_smem + (size_t)kScorerWarps * kScorerSmem + (size_t)pw * kPlannerSmem;
    E.s_pairs = (unsigned long long*)sm; E.s_b = (uint32_t*)(sm + kPairsShared * 8); E.s_p = E.s_b + kPairsShared;
  }
  E.n_sw_calls = E.n_sw_cells = E.n_pos_entries = E.n_lis_calls = E.n_spec_calls = E.n_spec_cells = E.n_rounds_b = E.w1_cyc = E.w1_cnt = 0;
  for (int i = 0; i < 8; ++i) E.cyc[i] = 0;
  const uint32_t nwork = s_bin_start[kCostBins];
  unsigned long long t_max = 0, t_sum = 0; const long long t_k0 = lis_clock<kInstr>();
  unsigned long long dbg_loc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, t_busy_max = 0;
  const bool single = (prm.is_forward != 0) != (prm.is_reverse != 0);
  bool in_a = (int)(planner % 8u) < SMR_SCHED_A; (void)in_a;   // which region this planner draws from
  for (;;) {
    uint32_t wi = 0;
#if SMR_SCHED_A
    {   // two cursors over the heaviest-first schedule (see the comment at SMR_SCHED_A); a planner whose region is exhausted helps in the other
      const uint32_t m = nwork >> SMR_SPLIT_SHIFT;
      bool got = false;
#pragma unroll 1
      for (int tries = 0; tries < 2 && !got; ++tries) {
        uint32_t a = 0;
        if (lane == 0) a = atomicAdd(in_a ? g.work_next : g.work_next_b, 1u);
        a = __shfl_sync(kFull, a, 0);
        if (in_a) { if (a < m) { wi = a; got = true; } else in_a = false; }
        else { if (a < nwork - m) { wi = m + a; got = true; } else in_a = true; }
      }
      if (!got) break;
    }
#else
    if (lane == 0) wi = atomicAdd(g.work_next, 1u);
    wi = __shfl_sync(kFull, wi, 0);
    if (wi >= nwork) break;
#endif
    uint32_t k = 0;
    while (wi >= s_bin_start[k + 1]) ++k;
    const uint32_t r = b.bins[(size_t)(kCostBins - 1 - k) * b.cnt_stride + (wi - s_bin_start[k])];
    const long long t_read0 = lis_clock<kInstr>();
    unsigned long long cyc0[6], calls0 = E.n_sw_calls, spec0 = E.n_spec_calls, ra0 = E.n_spec_cells;
    for (int i = 0; i < 6; ++i) cyc0[i] = E.cyc[i];
    ReadCtx rc;
    rc.r = r; rc.seq_base = b.seq_off[r]; rc.len = b.seq_off[r + 1] - rc.seq_base;
    rc.hasn = b.has_n[r] != 0; rc.flags = 0; rc.ovf_slots = false;
    for (uint32_t p = 0; p < g.nparts && !rc.flags; ++p) {
      const DevIndex& ix = g.parts[p];
      const ReadState st = b.state[r];
      if (st.is_done) break;                                                                  // processor.cpp:120-126
      if (rc.len < ix.lnwin) continue;                                                        // processor.cpp:109-114
      E.nh = b.hit_cnt[(size_t)p * b.cnt_stride + (r - b.r0)];
      if (E.nh == 0) continue;   // no window hit in this part: traverse() changes nothing that is persisted
      E.hits = b.hits + hit_base(b, p, r);
      E.ix = &ix;
      rc.reversed = false; rc.form04 = false;                                                 // a fresh Read per index pass (processor.cpp:107)
      rc.vcls[0] = rc.vcls[1] = rc.vcls[2] = kVarFwd; rc.pass_n = 0;
      rc.hit_seeds = st.hit_seeds; rc.min_index = st.min_index; rc.max_index = st.max_index; rc.n_align = st.n_align;  // load_db (read.cpp:467-539)
      rc.max_SW_count = st.max_SW_count; rc.is_done = false; rc.is_hit = st.is_hit != 0; rc.is_new_hit = false;
      rc.best = prm.min_lis > 0 ? prm.min_lis : 0;                                            // Read::init (read.cpp:264-271)
      const int num_strands = single ? 1 : 2;                                                 // processor.cpp:130-146
      for (int count = 0; count < num_strands && !rc.is_done && !rc.flags; ++count) {
        if ((single && prm.is_reverse) || count == 1) rc.reversed = true;
        traverse_dev<kInstr>(E, rc, single || count == 1);
      }
      if (rc.flags) break;
      if (rc.is_new_hit && rc.n_align > 0 && lane == 0) {                                     // kvdb.put (processor.cpp:150-155)
        ReadState ns;
        ns.lastIndex = ix.index_num; ns.lastPart = ix.part; ns.hit_seeds = rc.hit_seeds; ns.min_index = rc.min_index; ns.max_index = rc.max_index;
        ns.n_align = rc.n_align; ns.max_SW_count = (uint16_t)rc.max_SW_count; ns.is_done = rc.is_done ? 1 : 0; ns.is_hit = rc.is_hit ? 1 : 0;
        b.state[r] = ns;
      }
      __syncwarp();
    }
    if (rc.ovf_slots) rc.flags |= kOvfSlots;
    if (rc.flags && lane == 0) atomicOr(&b.flags[r], rc.flags);
    { const unsigned long long dt = (unsigned long long)(lis_clock<kInstr>() - t_read0);
      if (dt > t_max) { t_max = dt; for (int i = 0; i < 6; ++i) dbg_loc[i] = E.cyc[i] - cyc0[i]; dbg_loc[6] = E.n_sw_calls - calls0; dbg_loc[7] = E.n_spec_calls - spec0; dbg_loc[8] = E.n_spec_cells - ra0; dbg_loc[9] = r; }
      const unsigned long long busy = dt - (E.cyc[4] - cyc0[4]);   // without the time spent waiting for the scorers
      t_busy_max = busy > t_busy_max ? busy : t_busy_max;
      t_sum += dt; }
    if (kInstr && g.dbg && lane == 0) { const unsigned long long k = (tl_now() - E.tl0) / kTlBucketNs; if (k < (unsigned long long)kTlBuckets) atomicAdd(g.dbg + kTlBase + 4 * kTlBuckets + k, 1ull); }
    __syncwarp();
  }
  if (kInstr && g.dbg) tl_add(g.dbg + kTlBase + 5 * kTlBuckets, E.tl0, E.tl0, tl_now());
  if (lane == 0) {
    *E.epoch_ptr = E.epoch;
    atomicAdd(&b.counters[dcSwCalls], E.n_sw_calls); atomicAdd(&b.counters[dcSwCells], E.n_sw_cells);
    atomicAdd(&b.counters[dcPosEntries], E.n_pos_entries); atomicAdd(&b.counters[dcLisCalls], E.n_lis_calls);
    atomicAdd(&b.counters[dcSpecCalls], E.n_spec_calls); atomicAdd(&b.counters[dcRoundsA], E.n_spec_cells); atomicAdd(&b.counters[dcRoundsB], E.n_rounds_b);
    atomicAdd(&b.counters[dcW1Cyc], E.w1_cyc); atomicAdd(&b.counters[dcW1Cnt], E.w1_cnt); atomicMax(&b.counters[dcMaxReadBusy], t_busy_max);
    for (int i = 0; i < 6; ++i) atomicAdd(&b.counters[dcCycVote + i], E.cyc[i]);
    if (atomicMax(&b.counters[dcMaxReadCycles], t_max) < t_max && g.dbg) { g.dbg[0] = t_max; for (int i = 0; i < 10; ++i) g.dbg[1 + i] = dbg_loc[i]; }
    atomicAdd(&b.counters[dcSumReadCycles], t_sum);
    atomicMax(&b.counters[dcLisKernelCycles], (unsigned long long)(lis_clock<kInstr>() - t_k0));
    // the last planner out shuts the scorers down: one entry each
    const uint32_t nplanners = gridDim.x * kPlannerWarps, nscorers = gridDim.x * kScorerWarps;   // one shutdown entry per fetcher lane of each queue
    if (atomicAdd(g.planners_done, 1u) + 1u == nplanners) {
      for (uint32_t qi = 0; qi < 2; ++qi) {
        QSlot* ring = g.ring + (size_t)qi * kQueueCap;
        const uint32_t base = atomicAdd(g.q_tail + qi * 16, nscorers);
        for (uint32_t i = 0; i < nscorers; ++i) {
          const uint32_t idx = base + i;
          QSlot* sl = ring + (idx & (kQueueCap - 1));
          while (ld_volatile_u32(&sl->seq) != idx) __nanosleep(64);
          sl->planner = kPoison; sl->ta = kNoTask; sl->tb = kNoTask;
          __threadfence();
          st_volatile_u32(&sl->seq, idx + 1);
        }
      }
    }
  }
}

// unit-test kernel (smr_debug_sw_tasks): the scorer path of the candidate kernel on explicit task pairs.  One warp per chain of
// `chain` consecutive pairs, scored in order with one profile cache and the two input slots taken in turn, as one scorer warp does;
// lane 0 stages each pair as the fetcher does.  tasks: ref_abs into tcat, q_abs into qcat, meta = minus strand << 16.
// pairs[2k], pairs[2k + 1]: the task indices of pair k (B = kNoTask: none).  scores[t]: what the scorer publishes for task t;
// path[k]: 1 = packed 16-bit pass, 0 = s32 fallback.  rows: 2 * row_cap ints of fallback scratch per warp.
constexpr int kSwDebugWarps = 4;
__global__ void __launch_bounds__(kSwDebugWarps * 32)
sw_tasks_debug_kernel(const uint8_t* qcat, const uint8_t* tcat, const SwTask* tasks, const uint32_t* pairs, uint32_t npairs, uint32_t chain,
                      DevParams prm, int32_t* rows, uint32_t row_cap, uint32_t* scores, uint8_t* path) {
  extern __shared__ __align__(16) uint8_t dbg_smem[];   // kSwDebugWarps * kScorerSmem: the scorer layout, profiles then slots
  const unsigned lane = lane_id();
  const uint32_t w = threadIdx.x >> 5, warp = blockIdx.x * kSwDebugWarps + w;
  uint8_t* sm = dbg_smem + (size_t)w * kScorerSmem;
  uint32_t* s_prof = (uint32_t*)sm;
  ScSlot* slots = (ScSlot*)(sm + 2 * kPairProfWords * 4);
  if (lane < 2u) mbar_init(&slots[lane].bar, 1);
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  __syncwarp();
  const SwScore sc{prm.match, prm.mismatch, prm.score_N, prm.gap_open, prm.gap_ext, prm.one};
  int32_t* rowH = rows + (size_t)warp * 2 * row_cap; int32_t* rowF = rowH + row_cap;
  const auto ref_of = [&](const uint32_t&) { return tcat; };
  // identity of the query profile resident in each half: (q_abs, qlen | rev << 31, R)
  uint32_t keyq[2] = {0xFFFFFFFFu, 0xFFFFFFFFu}, keym[2] = {0xFFFFFFFFu, 0xFFFFFFFFu}; int keyR = 0;
  uint32_t par[2] = {0, 0};
  const uint64_t k0 = (uint64_t)warp * chain, k1 = min(k0 + chain, (uint64_t)npairs);
  for (uint64_t k = k0; k < k1; ++k) {
    const int s = (int)((k - k0) & 1u);
    ScSlot* sl = slots + s;
    const uint32_t ta = pairs[2 * k], tb = pairs[2 * k + 1];
    const bool two = tb != kNoTask;
    // the slot's previous pair was read (and its sentinels written) through the generic proxy; the bulk copies write through the async one
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) {
      const uint4 da = *(const uint4*)(tasks + ta);
      const uint32_t ma = tasks[ta].meta;
      uint4 db = make_uint4(0, 0, 0, 0); uint32_t mb = 0;
      if (two) { db = *(const uint4*)(tasks + tb); mb = tasks[tb].meta; }
      sl->planner = 0; sl->ta = ta; sl->tb = tb;
      stage_pair(sl, da, ma, two, db, mb, qcat, sc, ref_of);
    }
    while (!mbar_try_wait(&sl->bar, par[s])) {}
    par[s] ^= 1u;
    uint32_t sa, sb;
    const bool packed = score_slot(*sl, two, s_prof, keyq, keym, keyR, sc, qcat, ref_of, rowH, rowF, row_cap, [] {}, [] {}, sa, sb);
    __syncwarp();
    if (lane == 0) { scores[ta] = sa; if (two) scores[tb] = sb; path[k] = packed ? 1 : 0; }
  }
}

// queue / counter reset before every lis_kernel launch
__global__ void lis_reset_kernel(LisGlobals g, uint32_t nplanners) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < kQueueCap) { QSlot s; s.seq = i; s.planner = 0; s.ta = 0; s.tb = 0; g.ring[i] = s; g.ring[kQueueCap + i] = s; }
  if (i < nplanners) g.done[i] = 0;
  if (i == 0) { g.q_head[0] = 0; g.q_head[16] = 0; g.q_tail[0] = 0; g.q_tail[16] = 0; *g.planners_done = 0; }
}

}  // namespace smr
