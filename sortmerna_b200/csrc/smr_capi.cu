// C ABI of libsmr_b200.so (include/smr_b200.h): context, index residency, batch driver.
// Host side of the seam that replaces align() (src/sortmerna/processor.cpp:173-285).
#include "../../include/smr_b200.h"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "smr_decode.cuh"
#include "smr_inflate.cuh"
#include "smr_build.h"
#include "smr_build_dev.cuh"
#include "smr_final.cuh"
#include "smr_index.h"

using namespace smr;

namespace {

struct Part {
  DevIndex d{};
  std::vector<void*> owned;   // device allocations
  size_t bytes = 0, n_nodes = 0, n_entries = 0, n_ids = 0, n_pos = 0, n_refseq = 0;
};

struct DevBuf {
  void* p = nullptr; size_t cap = 0;
};
struct PinBuf {   // grow-only pinned host staging (page-locked once; pageable vectors cost a page-fault pass + a bounce copy per batch)
  void* p = nullptr; size_t cap = 0;
};

}  // namespace

struct smr_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  smr_params prm{};
  bool have_params = false;
  std::vector<Part> parts;
  uint32_t n_index_files = 0;
  int sm_count = 148;
  uint32_t chunk_reads = 1u << 20;
  uint32_t need_slots = 0;       // set with SMR_ERR_CAPACITY in all-alignments mode: the stride the batch needs
  uint32_t all_slots = 16;       // stride of the result layout when num_alignments == 0 (smr_set_aln_slots)
  uint32_t lis_ctas_per_sm = kLisMinCtas;   // persistent CTAs of the candidate kernel per SM (matches its __launch_bounds__)

  // resident batch
  uint32_t nreads = 0; uint64_t total_nt = 0; uint32_t max_len = 0;
  std::vector<uint8_t> h_seq; std::vector<uint64_t> h_off;    // host copy (scratch-overflow retries)
  std::vector<uint32_t> off32;                                // 32-bit read offsets of the resident batch
  DevBuf seq04, seq_off, pk03, pk03alt, pk_off, has_n, hit_cnt, flags, state, hit_db, aln_work, out_aln;
  DevBuf hits, cost, bins, scalars, counters, cigar_pool, parts_dev;
  size_t hits_stride = 0; uint32_t cnt_stride = 0;
  DevBuf lis_arena, lis_epochs, lis_queue, lis_done, lis_rows, lis_dbg, final_arena, lane_hits, tb_arena, tb_jobs, aln_stats;
  smr_aln_stats* host_stats = nullptr;   // optional output of the report arithmetic
  PinBuf h_state, h_flags, h_hitdb, h_outaln, h_stats, h_cigar, h_off32, h_pkoff;
  std::vector<uint64_t> h_coff;
  DevBuf d_text, d_cnt, d_scal, d_nl, d_hdr, d_sb, d_rec, d_spos, d_hdroff, scan_sums;   // input decode (smr_decode.cuh)
  DevBuf seed_ctr, d_gz, d_cand, d_res, d_sym, d_win, d_ids, d_off, d_cnt64, d_moff, d_mem, d_poff, d_plen, d_pcrc;   // gz inflate (smr_inflate.cuh)
  uint64_t text_bytes = 0;          // size of the text behind the resident batch (smr_upload_fastx / _gz)
  uint32_t inf_spans = 0, inf_candidates = 0; double t_inflate = 0;
  bool device_only_reads = false;   // the resident batch was decoded on the device: no host copy of the sequences yet
  double t_decode = 0;
  uint32_t tb_threads = 0, tb_cap_w = 0, tb_cap_cig = 0; size_t tb_cap_dir = 0, tb_stride = 0;
  uint32_t lis_warps = 0, final_warps = 0;
  size_t lis_stride = 0, final_stride = 0;
  uint32_t hist_cap = 0, cand_cap = 0, pair_cap = 0, row_cap = 0, pall_cap = 0, task_cap = 0, cap_w = 0, cap_cig = 0; size_t cap_dir = 0;
  uint32_t lis_ctas = 0;
  uint32_t lane_hits_cap = 0, lane_hits_warps = 0;
  uint64_t cigar_cap_dev = 0;
  uint32_t scale = 1;         // scratch scale of the current run (1 = fast path)
  bool instr = false;         // smr_set_instrumentation: seed kernel counts windows / lists / entries, candidate kernel accounts its phases (clock64)
  uint64_t flag_hist[6] = {0, 0, 0, 0, 0, 0};  // overflow causes seen so far (seed lane / seed region / pairs / trace / cigar / error)
  // timings
  std::vector<cudaEvent_t> ev;
  double t_total = 0, t_seed = 0, t_lis = 0, t_final = 0, t_h2d = 0, t_d2h = 0; uint64_t n_launch = 0;
};

namespace {

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) {                                                                       \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                               \
      return SMR_ERR_CUDA;                                                                         \
    }                                                                                              \
  } while (0)

// alignment slots per read in every flat result array: num_alignments, or the stride set for "all alignments" (0)
uint32_t slots_of(const smr_ctx* ctx) { return ctx->prm.num_alignments > 0 ? (uint32_t)ctx->prm.num_alignments : std::max(1u, ctx->all_slots); }

int ensure(smr_ctx* ctx, DevBuf& b, size_t bytes) {
  if (bytes <= b.cap && b.p) return SMR_OK;
  if (b.p) { cudaFree(b.p); b.p = nullptr; b.cap = 0; }
  size_t want = bytes + bytes / 8 + 256;
  CK(cudaMalloc(&b.p, want));
  b.cap = want;
  return SMR_OK;
}
void release(DevBuf& b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }
int ensure_pinned(smr_ctx* ctx, PinBuf& b, size_t bytes) {
  if (bytes <= b.cap && b.p) return SMR_OK;
  if (b.p) { cudaFreeHost(b.p); b.p = nullptr; b.cap = 0; }
  const size_t want = bytes + bytes / 8 + 256;
  CK(cudaHostAlloc(&b.p, want, cudaHostAllocDefault));
  b.cap = want;
  return SMR_OK;
}
void release(PinBuf& b) { if (b.p) cudaFreeHost(b.p); b.p = nullptr; b.cap = 0; }

template <class T>
int upload_vec(smr_ctx* ctx, Part& pt, const std::vector<T>& v, const T** out) {
  void* d = nullptr;
  size_t bytes = v.size() * sizeof(T) + 64;   // the seed kernel reads whole aligned groups of four list entries
  CK(cudaMalloc(&d, bytes));
  CK(cudaMemset(d, 0, bytes));
  if (!v.empty()) CK(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  pt.owned.push_back(d); pt.bytes += bytes;
  *out = (const T*)d;
  return SMR_OK;
}


// ---------------------------------------------------------------------------------------------------------------------
// index build on the device (smr_build_dev.cuh): orchestration of one part
// ---------------------------------------------------------------------------------------------------------------------
struct TempPool {   // device scratch of one build, freed on return
  std::vector<void*> v;
  ~TempPool() { for (void* p : v) cudaFree(p); }
  template <class T> cudaError_t get(T** out, size_t n) { void* p = nullptr; cudaError_t e = cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)); if (e == cudaSuccess) v.push_back(p); *out = (T*)p; return e; }
};

int build_part_device(smr_ctx* ctx, const std::vector<RefRecord>& recs, const std::vector<size_t>& members, const BuildOptions& opt, Part& pt) {
  BuildGeom g{};
  g.L = opt.lnwin; g.half = g.L / 2; g.pread = g.L + 1; g.interval = opt.interval; g.max_pos = opt.max_pos; g.burst_depth = g.pread - g.half - 3;
  g.nseq = (uint32_t)members.size();
  const uint32_t list_bits = 2 * g.half + 1, key_bits = list_bits + 2 * g.burst_depth;
  if (key_bits > 64 || 2 * g.pread > 62 || 2 * (g.half + 1) > 32) { ctx->err = "seed length too large for the device builder"; return SMR_ERR_UNSUPPORTED; }
  // host: concatenated builder codes + 0..4 codes, offsets, first window of every sequence
  std::vector<uint64_t> soff(g.nseq + 1, 0);
  std::vector<uint32_t> wstart(g.nseq + 1, 0);
  uint64_t total_win = 0;
  for (uint32_t k = 0; k < g.nseq; ++k) {
    const size_t len = recs[members[k]].seq.size();
    soff[k + 1] = soff[k] + len;
    total_win += (len - g.pread + g.interval) / g.interval;
    if (total_win >= (1ull << 31)) { ctx->err = "more than 2^31 windows in one index part"; return SMR_ERR_UNSUPPORTED; }
    wstart[k + 1] = (uint32_t)total_win;
  }
  if (soff[g.nseq] >= 0xFFFFFFFFull) { ctx->err = "reference part larger than 4 GB"; return SMR_ERR_UNSUPPORTED; }
  g.nwin = (uint32_t)total_win;
  std::vector<uint8_t> codes(soff[g.nseq]), c04(soff[g.nseq] + 64, 4);
  for (uint32_t k = 0; k < g.nseq; ++k) {
    const RefRecord& r = recs[members[k]];
    memcpy(codes.data() + soff[k], r.seq.data(), r.seq.size());
    memcpy(c04.data() + soff[k], r.seq04.data(), r.seq04.size());
  }
  std::vector<uint32_t> roff(g.nseq + 1);
  for (uint32_t k = 0; k <= g.nseq; ++k) roff[k] = (uint32_t)soff[k];
  TempPool tp;
  cudaStream_t st = ctx->stream;
  const uint32_t n = g.nwin;
  const unsigned tb = 256, gw = (n + tb - 1) / tb;
  uint8_t* d_codes; uint64_t* d_soff; uint32_t* d_wstart;
  CK(tp.get(&d_codes, codes.size() + 64)); CK(tp.get(&d_soff, soff.size())); CK(tp.get(&d_wstart, wstart.size()));
  CK(cudaMemcpyAsync(d_codes, codes.data(), codes.size(), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_soff, soff.data(), soff.size() * 8, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(d_wstart, wstart.data(), wstart.size() * 4, cudaMemcpyHostToDevice, st));
  uint64_t *keyA, *keyB; uint32_t *valA, *valB, *u0, *u1, *u2, *u3, *win_id;
  CK(tp.get(&keyA, n)); CK(tp.get(&keyB, n)); CK(tp.get(&valA, n)); CK(tp.get(&valB, n));
  CK(tp.get(&u0, n)); CK(tp.get(&u1, n)); CK(tp.get(&u2, n)); CK(tp.get(&u3, n)); CK(tp.get(&win_id, n));
  // cub scratch, sized for the largest call (entries: at most 2n)
  size_t cub_bytes = 0, need = 0;
  cub::DeviceRadixSort::SortPairs(nullptr, need, (uint64_t*)nullptr, (uint64_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, 2 * (size_t)n, 0, 64, st); cub_bytes = std::max(cub_bytes, need);
  cub::DeviceScan::InclusiveSum(nullptr, need, (uint32_t*)nullptr, (uint32_t*)nullptr, 2 * (size_t)n, st); cub_bytes = std::max(cub_bytes, need);
  cub::DeviceScan::InclusiveScan(nullptr, need, (uint32_t*)nullptr, (uint32_t*)nullptr, cuda::maximum<uint32_t>{}, 2 * (size_t)n, st); cub_bytes = std::max(cub_bytes, need);
  uint8_t* d_cub; CK(tp.get(&d_cub, cub_bytes + 256));
  // 1. windows sorted by value (stable: equal values keep scan order)
  bld_windows_kernel<<<gw, tb, 0, st>>>(d_codes, d_soff, d_wstart, g, keyA, valA);
  CK(cudaGetLastError());
  need = cub_bytes; CK(cub::DeviceRadixSort::SortPairs(d_cub, need, keyA, keyB, valA, valB, (size_t)n, 0, (int)(2 * g.pread), st));
  // 2. distinct (L+1)-mers, ids of the L-mers
  bld_heads_kernel<<<gw, tb, 0, st>>>(keyB, n, u0, u1);
  CK(cudaGetLastError());
  need = cub_bytes; CK(cub::DeviceScan::InclusiveSum(d_cub, need, u0, u2, (size_t)n, st));
  need = cub_bytes; CK(cub::DeviceScan::InclusiveSum(d_cub, need, u1, u3, (size_t)n, st));
  uint32_t nent = 0, nids = 0;
  CK(cudaMemcpyAsync(&nent, u2 + (n - 1), 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(&nids, u3 + (n - 1), 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const uint32_t E = 2 * nent;
  uint32_t *e_list, *e_pref, *e_text, *e_id, *e_arr, *e_tpar; uint8_t* e_leaf;
  CK(tp.get(&e_list, E)); CK(tp.get(&e_pref, E)); CK(tp.get(&e_text, E)); CK(tp.get(&e_id, E)); CK(tp.get(&e_arr, E)); CK(tp.get(&e_tpar, E)); CK(tp.get(&e_leaf, E));
  CK(cudaMemsetAsync(e_tpar, 0, (size_t)E * 4, st)); CK(cudaMemsetAsync(e_leaf, 0, E, st));
  bld_entries_kernel<<<gw, tb, 0, st>>>(keyB, valB, u0, u2, u3, g, nent, win_id, e_list, e_pref, e_text, e_id, e_arr);
  CK(cudaGetLastError());
  // 3. positions (persistent arrays)
  auto keep_alloc = [&](void** out, size_t bytes) -> cudaError_t { cudaError_t e = cudaMalloc(out, bytes + 64); if (e == cudaSuccess) { pt.owned.push_back(*out); pt.bytes += bytes + 64; e = cudaMemsetAsync(*out, 0, bytes + 64, st); } return e; };
  bld_poskeys_kernel<<<gw, tb, 0, st>>>(win_id, n, keyA);
  CK(cudaGetLastError());
  need = cub_bytes; CK(cub::DeviceRadixSort::SortKeys(d_cub, need, keyA, keyB, (size_t)n, 0, 64, st));
  bld_posflag_kernel<<<gw, tb, 0, st>>>(keyB, n, u0);
  CK(cudaGetLastError());
  need = cub_bytes; CK(cub::DeviceScan::InclusiveScan(d_cub, need, u0, u1, cuda::maximum<uint32_t>{}, (size_t)n, st));
  bld_poskeep_kernel<<<gw, tb, 0, st>>>(u1, n, g.max_pos, u2);
  CK(cudaGetLastError());
  need = cub_bytes; CK(cub::DeviceScan::InclusiveSum(d_cub, need, u2, u3, (size_t)n, st));
  uint32_t npos = 0;
  CK(cudaMemcpyAsync(&npos, u3 + (n - 1), 4, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  void *p_posoff = nullptr, *p_pos = nullptr, *p_flist = nullptr, *p_flookup = nullptr, *p_ref = nullptr, *p_roff = nullptr;
  CK(keep_alloc(&p_posoff, ((size_t)nids + 1) * 4)); CK(keep_alloc(&p_pos, (size_t)npos * 8));
  bld_poswrite_kernel<<<gw, tb, 0, st>>>(keyB, u1, u2, u3, d_wstart, g, nids, (uint32_t*)p_posoff, (uint2*)p_pos);
  CK(cudaGetLastError());
  // 4. burst-trie order of the entries: first occurrence order, then one stable sort + one decision pass per level
  const unsigned ge = (E + tb - 1) / tb;
  uint64_t *ekA, *ekB; uint32_t *pA, *pB;
  CK(tp.get(&ekA, E)); CK(tp.get(&ekB, E)); CK(tp.get(&pA, E)); CK(tp.get(&pB, E));
  bld_arrkey_kernel<<<ge, tb, 0, st>>>(e_arr, E, ekA, pA);
  CK(cudaGetLastError());
  need = cub_bytes; CK(cub::DeviceRadixSort::SortPairs(d_cub, need, ekA, ekB, pA, pB, (size_t)E, 0, 32, st));
  for (uint32_t d = 1; d <= g.burst_depth; ++d) {
    bld_levelkey_kernel<<<ge, tb, 0, st>>>(pB, e_list, e_pref, e_leaf, E, d, g.burst_depth, ekA, pA);
    CK(cudaGetLastError());
    need = cub_bytes; CK(cub::DeviceRadixSort::SortPairs(d_cub, need, ekA, ekB, pA, pB, (size_t)E, 0, (int)key_bits, st));
    if (d < g.burst_depth) { bld_level_kernel<<<ge, tb, 0, st>>>(ekB, pB, E, d, e_arr, e_tpar, e_leaf); CK(cudaGetLastError()); }
  }
  // 5. the lists and their lookup rows
  const size_t nk = (size_t)1 << (2 * g.half);
  CK(keep_alloc(&p_flist, (size_t)E * 8)); CK(keep_alloc(&p_flookup, nk * 16));
  bld_flist_kernel<<<ge, tb, 0, st>>>(pB, e_list, e_text, e_id, E, (uint2*)p_flist, (uint32_t*)p_flookup, 0);
  bld_flist_kernel<<<ge, tb, 0, st>>>(pB, e_list, e_text, e_id, E, (uint2*)p_flist, (uint32_t*)p_flookup, 1);
  CK(cudaGetLastError());
  // 6. references for the Smith-Waterman side
  CK(keep_alloc(&p_ref, c04.size())); CK(keep_alloc(&p_roff, roff.size() * 4));
  CK(cudaMemcpyAsync(p_ref, c04.data(), c04.size(), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(p_roff, roff.data(), roff.size() * 4, cudaMemcpyHostToDevice, st));
  CK(cudaStreamSynchronize(st));
  pt.d.lnwin = g.L; pt.d.partialwin = g.half; pt.d.nref = g.nseq; pt.d.nids = nids;
  pt.d.flookup = (const uint4*)p_flookup; pt.d.flist = (const uint2*)p_flist; pt.d.pos_off = (const uint32_t*)p_posoff; pt.d.pos = (const uint2*)p_pos;
  pt.d.refseq = (const uint8_t*)p_ref; pt.d.ref_off = (const uint32_t*)p_roff;
  pt.n_entries = E; pt.n_ids = nids; pt.n_pos = npos; pt.n_refseq = c04.size();
  return SMR_OK;
}

DevParams to_dev(const smr_params& p) {
  DevParams d;
  d.match = p.match; d.mismatch = p.mismatch; d.score_N = p.score_N; d.gap_open = p.gap_open; d.gap_ext = p.gap_ext;
  d.num_seeds = p.num_seeds; d.min_lis = p.min_lis; d.edges = p.edges; d.edges_is_percent = p.edges_is_percent;
  d.num_alignments = p.num_alignments; d.is_best = p.is_best; d.is_forward = p.is_forward; d.is_reverse = p.is_reverse;
  d.is_full_search = p.is_full_search;
  d.one = 1;
  return d;
}

uint32_t pow2_ge(uint32_t v) { uint32_t p = 1; while (p < v) p <<= 1; return p; }

cudaEvent_t get_event(smr_ctx* ctx, size_t i) {
  while (ctx->ev.size() <= i) { cudaEvent_t e; cudaEventCreate(&e); ctx->ev.push_back(e); }
  return ctx->ev[i];
}

// scalars block layout (u32): [0]=work_n [1]=lis work_next [2]=final work_next [3]=lis work_next of the second cursor ; cigar_used (u64) at byte 16 ; task queue cursors at 128..
struct Scalars { uint32_t* work_n; uint32_t* lis_next; uint32_t* fin_next; uint32_t* lis_next_b; unsigned long long* cigar_used; uint32_t* q_head; uint32_t* q_tail; uint32_t* planners_done; };
Scalars scalars_of(smr_ctx* ctx) {
  uint8_t* p = (uint8_t*)ctx->scalars.p;
  return Scalars{(uint32_t*)p, (uint32_t*)(p + 4), (uint32_t*)(p + 8), (uint32_t*)(p + 12), (unsigned long long*)(p + 16), (uint32_t*)(p + 128), (uint32_t*)(p + 256), (uint32_t*)(p + 384)};
}

int setup_arenas(smr_ctx* ctx) {
  uint32_t max_nref = 1;
  for (auto& pt : ctx->parts) max_nref = std::max(max_nref, pt.d.nref);
  ctx->hist_cap = max_nref;
  ctx->cand_cap = std::max(64u, max_nref);
  ctx->pair_cap = pow2_ge(4096u * ctx->scale);
  ctx->task_cap = 2 * ctx->pair_cap;
  // SW windows are at most read length + 2 * edges columns (alignment.cpp:272-357; edges may be a percentage of the read)
  const uint32_t edges = ctx->prm.edges_is_percent ? (uint32_t)((ctx->prm.edges / 100.0) * (double)ctx->max_len) : (uint32_t)std::max(0, ctx->prm.edges);
  ctx->row_cap = ctx->max_len + 2 * edges + 2 * 64 + 64;
  // planner and scorer warps wait for each other: EVERY CTA of the grid must be resident at once
  int occ = 0;
  CK(cudaFuncSetAttribute(lis_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kLisSmemBytes));
  CK(cudaFuncSetAttribute(lis_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kLisSmemBytes));
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lis_kernel<true>, kLisWarpsPerCta * 32, kLisSmemBytes));   // (same launch bounds and shared memory for both)
  if (occ < 1) { ctx->err = "lis_kernel does not fit on an SM"; return SMR_ERR_CUDA; }
  ctx->lis_ctas = (uint32_t)ctx->sm_count * std::min<uint32_t>(ctx->lis_ctas_per_sm, (uint32_t)occ);
  ctx->lis_warps = ctx->lis_ctas * kPlannerWarps;   // planner warps (each owns an arena)
  ctx->pall_cap = 32768u * ctx->scale;
  ctx->lis_stride = lis_arena_bytes(ctx->hist_cap, ctx->cand_cap, ctx->pair_cap, ctx->task_cap, ctx->pall_cap);
  // keep the arena total under ~16 GB (of 180): fewer persistent CTAs for huge reference sets
  const size_t budget = (size_t)16 << 30;
  while (ctx->lis_ctas > 16 && ctx->lis_stride * ctx->lis_warps > budget) { ctx->lis_ctas /= 2; ctx->lis_warps = ctx->lis_ctas * kPlannerWarps; }
  if (int rc = ensure(ctx, ctx->lis_arena, ctx->lis_stride * ctx->lis_warps)) return rc;
  if (int rc = ensure(ctx, ctx->lis_epochs, (size_t)ctx->lis_warps * 4)) return rc;
  if (int rc = ensure(ctx, ctx->lis_queue, (size_t)2 * kQueueCap * sizeof(QSlot) + 64)) return rc;
  if (int rc = ensure(ctx, ctx->lis_done, (size_t)ctx->lis_warps * 4 + 64)) return rc;
  const size_t dbg_bytes = (size_t)(kTlBase + kTlRows * kTlBuckets) * 8;
  if (int rc = ensure(ctx, ctx->lis_dbg, dbg_bytes)) return rc;
  CK(cudaMemsetAsync(ctx->lis_dbg.p, 0, dbg_bytes, ctx->stream));
  if (int rc = ensure(ctx, ctx->lis_rows, (size_t)ctx->lis_ctas * kScorerWarps * 2 * ctx->row_cap * 4)) return rc;
  // histogram epochs start at 0 over a zeroed histogram (every run: the arena layout depends on the scale of the run)
  CK(cudaMemset2DAsync(ctx->lis_arena.p, ctx->lis_stride, 0, lis_arena_zero_bytes(ctx->hist_cap), ctx->lis_warps, ctx->stream));   // votes + bitmaps only
  CK(cudaMemsetAsync(ctx->lis_epochs.p, 0, (size_t)ctx->lis_warps * 4, ctx->stream));
  ctx->cap_w = 2 * 256 * ctx->scale + 8;          // band widths up to 256*scale
  ctx->cap_cig = 2 * (ctx->max_len + 64) + 16;
  ctx->cap_dir = (size_t)65536 * ctx->scale + (size_t)ctx->max_len * 9 * 3 + 64;
  ctx->final_warps = (uint32_t)ctx->sm_count * kFinalCtasPerSm * kFinalWarpsPerCta;
  ctx->final_stride = final_arena_bytes(ctx->cap_w, ctx->cap_cig, ctx->row_cap, ctx->cap_dir);
  while (ctx->final_warps > 64 && ctx->final_stride * ctx->final_warps > budget) ctx->final_warps /= 2;
  if (int rc = ensure(ctx, ctx->final_arena, ctx->final_stride * ctx->final_warps)) return rc;
  // traceback stage: one thread per alignment, 1024 threads per SM
  ctx->tb_threads = (uint32_t)ctx->sm_count * 1024u;
  ctx->tb_cap_w = 2 * 32 * ctx->scale + 8;                       // band widths up to 32*scale
  ctx->tb_cap_cig = 128 * ctx->scale;
  ctx->tb_cap_dir = (size_t)32768 * ctx->scale;                  // (2*band+1) * readLen * 3 bytes: band 32 at 150 nt
  ctx->tb_stride = ((size_t)ctx->tb_cap_w * 12 + (size_t)ctx->tb_cap_cig * 4 + ctx->tb_cap_dir + 255) & ~(size_t)255;
  while (ctx->tb_threads > 4096 && ctx->tb_stride * ctx->tb_threads > budget) ctx->tb_threads /= 2;
  if (int rc = ensure(ctx, ctx->tb_arena, ctx->tb_stride * ctx->tb_threads)) return rc;
  ctx->lane_hits_cap = kLaneHitCap * ctx->scale;
  ctx->lane_hits_warps = ctx->scale == 1 ? (uint32_t)ctx->sm_count * kSeedCtasPerSm * kSeedWarpsPerCta : 1024u;
  if (int rc = ensure(ctx, ctx->lane_hits, (size_t)ctx->lane_hits_warps * ctx->lane_hits_cap * 32 * 4)) return rc;
  return SMR_OK;
}

int finish_upload(smr_ctx* ctx, uint32_t nreads, uint64_t w);

int upload_batch_impl(smr_ctx* ctx, const uint8_t* seq_cat, const uint64_t* seq_off, uint32_t nreads, bool keep_host) {
  if (nreads == 0) { ctx->nreads = 0; return SMR_OK; }
  const uint64_t total = seq_off[nreads] - seq_off[0];
  if (total >= 0xF0000000ull) { ctx->err = "batch larger than 2^32 nucleotides: split it"; return SMR_ERR_ARG; }
  cudaEvent_t e0 = get_event(ctx, 0), e1 = get_event(ctx, 1);
  CK(cudaEventRecord(e0, ctx->stream));
  std::vector<uint32_t>& off32 = ctx->off32; off32.resize(nreads + 1);
  { int prc; if ((prc = ensure_pinned(ctx, ctx->h_pkoff, (size_t)(nreads + 1) * 4))) return prc; if ((prc = ensure_pinned(ctx, ctx->h_off32, (size_t)(nreads + 1) * 4))) return prc; }
  uint32_t* pkoff = (uint32_t*)ctx->h_pkoff.p;
  uint32_t max_len = 0; uint64_t w = 0;
  for (uint32_t r = 0; r <= nreads; ++r) {
    off32[r] = (uint32_t)(seq_off[r] - seq_off[0]);
    pkoff[r] = (uint32_t)w;
    if (r < nreads) {
      const uint64_t len = seq_off[r + 1] - seq_off[r];
      max_len = std::max<uint32_t>(max_len, (uint32_t)len);
      w += (len + 15) / 16 + 2;     // +2 padding words: window_fwd reads three consecutive words
    }
  }
  if (w >= 0xFFFFFFFFull) { ctx->err = "batch too large"; return SMR_ERR_ARG; }
  ctx->nreads = nreads; ctx->total_nt = total; ctx->max_len = max_len;
  if (keep_host) {
    ctx->h_seq.assign(seq_cat + seq_off[0], seq_cat + seq_off[nreads]);
    ctx->h_off.resize(nreads + 1);
    for (uint32_t r = 0; r <= nreads; ++r) ctx->h_off[r] = seq_off[r] - seq_off[0];
  }
  const uint32_t slots = slots_of(ctx);
  int rc;
  if ((rc = ensure(ctx, ctx->seq04, total + 64))) return rc;
  if ((rc = ensure(ctx, ctx->seq_off, (size_t)(nreads + 1) * 4))) return rc;
  if ((rc = ensure(ctx, ctx->pk_off, (size_t)(nreads + 1) * 4))) return rc;
  CK(cudaMemcpyAsync(ctx->seq04.p, seq_cat + seq_off[0], total, cudaMemcpyHostToDevice, ctx->stream));
  memcpy(ctx->h_off32.p, off32.data(), (size_t)(nreads + 1) * 4);
  CK(cudaMemcpyAsync(ctx->seq_off.p, ctx->h_off32.p, (size_t)(nreads + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->pk_off.p, pkoff, (size_t)(nreads + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
  ctx->device_only_reads = false;
  if ((rc = finish_upload(ctx, nreads, w))) return rc;
  CK(cudaEventRecord(e1, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));   // off32/pkoff are stack-owned
  float ms = 0; cudaEventElapsedTime(&ms, e0, e1); ctx->t_h2d = ms;
  return SMR_OK;
}

// the part of an upload that does not depend on where the reads came from: seq04 / seq_off / pk_off are on the device,
// ctx->off32 (host) holds the offsets; sizes the per-batch buffers and 2-bit packs the reads
int finish_upload(smr_ctx* ctx, uint32_t nreads, uint64_t w) {
  const uint32_t slots = slots_of(ctx);
  const std::vector<uint32_t>& off32 = ctx->off32;
  int rc;
  if ((rc = ensure(ctx, ctx->pk03, (size_t)(w + 4) * 4))) return rc;
  if ((rc = ensure(ctx, ctx->pk03alt, (size_t)(w + 4) * 4))) return rc;
  if ((rc = ensure(ctx, ctx->has_n, nreads))) return rc;
  if ((rc = ensure(ctx, ctx->flags, (size_t)nreads * 4))) return rc;
  if ((rc = ensure(ctx, ctx->state, (size_t)nreads * sizeof(ReadState)))) return rc;
  if ((rc = ensure(ctx, ctx->hit_db, (size_t)nreads * 2))) return rc;
  if ((rc = ensure(ctx, ctx->aln_work, (size_t)nreads * slots * sizeof(AlnWork)))) return rc;
  if ((rc = ensure(ctx, ctx->out_aln, (size_t)nreads * slots * sizeof(OutAln)))) return rc;
  if ((rc = ensure(ctx, ctx->scalars, 512))) return rc;
  if ((rc = ensure(ctx, ctx->counters, (size_t)(dcCount + 64) * 8))) return rc;
  CK(cudaMemsetAsync(ctx->pk03.p, 0, (size_t)(w + 4) * 4, ctx->stream));
  CK(cudaMemsetAsync(ctx->pk03alt.p, 0, (size_t)(w + 4) * 4, ctx->stream));
  // hit regions are per chunk
  uint64_t max_chunk_nt = 0;
  for (uint32_t c0 = 0; c0 < nreads; c0 += ctx->chunk_reads) {
    const uint32_t c1 = std::min(nreads, c0 + ctx->chunk_reads);
    max_chunk_nt = std::max<uint64_t>(max_chunk_nt, off32[c1] - off32[c0]);
  }
  // one hit-region set per loaded (index,part): all parts are seeded before the candidate kernel runs read-major
  const uint32_t nparts = (uint32_t)std::max<size_t>(1, ctx->parts.size());
  ctx->cnt_stride = std::min(nreads, ctx->chunk_reads);
  ctx->hits_stride = (size_t)((uint64_t)ctx->scale * (2 * max_chunk_nt + 32ull * ctx->cnt_stride) + 64);
  if ((rc = ensure(ctx, ctx->hits, ctx->hits_stride * nparts * 8))) return rc;
  if ((rc = ensure(ctx, ctx->hit_cnt, (size_t)ctx->cnt_stride * nparts * 4))) return rc;
  if ((rc = ensure(ctx, ctx->cost, (size_t)ctx->cnt_stride * 4))) return rc;
  if ((rc = ensure(ctx, ctx->bins, (size_t)ctx->cnt_stride * kCostBins * 4 + (size_t)kCostBins * 4))) return rc;
  // 2-bit packing + N detection
  DevBatch b{};
  b.nreads = nreads; b.r0 = 0; b.seq04 = (const uint8_t*)ctx->seq04.p; b.seq_off = (const uint32_t*)ctx->seq_off.p;
  b.pk_off = (const uint32_t*)ctx->pk_off.p;
  pack_reads_kernel<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(b, (uint32_t*)ctx->pk03.p, (uint32_t*)ctx->pk03alt.p, (uint8_t*)ctx->has_n.p);
  CK(cudaGetLastError());
  return SMR_OK;
}

// exclusive scan of n u32 on the device (out may alias in); total (optional, device pointer) receives the sum
int device_scan(smr_ctx* ctx, const uint32_t* in, uint32_t* out, uint64_t n, uint32_t* total_dev) {
  const uint32_t ntiles = (uint32_t)((n + kScanTile - 1) / kScanTile);
  int rc;
  if ((rc = ensure(ctx, ctx->scan_sums, (size_t)std::max<uint32_t>(ntiles, 1) * 4))) return rc;
  if (ntiles == 0) { if (total_dev) CK(cudaMemsetAsync(total_dev, 0, 4, ctx->stream)); return SMR_OK; }
  scan_tile_sums_kernel<<<ntiles, kScanThreads, 0, ctx->stream>>>(in, n, (uint32_t*)ctx->scan_sums.p);
  scan_sums_kernel<<<1, 1024, 0, ctx->stream>>>((uint32_t*)ctx->scan_sums.p, ntiles, total_dev);
  scan_apply_kernel<<<ntiles, kScanThreads, 0, ctx->stream>>>(in, n, (const uint32_t*)ctx->scan_sums.p, out);
  CK(cudaGetLastError());
  return SMR_OK;
}

// FASTA / FASTQ text -> resident batch (smr_decode.cuh)
// text == nullptr: the text is already in ctx->d_text (inflated on the device), first byte given
int upload_fastx_impl(smr_ctx* ctx, const char* text, uint64_t nbytes, uint32_t* nreads_out, char first_byte = 0) {
  *nreads_out = 0;
  ctx->nreads = 0;
  ctx->text_bytes = nbytes;
  if (nbytes == 0) return SMR_OK;
  if (nbytes >= 0xF0000000ull) { ctx->err = "text batch of 2^32 bytes or more: split it (line counts and sequence offsets are 32-bit on the device)"; return SMR_ERR_ARG; }
  const char c0 = text ? text[0] : first_byte;
  const uint32_t fmt = c0 == '@' ? kFmtFastq : kFmtFasta;
  if (c0 != '@' && c0 != '>') { ctx->err = "reads text must start with '@' (FASTQ) or '>' (FASTA)"; return SMR_ERR_ARG; }
  cudaEvent_t e0 = get_event(ctx, 0), e1 = get_event(ctx, 1), e2 = get_event(ctx, 2);
  int rc;
  CK(cudaEventRecord(e0, ctx->stream));
  if (text) {
    if ((rc = ensure(ctx, ctx->d_text, nbytes + 64))) return rc;
    CK(cudaMemcpyAsync(ctx->d_text.p, text, nbytes, cudaMemcpyHostToDevice, ctx->stream));
  }
  CK(cudaEventRecord(e1, ctx->stream));
  const uint8_t* dt = (const uint8_t*)ctx->d_text.p;
  const uint64_t nchunks = nbytes / 32 + 1;
  if ((rc = ensure(ctx, ctx->d_cnt, nchunks * 4))) return rc;
  if ((rc = ensure(ctx, ctx->d_scal, 64))) return rc;
  uint32_t* scal = (uint32_t*)ctx->d_scal.p;   // [0] nlines [1] nrec [2] total nt [3] err [4] words [5] max_len
  CK(cudaMemsetAsync(scal, 0, 64, ctx->stream));
  const int grid = ctx->sm_count * 8;
  count_newlines_kernel<<<grid, 256, 0, ctx->stream>>>(dt, nbytes, (uint32_t*)ctx->d_cnt.p, nchunks);
  if ((rc = device_scan(ctx, (const uint32_t*)ctx->d_cnt.p, (uint32_t*)ctx->d_cnt.p, nchunks, scal + 0))) return rc;
  uint32_t h[8];
  CK(cudaMemcpyAsync(h, scal, 32, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  const uint32_t nlines = h[0];
  if (nlines == 0) return SMR_OK;
  if ((rc = ensure(ctx, ctx->d_nl, (size_t)nlines * 8))) return rc;
  if ((rc = ensure(ctx, ctx->d_hdr, (size_t)nlines * 4))) return rc;
  if ((rc = ensure(ctx, ctx->d_sb, (size_t)nlines * 4))) return rc;
  if ((rc = ensure(ctx, ctx->d_rec, (size_t)nlines * 4))) return rc;
  if ((rc = ensure(ctx, ctx->d_spos, (size_t)nlines * 4))) return rc;
  write_newlines_kernel<<<grid, 256, 0, ctx->stream>>>(dt, nbytes, (const uint32_t*)ctx->d_cnt.p, nchunks, (uint64_t*)ctx->d_nl.p);
  line_info_kernel<<<grid, 256, 0, ctx->stream>>>(dt, (const uint64_t*)ctx->d_nl.p, nlines, fmt, (uint32_t*)ctx->d_hdr.p, (uint32_t*)ctx->d_sb.p, scal + 3);
  if ((rc = device_scan(ctx, (const uint32_t*)ctx->d_hdr.p, (uint32_t*)ctx->d_rec.p, nlines, scal + 1))) return rc;
  if ((rc = device_scan(ctx, (const uint32_t*)ctx->d_sb.p, (uint32_t*)ctx->d_spos.p, nlines, scal + 2))) return rc;
  CK(cudaMemcpyAsync(h, scal, 32, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  const uint32_t nreads = h[1], total = h[2], err = h[3];
  if (err) { ctx->err = err & kDecBadHeader ? "reads text: a record does not start with its header character" : "reads text: FASTQ separator line '+' missing"; return SMR_ERR_ARG; }
  if (total >= 0xF0000000u) { ctx->err = "batch larger than 2^32 nucleotides: split it"; return SMR_ERR_ARG; }
  if (nreads == 0) return SMR_OK;
  if ((rc = ensure(ctx, ctx->seq04, (size_t)total + 64))) return rc;
  if ((rc = ensure(ctx, ctx->seq_off, (size_t)(nreads + 1) * 4))) return rc;
  if ((rc = ensure(ctx, ctx->pk_off, (size_t)(nreads + 1) * 4))) return rc;
  if ((rc = ensure(ctx, ctx->d_hdroff, (size_t)nreads * 8))) return rc;
  scatter_lines_kernel<<<grid, 256, 0, ctx->stream>>>(dt, (const uint64_t*)ctx->d_nl.p, nlines, (const uint32_t*)ctx->d_hdr.p, (const uint32_t*)ctx->d_rec.p,
                                                       (const uint32_t*)ctx->d_sb.p, (const uint32_t*)ctx->d_spos.p, (uint8_t*)ctx->seq04.p,
                                                       (uint32_t*)ctx->seq_off.p, (uint64_t*)ctx->d_hdroff.p);
  CK(cudaMemcpyAsync((uint32_t*)ctx->seq_off.p + nreads, scal + 2, 4, cudaMemcpyDeviceToDevice, ctx->stream));
  // packed-word offsets and the longest read (what upload_batch_impl computes on the host)
  if ((rc = ensure(ctx, ctx->d_cnt, (size_t)(nreads + 1) * 4))) return rc;
  record_words_kernel<<<grid, 256, 0, ctx->stream>>>((const uint32_t*)ctx->seq_off.p, nreads, (uint32_t*)ctx->d_cnt.p, scal + 5);
  if ((rc = device_scan(ctx, (const uint32_t*)ctx->d_cnt.p, (uint32_t*)ctx->pk_off.p, (uint64_t)nreads + 1, scal + 4))) return rc;
  ctx->off32.resize((size_t)nreads + 1);
  if ((rc = ensure_pinned(ctx, ctx->h_off32, (size_t)(nreads + 1) * 4))) return rc;
  CK(cudaMemcpyAsync(ctx->h_off32.p, ctx->seq_off.p, (size_t)(nreads + 1) * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(h, scal, 32, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaEventRecord(e2, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  memcpy(ctx->off32.data(), ctx->h_off32.p, (size_t)(nreads + 1) * 4);
  ctx->nreads = nreads; ctx->total_nt = total; ctx->max_len = h[5];
  ctx->h_seq.clear(); ctx->h_off.clear(); ctx->device_only_reads = true;
  if ((rc = finish_upload(ctx, nreads, h[4]))) return rc;
  CK(cudaStreamSynchronize(ctx->stream));
  float ms = 0; cudaEventElapsedTime(&ms, e0, e1); if (text) ctx->t_h2d = ms;
  cudaEventElapsedTime(&ms, e1, e2); ctx->t_decode = ms;
  *nreads_out = nreads;
  return SMR_OK;
}

const char* inf_status_text(uint32_t st) {
  switch (st) {
    case kInfErrCode: return "invalid Huffman code";
    case kInfErrHeader: return "invalid block header";
    case kInfErrOverrun: return "compressed data ends inside a block (truncated file)";
    case kInfErrDistance: return "invalid distance too far back";
    case kInfErrStored: return "invalid stored block lengths";
    case kInfErrMember: return "not a gzip member";
    case kInfErrCrc: return "CRC-32 of a member disagrees with its data";
    case kInfErrSize: return "size field (ISIZE) of a member disagrees with its data";
    default: return "internal error";
  }
}

// gzip file (host bytes) -> inflated bytes in ctx->d_text.  The five steps of smr_inflate.h; the host only walks the list of
// spans (a few thousand entries) between the COUNT and the WRITE pass.
int inflate_impl(smr_ctx* ctx, const void* gz, uint64_t nbytes, uint64_t chunk_bytes, uint64_t* out_bytes) {
  *out_bytes = 0;
  ctx->inf_spans = ctx->inf_candidates = 0;
  if (nbytes < 18) { ctx->err = "gz input: shorter than a gzip header and trailer"; return SMR_ERR_ARG; }
  if (chunk_bytes < 1024) chunk_bytes = 1024;
  int rc;
  cudaEvent_t e0 = get_event(ctx, 0), e1 = get_event(ctx, 1), e2 = get_event(ctx, 2);
  CK(cudaEventRecord(e0, ctx->stream));
  const size_t padded = (nbytes + 3) / 4 * 4 + 128;
  if ((rc = ensure(ctx, ctx->d_gz, padded))) return rc;
  CK(cudaMemsetAsync((uint8_t*)ctx->d_gz.p + nbytes / 4 * 4, 0, padded - nbytes / 4 * 4, ctx->stream));
  CK(cudaMemcpyAsync(ctx->d_gz.p, gz, nbytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaEventRecord(e1, ctx->stream));
  const uint32_t* w = (const uint32_t*)ctx->d_gz.p;
  // FIND
  const uint64_t nchunks = (nbytes + chunk_bytes - 1) / chunk_bytes;
  if (nchunks > (1u << 24)) { ctx->err = "gz input: too many chunks"; return SMR_ERR_ARG; }
  std::vector<uint64_t> cand;
  if (nchunks > 1) {
    if ((rc = ensure(ctx, ctx->d_cand, nchunks * 8))) return rc;
    inf_find_kernel<<<(unsigned)(nchunks - 1), 256, 0, ctx->stream>>>(w, nbytes, chunk_bytes, (uint64_t*)ctx->d_cand.p);
    CK(cudaGetLastError());
    std::vector<uint64_t> raw(nchunks - 1);
    CK(cudaMemcpyAsync(raw.data(), ctx->d_cand.p, (nchunks - 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (uint64_t p : raw) if (p != kInfNone) cand.push_back(p);   // chunk order = position order
    if (!cand.empty()) CK(cudaMemcpyAsync(ctx->d_cand.p, cand.data(), cand.size() * 8, cudaMemcpyHostToDevice, ctx->stream));
  } else if ((rc = ensure(ctx, ctx->d_cand, 8))) return rc;
  const uint32_t ncand = (uint32_t)cand.size(), ns = ncand + 1;
  // COUNT
  CK(cudaFuncSetAttribute(inf_span_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kInfSpanSmem));   // per device
  CK(cudaFuncSetAttribute(inf_span_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kInfSpanSmem));
  if ((rc = ensure(ctx, ctx->d_res, (size_t)ns * sizeof(SpanResult)))) return rc;
  const unsigned ctas = (ns + kInfSpanThreads - 1) / kInfSpanThreads;
  inf_span_kernel<false><<<ctas, kInfSpanThreads, kInfSpanSmem, ctx->stream>>>(w, nbytes, (const uint64_t*)ctx->d_cand.p, ncand, nullptr, nullptr, nullptr, nullptr, nullptr, ns,
                                                                               nullptr, (SpanResult*)ctx->d_res.p);
  CK(cudaGetLastError());
  std::vector<SpanResult> res(ns);
  CK(cudaMemcpyAsync(res.data(), ctx->d_res.p, (size_t)ns * sizeof(SpanResult), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  std::vector<uint32_t> real(ns); std::vector<uint64_t> off(ns), cnt(ns);
  uint32_t nreal = 0, why = 0;
  const uint64_t total = inf_chain(cand.data(), ncand, res.data(), real.data(), off.data(), nreal, &why);
  if (total == kInfNone) { ctx->err = std::string("gz input: ") + inf_status_text(why); return SMR_ERR_ARG; }
  std::vector<uint32_t> moff(nreal + 1, 0);
  for (uint32_t k = 0; k < nreal; ++k) { cnt[k] = res[real[k]].out_n; moff[k + 1] = moff[k] + res[real[k]].members; }
  const uint32_t nmembers = moff[nreal];
  ctx->inf_spans = nreal; ctx->inf_candidates = ncand;
  if ((rc = ensure(ctx, ctx->d_text, total + 64))) return rc;
  if (total) {
    // WRITE
    if ((rc = ensure(ctx, ctx->d_ids, (size_t)nreal * 4))) return rc;
    if ((rc = ensure(ctx, ctx->d_off, (size_t)nreal * 8))) return rc;
    if ((rc = ensure(ctx, ctx->d_cnt64, (size_t)nreal * 8))) return rc;
    if ((rc = ensure(ctx, ctx->d_sym, (total + 8) * 2))) return rc;
    if ((rc = ensure(ctx, ctx->d_win, (size_t)(nreal + 1) * kInfWindow))) return rc;
    CK(cudaMemcpyAsync(ctx->d_ids.p, real.data(), (size_t)nreal * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_off.p, off.data(), (size_t)nreal * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_cnt64.p, cnt.data(), (size_t)nreal * 8, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = ensure(ctx, ctx->d_moff, (size_t)(nreal + 1) * 4))) return rc;
    if ((rc = ensure(ctx, ctx->d_mem, (size_t)(nmembers + 1) * sizeof(MemberEnd)))) return rc;
    CK(cudaMemcpyAsync(ctx->d_moff.p, moff.data(), (size_t)(nreal + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
    inf_span_kernel<true><<<(nreal + kInfSpanThreads - 1) / kInfSpanThreads, kInfSpanThreads, kInfSpanSmem, ctx->stream>>>(
        w, nbytes, (const uint64_t*)ctx->d_cand.p, ncand, (const uint32_t*)ctx->d_ids.p, (const uint64_t*)ctx->d_off.p, (const uint64_t*)ctx->d_cnt64.p,
        (const uint32_t*)ctx->d_moff.p, (MemberEnd*)ctx->d_mem.p, nreal, (uint16_t*)ctx->d_sym.p, (SpanResult*)ctx->d_res.p);
    CK(cudaGetLastError());
    // WINDOW, RESOLVE
    inf_window_kernel<<<1, 1024, 0, ctx->stream>>>((const uint16_t*)ctx->d_sym.p, (const uint64_t*)ctx->d_off.p, (const uint64_t*)ctx->d_cnt64.p, nreal, (uint8_t*)ctx->d_win.p);
    CK(cudaGetLastError());
    const uint64_t avg = total / nreal + 1;
    const unsigned pieces = (unsigned)std::min<uint64_t>(64, std::max<uint64_t>(1, avg / 8192));
    inf_resolve_kernel<<<dim3(pieces, nreal), 256, 0, ctx->stream>>>((const uint16_t*)ctx->d_sym.p, (const uint64_t*)ctx->d_off.p, (const uint64_t*)ctx->d_cnt64.p,
                                                                     (const uint8_t*)ctx->d_win.p, (uint8_t*)ctx->d_text.p);
    CK(cudaGetLastError());
    std::vector<SpanResult> res2(nreal);
    std::vector<MemberEnd> ends(nmembers);
    CK(cudaMemcpyAsync(res2.data(), ctx->d_res.p, (size_t)nreal * sizeof(SpanResult), cudaMemcpyDeviceToHost, ctx->stream));
    if (nmembers) CK(cudaMemcpyAsync(ends.data(), ctx->d_mem.p, (size_t)nmembers * sizeof(MemberEnd), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (uint32_t k = 0; k < nreal; ++k) {
      if (res2[k].status != res[real[k]].status || res2[k].out_n != cnt[k] || res2[k].end_bit != res[real[k]].end_bit || res2[k].members != res[real[k]].members) {
        ctx->err = "gz inflate: the write pass disagrees with the count pass"; return SMR_ERR_CUDA;
      }
      for (uint32_t m = moff[k]; m < moff[k + 1]; ++m) ends[m].out_end += off[k];
    }
    // CRC-32 + ISIZE of every member (RFC 1952 2.3.1): pieces on the device, joined here
    std::vector<uint64_t> poff; std::vector<uint32_t> plen, first;
    inf_crc_plan(ends, 32768, poff, plen, first);
    const uint32_t npieces = (uint32_t)poff.size();
    std::vector<uint32_t> crcs(npieces);
    if (npieces) {
      if ((rc = ensure(ctx, ctx->d_poff, (size_t)npieces * 8))) return rc;
      if ((rc = ensure(ctx, ctx->d_plen, (size_t)npieces * 4))) return rc;
      if ((rc = ensure(ctx, ctx->d_pcrc, (size_t)npieces * 4))) return rc;
      CK(cudaMemcpyAsync(ctx->d_poff.p, poff.data(), (size_t)npieces * 8, cudaMemcpyHostToDevice, ctx->stream));
      CK(cudaMemcpyAsync(ctx->d_plen.p, plen.data(), (size_t)npieces * 4, cudaMemcpyHostToDevice, ctx->stream));
      inf_crc_kernel<<<(npieces + 127) / 128, 128, 0, ctx->stream>>>((const uint8_t*)ctx->d_text.p, (const uint64_t*)ctx->d_poff.p, (const uint32_t*)ctx->d_plen.p, npieces,
                                                                       (uint32_t*)ctx->d_pcrc.p);
      CK(cudaGetLastError());
      CK(cudaMemcpyAsync(crcs.data(), ctx->d_pcrc.p, (size_t)npieces * 4, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaEventRecord(e2, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (const uint32_t bad = inf_crc_verify(ends, plen, first, crcs.data())) { ctx->err = std::string("gz input: ") + inf_status_text(bad); return SMR_ERR_ARG; }
  } else {
    CK(cudaEventRecord(e2, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  float ms = 0; cudaEventElapsedTime(&ms, e0, e1); ctx->t_h2d = ms;
  cudaEventElapsedTime(&ms, e1, e2); ctx->t_inflate = ms;
  *out_bytes = total;
  return SMR_OK;
}

DevBatch make_batch(smr_ctx* ctx, uint32_t c0, uint32_t n) {
  DevBatch b{};
  b.nreads = n; b.r0 = c0;
  b.seq04 = (const uint8_t*)ctx->seq04.p; b.seq_off = (const uint32_t*)ctx->seq_off.p;
  b.pk03 = (const uint32_t*)ctx->pk03.p; b.pk03alt = (const uint32_t*)ctx->pk03alt.p; b.pk_off = (const uint32_t*)ctx->pk_off.p;
  b.has_n = (const uint8_t*)ctx->has_n.p; b.hit_scale = ctx->scale; b.hits = (uint2*)ctx->hits.p;
  b.hit_cnt = (uint32_t*)ctx->hit_cnt.p; b.flags = (uint32_t*)ctx->flags.p; b.state = (ReadState*)ctx->state.p;
  b.hit_db = (uint16_t*)ctx->hit_db.p; b.counters = (unsigned long long*)ctx->counters.p;
  b.hits_stride = ctx->hits_stride; b.cnt_stride = ctx->cnt_stride; b.cost = (uint32_t*)ctx->cost.p;
  b.bins = (uint32_t*)ctx->bins.p; b.bin_count = (uint32_t*)ctx->bins.p + (size_t)ctx->cnt_stride * kCostBins;
  return b;
}

// Several contexts may share a device (two per GPU let the copies and the host-side result packing of one batch run under the
// kernels of the other).  Their KERNEL sections are serialised: the candidate kernel is persistent and needs every one of its CTAs
// resident at once (planner and scorer warps wait for each other), which two such kernels sharing the SMs could not guarantee.
std::mutex& device_kernel_mutex(int device) {
  static std::mutex m[64];
  return m[device & 63];
}

// all kernels of one pass over the resident batch
int run_impl(smr_ctx* ctx) {
  if (!ctx->have_params) { ctx->err = "smr_set_params not called"; return SMR_ERR_ARG; }
  if (ctx->parts.empty()) { ctx->err = "no index loaded"; return SMR_ERR_ARG; }
  if (ctx->prm.num_alignments < 0) { ctx->err = "num_alignments < 0"; return SMR_ERR_ARG; }
  if (ctx->prm.minoccur != 0) { ctx->err = "minoccur != 0 is not supported"; return SMR_ERR_UNSUPPORTED; }
  ctx->t_seed = ctx->t_lis = ctx->t_final = ctx->t_total = 0; ctx->n_launch = 0;
  const uint32_t nreads = ctx->nreads;
  if (nreads == 0) return SMR_OK;
  const uint32_t slots = slots_of(ctx);
  std::lock_guard<std::mutex> dev_lock(device_kernel_mutex(ctx->device));   // held until the stream has drained
  int rc;
  if ((rc = setup_arenas(ctx))) return rc;
  // device copy of the part table (finalize looks parts up by slot)
  std::vector<DevIndex> hp;
  for (size_t i = 0; i < ctx->parts.size(); ++i) {
    DevIndex d = ctx->parts[i].d; d.slot = (uint32_t)i; d.is_last = (i + 1 == ctx->parts.size()) ? 1u : 0u;
    hp.push_back(d);
  }
  if ((rc = ensure(ctx, ctx->parts_dev, hp.size() * sizeof(DevIndex)))) return rc;
  CK(cudaMemcpyAsync(ctx->parts_dev.p, hp.data(), hp.size() * sizeof(DevIndex), cudaMemcpyHostToDevice, ctx->stream));
  // cigar pool on the device: generous fixed share per alignment slot
  ctx->cigar_cap_dev = (uint64_t)nreads * slots * 24 * ctx->scale + 4096;
  if (ctx->cigar_cap_dev >= 0xFFFFFFFFull) { ctx->err = "CIGAR pool of this batch would pass 2^32 words (smr_aln.cigar_off is 32-bit): use smaller batches"; return SMR_ERR_CAPACITY; }
  if ((rc = ensure(ctx, ctx->cigar_pool, ctx->cigar_cap_dev * 4))) return rc;
  const Scalars sc = scalars_of(ctx);
  CK(cudaMemsetAsync(ctx->scalars.p, 0, 512, ctx->stream));
  CK(cudaMemsetAsync(ctx->counters.p, 0, (size_t)(dcCount + 64) * 8, ctx->stream));
  CK(cudaMemsetAsync(ctx->state.p, 0, (size_t)nreads * sizeof(ReadState), ctx->stream));
  CK(cudaMemsetAsync(ctx->flags.p, 0, (size_t)nreads * 4, ctx->stream));
  CK(cudaMemsetAsync(ctx->hit_db.p, 0xFF, (size_t)nreads * 2, ctx->stream));
  const DevParams dp = to_dev(ctx->prm);
  size_t evi = 2;
  std::vector<std::pair<size_t, int>> spans;   // (event index of start, kind) ; end = start+1
  cudaEvent_t eb = get_event(ctx, evi++); CK(cudaEventRecord(eb, ctx->stream));
  for (uint32_t c0 = 0; c0 < nreads; c0 += ctx->chunk_reads) {
    const uint32_t n = std::min(ctx->chunk_reads, nreads - c0);
    DevBatch b = make_batch(ctx, c0, n);
    b.seq_base0 = ctx->off32[c0];
    CK(cudaMemsetAsync(sc.work_n, 0, 16, ctx->stream));  // (unused word), the two cursors of the candidate kernel's read schedule, finalize's cursor (zeroed again before it runs)
    CK(cudaMemsetAsync(b.cost, 0, (size_t)n * 4, ctx->stream));
    CK(cudaMemsetAsync(b.bin_count, 0, (size_t)kCostBins * 4, ctx->stream));
    cudaEvent_t s0 = get_event(ctx, evi), s1 = get_event(ctx, evi + 1), s2 = get_event(ctx, evi + 2); evi += 3;
    CK(cudaEventRecord(s0, ctx->stream));
    if ((rc = ensure(ctx, ctx->seed_ctr, hp.size() * 4))) return rc;
    CK(cudaMemsetAsync(ctx->seed_ctr.p, 0, hp.size() * 4, ctx->stream));   // one work counter per seed launch
    for (size_t pi = 0; pi < hp.size(); ++pi) {
      const int ctas = (int)(ctx->lane_hits_warps / kSeedWarpsPerCta);
      uint32_t* next_read = (uint32_t*)ctx->seed_ctr.p + pi;
      if (ctx->instr) seed_kernel<true><<<ctas, kSeedWarpsPerCta * 32, 0, ctx->stream>>>(hp[pi], b, dp, (uint32_t*)ctx->lane_hits.p, ctx->lane_hits_cap, next_read);
      else seed_kernel<false><<<ctas, kSeedWarpsPerCta * 32, 0, ctx->stream>>>(hp[pi], b, dp, (uint32_t*)ctx->lane_hits.p, ctx->lane_hits_cap, next_read);
      CK(cudaGetLastError());
      ctx->n_launch += 1;
    }
    bin_kernel<<<(n + 255) / 256, 256, 0, ctx->stream>>>(b);
    CK(cudaGetLastError());
    CK(cudaEventRecord(s1, ctx->stream));
    {
      LisGlobals lg{};
      lg.arena_base = (uint8_t*)ctx->lis_arena.p; lg.arena_stride = ctx->lis_stride;
      lg.hist_cap = ctx->hist_cap; lg.cand_cap = ctx->cand_cap; lg.pair_cap = ctx->pair_cap; lg.row_cap = ctx->row_cap; lg.pall_cap = ctx->pall_cap;
      lg.task_cap = ctx->task_cap;
      lg.epochs = (uint32_t*)ctx->lis_epochs.p; lg.aln_work = (AlnWork*)ctx->aln_work.p; lg.slots = slots; lg.work_next = sc.lis_next; lg.work_next_b = sc.lis_next_b;
      lg.parts = (const DevIndex*)ctx->parts_dev.p; lg.nparts = (uint32_t)hp.size();
      lg.ring = (QSlot*)ctx->lis_queue.p; lg.done = (uint32_t*)ctx->lis_done.p; lg.score_rows = (int32_t*)ctx->lis_rows.p;
      lg.dbg = (getenv("SMR_TIMELINE") || getenv("SMR_VERBOSE")) ? (unsigned long long*)ctx->lis_dbg.p : nullptr;   // (the timeline costs the instrumented kernel an atomic per scored pair)
      lg.q_head = sc.q_head; lg.q_tail = sc.q_tail; lg.planners_done = sc.planners_done;
      lis_reset_kernel<<<kQueueCap / 256, 256, 0, ctx->stream>>>(lg, ctx->lis_warps);
      CK(cudaGetLastError());
      if (ctx->instr) lis_kernel<true><<<ctx->lis_ctas, kLisWarpsPerCta * 32, kLisSmemBytes, ctx->stream>>>(b, dp, lg);
      else lis_kernel<false><<<ctx->lis_ctas, kLisWarpsPerCta * 32, kLisSmemBytes, ctx->stream>>>(b, dp, lg);
      CK(cudaGetLastError());
      CK(cudaEventRecord(s2, ctx->stream));
      spans.push_back({evi - 3, 0});
      ctx->n_launch += 2;
    }
    // finalize this chunk
    CK(cudaMemsetAsync(sc.fin_next, 0, 4, ctx->stream));
    cudaEvent_t f0 = get_event(ctx, evi), f1 = get_event(ctx, evi + 1); evi += 2;
    CK(cudaEventRecord(f0, ctx->stream));
    FinalGlobals fg{};
    fg.arena_base = (uint8_t*)ctx->final_arena.p; fg.arena_stride = ctx->final_stride;
    fg.cap_w = ctx->cap_w; fg.cap_cig = ctx->cap_cig; fg.row_cap = ctx->row_cap; fg.cap_dir = ctx->cap_dir;
    fg.parts = (const DevIndex*)ctx->parts_dev.p; fg.aln_work = (const AlnWork*)ctx->aln_work.p; fg.out = (OutAln*)ctx->out_aln.p;
    fg.slots = slots; fg.cigar_pool = (uint32_t*)ctx->cigar_pool.p; fg.cigar_cap = ctx->cigar_cap_dev; fg.cigar_used = sc.cigar_used;
    fg.work_next = sc.fin_next;
    if ((rc = ensure(ctx, ctx->tb_jobs, (size_t)n * slots * sizeof(TraceJob)))) return rc;
    fg.jobs = (TraceJob*)ctx->tb_jobs.p; fg.tb_arena = (uint8_t*)ctx->tb_arena.p; fg.tb_stride = ctx->tb_stride;
    fg.tb_cap_w = ctx->tb_cap_w; fg.tb_cap_cig = ctx->tb_cap_cig; fg.tb_cap_dir = ctx->tb_cap_dir;
    fg.stats = nullptr;
    if (ctx->host_stats) {
      if ((rc = ensure(ctx, ctx->aln_stats, (size_t)nreads * slots * sizeof(AlnStats)))) return rc;
      fg.stats = (AlnStats*)ctx->aln_stats.p;
    }
    finalize_kernel<<<ctx->final_warps / kFinalWarpsPerCta, kFinalWarpsPerCta * 32, 0, ctx->stream>>>(b, dp, fg);
    CK(cudaGetLastError());
    traceback_kernel<<<ctx->tb_threads / 128, 128, 0, ctx->stream>>>(b, dp, fg);
    CK(cudaGetLastError());
    ctx->n_launch += 1;
    CK(cudaEventRecord(f1, ctx->stream));
    spans.push_back({evi - 2, 1});
    ctx->n_launch += 1;
  }
  cudaEvent_t ee = get_event(ctx, evi++); CK(cudaEventRecord(ee, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  float ms = 0;
  cudaEventElapsedTime(&ms, eb, ee); ctx->t_total = ms;
  if (getenv("SMR_VERBOSE")) {
    unsigned long long d[16]; cudaMemcpy(d, ctx->lis_dbg.p, 128, cudaMemcpyDeviceToHost);
    fprintf(stderr, "[smr] slowest read %llu: %.2f ms; cycles vote %llu order %llu group %llu plan %llu wait %llu replay %llu; sw calls %llu, tasks scored %llu, rounds %llu\n", d[10], d[0] / 1.965e6, d[1], d[2], d[3], d[4], d[5], d[6], d[7], d[8], d[9]);
  }
  if (ctx->instr && getenv("SMR_TIMELINE")) {   // ns per role and state in 1 ms buckets since the kernel's start (this run's candidate launches summed)
    std::vector<unsigned long long> tl((size_t)kTlRows * kTlBuckets);
    cudaMemcpy(tl.data(), (const unsigned long long*)ctx->lis_dbg.p + kTlBase, tl.size() * 8, cudaMemcpyDeviceToHost);
    static const char* names[kTlRows] = {"scorer_wait_ns", "scorer_busy_ns", "planner_wait_ns", "planner_vote_group_ns", "reads_done", "planner_alive_ns"};
    for (int r = 0; r < kTlRows; ++r) {
      int last = 0; for (int k = 0; k < kTlBuckets; ++k) if (tl[(size_t)r * kTlBuckets + k]) last = k + 1;
      fprintf(stderr, "[smr timeline] %s", names[r]);
      for (int k = 0; k < last; ++k) fprintf(stderr, " %llu", tl[(size_t)r * kTlBuckets + k]);
      fprintf(stderr, "\n");
    }
  }
  for (auto& s : spans) {
    if (s.second == 0) {
      cudaEventElapsedTime(&ms, ctx->ev[s.first], ctx->ev[s.first + 1]); ctx->t_seed += ms;
      cudaEventElapsedTime(&ms, ctx->ev[s.first + 1], ctx->ev[s.first + 2]); ctx->t_lis += ms;
    } else { cudaEventElapsedTime(&ms, ctx->ev[s.first], ctx->ev[s.first + 1]); ctx->t_final += ms; }
  }
  return SMR_OK;
}

struct HostOut {
  smr_read_result* results; smr_aln* alns; uint32_t* cigar_pool; uint64_t cigar_cap; uint64_t cigar_used;
  uint64_t* counters; uint32_t n_counters;
};

// copies results of the resident batch to the host; returns the indices of reads whose scratch overflowed
int download_impl(smr_ctx* ctx, HostOut& out, std::vector<uint32_t>& flagged, const uint32_t* map /*local->caller index or null*/) {
  const uint32_t n = ctx->nreads;
  flagged.clear();
  if (n == 0) return SMR_OK;
  const uint32_t slots = slots_of(ctx);
  cudaEvent_t e0 = get_event(ctx, 0), e1 = get_event(ctx, 1);
  CK(cudaEventRecord(e0, ctx->stream));
  int prc;
  if ((prc = ensure_pinned(ctx, ctx->h_state, (size_t)n * sizeof(ReadState)))) return prc;
  if ((prc = ensure_pinned(ctx, ctx->h_flags, (size_t)n * 4))) return prc;
  if ((prc = ensure_pinned(ctx, ctx->h_hitdb, (size_t)n * 2))) return prc;
  if ((prc = ensure_pinned(ctx, ctx->h_outaln, (size_t)n * slots * sizeof(OutAln)))) return prc;
  const ReadState* st = (const ReadState*)ctx->h_state.p; const uint32_t* fl = (const uint32_t*)ctx->h_flags.p;
  const uint16_t* hdb = (const uint16_t*)ctx->h_hitdb.p; const OutAln* oa = (const OutAln*)ctx->h_outaln.p;
  const AlnStats* ast = nullptr;
  if (ctx->host_stats) {
    if ((prc = ensure_pinned(ctx, ctx->h_stats, (size_t)n * slots * sizeof(AlnStats)))) return prc;
    ast = (const AlnStats*)ctx->h_stats.p;
    CK(cudaMemcpyAsync(ctx->h_stats.p, ctx->aln_stats.p, (size_t)n * slots * sizeof(AlnStats), cudaMemcpyDeviceToHost, ctx->stream));
  }
  unsigned long long used = 0;
  std::vector<unsigned long long> cnt(dcCount + 64);
  CK(cudaMemcpyAsync(ctx->h_state.p, ctx->state.p, (size_t)n * sizeof(ReadState), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(ctx->h_flags.p, ctx->flags.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(ctx->h_hitdb.p, ctx->hit_db.p, (size_t)n * 2, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(ctx->h_outaln.p, ctx->out_aln.p, (size_t)n * slots * sizeof(OutAln), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(&used, scalars_of(ctx).cigar_used, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(cnt.data(), ctx->counters.p, cnt.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  used = std::min<unsigned long long>(used, ctx->cigar_cap_dev);
  if ((prc = ensure_pinned(ctx, ctx->h_cigar, (size_t)used * 4 + 16))) return prc;
  const uint32_t* cig = (const uint32_t*)ctx->h_cigar.p;
  if (used) CK(cudaMemcpyAsync(ctx->h_cigar.p, ctx->cigar_pool.p, used * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaEventRecord(e1, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  float ms = 0; cudaEventElapsedTime(&ms, e0, e1); ctx->t_d2h = ms;
  int rc = SMR_OK;
  // pass 1 (sequential, cheap): flagged reads, cigar offsets in the caller's pool (running sum in read order), counters
  std::vector<uint64_t>& coff = ctx->h_coff; coff.resize((size_t)n + 1);
  uint64_t run = out.cigar_used;
  uint32_t need_slots = 0;
  for (uint32_t r = 0; r < n; ++r) {
    coff[r] = run;
    if (fl[r] & kErrTrace) { ctx->err = "trace back error (ssw.c:707 is fatal in the reference too)"; rc = SMR_ERR_INDEX; }
    if (fl[r] & kOvfSlots) { need_slots = std::max(need_slots, st[r].n_align); continue; }   // not retried: the stride is the caller's
    if (fl[r]) { flagged.push_back(r); for (int bit = 0; bit < 6; ++bit) if (fl[r] & (1u << bit)) ctx->flag_hist[bit]++; continue; }
    const ReadState& s = st[r];
    for (uint32_t k = 0; k < slots && k < s.n_align; ++k) run += oa[(size_t)r * slots + k].cigar_len;
    if (s.is_hit && out.counters) {
      if (out.n_counters > SMR_CNT_NUM_ALIGNED) out.counters[SMR_CNT_NUM_ALIGNED]++;
      const uint32_t ci = SMR_CNT_FIXED + hdb[r];
      if (hdb[r] != 0xFFFF && ci < out.n_counters) out.counters[ci]++;
    }
  }
  coff[n] = run;
  if (need_slots) {
    ctx->err = "all-alignments mode: a read stored " + std::to_string(need_slots) + " alignments, the result stride is " + std::to_string(slots) +
               " (smr_set_aln_slots(" + std::to_string(need_slots) + ") or more, then call again)";
    ctx->need_slots = need_slots;
    return SMR_ERR_CAPACITY;
  }
  if (run > out.cigar_cap) { ctx->err = "cigar pool too small"; return SMR_ERR_CAPACITY; }
  if (run >= 0xFFFFFFFFull) { ctx->err = "CIGAR pool offset passes 2^32 words (smr_aln.cigar_off is 32-bit): use smaller batches"; return SMR_ERR_CAPACITY; }
  out.cigar_used = run;
  // pass 2: results, alignments and cigars of disjoint read ranges, by a few host threads for large batches
  auto pack = [&](uint32_t lo, uint32_t hi) {
    for (uint32_t r = lo; r < hi; ++r) {
      if (fl[r]) continue;
      const uint32_t dst = map ? map[r] : r;
      smr_read_result& o = out.results[dst];
      const ReadState& s = st[r];
      o.lastIndex = s.lastIndex; o.lastPart = s.lastPart; o.hit_seeds = s.hit_seeds; o.min_index = s.min_index; o.max_index = s.max_index;
      o.n_align = s.n_align; o.max_SW_count = s.max_SW_count; o.is_done = s.is_done; o.is_hit = s.is_hit;
      uint64_t at = coff[r];
      for (uint32_t k = 0; k < slots; ++k) {
        smr_aln& a = out.alns[(size_t)dst * slots + k];
        memset(&a, 0, sizeof(a));
        if (k >= s.n_align) continue;
        const OutAln& d = oa[(size_t)r * slots + k];
        memcpy(out.cigar_pool + at, cig + d.cigar_off, (size_t)d.cigar_len * 4);
        a.cigar_off = (uint32_t)at; a.cigar_len = d.cigar_len; at += d.cigar_len;
        a.ref_num = d.ref_num; a.ref_begin1 = d.ref_begin1; a.ref_end1 = d.ref_end1; a.read_begin1 = d.read_begin1; a.read_end1 = d.read_end1;
        a.readlen = d.readlen; a.score1 = d.score1; a.part = d.part; a.index_num = d.index_num; a.strand = d.strand;
        if (ctx->host_stats) { const AlnStats& st2 = ast[(size_t)r * slots + k]; ctx->host_stats[(size_t)dst * slots + k] = smr_aln_stats{st2.n_miss, st2.n_gap, st2.n_match, st2.n_match_denovo}; }
      }
    }
  };
  const uint32_t nthr = n >= (1u << 16) ? std::min<uint32_t>(8, std::max<uint32_t>(1, std::thread::hardware_concurrency() / 2)) : 1;
  if (nthr <= 1) pack(0, n);
  else {
    std::vector<std::thread> pool;
    for (uint32_t t = 0; t < nthr; ++t) pool.emplace_back(pack, (uint32_t)((uint64_t)n * t / nthr), (uint32_t)((uint64_t)n * (t + 1) / nthr));
    for (auto& th : pool) th.join();
  }
  if (out.counters) {
    static const int mapc[][2] = {{SMR_CNT_NUM_SHORT, dcNumShort}, {SMR_CNT_SW_CALLS, dcSwCalls}, {SMR_CNT_SW_CELLS, dcSwCells},
                                  {SMR_CNT_WINDOWS, dcWindows}, {SMR_CNT_TRIE_NODES, dcNodes}, {SMR_CNT_BUCKETS, dcBuckets},
                                  {SMR_CNT_BUCKET_ENTRIES, dcEntries}, {SMR_CNT_POS_ENTRIES, dcPosEntries}, {SMR_CNT_LIS_CALLS, dcLisCalls},
                                  {10, dcMaxReadCycles}, {11, dcSumReadCycles}, {12, dcLisKernelCycles},
                                  {13, dcCycVote}, {14, dcCycOrder}, {15, dcCycGroup}, {16, dcCycPlan}, {17, dcCycWait}, {18, dcCycReplay}, {19, dcSpecCalls},
                                  {20, dcSpecCells}, {21, dcSpecPairs}, {22, dcSlowPairs}, {23, dcScWait}, {24, dcScLoad}, {25, dcScSw}, {26, dcScPub}, {27, dcRoundsA}, {28, dcRoundsB}, {29, dcW1Cyc}, {30, dcW1Cnt}, {31, dcMaxReadBusy}};
    for (auto& m : mapc) if ((uint32_t)m[0] < out.n_counters) out.counters[m[0]] += cnt[m[1]];
  }
  return rc;
}

// align a host batch, retrying reads whose scratch overflowed with a larger scale
int align_impl(smr_ctx* ctx, const uint8_t* seq_cat, const uint64_t* seq_off, uint32_t nreads, HostOut& out, const uint32_t* map, int depth) {
  int rc = upload_batch_impl(ctx, seq_cat, seq_off, nreads, false);
  if (rc) return rc;
  const double h2d = ctx->t_h2d;
  if ((rc = run_impl(ctx))) return rc;
  std::vector<uint32_t> flagged;
  if ((rc = download_impl(ctx, out, flagged, map))) return rc;
  ctx->t_h2d = h2d;
  if (flagged.empty()) return SMR_OK;
  if (getenv("SMR_VERBOSE")) fprintf(stderr, "[smr] %zu reads overflowed their scratch at scale %u: retrying with scale %u (causes so far: lane %llu region %llu pairs %llu trace %llu cigar %llu err %llu)\n", flagged.size(), ctx->scale, ctx->scale * 8,
      (unsigned long long)ctx->flag_hist[0], (unsigned long long)ctx->flag_hist[1], (unsigned long long)ctx->flag_hist[2], (unsigned long long)ctx->flag_hist[3], (unsigned long long)ctx->flag_hist[4], (unsigned long long)ctx->flag_hist[5]);
  if (depth >= 3) { ctx->err = "scratch overflow persists after 3 retries (" + std::to_string(flagged.size()) + " reads)"; return SMR_ERR_CAPACITY; }
  // sub-batch of the flagged reads, 8x the scratch
  std::vector<uint8_t> sseq; std::vector<uint64_t> soff(1, 0); std::vector<uint32_t> smap;
  for (uint32_t r : flagged) {
    sseq.insert(sseq.end(), seq_cat + seq_off[r], seq_cat + seq_off[r + 1]);
    soff.push_back(sseq.size());
    smap.push_back(map ? map[r] : r);
  }
  const uint32_t old_scale = ctx->scale;
  const double tt = ctx->t_total, ts = ctx->t_seed, tl = ctx->t_lis, tf = ctx->t_final, td = ctx->t_d2h; const uint64_t nl = ctx->n_launch;
  ctx->scale = old_scale * 8;
  rc = align_impl(ctx, sseq.data(), soff.data(), (uint32_t)flagged.size(), out, smap.data(), depth + 1);
  ctx->scale = old_scale;
  ctx->t_total += tt; ctx->t_seed += ts; ctx->t_lis += tl; ctx->t_final += tf; ctx->t_d2h += td; ctx->t_h2d += h2d; ctx->n_launch += nl;
  return rc;
}

}  // namespace

extern "C" {

// No exception crosses the C ABI: the batch entry points below are function-try-blocks that turn a failed host allocation (the result
// vectors of a 2^32-nt batch, the retry copies) or any other std::exception into a status and an error text.
#define SMR_CATCH(ctx) \
  catch (const std::bad_alloc&) { if (ctx) (ctx)->err = "out of host memory"; return SMR_ERR_CAPACITY; } \
  catch (const std::exception& ex) { if (ctx) (ctx)->err = std::string("internal error: ") + ex.what(); return SMR_ERR_CUDA; }

int smr_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int smr_init(int device, smr_ctx** out) {
  if (!out) return SMR_ERR_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0 || device < 0 || device >= n) return SMR_ERR_NO_DEVICE;
  smr_ctx* ctx = new smr_ctx();
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return SMR_ERR_NO_DEVICE; }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return SMR_ERR_NO_DEVICE; }
  ctx->sm_count = prop.multiProcessorCount;
  if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return SMR_ERR_CUDA; }
  if (const char* e = getenv("SMR_CHUNK_READS")) { const long v = atol(e); if (v >= 32 && v <= (1l << 22)) ctx->chunk_reads = (uint32_t)v; }   // tests: several chunks per batch
  if (const char* e = getenv("SMR_INSTR")) ctx->instr = atoi(e) != 0;   // instrumented instantiations of the seed and candidate kernels (smr_set_instrumentation)
  if (const char* e = getenv("SMR_LIS_CTAS_PER_SM")) { const int v = atoi(e); if (v >= 1 && v <= 16) ctx->lis_ctas_per_sm = (uint32_t)v; }
  *out = ctx;
  return SMR_OK;
}

void smr_destroy(smr_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  for (auto& pt : ctx->parts) for (void* p : pt.owned) cudaFree(p);
  DevBuf* bufs[] = {&ctx->seq04, &ctx->seq_off, &ctx->pk03, &ctx->pk03alt, &ctx->pk_off, &ctx->has_n, &ctx->hit_cnt, &ctx->flags, &ctx->state,
                    &ctx->hit_db, &ctx->aln_work, &ctx->out_aln, &ctx->hits, &ctx->cost, &ctx->bins, &ctx->scalars, &ctx->counters, &ctx->cigar_pool,
                    &ctx->parts_dev, &ctx->lis_arena, &ctx->lis_epochs, &ctx->lis_queue, &ctx->lis_done, &ctx->lis_rows, &ctx->lis_dbg, &ctx->final_arena, &ctx->lane_hits, &ctx->tb_arena, &ctx->tb_jobs, &ctx->aln_stats,
                    &ctx->d_text, &ctx->d_cnt, &ctx->d_scal, &ctx->d_nl, &ctx->d_hdr, &ctx->d_sb, &ctx->d_rec, &ctx->d_spos, &ctx->d_hdroff, &ctx->scan_sums,
                    &ctx->d_gz, &ctx->d_cand, &ctx->d_res, &ctx->d_sym, &ctx->d_win, &ctx->d_ids, &ctx->d_off, &ctx->d_cnt64,
                    &ctx->d_moff, &ctx->d_mem, &ctx->d_poff, &ctx->d_plen, &ctx->d_pcrc, &ctx->seed_ctr};
  for (DevBuf* b : bufs) release(*b);
  PinBuf* pins[] = {&ctx->h_state, &ctx->h_flags, &ctx->h_hitdb, &ctx->h_outaln, &ctx->h_stats, &ctx->h_cigar, &ctx->h_off32, &ctx->h_pkoff};
  for (PinBuf* b : pins) release(*b);
  for (cudaEvent_t e : ctx->ev) cudaEventDestroy(e);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* smr_last_error(const smr_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int smr_load_index_part(smr_ctx* ctx, uint32_t index_num, uint32_t part, const void* kmer_file, size_t kmer_bytes,
                        const void* bursttrie_file, size_t bursttrie_bytes, const void* pos_file, size_t pos_bytes,
                        const uint8_t* refseq_cat, const uint64_t* ref_off, uint32_t nref, uint32_t lnwin, uint32_t minimal_score,
                        const uint32_t skiplengths[3]) {
  if (!ctx || !kmer_file || !bursttrie_file || !pos_file || !refseq_cat || !ref_off || !skiplengths) return SMR_ERR_ARG;
  if (skiplengths[0] == 0 || skiplengths[1] == 0 || skiplengths[2] == 0) { ctx->err = "skiplengths must be positive"; return SMR_ERR_ARG; }
  CK(cudaSetDevice(ctx->device));
  FlatIndex fx;
  std::string e;
  try {
    e = flatten_index(kmer_file, kmer_bytes, bursttrie_file, bursttrie_bytes, pos_file, pos_bytes, lnwin, fx);
  } catch (const std::exception& ex) { e = std::string("index files could not be read: ") + ex.what(); }   // bad_alloc / length_error on a malformed file
  if (!e.empty()) { ctx->err = e; return SMR_ERR_INDEX; }
  const uint64_t ref_total = ref_off[nref] - ref_off[0];
  if (ref_total >= 0xFFFFFFFFull) { ctx->err = "reference part larger than 4 GB"; return SMR_ERR_UNSUPPORTED; }
  for (const auto& sp : fx.pos) if (sp.seq >= nref) { ctx->err = "position table names a sequence beyond the references"; return SMR_ERR_INDEX; }
  Part pt;
  pt.d.index_num = index_num; pt.d.part = part; pt.d.lnwin = lnwin; pt.d.partialwin = lnwin / 2; pt.d.minimal_score = minimal_score;
  for (int i = 0; i < 3; ++i) pt.d.skip[i] = skiplengths[i];
  pt.d.nref = nref; pt.d.nids = (uint32_t)(fx.pos_off.size() - 1);
  std::vector<uint32_t> roff(nref + 1);
  for (uint32_t i = 0; i <= nref; ++i) roff[i] = (uint32_t)(ref_off[i] - ref_off[0]);
  std::vector<uint8_t> rseq(refseq_cat + ref_off[0], refseq_cat + ref_off[nref]);
  rseq.resize(rseq.size() + 64, 4);
  int rc;
  const uint32_t* lk = nullptr; const Entry* en = nullptr; const uint32_t* po = nullptr; const SeqPos* ps = nullptr;
  const uint8_t* rs = nullptr; const uint32_t* ro = nullptr;
  if ((rc = upload_vec(ctx, pt, fx.flookup, &lk))) return rc;
  if ((rc = upload_vec(ctx, pt, fx.flist, &en))) return rc;
  if ((rc = upload_vec(ctx, pt, fx.pos_off, &po))) return rc;
  if ((rc = upload_vec(ctx, pt, fx.pos, &ps))) return rc;
  if ((rc = upload_vec(ctx, pt, rseq, &rs))) return rc;
  if ((rc = upload_vec(ctx, pt, roff, &ro))) return rc;
  pt.d.flookup = (const uint4*)lk; pt.d.flist = (const uint2*)en; pt.d.pos_off = po; pt.d.pos = (const uint2*)ps;
  pt.d.refseq = rs; pt.d.ref_off = ro;
  pt.n_refseq = rseq.size();
  pt.n_nodes = fx.nodes.size(); pt.n_entries = fx.entries.size(); pt.n_ids = pt.d.nids; pt.n_pos = fx.pos.size();
  ctx->parts.push_back(std::move(pt));
  ctx->n_index_files = std::max(ctx->n_index_files, index_num + 1);
  return SMR_OK;
}

int smr_build_index_device(smr_ctx* ctx, uint32_t index_num, const char* fasta_path, uint32_t lnwin, uint32_t interval, uint32_t max_pos, double max_mb,
                           const uint32_t skiplengths[3], uint32_t minimal_score, uint32_t* nparts, uint64_t report6[6]) {
  if (!ctx || !fasta_path || !skiplengths) return SMR_ERR_ARG;
  if (skiplengths[0] == 0 || skiplengths[1] == 0 || skiplengths[2] == 0) { ctx->err = "skiplengths must be positive"; return SMR_ERR_ARG; }
  if (lnwin < 8 || lnwin > 26 || (lnwin & 1)) { ctx->err = "unsupported seed length"; return SMR_ERR_ARG; }
  if (interval == 0) { ctx->err = "interval must be >= 1"; return SMR_ERR_ARG; }
  CK(cudaSetDevice(ctx->device));
  BuildOptions opt; opt.lnwin = lnwin; opt.interval = interval; opt.max_pos = max_pos; opt.max_mb = max_mb;
  std::vector<RefRecord> recs;
  double freq[4] = {0, 0, 0, 0};
  uint64_t full_len = 0; size_t fsize = 0;
  std::string e;
  try {
    e = parse_reference_fasta(fasta_path, lnwin + 1, true, recs, freq, full_len, fsize);
  } catch (const std::exception& ex) { e = std::string("index build failed: ") + ex.what(); }
  if (!e.empty()) { ctx->err = e; return SMR_ERR_INDEX; }
  uint32_t part = 0;
  uint64_t rep[6] = {0, recs.size(), 0, 0, 0, 0};
  size_t first = 0;
  while (first < recs.size()) {
    std::vector<size_t> members; size_t next = first; uint64_t start_part = 0, seq_part_size = 0;
    e = next_index_part(recs, first, lnwin + 1, max_mb, members, next, start_part, seq_part_size);
    if (!e.empty()) { ctx->err = e; return SMR_ERR_INDEX; }
    if (members.empty()) break;
    Part pt;
    int rc = build_part_device(ctx, recs, members, opt, pt);
    if (rc) { for (void* p : pt.owned) cudaFree(p); return rc; }
    pt.d.index_num = index_num; pt.d.part = part; pt.d.minimal_score = minimal_score;
    for (int i = 0; i < 3; ++i) pt.d.skip[i] = skiplengths[i];
    rep[3] += pt.n_ids; rep[5] += pt.bytes;
    ctx->parts.push_back(std::move(pt));
    ctx->n_index_files = std::max(ctx->n_index_files, index_num + 1);
    ++part; first = next;
  }
  if (part == 0) { ctx->err = "no index was created"; return SMR_ERR_INDEX; }
  rep[0] = part;
  if (nparts) *nparts = part;
  if (report6) memcpy(report6, rep, sizeof(rep));
  return SMR_OK;
}

int smr_debug_index_array(smr_ctx* ctx, uint32_t slot, uint32_t which, void* out, uint64_t cap_bytes, uint64_t* nbytes) {
  if (!ctx || !nbytes || slot >= ctx->parts.size()) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  const Part& pt = ctx->parts[slot];
  const void* src = nullptr; uint64_t n = 0;
  switch (which) {
    case 0: src = pt.d.flookup; n = ((uint64_t)16) << (2 * pt.d.partialwin); break;
    case 1: src = pt.d.flist; n = (uint64_t)pt.n_entries * 8; break;
    case 2: src = pt.d.pos_off; n = ((uint64_t)pt.n_ids + 1) * 4; break;
    case 3: src = pt.d.pos; n = (uint64_t)pt.n_pos * 8; break;
    case 4: src = pt.d.refseq; n = pt.n_refseq; break;
    case 5: src = pt.d.ref_off; n = ((uint64_t)pt.d.nref + 1) * 4; break;
    default: ctx->err = "no such array"; return SMR_ERR_ARG;
  }
  *nbytes = n;
  if (!out) return SMR_OK;
  if (cap_bytes < n) { ctx->err = "buffer too small"; return SMR_ERR_CAPACITY; }
  if (n) CK(cudaMemcpy(out, src, n, cudaMemcpyDeviceToHost));
  return SMR_OK;
}

int smr_set_minimal_score(smr_ctx* ctx, uint32_t index_num, uint32_t minimal_score) {
  if (!ctx) return SMR_ERR_ARG;
  bool any = false;
  for (auto& pt : ctx->parts) if (pt.d.index_num == index_num) { pt.d.minimal_score = minimal_score; any = true; }
  if (!any) { ctx->err = "no such index"; return SMR_ERR_ARG; }
  return SMR_OK;
}

int smr_set_params(smr_ctx* ctx, const smr_params* p) {
  if (!ctx || !p) return SMR_ERR_ARG;
  if (p->match < -128 || p->match > 127 || p->gap_open < 0 || p->gap_ext < 0) { ctx->err = "scores out of range"; return SMR_ERR_ARG; }
  ctx->prm = *p; ctx->have_params = true;
  return SMR_OK;
}

int smr_set_aln_slots(smr_ctx* ctx, uint32_t slots) {
  if (!ctx || slots == 0 || slots > (1u << 20)) return SMR_ERR_ARG;
  ctx->all_slots = slots;
  return SMR_OK;
}

uint32_t smr_aln_slots(const smr_ctx* ctx) { return ctx ? slots_of(ctx) : 0; }
uint32_t smr_aln_slots_needed(const smr_ctx* ctx) { return ctx ? ctx->need_slots : 0; }

int smr_index_info(const smr_ctx* ctx, uint64_t out[6]) {
  if (!ctx || !out) return SMR_ERR_ARG;
  memset(out, 0, 6 * sizeof(uint64_t));
  out[0] = ctx->parts.size();
  for (auto& pt : ctx->parts) { out[1] += pt.bytes; out[2] += pt.n_nodes; out[3] += pt.n_entries; out[4] += pt.n_ids; out[5] += pt.n_pos; }
  return SMR_OK;
}

int smr_align_batch(smr_ctx* ctx, const uint8_t* seq_cat, const uint64_t* seq_off, uint32_t nreads, smr_read_result* results, smr_aln* alns,
                    uint32_t* cigar_pool, uint64_t cigar_cap, uint64_t* cigar_used, uint64_t* counters, uint32_t n_counters) try {
  if (!ctx || !seq_cat || !seq_off || !results || !alns || (!cigar_pool && cigar_cap)) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  const uint32_t slots = slots_of(ctx);
  memset(results, 0, (size_t)nreads * sizeof(smr_read_result));
  memset(alns, 0, (size_t)nreads * slots * sizeof(smr_aln));
  HostOut out{results, alns, cigar_pool, cigar_cap, 0, counters, n_counters};
  ctx->scale = 1;
  int rc = align_impl(ctx, seq_cat, seq_off, nreads, out, nullptr, 0);
  if (cigar_used) *cigar_used = out.cigar_used;
  return rc;
} SMR_CATCH(ctx)

int smr_set_instrumentation(smr_ctx* ctx, int on) {
  if (!ctx) return SMR_ERR_ARG;
  ctx->instr = on != 0;
  return SMR_OK;
}

int smr_set_stats_buffer(smr_ctx* ctx, smr_aln_stats* stats) {
  if (!ctx) return SMR_ERR_ARG;
  ctx->host_stats = stats;
  return SMR_OK;
}

int smr_upload_batch(smr_ctx* ctx, const uint8_t* seq_cat, const uint64_t* seq_off, uint32_t nreads) try {
  if (!ctx || !seq_cat || !seq_off) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  ctx->scale = 1;
  return upload_batch_impl(ctx, seq_cat, seq_off, nreads, true);
} SMR_CATCH(ctx)

int smr_upload_fastx(smr_ctx* ctx, const char* text, uint64_t nbytes, uint32_t* nreads) try {
  if (!ctx || (!text && nbytes) || !nreads) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  ctx->scale = 1;
  return upload_fastx_impl(ctx, text, nbytes, nreads);
} SMR_CATCH(ctx)

int smr_upload_fastx_gz(smr_ctx* ctx, const void* gz, uint64_t nbytes, uint32_t* nreads) try {
  if (!ctx || !gz || !nreads) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  ctx->scale = 1;
  *nreads = 0; ctx->nreads = 0; ctx->text_bytes = 0;
  uint64_t total = 0;
  const char* e = getenv("SMR_INFLATE_CHUNK");
  // distance of the speculative block searches: 64 KB for large files, down to 8 KB so that a small file still makes thousands of spans
  const uint64_t chunk = e ? strtoull(e, nullptr, 10) : std::min<uint64_t>(65536, std::max<uint64_t>(8192, nbytes / 8192));
  int rc = inflate_impl(ctx, gz, nbytes, chunk, &total);
  if (rc) return rc;
  if (total == 0) return SMR_OK;
  char c0 = 0;
  CK(cudaMemcpy(&c0, ctx->d_text.p, 1, cudaMemcpyDeviceToHost));
  return upload_fastx_impl(ctx, nullptr, total, nreads, c0);
} SMR_CATCH(ctx)

int smr_resident_text(smr_ctx* ctx, char* text, uint64_t cap, uint64_t* nbytes) {
  if (!ctx || !nbytes) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  *nbytes = ctx->text_bytes;
  if (!text || ctx->text_bytes == 0) return SMR_OK;
  if (cap < ctx->text_bytes) { ctx->err = "text buffer too small"; return SMR_ERR_CAPACITY; }
  CK(cudaMemcpy(text, ctx->d_text.p, ctx->text_bytes, cudaMemcpyDeviceToHost));
  return SMR_OK;
}

int smr_debug_inflate(smr_ctx* ctx, const void* gz, uint64_t nbytes, uint64_t chunk_bytes, uint8_t* out, uint64_t out_cap, uint64_t* out_bytes, uint32_t info[4]) try {
  if (!ctx || !gz || !out_bytes) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  ctx->nreads = 0; ctx->text_bytes = 0;
  if (chunk_bytes == 0) chunk_bytes = std::min<uint64_t>(65536, std::max<uint64_t>(8192, nbytes / 8192));   // as smr_upload_fastx_gz
  int rc = inflate_impl(ctx, gz, nbytes, chunk_bytes, out_bytes);
  if (rc) return rc;
  if (info) { info[0] = ctx->inf_spans; info[1] = ctx->inf_candidates; info[2] = (uint32_t)(ctx->t_inflate * 1000.0); info[3] = (uint32_t)(ctx->t_h2d * 1000.0); }
  if (out && *out_bytes) {
    if (out_cap < *out_bytes) { ctx->err = "output buffer too small"; return SMR_ERR_CAPACITY; }
    CK(cudaMemcpy(out, ctx->d_text.p, *out_bytes, cudaMemcpyDeviceToHost));
  }
  return SMR_OK;
} SMR_CATCH(ctx)

int smr_resident_layout(smr_ctx* ctx, uint64_t* header_text_off, uint64_t* read_off, uint8_t* seq04, uint64_t seq_cap) try {
  if (!ctx) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  const uint32_t n = ctx->nreads;
  if (read_off) for (uint32_t r = 0; r <= n; ++r) read_off[r] = n ? ctx->off32[r] : 0;
  if (header_text_off && n) {
    if (!ctx->device_only_reads) { ctx->err = "the resident batch was not uploaded as text"; return SMR_ERR_ARG; }
    CK(cudaMemcpy(header_text_off, ctx->d_hdroff.p, (size_t)n * 8, cudaMemcpyDeviceToHost));
  }
  if (seq04 && n) {
    if (seq_cap < ctx->total_nt) { ctx->err = "sequence buffer too small"; return SMR_ERR_CAPACITY; }
    CK(cudaMemcpy(seq04, ctx->seq04.p, ctx->total_nt, cudaMemcpyDeviceToHost));
  }
  return SMR_OK;
} SMR_CATCH(ctx)

int smr_run_resident(smr_ctx* ctx) try {
  if (!ctx) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  return run_impl(ctx);
} SMR_CATCH(ctx)

int smr_download_results(smr_ctx* ctx, smr_read_result* results, smr_aln* alns, uint32_t* cigar_pool, uint64_t cigar_cap, uint64_t* cigar_used,
                         uint64_t* counters, uint32_t n_counters) try {
  if (!ctx || !results || !alns) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  const uint32_t slots = slots_of(ctx);
  const uint32_t n = ctx->nreads;
  memset(results, 0, (size_t)n * sizeof(smr_read_result));
  memset(alns, 0, (size_t)n * slots * sizeof(smr_aln));
  HostOut out{results, alns, cigar_pool, cigar_cap, 0, counters, n_counters};
  std::vector<uint32_t> flagged;
  int rc = download_impl(ctx, out, flagged, nullptr);
  if (rc == SMR_OK && !flagged.empty()) {
    if (getenv("SMR_VERBOSE")) fprintf(stderr, "[smr] %zu reads overflowed their scratch (resident batch): retrying with scale 8 (causes so far: lane %llu region %llu pairs %llu trace %llu cigar %llu err %llu)\n", flagged.size(),
      (unsigned long long)ctx->flag_hist[0], (unsigned long long)ctx->flag_hist[1], (unsigned long long)ctx->flag_hist[2], (unsigned long long)ctx->flag_hist[3], (unsigned long long)ctx->flag_hist[4], (unsigned long long)ctx->flag_hist[5]);
    // redo the overflowed reads from the retained host copy with larger scratch
    if (ctx->device_only_reads) {   // decoded on the device: fetch the sequences now (only when a retry is needed)
      ctx->h_seq.resize(ctx->total_nt);
      CK(cudaMemcpy(ctx->h_seq.data(), ctx->seq04.p, ctx->total_nt, cudaMemcpyDeviceToHost));
      ctx->h_off.assign(ctx->off32.begin(), ctx->off32.end());
    }
    std::vector<uint8_t> hs; std::vector<uint64_t> ho;
    hs.swap(ctx->h_seq); ho.swap(ctx->h_off);
    std::vector<uint8_t> sseq; std::vector<uint64_t> soff(1, 0);
    for (uint32_t r : flagged) { sseq.insert(sseq.end(), hs.begin() + ho[r], hs.begin() + ho[r + 1]); soff.push_back(sseq.size()); }
    ctx->scale = 8;
    rc = align_impl(ctx, sseq.data(), soff.data(), (uint32_t)flagged.size(), out, flagged.data(), 1);
    ctx->scale = 1;
    // the resident batch was replaced by the retry batch: upload again before the next smr_run_resident
    ctx->nreads = 0;
  }
  if (cigar_used) *cigar_used = out.cigar_used;
  return rc;
} SMR_CATCH(ctx)

int smr_last_timings(const smr_ctx* ctx, double out[8]) {
  if (!ctx || !out) return SMR_ERR_ARG;
  out[0] = ctx->t_total; out[1] = ctx->t_seed; out[2] = ctx->t_lis; out[3] = ctx->t_final; out[4] = ctx->t_h2d; out[5] = ctx->t_d2h;
  out[6] = (double)ctx->n_launch; out[7] = ctx->t_decode;
  return SMR_OK;
}

int smr_debug_dpx_peak(smr_ctx* ctx, double* giga_ops_per_s) {
  if (!ctx || !giga_ops_per_s) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  int32_t* d = nullptr;
  CK(cudaMalloc(&d, 64));
  const int iters = 1 << 14, ctas = ctx->sm_count * 8, thr = 256;
  cudaEvent_t e0 = get_event(ctx, 0), e1 = get_event(ctx, 1);
  double best = 0;
  for (int rep = 0; rep < 4; ++rep) {
    CK(cudaEventRecord(e0, ctx->stream));
    dpx_peak_kernel<<<ctas, thr, 0, ctx->stream>>>(d, iters, -2, -1000000);
    CK(cudaGetLastError());
    CK(cudaEventRecord(e1, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    const double ops = (double)ctas * thr * iters * 8.0;
    if (rep > 0) best = std::max(best, ops / (ms * 1e-3) / 1e9);
  }
  cudaFree(d);
  *giga_ops_per_s = best;
  return SMR_OK;
}

int smr_debug_seed_windows(smr_ctx* ctx, uint32_t part_slot, const uint8_t* seq_cat, const uint64_t* seq_off, uint32_t nreads,
                           const uint32_t* win_read, const uint32_t* win_pos, uint32_t nwin, uint32_t* ids, uint32_t cap, uint32_t* counts,
                           uint8_t* zero) {
  if (!ctx || part_slot >= ctx->parts.size() || !seq_cat || !seq_off || !win_read || !win_pos || !ids || !counts || !zero) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  const uint32_t cap_arg = cap;
  cap &= 0x7FFFFFFFu;
  const uint64_t total = seq_off[nreads] - seq_off[0];
  std::vector<uint32_t> off32(nreads + 1);
  for (uint32_t r = 0; r <= nreads; ++r) off32[r] = (uint32_t)(seq_off[r] - seq_off[0]);
  uint8_t *d_seq = nullptr, *d_zero = nullptr; uint32_t *d_off = nullptr, *d_wr = nullptr, *d_wp = nullptr, *d_ids = nullptr, *d_cnt = nullptr;
  CK(cudaMalloc(&d_seq, total + 64)); CK(cudaMalloc(&d_off, (size_t)(nreads + 1) * 4)); CK(cudaMalloc(&d_wr, (size_t)nwin * 4 + 4));
  CK(cudaMalloc(&d_wp, (size_t)nwin * 4 + 4)); CK(cudaMalloc(&d_ids, (size_t)nwin * cap * 4 + 4)); CK(cudaMalloc(&d_cnt, (size_t)nwin * 4 + 4));
  CK(cudaMalloc(&d_zero, nwin + 4));
  CK(cudaMemcpy(d_seq, seq_cat + seq_off[0], total, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_off, off32.data(), (size_t)(nreads + 1) * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_wr, win_read, (size_t)nwin * 4, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_wp, win_pos, (size_t)nwin * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(d_ids, 0, (size_t)nwin * cap * 4));
  DevIndex d = ctx->parts[part_slot].d;
  const int mode = cap_arg >= 0x80000000u ? 1 : 0;   // high bit of cap selects the per-lane fallback path (tests exercise both)
  seed_debug_kernel<<<(nwin + kSeedWarpsPerCta * 32 - 1) / (kSeedWarpsPerCta * 32), kSeedWarpsPerCta * 32, 0, ctx->stream>>>(
      d, d_seq, d_off, d_wr, d_wp, nwin, d_ids, cap, d_cnt, d_zero, ctx->have_params ? ctx->prm.is_full_search : 0, mode);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(ids, d_ids, (size_t)nwin * cap * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(counts, d_cnt, (size_t)nwin * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(zero, d_zero, nwin, cudaMemcpyDeviceToHost));
  cudaFree(d_seq); cudaFree(d_off); cudaFree(d_wr); cudaFree(d_wp); cudaFree(d_ids); cudaFree(d_cnt); cudaFree(d_zero);
  return SMR_OK;
}

int smr_debug_ssw(smr_ctx* ctx, const uint8_t* q_cat, const uint64_t* q_off, const uint8_t* t_cat, const uint64_t* t_off, uint32_t npairs,
                  uint32_t filters, int32_t* out, uint32_t* cigars, uint32_t cigar_cap) {
  if (!ctx || !q_cat || !q_off || !t_cat || !t_off || !out || !cigars || !ctx->have_params) return SMR_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  const uint64_t qt = q_off[npairs] - q_off[0], tt = t_off[npairs] - t_off[0];
  std::vector<uint32_t> qo(npairs + 1), to(npairs + 1);
  uint32_t maxlen = 0;
  for (uint32_t i = 0; i <= npairs; ++i) { qo[i] = (uint32_t)(q_off[i] - q_off[0]); to[i] = (uint32_t)(t_off[i] - t_off[0]); }
  for (uint32_t i = 0; i < npairs; ++i) maxlen = std::max(maxlen, std::max(qo[i + 1] - qo[i], to[i + 1] - to[i]));
  uint8_t *dq = nullptr, *dt = nullptr, *arena = nullptr; uint32_t *dqo = nullptr, *dto = nullptr, *dc = nullptr; int32_t* dout = nullptr;
  FinalGlobals g{};
  g.cap_w = 2 * 2048 + 8; g.cap_cig = 2 * (maxlen + 64) + 16; g.row_cap = maxlen + 128; g.cap_dir = (size_t)(2 * 64 + 1) * (maxlen + 8) * 3 + 65536;
  const uint32_t nwarps = 512;
  g.arena_stride = final_arena_bytes(g.cap_w, g.cap_cig, g.row_cap, g.cap_dir);
  CK(cudaMalloc(&arena, g.arena_stride * nwarps)); g.arena_base = arena;
  CK(cudaMalloc(&dq, qt + 64)); CK(cudaMalloc(&dt, tt + 64)); CK(cudaMalloc(&dqo, (size_t)(npairs + 1) * 4)); CK(cudaMalloc(&dto, (size_t)(npairs + 1) * 4));
  CK(cudaMalloc(&dc, (size_t)npairs * cigar_cap * 4 + 4)); CK(cudaMalloc(&dout, (size_t)npairs * 6 * 4 + 4));
  CK(cudaMemcpy(dq, q_cat + q_off[0], qt, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dt, t_cat + t_off[0], tt, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(dqo, qo.data(), (size_t)(npairs + 1) * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dto, to.data(), (size_t)(npairs + 1) * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(dc, 0, (size_t)npairs * cigar_cap * 4));
  ssw_debug_kernel<<<nwarps / kFinalWarpsPerCta, kFinalWarpsPerCta * 32, 0, ctx->stream>>>(dq, dqo, dt, dto, npairs, filters, to_dev(ctx->prm), dout, dc,
                                                                                           cigar_cap, g);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(out, dout, (size_t)npairs * 6 * 4, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(cigars, dc, (size_t)npairs * cigar_cap * 4, cudaMemcpyDeviceToHost));
  cudaFree(dq); cudaFree(dt); cudaFree(dqo); cudaFree(dto); cudaFree(dc); cudaFree(dout); cudaFree(arena);
  return SMR_OK;
}

int smr_debug_sw_tasks(smr_ctx* ctx, const uint8_t* q_cat, uint64_t q_len, const uint8_t* t_cat, uint64_t t_len, const uint32_t* tasks,
                       uint32_t ntasks, const uint32_t* pairs, uint32_t npairs, uint32_t chain, uint32_t* scores, uint8_t* path) {
  if (!ctx || !q_cat || !t_cat || (ntasks && (!tasks || !scores)) || (npairs && (!pairs || !path)) || chain == 0 || !ctx->have_params) return SMR_ERR_ARG;
  if (ntasks >= kNoTask || q_len >= 0x80000000ull || t_len >= 0x80000000ull) return SMR_ERR_ARG;
  std::vector<SwTask> tv(ntasks);
  uint32_t row_cap = 1;
  for (uint32_t i = 0; i < ntasks; ++i) {
    const uint64_t ref = tasks[5 * i], qa = tasks[5 * i + 1], n = tasks[5 * i + 2], m = tasks[5 * i + 3], minus = tasks[5 * i + 4];
    if (minus > 1 || ref + n > t_len) return SMR_ERR_ARG;
    if (m == 0 ? qa > q_len : (minus ? qa >= q_len || qa + 1 < m : qa + m > q_len)) return SMR_ERR_ARG;   // minus strand: the query ends at q_abs
    SwTask t{};
    t.ref_abs = (uint32_t)ref; t.q_abs = (uint32_t)qa; t.alen = (uint32_t)n; t.qlen = (uint32_t)m; t.meta = (uint32_t)minus << 16;
    tv[i] = t;
    row_cap = std::max(row_cap, (uint32_t)n);
  }
  std::vector<uint32_t> pv(2 * (size_t)npairs);
  for (uint32_t k = 0; k < npairs; ++k) {
    const uint32_t a = pairs[2 * k], b = pairs[2 * k + 1];
    if (a >= ntasks || (b != 0xFFFFFFFFu && b >= ntasks)) return SMR_ERR_ARG;
    pv[2 * k] = a; pv[2 * k + 1] = b == 0xFFFFFFFFu ? kNoTask : b;
  }
  CK(cudaSetDevice(ctx->device));
  const uint64_t nchains = ((uint64_t)npairs + chain - 1) / chain, ctas = std::max<uint64_t>(1, (nchains + kSwDebugWarps - 1) / kSwDebugWarps);
  uint8_t *dq = nullptr, *dt = nullptr, *dpath = nullptr; SwTask* dtask = nullptr; uint32_t *dpairs = nullptr, *dscore = nullptr; int32_t* drows = nullptr;
  // padded as the product pads its reads (seq04: +64 bytes) and references (refseq: +64 bytes of N), so that a window or query at the end
  // of a buffer is staged exactly as in a run
  CK(cudaMalloc(&dq, q_len + 64)); CK(cudaMalloc(&dt, t_len + 64));
  CK(cudaMemset(dq + q_len, 0, 64)); CK(cudaMemset(dt + t_len, 4, 64));
  if (q_len) CK(cudaMemcpy(dq, q_cat, q_len, cudaMemcpyHostToDevice));
  if (t_len) CK(cudaMemcpy(dt, t_cat, t_len, cudaMemcpyHostToDevice));
  CK(cudaMalloc(&dtask, (size_t)ntasks * sizeof(SwTask) + sizeof(SwTask))); CK(cudaMalloc(&dpairs, pv.size() * 4 + 8));
  CK(cudaMalloc(&dscore, (size_t)ntasks * 4 + 4)); CK(cudaMalloc(&dpath, (size_t)npairs + 4));
  CK(cudaMalloc(&drows, (size_t)ctas * kSwDebugWarps * 2 * row_cap * 4));
  if (ntasks) CK(cudaMemcpy(dtask, tv.data(), (size_t)ntasks * sizeof(SwTask), cudaMemcpyHostToDevice));
  if (npairs) CK(cudaMemcpy(dpairs, pv.data(), pv.size() * 4, cudaMemcpyHostToDevice));
  CK(cudaMemset(dscore, 0xFF, (size_t)ntasks * 4 + 4)); CK(cudaMemset(dpath, 0xFF, (size_t)npairs + 4));   // a task no pair scores reads 0xFFFFFFFF
  if (npairs) {
    sw_tasks_debug_kernel<<<(unsigned)ctas, kSwDebugWarps * 32, kSwDebugWarps * kScorerSmem, ctx->stream>>>(dq, dt, dtask, dpairs, npairs, chain, to_dev(ctx->prm),
                                                                                                          drows, row_cap, dscore, dpath);
    CK(cudaGetLastError());
  }
  CK(cudaStreamSynchronize(ctx->stream));
  if (ntasks) CK(cudaMemcpy(scores, dscore, (size_t)ntasks * 4, cudaMemcpyDeviceToHost));
  if (npairs) CK(cudaMemcpy(path, dpath, npairs, cudaMemcpyDeviceToHost));
  cudaFree(dq); cudaFree(dt); cudaFree(dtask); cudaFree(dpairs); cudaFree(dscore); cudaFree(dpath); cudaFree(drows);
  return SMR_OK;
}

}  // extern "C"
