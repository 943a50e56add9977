/*
 * include/smr_b200.h -- C ABI of the B200-native alignment hot path (libsmr_b200.so).
 *
 * The reference (sortmerna v5.0.0) has no FFI; the seam this library replaces is the C++ call
 *     void align(Readfeed&, Readstats&, Index&, KeyValueDatabase&, Runopts&)
 *         (src/sortmerna/processor.cpp:173, called from src/sortmerna/main.cpp:88,99,105)
 * whose unit of work is
 *     void traverse(Runopts&, Index&, References&, Readstats&, Refstats&, Read&, bool)
 *         (src/sortmerna/paralleltraversal.cpp:81-90).
 * Each entry point below names the reference code it stands in for.  All functions return 0 on
 * success and a non-zero smr_status otherwise (the reference prints and exit()s; a host wrapper
 * maps non-zero to that).  Plain pointers and sizes only; no C++ or torch types.  Every compute
 * entry point requires a CUDA device: there is no CPU fallback.
 */
#ifndef SMR_B200_H
#define SMR_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct smr_ctx smr_ctx; /* opaque; one per GPU, driven by one host thread */

enum smr_status {
  SMR_OK = 0,
  SMR_ERR_CUDA = 1,        /* a CUDA call failed (smr_last_error has the text) */
  SMR_ERR_ARG = 2,         /* invalid argument */
  SMR_ERR_INDEX = 3,       /* malformed index file (index.cpp:282-286 is fatal in the reference too) */
  SMR_ERR_UNSUPPORTED = 4, /* option combination outside this build (see DESIGN.md) */
  SMR_ERR_CAPACITY = 5,    /* caller-provided output buffer too small */
  SMR_ERR_NO_DEVICE = 6    /* no CUDA device / extension cannot run: fail loudly, never fall back */
};

/* The opts.* fields that cross the seam (SURVEY 8(b)); defaults are those of
 * Runopts::validate (src/sortmerna/options.cpp:1684-1738). */
typedef struct {
  int32_t match, mismatch, score_N, gap_open, gap_ext; /* --match --mismatch -N --gap_open --gap_ext */
  int32_t num_seeds, min_lis, edges, edges_is_percent; /* --num_seeds --min_lis --edges */
  int32_t num_alignments, is_best;                     /* --num_alignments / --best / --no-best */
  int32_t is_forward, is_reverse, is_full_search;      /* -F -R --full_search */
  int32_t minoccur;                                    /* include/options.hpp:572 (no CLI option) */
} smr_params;

/* Per-read result = the fields Read::toBinString persists (src/sortmerna/read.cpp:429-462), i.e.
 * what the unchanged report stage reads back through Read::load_db. */
typedef struct {
  uint32_t lastIndex, lastPart;
  uint32_t hit_seeds;
  uint32_t min_index, max_index; /* alignment_struct2 (include/ssw.hpp:157-159) */
  uint32_t n_align;              /* alignv.size() */
  uint16_t max_SW_count;
  uint8_t is_done, is_hit;
} smr_read_result;

/* One stored alignment = s_align2 (include/ssw.hpp:44-56); slot (read * max(1,num_alignments) + k) */
typedef struct {
  uint32_t cigar_off, cigar_len; /* into the cigar pool; BAM style len<<4|op, op 0=M 1=I 2=D (ssw.c:750-758) */
  uint32_t ref_num;
  int32_t ref_begin1, ref_end1, read_begin1, read_end1;
  uint32_t readlen;
  uint16_t score1, part, index_num;
  uint8_t strand, pad;
} smr_aln;

/* Index builder (host code, no GPU needed; SURVEY 8(f)(3)).  Replaces build_index (src/sortmerna/indexdb.cpp:1119-2095): writes
 * <out_prefix>.kmer_P.dat / .bursttrie_P.dat / .pos_P.dat for every part P and <out_prefix>.stats in the reference's on-disk
 * format -- the files Index::load (index.cpp:143-357), Refstats::load (refstats.cpp:103-190) and smr_load_index_part read.
 * Content is that of the reference's builder (same windows, alphabet map, burst tries, counts, position lists, part split);
 * only the arbitrary numbering of the unique L-mers differs (order of first occurrence instead of a CMPH hash value).
 * lnwin = -L (18), interval = -interval (1), max_pos = -max_pos (10000; 0 = all), max_mb = -m (3072); threads: 2*threads
 * workers build the tries of disjoint 9-mer classes (0 = cores/8 clamped to 1..8); the files do not depend on it.
 * report6 (optional): parts, sequences, windows, unique L-mers, trie nodes, bytes written.  err: message buffer. */
int smr_build_index(const char* fasta_path, const char* out_prefix, uint32_t lnwin, uint32_t interval, uint32_t max_pos,
                    double max_mb, uint32_t threads, uint64_t* report6, char* err, size_t err_cap);

/* KVDB blob writer (host code; SURVEY 8(f)(4)): for every read of a batch the byte string Read::toBinString() would store
 * under its id (src/sortmerna/read.cpp:429-462; alignment_struct2::toString read.cpp:79-101; s_align2::toString
 * include/ssw.hpp:106-140), written straight from the result buffers, so Read::load_db (read.cpp:467-539) reads back what the
 * CPU path would have stored.  Reads without a stored alignment get an empty blob (read.cpp:431-432).
 * num_alignments = opts.num_alignments; denovo4 (optional) = per read {c_yid_ycov, n_yid_ncov, n_nid_ycov, n_denovo}
 * (zero while aligning; set by denovo_stats).  blob_off[0..nreads] receives the offsets; call with out == nullptr to size. */
int smr_pack_kvdb_blobs(const smr_read_result* results, const smr_aln* alns, const uint32_t* cigar_pool, uint32_t nreads,
                        uint32_t slots, int32_t num_alignments, const uint32_t* denovo4, uint8_t* out, uint64_t out_cap,
                        uint64_t* blob_off);

/* Report-side arithmetic of one stored alignment = Read::calc_miss_gap_match (src/sortmerna/read.cpp:547-589), computed on the
 * GPU from the CIGAR it has just produced (SURVEY 8(f)(1)): what %id / %cov / NM:i / BLAST columns 3,5,6 are derived from. */
typedef struct {
  uint32_t n_miss, n_gap, n_match;
  /* n_match as denovo_stats_run obtains it (src/sortmerna/processor.cpp:329-357): that caller does NOT reverse-complement
   * the read first, so for a reverse-strand alignment the CIGAR is walked over the forward read.  Reproduced as is, because
   * n_yid_ycov / n_yid_ncov / n_nid_ycov / n_denovo and aligned_denovo.* depend on it; equals n_match on the forward strand. */
  uint32_t n_match_denovo;
} smr_aln_stats;

/* Counters.  The first block is Readstats (include/readstats.hpp:77-84) as mutated by this path;
 * it is what the single NCCL all-reduce sums across GPUs.  The second block is instrumentation
 * used for the roofline arithmetic (SURVEY 8(d)). */
enum {
  SMR_CNT_NUM_ALIGNED = 0,   /* readstats.num_aligned (alignment.cpp:414) */
  SMR_CNT_NUM_SHORT = 1,     /* readstats.num_short of the LAST index pass (processor.cpp:109-114,228) */
  SMR_CNT_SW_CALLS = 2,      /* ssw_align-equivalent calls */
  SMR_CNT_SW_CELLS = 3,      /* sum refLen*readLen over those calls (forward pass only) */
  SMR_CNT_WINDOWS = 4,       /* seed windows searched (speculative windows included) */
  SMR_CNT_TRIE_NODES = 5,    /* trie nodes visited */
  SMR_CNT_BUCKETS = 6,       /* buckets visited */
  SMR_CNT_BUCKET_ENTRIES = 7,/* bucket entries visited */
  SMR_CNT_POS_ENTRIES = 8,   /* position entries touched by candidate voting */
  SMR_CNT_LIS_CALLS = 9,     /* compute_lis_alignment-equivalent calls */
  /* 10..22: warp-cycle accounting of the candidate kernel (max per read, sum, kernel, then per phase) */
  SMR_CNT_FIXED = 32         /* reads_matched_per_db[i] lives at counters[SMR_CNT_FIXED + i] */
};

/* -- lifetime ------------------------------------------------------------------------------- */
int smr_init(int device, smr_ctx** out);
void smr_destroy(smr_ctx*);
const char* smr_last_error(const smr_ctx*); /* text of the last failure on this context */
int smr_device_count(void);                 /* number of visible CUDA devices (0 if none) */

/* -- index + references: Index::load (src/sortmerna/index.cpp:143-357) and References::load
 *    (src/sortmerna/references.cpp:55-164) for one (index_num, part), in --ref order.  Takes the
 *    raw bytes of <idx>.kmer_<p>.dat / .bursttrie_<p>.dat / .pos_<p>.dat, flattens them to
 *    contiguous HBM arrays and keeps them resident (all indexes stay loaded; the reference loads
 *    and unloads one at a time, processor.cpp:225-266).
 *    refseq_cat: reference sequences in the 0..4 alphabet (nt_table, common.hpp:68-77), concatenated;
 *    ref_off[nref+1] offsets.  minimal_score / lnwin / skiplengths come from Refstats
 *    (src/sortmerna/refstats.cpp:147-166,259-265). */
int smr_load_index_part(smr_ctx*, uint32_t index_num, uint32_t part,
                        const void* kmer_file, size_t kmer_bytes,
                        const void* bursttrie_file, size_t bursttrie_bytes,
                        const void* pos_file, size_t pos_bytes,
                        const uint8_t* refseq_cat, const uint64_t* ref_off, uint32_t nref,
                        uint32_t lnwin, uint32_t minimal_score, const uint32_t skiplengths[3]);
/* Index build on the device (SURVEY 8(f)(3)): what smr_build_index + smr_load_index_part do for every part of the index of
 * `fasta_path`, without the files -- the FASTA is parsed on the host (records, alphabet maps, the part split rule of
 * indexdb.cpp:1381-1431), then windows, unique L-mers, position lists and the burst-trie order of every list are computed on the
 * device with sorts (sortmerna_b200/csrc/smr_build_dev.cuh) and stay resident.  Replaces build_index (src/sortmerna/indexdb.cpp:
 * 1119-2095) + Index::load (index.cpp:143-357) + References::load (references.cpp:55-154) for this index.  The arrays equal those
 * smr_load_index_part makes from the reference builder's files up to the numbering of the L-mer ids.
 * *nparts = parts made (ordinals continue the context's part list); report6 as for smr_build_index (nodes: 0). */
int smr_build_index_device(smr_ctx*, uint32_t index_num, const char* fasta_path, uint32_t lnwin, uint32_t interval, uint32_t max_pos, double max_mb,
                           const uint32_t skiplengths[3], uint32_t minimal_score, uint32_t* nparts, uint64_t report6[6]);
/* Test hook: resident array `which` of loaded part `slot` (0 flookup, 1 flist, 2 pos_off, 3 pos, 4 refseq, 5 ref_off). */
int smr_debug_index_array(smr_ctx*, uint32_t slot, uint32_t which, void* out, uint64_t cap_bytes, uint64_t* nbytes);
/* refstats.minimal_score depends on the read set (refstats.cpp:247-265): update without reloading */
int smr_set_minimal_score(smr_ctx*, uint32_t index_num, uint32_t minimal_score);
int smr_set_params(smr_ctx*, const smr_params*);
/* out[0]=#parts loaded [1]=bytes resident in HBM [2]=trie nodes [3]=bucket entries [4]=ids [5]=positions */
int smr_index_info(const smr_ctx*, uint64_t out[6]);

/* -- the hot path: align() (processor.cpp:173-285) over one batch of reads, read-major.
 *    For each read: for each loaded (index,part) in order: forward then reverse strand through
 *    traverse() with KVDB-equivalent carry-over (read.cpp:429-539).
 *    seq_cat: reads in 0..4 (4 = ambiguous, as nt_table yields), concatenated; seq_off[nreads+1].
 *    Host buffers; the call copies host->device, runs, and copies the results back.
 *    results[nreads]; alns[nreads * smr_aln_slots()] (= num_alignments per read; see smr_set_aln_slots for 0); cigar_pool[cigar_cap] u32 words;
 *    counters[SMR_CNT_FIXED + n_index_files] are ADDED to (caller zeroes them). */
int smr_align_batch(smr_ctx*, const uint8_t* seq_cat, const uint64_t* seq_off, uint32_t nreads,
                    smr_read_result* results, smr_aln* alns,
                    uint32_t* cigar_pool, uint64_t cigar_cap, uint64_t* cigar_used,
                    uint64_t* counters, uint32_t n_counters);

/* "All alignments" (opts.num_alignments == 0, src/sortmerna/alignment.cpp:420-424: every accepted alignment is appended, nothing
 * stops the candidate loop, scripts/test.jinja t9): the number of alignments of a read is unbounded, so the flat result layout needs
 * a stride.  smr_set_aln_slots sets it (default 16); alns[] / stats then hold nreads * slots entries, results[r].n_align of them
 * used.  If a read accepts more, the call fails with SMR_ERR_CAPACITY and smr_aln_slots_needed() names the stride that batch
 * needs (nothing is truncated silently).  smr_aln_slots() = the stride in effect: num_alignments when > 0, else the value set. */
int smr_set_aln_slots(smr_ctx*, uint32_t slots);
uint32_t smr_aln_slots(const smr_ctx*);
uint32_t smr_aln_slots_needed(const smr_ctx*);

/* Instrumentation (default OFF; the environment variable SMR_INSTR=1 turns it on at smr_init).  With it, the seed kernel counts
 * SMR_CNT_WINDOWS / BUCKETS / BUCKET_ENTRIES and the candidate kernel accounts its phases with the cycle counter (the SMR_CNT_*
 * entries from DBG_MAX_READ_CYCLES on): separate instantiations of both kernels, 2-3 % slower.  Everything a caller of the
 * reference would see -- results, Readstats counters, SW_CALLS / SW_CELLS / POS_ENTRIES / LIS_CALLS -- is identical either way. */
int smr_set_instrumentation(smr_ctx*, int on);

/* Optional: where the next smr_align_batch / smr_download_results stores smr_aln_stats for every stored alignment (same
 * indexing as alns[]; nullptr = do not compute).  Host buffer of nreads * max(1,num_alignments) entries. */
int smr_set_stats_buffer(smr_ctx*, smr_aln_stats* stats);

/* Input decode on the device (SURVEY 8(f)(2)): `text` = the bytes of an uncompressed FASTA or FASTQ file (or a record-aligned
 * piece of one).  Replaces, for the reads of this batch, the record split of Readfeed (src/sortmerna/readfeed.cpp:683-770),
 * Read::Read(readstr) (read.cpp:141-176) and the nt_table encoding of Read::init (read.cpp:264-288, common.hpp:68-77):
 * the text is copied to the device once and newline indexing, record split and 0-4 encoding run there; the decoded batch
 * becomes the resident batch (as after smr_upload_batch): follow with smr_run_resident / smr_download_results.
 * FASTQ: 4 lines per record; FASTA: '>' header + any number of sequence lines; CR LF tolerated; a missing final newline is
 * fine; trailing blank lines are ignored.  *nreads = records found. */
int smr_upload_fastx(smr_ctx*, const char* text, uint64_t nbytes, uint32_t* nreads);

/* The same from a gzip file: `gz` = the bytes of a .fastq.gz / .fasta.gz (one or several gzip members, RFC 1952).  Replaces the
 * inflate of the reference's read feed (Readfeed::next_gz, src/sortmerna/readfeed.cpp:683-770, izlib.cpp / rapidgzip): the
 * compressed bytes are copied to the device and inflated there -- block starts found speculatively in every 64 KB of the file, one
 * decoder thread per span, back-references into not-yet-known history resolved in a second step (sortmerna_b200/csrc/smr_inflate.h)
 * -- then decoded as in smr_upload_fastx.  The CRC-32 and ISIZE of every member are checked on the inflated bytes; a corrupt or
 * truncated file fails with SMR_ERR_ARG. */
int smr_upload_fastx_gz(smr_ctx*, const void* gz, uint64_t nbytes, uint32_t* nreads);
/* The text behind the resident batch (what smr_upload_fastx was given / what smr_upload_fastx_gz inflated): *nbytes = its size;
 * copied to `text` when that is not null (cap bytes available).  header_text_off of smr_resident_layout indexes it. */
int smr_resident_text(smr_ctx*, char* text, uint64_t cap, uint64_t* nbytes);
/* Test hook: inflate only.  chunk_bytes = distance of the speculative block searches (>= 1024; 0 = the default of smr_upload_fastx_gz); info = {spans decoded,
 * candidates found, device time in us, H2D time in us}. */
int smr_debug_inflate(smr_ctx*, const void* gz, uint64_t nbytes, uint64_t chunk_bytes, uint8_t* out, uint64_t out_cap, uint64_t* out_bytes, uint32_t info[4]);

/* Where the resident reads are: header_text_off[r] = offset of record r's header line in the text given to
 * smr_upload_fastx (for Read::getSeqId / report writers; nullptr = skip; only after smr_upload_fastx), read_off[0..nreads] =
 * offsets into the concatenated 0-4 codes, seq04 (optional) = those codes (seq_cap bytes available). */
int smr_resident_layout(smr_ctx*, uint64_t* header_text_off, uint64_t* read_off, uint8_t* seq04, uint64_t seq_cap);

/* Same work with the batch already resident: upload once, run many times (bench `value` leg). */
int smr_upload_batch(smr_ctx*, const uint8_t* seq_cat, const uint64_t* seq_off, uint32_t nreads);
int smr_run_resident(smr_ctx*);                       /* all kernels of one pass over the resident batch */
int smr_download_results(smr_ctx*, smr_read_result* results, smr_aln* alns, uint32_t* cigar_pool,
                         uint64_t cigar_cap, uint64_t* cigar_used, uint64_t* counters, uint32_t n_counters);

/* Device-side timings of the last smr_run_resident / smr_align_batch, CUDA events on the
 * library's stream, milliseconds: out[0]=total [1]=seed kernels [2]=candidate/SW kernels
 * [3]=finalize (reverse SW + traceback) [4]=h2d [5]=d2h; out[6]=number of kernel launches */
int smr_last_timings(const smr_ctx*, double out[8]);

/* -- multi-GPU: the only cross-read state is the counter vector (SURVEY 8(e)).  The library
 *    shards nothing itself: each rank calls smr_align_batch on its own reads and the host sums
 *    `counters` with one all-reduce (torch.distributed / NCCL, see INTEGRATION.md). */

/* -- unit-test entry points (run the same device functions the hot path uses) ------------------ */
/* seed search of explicit windows: for window k, sequence seq03 (0..3, length >= win_pos+lnwin) of
 * read read_of[k]; returns ids per window into ids[k*cap .. ), counts[k] (may exceed cap),
 * zero[k] = accept_zero_kmer.  Bit 31 of cap selects the per-lane fallback search instead of the cooperative one. */
int smr_debug_seed_windows(smr_ctx*, uint32_t part_slot, const uint8_t* seq_cat, const uint64_t* seq_off,
                           uint32_t nreads, const uint32_t* win_read, const uint32_t* win_pos, uint32_t nwin,
                           uint32_t* ids, uint32_t cap, uint32_t* counts, uint8_t* zero);
/* measured peak of dependent-free DPX (VIADDMNMX) thread-operations per second on this device, in 1e9/s:
 * the denominator of the Smith-Waterman roofline (SURVEY 8(d)) */
int smr_debug_dpx_peak(smr_ctx*, double* giga_ops_per_s);
/* ssw_align(flag=2) equivalents on explicit (query, target) pairs:
 * out[k*6..] = score1, ref_begin1, ref_end1, read_begin1, read_end1, cigar_len; cigars at k*cigar_cap */
int smr_debug_ssw(smr_ctx*, const uint8_t* q_cat, const uint64_t* q_off, const uint8_t* t_cat,
                  const uint64_t* t_off, uint32_t npairs, uint32_t filters, int32_t* out, uint32_t* cigars,
                  uint32_t cigar_cap);
/* the candidate kernel's scorer path (fetcher staging + packed 16-bit pass or s32 fallback) on explicit tasks.
 * q_cat: reads (codes 0..4, q_len bytes), t_cat: reference bytes (0..4, t_len bytes).  tasks[5*i..]: ref_abs, q_abs, n (window
 * columns), m (query rows), minus -- minus = 1: q_abs names query element 0, read backwards and complemented.  pairs[2*k..]: task A,
 * task B (0xFFFFFFFF: none).  One warp scores each run of `chain` consecutive pairs in order, as one scorer warp does (its query
 * profile cache carries over).  scores[i]: the score published for task i; path[k]: 1 = packed pass, 0 = s32 fallback.
 * SMR_ERR_ARG if a task reaches outside its buffer. */
int smr_debug_sw_tasks(smr_ctx*, const uint8_t* q_cat, uint64_t q_len, const uint8_t* t_cat, uint64_t t_len,
                       const uint32_t* tasks, uint32_t ntasks, const uint32_t* pairs, uint32_t npairs, uint32_t chain,
                       uint32_t* scores, uint8_t* path);

#ifdef __cplusplus
}
#endif
#endif
