"""ctypes binding of libsmr_b200.so (include/smr_b200.h) and a host-side driver that mirrors the
reference's `align()` call (src/sortmerna/processor.cpp:173-285): load every (index, part) given
with --ref, then push batches of reads through the GPU hot path.

There is NO CPU fallback: importing this module without the built extension, or creating an
`Aligner` without a CUDA device, raises.  (The CPU oracle lives under oracle/ and is test
infrastructure; nothing here imports it.)
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import hostio

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SMR_LIB_PATH") or os.path.join(HERE, "libsmr_b200.so")  # override: kernel-variant experiments only

STATUS = {0: "SMR_OK", 1: "SMR_ERR_CUDA", 2: "SMR_ERR_ARG", 3: "SMR_ERR_INDEX", 4: "SMR_ERR_UNSUPPORTED",
          5: "SMR_ERR_CAPACITY", 6: "SMR_ERR_NO_DEVICE"}

# every symbol include/smr_b200.h declares
SYMBOLS = ["smr_init", "smr_destroy", "smr_last_error", "smr_device_count", "smr_load_index_part",
           "smr_set_minimal_score", "smr_set_params", "smr_index_info", "smr_align_batch", "smr_upload_batch",
           "smr_run_resident", "smr_download_results", "smr_last_timings", "smr_debug_seed_windows", "smr_debug_ssw",
           "smr_debug_dpx_peak", "smr_set_stats_buffer", "smr_build_index", "smr_upload_fastx", "smr_resident_layout", "smr_pack_kvdb_blobs",
           "smr_set_aln_slots", "smr_aln_slots", "smr_aln_slots_needed", "smr_upload_fastx_gz", "smr_resident_text", "smr_debug_inflate",
           "smr_build_index_device", "smr_debug_index_array", "smr_set_instrumentation", "smr_debug_sw_tasks"]

CNT_NAMES = ("num_aligned", "num_short", "sw_calls", "sw_cells", "windows", "trie_nodes", "buckets",
             "bucket_entries", "pos_entries", "lis_calls", "dbg_max_read_cycles", "dbg_sum_read_cycles", "dbg_lis_kernel_cycles",
             "cyc_vote", "cyc_order", "cyc_group", "cyc_plan", "cyc_wait", "cyc_replay", "spec_calls", "spec_cells", "spec_pairs", "slow_pairs",
             "sc_wait", "sc_load", "sc_sw", "sc_pub", "rounds_a", "rounds_b", "w1_cyc", "w1_cnt", "dbg_max_read_busy_cycles")
CNT_FIXED = 32


class Params(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "match", "mismatch", "score_N", "gap_open", "gap_ext", "num_seeds", "min_lis", "edges",
        "edges_is_percent", "num_alignments", "is_best", "is_forward", "is_reverse", "is_full_search",
        "minoccur")]


def default_params(**kw) -> Params:
    """Runopts::validate defaults (src/sortmerna/options.cpp:1684-1738)."""
    p = Params(match=2, mismatch=-3, score_N=-3, gap_open=5, gap_ext=2, num_seeds=2, min_lis=2, edges=4,
               edges_is_percent=0, num_alignments=1, is_best=1, is_forward=1, is_reverse=1, is_full_search=0,
               minoccur=0)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


RESULT_DTYPE = np.dtype([("lastIndex", "<u4"), ("lastPart", "<u4"), ("hit_seeds", "<u4"), ("min_index", "<u4"),
                         ("max_index", "<u4"), ("n_align", "<u4"), ("max_SW_count", "<u2"), ("is_done", "u1"),
                         ("is_hit", "u1")])
ALN_DTYPE = np.dtype([("cigar_off", "<u4"), ("cigar_len", "<u4"), ("ref_num", "<u4"), ("ref_begin1", "<i4"),
                      ("ref_end1", "<i4"), ("read_begin1", "<i4"), ("read_end1", "<i4"), ("readlen", "<u4"),
                      ("score1", "<u2"), ("part", "<u2"), ("index_num", "<u2"), ("strand", "u1"), ("pad", "u1")])

STATS_DTYPE = np.dtype([("n_miss", "<u4"), ("n_gap", "<u4"), ("n_match", "<u4"), ("n_match_denovo", "<u4")])

_lib = None


def load_library():
    """Load the extension; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(nvcc, sm_100a). There is no CPU fallback for the alignment hot path.")
        L = C.CDLL(LIB_PATH)
        L.smr_last_error.restype = C.c_char_p
        L.smr_last_error.argtypes = [C.c_void_p]
        L.smr_init.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.smr_destroy.argtypes = [C.c_void_p]
        L.smr_destroy.restype = None
        L.smr_aln_slots.restype = C.c_uint32
        L.smr_aln_slots.argtypes = [C.c_void_p]
        L.smr_aln_slots_needed.restype = C.c_uint32
        L.smr_aln_slots_needed.argtypes = [C.c_void_p]
        L.smr_set_aln_slots.argtypes = [C.c_void_p, C.c_uint32]
        L.smr_set_instrumentation.argtypes = [C.c_void_p, C.c_int]
        for name in SYMBOLS:
            getattr(L, name)  # AttributeError if the build is stale
        _lib = L
    return _lib


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def build_index(fasta: str, out_prefix: str, lnwin: int = 18, interval: int = 1, max_pos: int = 10000, max_mb: float = 3072.0,
                threads: int = 0) -> dict:
    """smr_build_index: the native stand-in for the reference's `build_index` (indexdb.cpp:1119-2095).  Host code only (no GPU
    needed); writes <out_prefix>.{kmer,bursttrie,pos}_P.dat + .stats.  Defaults = the reference's (-L 18 -interval 1 -max_pos 10000 -m 3072)."""
    L = load_library()
    L.smr_build_index.argtypes = [C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, C.c_uint32, C.POINTER(C.c_uint64),
                                  C.c_char_p, C.c_size_t]
    rep = (C.c_uint64 * 6)()
    err = C.create_string_buffer(1024)
    rc = L.smr_build_index(os.fsencode(fasta), os.fsencode(out_prefix), lnwin, interval, max_pos, float(max_mb), threads, rep, err, len(err))
    if rc != 0:
        raise SmrError(f"smr_build_index({fasta}): {err.value.decode(errors='replace')}")
    return dict(zip(("parts", "numseq", "windows", "unique_lmers", "trie_nodes", "bytes_written"), (int(x) for x in rep)))


def pack_kvdb_blobs(out: dict, num_alignments: int, denovo: np.ndarray | None = None):
    """smr_pack_kvdb_blobs: Read::toBinString() of every read of a result dict (align() / download() / the oracle's), as
    (blob bytes, offsets[nreads+1]).  denovo: optional (nreads, 4) uint32 counters of hostio.denovo_classes."""
    L = load_library()
    res, alns, cig, slots = out["res"], out["alns"], np.ascontiguousarray(out["cigar"], np.uint32), int(out["slots"])
    n = res.shape[0]
    off = np.zeros(n + 1, np.uint64)
    dn = np.ascontiguousarray(denovo, np.uint32) if denovo is not None else None
    args = [_ptr(res), _ptr(alns), _ptr(cig) if cig.size else C.c_void_p(0), C.c_uint32(n), C.c_uint32(slots), C.c_int32(num_alignments),
            _ptr(dn) if dn is not None else C.c_void_p(0)]
    rc = L.smr_pack_kvdb_blobs(*args, C.c_void_p(0), C.c_uint64(0), _ptr(off))
    if rc != 0:
        raise SmrError(f"smr_pack_kvdb_blobs: {STATUS.get(rc, rc)}")
    buf = np.zeros(int(off[n]), np.uint8)
    rc = L.smr_pack_kvdb_blobs(*args, _ptr(buf) if buf.size else C.c_void_p(0), C.c_uint64(buf.size), _ptr(off))
    if rc != 0:
        raise SmrError(f"smr_pack_kvdb_blobs: {STATUS.get(rc, rc)}")
    return buf, off


class SmrError(RuntimeError):
    pass


class Aligner:
    """One GPU context.  Mirrors the objects `align()` receives: Index (+References, Refstats) via
    load_index_part, Runopts via set_params, Readfeed batches via align()."""

    def __init__(self, device: int = 0):
        self.L = load_library()
        self.h = C.c_void_p()
        rc = self.L.smr_init(device, C.byref(self.h))
        if rc != 0:
            raise SmrError(f"smr_init(device={device}) failed: {STATUS.get(rc, rc)} -- a CUDA device is required; "
                           "there is no CPU fallback")
        self.params = None
        self.n_index_files = 0
        self.refs_by_index = {}
        self._keep = []

    def _check(self, rc, what):
        if rc != 0:
            raise SmrError(f"{what}: {STATUS.get(rc, rc)}: {self.L.smr_last_error(self.h).decode()}")

    def close(self):
        if self.h:
            self.L.smr_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_params(self, params: Params):
        self.params = params
        self._check(self.L.smr_set_params(self.h, C.byref(params)), "smr_set_params")

    def set_instrumentation(self, on: bool):
        """smr_set_instrumentation: the instrumented instantiations of the seed and candidate kernels (seed-side counters and the
        cycle shares in `counters`); default off."""
        self._check(self.L.smr_set_instrumentation(self.h, C.c_int(1 if on else 0)), "smr_set_instrumentation")

    def set_aln_slots(self, slots: int):
        """smr_set_aln_slots: stride of the result layout in the all-alignments mode (num_alignments == 0)."""
        self._check(self.L.smr_set_aln_slots(self.h, C.c_uint32(slots)), "smr_set_aln_slots")

    def load_index_part(self, index_num: int, part: int, prefix: str, refs: hostio.References, minimal_score: int,
                        skiplengths=(18, 9, 3), lnwin: int = 18):
        sfx = f"_{part}.dat"
        bufs = [np.fromfile(prefix + ext + sfx, dtype=np.uint8) for ext in (".kmer", ".bursttrie", ".pos")]
        sk = (C.c_uint32 * 3)(*skiplengths)
        cat = np.ascontiguousarray(refs.cat, np.uint8)
        off = np.ascontiguousarray(refs.off, np.uint64)
        rc = self.L.smr_load_index_part(self.h, C.c_uint32(index_num), C.c_uint32(part),
                                        _ptr(bufs[0]), C.c_size_t(bufs[0].size), _ptr(bufs[1]), C.c_size_t(bufs[1].size),
                                        _ptr(bufs[2]), C.c_size_t(bufs[2].size), _ptr(cat), _ptr(off), C.c_uint32(refs.n),
                                        C.c_uint32(lnwin), C.c_uint32(minimal_score), sk)
        self._check(rc, f"smr_load_index_part({prefix})")
        self.n_index_files = max(self.n_index_files, index_num + 1)
        self.refs_by_index[index_num] = refs

    def build_index_device(self, index_num: int, fasta: str, refs=None, minimal_score: int = 0, skiplengths=(18, 9, 3), lnwin: int = 18,
                           interval: int = 1, max_pos: int = 10000, max_mb: float = 3072.0) -> int:
        """smr_build_index_device: the index of `fasta` built on the device and kept resident (every part); returns the number of
        parts.  refs: what the result formatters use for this index (a References, or the per-part list of hostio.split_by_parts)."""
        sk = (C.c_uint32 * 3)(*skiplengths)
        nparts = C.c_uint32(0)
        rep = (C.c_uint64 * 6)()
        self.L.smr_build_index_device.argtypes = [C.c_void_p, C.c_uint32, C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, C.c_void_p, C.c_uint32,
                                                  C.c_void_p, C.c_void_p]
        rc = self.L.smr_build_index_device(self.h, index_num, os.fsencode(fasta), lnwin, interval, max_pos, float(max_mb), C.cast(sk, C.c_void_p), minimal_score,
                                           C.cast(C.byref(nparts), C.c_void_p), C.cast(rep, C.c_void_p))
        self._check(rc, f"smr_build_index_device({fasta})")
        self.n_index_files = max(self.n_index_files, index_num + 1)
        if refs is not None:
            self.refs_by_index[index_num] = refs
        self.last_build_report = dict(zip(("parts", "numseq", "windows", "unique_lmers", "trie_nodes", "hbm_bytes"), (int(x) for x in rep)))
        return int(nparts.value)

    def index_array(self, slot: int, which: str) -> np.ndarray:
        """smr_debug_index_array: a resident array of loaded part `slot` (flookup u32x4 rows, flist {text,id}, pos_off, pos {pos,seq}, refseq, ref_off)."""
        k = ("flookup", "flist", "pos_off", "pos", "refseq", "ref_off").index(which)
        nb = C.c_uint64(0)
        self._check(self.L.smr_debug_index_array(self.h, C.c_uint32(slot), C.c_uint32(k), C.c_void_p(0), C.c_uint64(0), C.byref(nb)), "smr_debug_index_array")
        out = np.zeros(int(nb.value), np.uint8)
        if out.size:
            self._check(self.L.smr_debug_index_array(self.h, C.c_uint32(slot), C.c_uint32(k), _ptr(out), C.c_uint64(out.size), C.byref(nb)), "smr_debug_index_array")
        if which == "refseq":
            return out
        a = out.view(np.uint32)
        return a.reshape(-1, {"flookup": 4, "flist": 2, "pos": 2}.get(which, 1)) if which in ("flookup", "flist", "pos") else a

    def set_minimal_score(self, index_num: int, score: int):
        self._check(self.L.smr_set_minimal_score(self.h, C.c_uint32(index_num), C.c_uint32(score)), "smr_set_minimal_score")

    def index_info(self):
        out = np.zeros(6, np.uint64)
        self._check(self.L.smr_index_info(self.h, _ptr(out)), "smr_index_info")
        return dict(zip(("parts", "hbm_bytes", "nodes", "entries", "ids", "positions"), map(int, out)))

    def _outputs(self, n, reuse=False):
        slots = int(self.L.smr_aln_slots(self.h))   # num_alignments, or the stride of the all-alignments mode (0)
        if reuse:   # the same host buffers for every call of this shape (a streaming caller consumes a batch before the next)
            key = (n, slots, self.n_index_files)
            if getattr(self, "_out_key", None) != key:
                self._out_key, self._out_bufs = key, self._outputs(n)
            bufs = self._out_bufs
            bufs[5][:] = 0
            return bufs
        res = np.zeros(n, RESULT_DTYPE)
        alns = np.zeros(n * slots, ALN_DTYPE)
        cap = 48 * n * slots + 4096
        pool = np.zeros(cap, np.uint32)
        counters = np.zeros(CNT_FIXED + max(1, self.n_index_files), np.uint64)
        return slots, res, alns, pool, cap, counters

    def _pack(self, res, alns, pool, used, counters, slots):
        cnt = {k: int(counters[i]) for i, k in enumerate(CNT_NAMES)}
        return dict(res=res, alns=alns, cigar=pool[: used], matched=counters[CNT_FIXED:].copy(), counters=cnt,
                    slots=slots, timings=self.timings())

    def align(self, cat: np.ndarray, off: np.ndarray, with_stats: bool = False, reuse_outputs: bool = False):
        """smr_align_batch: host buffers in, host results out (H2D and D2H inside the call).
        with_stats: also return calc_miss_gap_match per stored alignment (out["stats"], computed on the GPU).
        reuse_outputs: write into the result buffers of the previous call of the same shape (valid until the next call)
        instead of allocating ~260 B/read of fresh zeroed host memory per call."""
        cat = np.ascontiguousarray(cat, np.uint8)
        off = np.ascontiguousarray(off, np.uint64)
        n = off.size - 1
        while True:
            slots, res, alns, pool, cap, counters = self._outputs(n, reuse_outputs)
            stats = np.zeros(n * slots, STATS_DTYPE) if with_stats else None
            self._check(self.L.smr_set_stats_buffer(self.h, _ptr(stats) if with_stats else C.c_void_p(0)), "smr_set_stats_buffer")
            used = C.c_uint64(0)
            rc = self.L.smr_align_batch(self.h, _ptr(cat), _ptr(off), C.c_uint32(n), _ptr(res), _ptr(alns), _ptr(pool),
                                        C.c_uint64(cap), C.byref(used), _ptr(counters), C.c_uint32(counters.size))
            need = int(self.L.smr_aln_slots_needed(self.h)) if rc == 5 and self.params.num_alignments == 0 else 0
            if need > slots:   # all-alignments mode: the library names the stride this batch needs; allocate and run again
                self.set_aln_slots(need)
                continue
            break
        self._check(rc, "smr_align_batch")
        self.L.smr_set_stats_buffer(self.h, C.c_void_p(0))
        out = self._pack(res, alns, pool, used.value, counters, slots)
        if with_stats:
            out["stats"] = stats
        return out

    def upload(self, cat: np.ndarray, off: np.ndarray):
        cat = np.ascontiguousarray(cat, np.uint8)
        off = np.ascontiguousarray(off, np.uint64)
        self._n_resident = off.size - 1
        self._check(self.L.smr_upload_batch(self.h, _ptr(cat), _ptr(off), C.c_uint32(off.size - 1)), "smr_upload_batch")

    def upload_fastx(self, text: bytes) -> int:
        """smr_upload_fastx: the bytes of an uncompressed FASTA / FASTQ file; record split and 0-4 encoding run on the device.
        Returns the number of reads; continue with run_resident() / download()."""
        n = C.c_uint32(0)
        buf = np.frombuffer(text, dtype=np.uint8)
        self._check(self.L.smr_upload_fastx(self.h, _ptr(buf), C.c_uint64(buf.size), C.byref(n)), "smr_upload_fastx")
        self._n_resident = int(n.value)
        return self._n_resident

    def upload_fastx_gz(self, gz: bytes) -> int:
        """smr_upload_fastx_gz: the bytes of a .fastq.gz / .fasta.gz; gzip inflate, record split and 0-4 encoding run on the device."""
        n = C.c_uint32(0)
        buf = np.frombuffer(gz, dtype=np.uint8)
        self._check(self.L.smr_upload_fastx_gz(self.h, _ptr(buf), C.c_uint64(buf.size), C.byref(n)), "smr_upload_fastx_gz")
        self._n_resident = int(n.value)
        return self._n_resident

    def resident_text(self) -> bytes:
        """smr_resident_text: the (inflated) text behind the resident batch; header offsets of resident_layout() index it."""
        nb = C.c_uint64(0)
        self._check(self.L.smr_resident_text(self.h, C.c_void_p(0), C.c_uint64(0), C.byref(nb)), "smr_resident_text")
        out = np.zeros(int(nb.value), np.uint8)
        if out.size:
            self._check(self.L.smr_resident_text(self.h, _ptr(out), C.c_uint64(out.size), C.byref(nb)), "smr_resident_text")
        return out.tobytes()

    def debug_inflate(self, gz: bytes, chunk_bytes: int = 65536, cap: int = 0):
        """smr_debug_inflate: (inflated bytes, {spans, candidates, device_us, h2d_us})."""
        buf = np.frombuffer(gz, dtype=np.uint8)
        nb = C.c_uint64(0)
        info = (C.c_uint32 * 4)()
        self._check(self.L.smr_debug_inflate(self.h, _ptr(buf), C.c_uint64(buf.size), C.c_uint64(chunk_bytes), C.c_void_p(0), C.c_uint64(0), C.byref(nb), info),
                    "smr_debug_inflate")
        out = np.zeros(int(nb.value), np.uint8)
        if out.size:   # the inflated text is still in the context's buffer
            nb2 = C.c_uint64(0)
            self.L.smr_resident_text.restype = C.c_int
            self._check(self.L.smr_debug_inflate(self.h, _ptr(buf), C.c_uint64(buf.size), C.c_uint64(chunk_bytes), _ptr(out), C.c_uint64(out.size), C.byref(nb2), info),
                        "smr_debug_inflate")
        return out.tobytes(), {"spans": info[0], "candidates": info[1], "device_us": info[2], "h2d_us": info[3]}

    def resident_layout(self, with_headers: bool = True, with_seq: bool = True):
        """smr_resident_layout: (header offsets in the uploaded text, read offsets, concatenated 0-4 codes) of the resident batch."""
        n = self._n_resident
        hdr = np.zeros(n, np.uint64) if with_headers else None
        off = np.zeros(n + 1, np.uint64)
        self._check(self.L.smr_resident_layout(self.h, _ptr(hdr) if with_headers and n else C.c_void_p(0), _ptr(off), C.c_void_p(0), C.c_uint64(0)),
                    "smr_resident_layout")
        seq = None
        if with_seq:
            seq = np.zeros(int(off[n]), np.uint8)
            if seq.size:
                self._check(self.L.smr_resident_layout(self.h, C.c_void_p(0), C.c_void_p(0), _ptr(seq), C.c_uint64(seq.size)), "smr_resident_layout")
        return hdr, off, seq

    def run_resident(self):
        self._check(self.L.smr_run_resident(self.h), "smr_run_resident")

    def download(self):
        n = self._n_resident
        slots, res, alns, pool, cap, counters = self._outputs(n)
        used = C.c_uint64(0)
        rc = self.L.smr_download_results(self.h, _ptr(res), _ptr(alns), _ptr(pool), C.c_uint64(cap), C.byref(used),
                                         _ptr(counters), C.c_uint32(counters.size))
        self._check(rc, "smr_download_results")
        return self._pack(res, alns, pool, used.value, counters, slots)

    def timings(self):
        out = np.zeros(8, np.float64)
        self.L.smr_last_timings(self.h, _ptr(out))
        return dict(total_ms=out[0], seed_ms=out[1], lis_ms=out[2], final_ms=out[3], h2d_ms=out[4], d2h_ms=out[5],
                    launches=int(out[6]), decode_ms=out[7])

    def dpx_peak(self) -> float:
        """measured dependent-free DPX thread-ops/s (1e9/s) on this device"""
        v = C.c_double(0)
        self._check(self.L.smr_debug_dpx_peak(self.h, C.byref(v)), "smr_debug_dpx_peak")
        return v.value

    # ---- unit-test entry points ----
    def debug_seed_windows(self, part_slot, cat03, off, win_read, win_pos, cap=64, fallback_path=False):
        cat03 = np.ascontiguousarray(cat03, np.uint8)
        off = np.ascontiguousarray(off, np.uint64)
        win_read = np.ascontiguousarray(win_read, np.uint32)
        win_pos = np.ascontiguousarray(win_pos, np.uint32)
        nwin = win_read.size
        ids = np.zeros(nwin * cap, np.uint32)
        counts = np.zeros(nwin, np.uint32)
        zero = np.zeros(nwin, np.uint8)
        rc = self.L.smr_debug_seed_windows(self.h, C.c_uint32(part_slot), _ptr(cat03), _ptr(off), C.c_uint32(off.size - 1),
                                           _ptr(win_read), _ptr(win_pos), C.c_uint32(nwin), _ptr(ids),
                                           C.c_uint32(cap | (0x80000000 if fallback_path else 0)), _ptr(counts), _ptr(zero))
        self._check(rc, "smr_debug_seed_windows")
        return ids.reshape(nwin, cap), counts, zero

    def debug_ssw(self, q_cat, q_off, t_cat, t_off, filters=0, cigar_cap=256):
        q_cat = np.ascontiguousarray(q_cat, np.uint8)
        t_cat = np.ascontiguousarray(t_cat, np.uint8)
        q_off = np.ascontiguousarray(q_off, np.uint64)
        t_off = np.ascontiguousarray(t_off, np.uint64)
        n = q_off.size - 1
        out = np.zeros(n * 6, np.int32)
        cig = np.zeros(n * cigar_cap, np.uint32)
        rc = self.L.smr_debug_ssw(self.h, _ptr(q_cat), _ptr(q_off), _ptr(t_cat), _ptr(t_off), C.c_uint32(n),
                                  C.c_uint32(filters), _ptr(out), _ptr(cig), C.c_uint32(cigar_cap))
        self._check(rc, "smr_debug_ssw")
        return out.reshape(n, 6), cig.reshape(n, cigar_cap)

    def debug_sw_tasks(self, q_cat, t_cat, tasks, pairs, chain=1):
        """The candidate kernel's scorer path on explicit tasks.  tasks: (ntasks, 5) rows (ref_abs, q_abs, n, m, minus) into t_cat /
        q_cat (codes 0..4); pairs: (npairs, 2) task indices, -1 = no task B.  Returns (score per task, packed-path flag per pair)."""
        q_cat = np.ascontiguousarray(q_cat, np.uint8)
        t_cat = np.ascontiguousarray(t_cat, np.uint8)
        tasks = np.ascontiguousarray(np.asarray(tasks, np.int64).reshape(-1, 5).astype(np.uint32))
        pairs = np.ascontiguousarray(np.asarray(pairs, np.int64).reshape(-1, 2).astype(np.uint32))
        scores = np.zeros(tasks.shape[0], np.uint32)
        path = np.zeros(pairs.shape[0], np.uint8)
        rc = self.L.smr_debug_sw_tasks(self.h, _ptr(q_cat), C.c_uint64(q_cat.size), _ptr(t_cat), C.c_uint64(t_cat.size), _ptr(tasks),
                                       C.c_uint32(tasks.shape[0]), _ptr(pairs), C.c_uint32(pairs.shape[0]), C.c_uint32(chain),
                                       _ptr(scores), _ptr(path))
        self._check(rc, "smr_debug_sw_tasks")
        return scores.astype(np.int64), path.astype(bool)


def align_files(aligner: Aligner, batch: hostio.ReadBatch):
    """Convenience: align a parsed read batch and return results + SAM rows."""
    out = aligner.align(batch.cat, batch.off)
    refs = [aligner.refs_by_index[i] for i in range(aligner.n_index_files)]
    out["sam"] = hostio.format_sam_rows(batch, refs, out["res"], out["alns"], out["cigar"], out["slots"])
    return out
