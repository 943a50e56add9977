#!/usr/bin/env python
"""bench.py -- reads/sec of the alignment hot path (150 bp reads vs the 8 bundled rRNA databases).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--reads R] [--impl ours|reference] [--db-dir DIR] [--work-dir DIR]
                  [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of R/K synthetic reads per GPU (default: BASELINE.json
config "10 M synthetic 150 bp Illumina reads vs all 8 data/rRNA_databases refs, 1xB200").  The 8 databases are the FASTA
files of --db-dir (the reference's data/rRNA_databases, e.g. as tools/stage_data.py stages them) or, by default, the seeded
synthetic stand-ins of tools/synth_db.py; they and their index files live in a temporary directory for the run, or in
--work-dir, where a later run finds and reuses them.
  value  : whole-job reads/s, kernels only, batch resident in HBM (CUDA events inside the C ABI)
  e2e    : reads/s through smr_align_batch with pinned HOST buffers (H2D + kernels + D2H inside the timed region)
  roofline: the seed-search kernel (dominant) against the measured HBM peak
  cpu_baseline: the reference CPU build (oracle/_ref/sortmerna_ref), all host threads, bounded sample
--impl reference times that same reference build only (rank 0), one bounded sample per step.
"""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from sortmerna_b200 import hostio  # noqa: E402
from tools import stage_data, synth_db  # noqa: E402

READ_LEN = 150
GEN_SEED = 20260924
METRIC = "reads/sec (150 bp vs SILVA-8)"
METRIC_SYNTHETIC = "reads/sec (150 bp vs synthetic SILVA-8)"


# ------------------------------------------------------------------------------------------------
# workload: synthetic Illumina-like reads (SURVEY 8(d) config 3): 1/3 at 1 % substitutions + 0.1 % indels,
# 1/3 at 10 % + 1 %, 1/3 i.i.d. uniform ACGT; sources sampled uniformly over the nucleotides of the 8
# databases (sequences >= 150 nt), random strand.  Returned in the 0..3 alphabet the C ABI takes.
# ------------------------------------------------------------------------------------------------
class DbPool:
    def __init__(self, refs_list):
        self.cat = np.concatenate([r.cat for r in refs_list])
        starts = []
        base = 0
        for r in refs_list:
            off = r.off.astype(np.int64)
            for i in range(r.n):
                n = int(off[i + 1] - off[i])
                if n >= READ_LEN:
                    starts.append((base + int(off[i]), n - READ_LEN + 1))
            base += int(off[-1])
        s = np.array(starts, dtype=np.int64)
        self.seq_start, self.seq_nwin = s[:, 0], s[:, 1]
        self.cum = np.cumsum(self.seq_nwin)

    def sample_starts(self, rng, n):
        u = rng.integers(0, int(self.cum[-1]), n)
        k = np.searchsorted(self.cum, u, side="right")
        prev = np.where(k > 0, self.cum[k - 1], 0)
        return self.seq_start[k] + (u - prev)


def gen_reads(pool, n, seed):
    """Returns an (n, 150) uint8 array in the 0..3 alphabet.  Generated with torch on the GPU when one is
    visible (10 M reads in about a second), else on the CPU (only ever used for small samples there)."""
    import torch
    if not torch.cuda.is_available():
        return _gen_reads_numpy(pool, n, seed)
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev); g.manual_seed(seed)
    if not hasattr(pool, "_t") or pool._t.device != dev:
        pool._t = torch.from_numpy(pool.cat).to(dev)
        pool._start = torch.from_numpy(pool.seq_start).to(dev)
        pool._cum = torch.from_numpy(pool.cum).to(dev)
    out = np.empty((n, READ_LEN), dtype=np.uint8)
    W = READ_LEN + 2
    col = torch.arange(READ_LEN, device=dev)[None, :]
    colw = torch.arange(W, device=dev)[None, :]
    CH = 1 << 20
    for c0 in range(0, n, CH):
        m = min(CH, n - c0)
        cls = torch.randint(0, 3, (m,), generator=g, device=dev)
        u = torch.randint(0, int(pool.cum[-1]), (m,), generator=g, device=dev)
        k = torch.searchsorted(pool._cum, u, right=True)
        prev = torch.where(k > 0, pool._cum[(k - 1).clamp(min=0)], torch.zeros_like(u))
        st = pool._start[k] + (u - prev)
        idx = (st[:, None] + colw).clamp(max=pool._t.numel() - 1)
        src = pool._t[idx]                                         # 152 columns: room for one deletion
        rnd_w = torch.randint(0, 4, (m, W), generator=g, device=dev, dtype=torch.uint8)
        src = torch.where(src > 3, rnd_w, src)
        sub_p = torch.where(cls == 0, 0.01, 0.10)[:, None]
        sub = torch.rand((m, W), generator=g, device=dev) < sub_p
        src = torch.where(sub, torch.randint(0, 4, (m, W), generator=g, device=dev, dtype=torch.uint8), src)
        # one indel event per read with probability 150 * rate (0.1 % / 1 %)
        ind_p = torch.where(cls == 0, 0.001, 0.01) * READ_LEN
        has = torch.rand((m,), generator=g, device=dev) < ind_p
        pos = torch.randint(5, READ_LEN - 5, (m,), generator=g, device=dev)[:, None]
        is_del = (torch.rand((m,), generator=g, device=dev) < 0.5)
        hd, hi = (has & is_del)[:, None], (has & ~is_del)[:, None]
        take = torch.where(hd, col + (col >= pos).long(), torch.where(hi, col - (col > pos).long(), col.expand(m, -1)))
        r = torch.gather(src, 1, take)
        rnd = torch.randint(0, 4, (m, READ_LEN), generator=g, device=dev, dtype=torch.uint8)
        r = torch.where(hi & (col == pos), rnd, r)                 # the inserted base
        r = torch.where((cls == 2)[:, None], torch.randint(0, 4, (m, READ_LEN), generator=g, device=dev, dtype=torch.uint8), r)
        flip = (torch.rand((m,), generator=g, device=dev) < 0.5)[:, None]
        r = torch.where(flip, (3 - r).flip(1), r)
        out[c0:c0 + m] = r.cpu().numpy()
    return out


def _gen_reads_numpy(pool, n, seed):
    """CPU twin of gen_reads (same mixture, numpy generator)."""
    rng = np.random.default_rng(seed)
    out = np.empty((n, READ_LEN), dtype=np.uint8)
    W = READ_LEN + 2
    CH = 1 << 18
    col = np.arange(READ_LEN)[None, :]
    for c0 in range(0, n, CH):
        m = min(CH, n - c0)
        cls = rng.integers(0, 3, m)
        st = pool.sample_starts(rng, m)
        idx = np.minimum(st[:, None] + np.arange(W)[None, :], pool.cat.size - 1)
        src = pool.cat[idx]
        src = np.where(src > 3, rng.integers(0, 4, src.shape, dtype=np.uint8), src)
        sub = rng.random((m, W), dtype=np.float32) < np.where(cls == 0, 0.01, 0.10)[:, None]
        src = np.where(sub, rng.integers(0, 4, src.shape, dtype=np.uint8), src)
        has = rng.random(m) < np.where(cls == 0, 0.001, 0.01) * READ_LEN
        pos = rng.integers(5, READ_LEN - 5, m)[:, None]
        is_del = rng.random(m) < 0.5
        hd, hi = (has & is_del)[:, None], (has & ~is_del)[:, None]
        take = np.where(hd, col + (col >= pos), np.where(hi, col - (col > pos), col))
        r = np.take_along_axis(src, take, axis=1)
        r = np.where(hi & (col == pos), rng.integers(0, 4, r.shape, dtype=np.uint8), r)
        r = np.where((cls == 2)[:, None], rng.integers(0, 4, (m, READ_LEN), dtype=np.uint8), r)
        flip = (rng.random(m) < 0.5)[:, None]
        out[c0:c0 + m] = np.where(flip, (3 - r)[:, ::-1], r)
    return out


def write_fastq(path, reads):
    """Illumina-like 4-line FASTQ, constant quality 'I', fixed-width ids (records of equal size: written as one array)."""
    n = reads.shape[0]
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    rec = np.empty((n, 10 + 1 + READ_LEN + 3 + READ_LEN + 1), dtype=np.uint8)
    ids = np.char.zfill(np.arange(n).astype("S9"), 9)
    rec[:, 0] = ord("@"); rec[:, 1:10] = np.frombuffer(ids.tobytes(), dtype=np.uint8).reshape(n, 9); rec[:, 10] = 10
    rec[:, 11:11 + READ_LEN] = lut[reads]
    o = 11 + READ_LEN
    rec[:, o] = 10; rec[:, o + 1] = ord("+"); rec[:, o + 2] = 10
    rec[:, o + 3:o + 3 + READ_LEN] = ord("I"); rec[:, o + 3 + READ_LEN] = 10
    with open(path, "wb") as f:
        f.write(rec.tobytes())


# ------------------------------------------------------------------------------------------------
def load_databases(tmp, db_dir=None, native_index=True):
    """The 8 databases in --ref order: the FASTA files of db_dir, or the synthetic ones written under tmp; index files under tmp.
    What tmp already holds is reused."""
    if db_dir:
        fastas = [os.path.join(db_dir, n + ".fasta") for n in stage_data.DBS]
        missing = [f for f in fastas if not os.path.exists(f)]
        if missing:
            raise SystemExit(f"missing database FASTA files {missing}")
    else:
        fastas = synth_db.write_databases(os.path.join(tmp, "databases"))
    if not native_index:
        return fastas, None, None, [hostio.load_references(f) for f in fastas], None, {}
    idx_dir, built = stage_data.ensure_indexes(fastas, os.path.join(tmp, "idx"))   # smr_build_index (our builder), 8 databases in parallel
    pre = hostio.find_index_prefixes(idx_dir)
    refs = [hostio.load_references(f) for f in fastas]
    stats = [hostio.parse_stats(pre[os.path.basename(f)]) for f in fastas]
    return fastas, idx_dir, [pre[os.path.basename(f)] for f in fastas], refs, stats, built


def load_resident_index(al, source, fastas, prefixes, refs, ms, stats):
    """The 8 databases resident in HBM: built on the device from the FASTA files, or flattened from the on-disk index."""
    for k in range(len(fastas)):
        if source == "device":
            if al.build_index_device(k, fastas[k], refs[k], ms[k], (18, 9, 3), stats[k].lnwin) != 1:
                raise SystemExit("the benchmark databases are single-part indexes")
        else:
            al.load_index_part(k, 0, prefixes[k], refs[k], ms[k], (18, 9, 3), stats[k].lnwin)


def survey_8d_seed(fastas, prefixes, refs, ms, stats, reads03, threads, reads_per_step, seed_ms, peak_gbs):
    """Bytes per read of SURVEY 8(d)'s seed figure: windows x 8 B (two k-mer counts) + visited trie nodes x 4 B + visited buckets x
    (4 B + 8 B x entries) + read bases 1 B/nt per (strand, index part), counted by the oracle's walk (oracle/smr_oracle.cpp: the
    reference's pass schedule and pruned DFS) -- and the rate / fraction of the HBM peak the seed kernels reach measured against it."""
    from oracle import ora
    n = reads03.shape[0]
    batch = hostio.ReadBatch([f"@r{i}" for i in range(n)], [b""] * n, [b""] * n, np.ascontiguousarray(reads03.reshape(-1)),
                             (np.arange(n + 1, dtype=np.uint64) * READ_LEN))
    oix = [ora.OracleIndex(p, 0, st.lnwin) for p, st in zip(prefixes, stats)]
    k = len(oix)
    got = ora.align(oix, list(range(k)), [0] * k, k, refs, ms, [18, 9, 3] * k, ora.default_params(), batch, nthreads=max(1, min(threads, 16)))
    c = got["counters"]
    per_read = (c["windows"] * 8 + c["trie_nodes"] * 4 + c["buckets"] * 4 + c["bucket_entries"] * 8) / n + READ_LEN * 2 * k
    ach = per_read * reads_per_step / (seed_ms / 1e3) / 1e9
    return {"bytes_per_read": round(per_read, 1), "achieved": ach, "unit": "GB/s", "frac": ach / peak_gbs,
            "per_read": {kk: round(c[kk] / n, 1) for kk in ("windows", "trie_nodes", "buckets", "bucket_entries")},
            "sample": f"oracle walk (reference pass schedule + pruned DFS) on the first {n} reads of the workload, 8 databases"}


def db_source(args):
    return os.path.abspath(args.db_dir) if args.db_dir else f"synthetic (tools/synth_db.py, seed {synth_db.SEED})"


def db_words(args):
    return "all 8 data/rRNA_databases refs" if args.db_dir else "synthetic stand-ins of the 8 data/rRNA_databases refs"


def reference_index_dir(fastas, tmp):
    """The reference legs (cpu_baseline, --impl reference) run the unmodified binary on the index ITS OWN builder makes
    (<tmp>/idx_ref; one process per database, outside every timed region) -- never on files our builder wrote."""
    d, _ = stage_data.ensure_indexes(fastas, os.path.join(tmp, "idx_ref"), builder="reference")
    return d


def minimal_scores(stats, fastas, nreads_total):
    g = json.load(open(os.path.join(ROOT, "sortmerna_b200", "gumbel_defaults.json")))["gumbel"]
    return [hostio.minimal_score(st, g[os.path.basename(f)]["lambda_"], g[os.path.basename(f)]["K"], nreads_total * READ_LEN, nreads_total)
            for st, f in zip(stats, fastas)]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, dev):
        super().__init__(daemon=True)
        self.dev, self.rows, self.stop_flag = dev, [], False

    def run(self):
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                   stdout=subprocess.PIPE, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = []
        for i, n in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")):
            if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows):
                reasons.append(n)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons, samples=len(self.rows))


def run_reference_sample(fastas, idx_dir, reads, threads):
    """The reference's own align() on a bounded sample: returns (reads/s over the per-index alignment loops,
    seconds, 'Done alignment' seconds incl. index loading)."""
    from oracle import ora
    with tempfile.TemporaryDirectory(prefix="smr_ref_") as d:
        fq = os.path.join(d, "sample.fq")
        write_fastq(fq, reads)
        r = ora.run_reference(fastas, fq, os.path.join(d, "w"), extra=["-fastx"], threads=threads, idx_dir=idx_dir)
        per_idx = [float(x) for x in re.findall(r"done index: \d+ part: \d+ in ([0-9.eE+-]+) sec", r["stdout"])]
        m = re.search(r"Done alignment in ([0-9.eE+-]+) sec", r["stdout"])
        total = float(m.group(1)) if m else float("nan")
        t = sum(per_idx) if per_idx else total
        log = ora.parse_log(r["log"])
    return reads.shape[0] / t, t, total, log


def host_cores():
    """Threads the reference CPU arm may really use: the affinity mask AND the cgroup CPU quota (os.cpu_count() ignores both).
    Returns (threads to use, description)."""
    ncpu = os.cpu_count() or 1
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = ncpu
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                      # cgroup v2: "<quota> <period>" or "max <period>"
            q, per = f.read().split()[:2]
            if q != "max":
                quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    eff = aff if quota is None else max(1, min(aff, int(quota + 0.5)))
    try:
        load = os.getloadavg()[0]
    except Exception:
        load = float("nan")
    return eff, dict(os_cpu_count=ncpu, affinity=aff, cgroup_quota=quota, threads_used=eff, loadavg_1m=load)


def cli_e2e(args, cores, core_info, tmp):
    """What a user runs: the reference's host program with the binding (oracle/_ref/sortmerna_gpu -ref x8 -reads file.fq) against
    the unmodified reference binary on the same file -- 'Done alignment' seconds and total wall, flat FASTQ (and .gz with
    --cli-gz).  The CPU binary gets a bounded prefix of the same file (its cost is linear in reads)."""
    import gzip
    import shutil
    from oracle import ora
    fastas, idx_dir, _, refs, _, _ = load_databases(tmp, args.db_dir)
    ref_idx = reference_index_dir(fastas, tmp)
    pool = DbPool(refs)
    n = args.cli_reads
    gpu_bin = os.path.join(ROOT, "oracle", "_ref", "sortmerna_gpu")
    out = {"reads": n, "gpus": args.cli_gpus, "host": core_info}
    with tempfile.TemporaryDirectory(prefix="smr_cli_") as d:
        reads = gen_reads(pool, n, GEN_SEED + 4242)
        fq = os.path.join(d, "reads.fq")
        write_fastq(fq, reads)
        inputs = [("flat", fq)]
        if args.cli_gz:
            gz = fq + ".gz"
            with open(fq, "rb") as fi, gzip.open(gz, "wb", compresslevel=1) as fo:
                shutil.copyfileobj(fi, fo, 1 << 24)
            inputs.append(("gz", gz))
        env = dict(os.environ, SMR_GPUS=str(args.cli_gpus))
        for name, path in inputs:
            cmd = [gpu_bin] + sum((["-ref", f] for f in fastas), []) + ["-reads", path, "-workdir", os.path.join(d, "w_" + name), "-idx-dir", idx_dir,
                                                                      "-threads", str(cores), "-task", "4", "-fastx", "-sam"]
            t0 = time.perf_counter()
            p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env, timeout=3000)
            wall = time.perf_counter() - t0
            if p.returncode != 0:
                raise SystemExit("sortmerna_gpu failed:\n" + p.stdout[-3000:])
            m = re.search(r"Done alignment in ([0-9.eE+-]+) sec", p.stdout)
            m2 = re.search(r"resident on \d+ GPU\(s\) in ([0-9.eE+-]+) sec; reads streamed, aligned and stored in ([0-9.eE+-]+) sec", p.stdout)
            log = ora.parse_log(open(os.path.join(d, "w_" + name, "out", "aligned.log")).read())
            out["gpu_" + name] = {"wall_s": wall, "done_alignment_s": float(m.group(1)) if m else None, "index_load_s": float(m2.group(1)) if m2 else None,
                                  "stream_align_store_s": float(m2.group(2)) if m2 else None, "reads_per_s_alignment": n / float(m2.group(2)) if m2 else None,
                                  "reads_per_s_wall": n / wall, "passing": log["passing"], "failing": log["failing"]}
        ncpu = min(n, args.cli_cpu_reads)
        fq_cpu = os.path.join(d, "reads_cpu.fq")
        write_fastq(fq_cpu, reads[:ncpu])
        t0 = time.perf_counter()
        r = ora.run_reference(fastas, fq_cpu, os.path.join(d, "w_cpu"), extra=["-fastx", "-sam"], threads=cores, idx_dir=ref_idx)
        wall = time.perf_counter() - t0
        m = re.search(r"Done alignment in ([0-9.eE+-]+) sec", r["stdout"])
        log = ora.parse_log(r["log"])
        out["cpu_flat"] = {"reads": ncpu, "threads": cores, "wall_s": wall, "done_alignment_s": float(m.group(1)) if m else None,
                           "reads_per_s_alignment": ncpu / float(m.group(1)) if m else None, "reads_per_s_wall": ncpu / wall,
                           "passing": log["passing"], "failing": log["failing"]}
    return out


# counters only the instrumented instantiations of the kernels fill (include/smr_b200.h: smr_set_instrumentation)
INSTR_ONLY = ("windows", "trie_nodes", "buckets", "bucket_entries", "dbg_max_read_cycles", "dbg_sum_read_cycles", "dbg_lis_kernel_cycles",
              "cyc_vote", "cyc_order", "cyc_group", "cyc_plan", "cyc_wait", "cyc_replay", "sc_wait", "sc_load", "sc_sw", "sc_pub", "w1_cyc",
              "dbg_max_read_busy_cycles")


# the per-read and per-alignment fields --dump-outputs writes (cigar_off is a position in the batch's CIGAR pool: the words
# themselves are written instead), and the counters that count algorithmic work (the same in every run of the same inputs)
DUMP_RES_FIELDS = ["lastIndex", "lastPart", "hit_seeds", "min_index", "max_index", "n_align", "max_SW_count", "is_done", "is_hit"]
DUMP_ALN_FIELDS = ["cigar_len", "ref_num", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "readlen", "score1", "part", "index_num", "strand"]
DUMP_COUNTERS = ("num_aligned", "sw_calls", "sw_cells", "pos_entries", "lis_calls")
DUMP_READS = 1 << 16


def dump_outputs(out_dir, res, read0):
    """What the last timed step returned to its caller (api.Aligner.download()), as float64 .npy files: every field of
    the per-read results and of the stored alignments of a fixed, seeded sample of DUMP_READS reads, their CIGAR words,
    the per-database match counts and the algorithmic counters of the whole batch.  read0: global number of the batch's
    first read."""
    os.makedirs(out_dir, exist_ok=True)
    n, slots = res["res"].shape[0], int(res["slots"])
    pick = np.sort(np.random.default_rng(GEN_SEED).choice(n, min(n, DUMP_READS), replace=False))
    arrays = {"read_index": pick + read0}
    for f in DUMP_RES_FIELDS:
        arrays["res." + f] = res["res"][f][pick]
    alns = res["alns"].reshape(n, slots)[pick] if slots else res["alns"][:0]
    for f in DUMP_ALN_FIELDS:
        arrays["alns." + f] = alns[f]
    flat = alns.reshape(-1)
    cig = res["cigar"]
    arrays["cigar"] = np.concatenate([cig[int(o):int(o) + int(k)] for o, k in zip(flat["cigar_off"], flat["cigar_len"])] or [cig[:0]])
    arrays["matched"] = res["matched"]
    for k in DUMP_COUNTERS:
        arrays["counters." + k] = np.array([res["counters"][k]])
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per GPU in the whole job; one step = reads/steps of them")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--index-source", default="device", choices=["device", "files"],
                    help="device: every database indexed on the GPU straight from its FASTA (smr_build_index_device); files: the on-disk index "
                         "(smr_build_index) flattened by smr_load_index_part.  Same resident arrays up to the id numbering; untimed either way")
    ap.add_argument("--cpu-sample", type=int, default=0, help="reads in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cli-e2e", action="store_true", help="time the drop-in host program (oracle/_ref/sortmerna_gpu) against the reference binary and exit")
    ap.add_argument("--cli-reads", type=int, default=2_000_000)
    ap.add_argument("--cli-cpu-reads", type=int, default=100_000)
    ap.add_argument("--cli-gpus", type=int, default=1)
    ap.add_argument("--cli-gz", action="store_true")
    ap.add_argument("--db-dir", default=None, help="directory of the 8 database FASTA files (default: the synthetic databases of tools/synth_db.py)")
    ap.add_argument("--work-dir", default=None, help="where the databases and their index files are written, and reused by later runs "
                                                     "(default: a temporary directory of this run)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step returned (a seeded sample of the reads, every result field) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    tmp = tempfile.mkdtemp(prefix="smr_bench_")     # databases, index files, reference work directories: never in the tree
    try:
        run(args, tmp)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run(args, tmp):
    # stdout carries exactly ONE JSON line: everything else that writes to fd 1 (NCCL's version banner, library chatter) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores, core_info = host_cores()

    work = args.work_dir or tmp
    if args.cli_e2e:
        emit({"cli_e2e": cli_e2e(args, cores, core_info, work)})
        return

    if args.impl == "reference":
        if rank != 0:
            return
        fastas, _, _, refs, _, _ = load_databases(work, args.db_dir, native_index=False)
        idx_dir = reference_index_dir(fastas, work)
        pool = DbPool(refs)
        # ~10 s of reference CPU time per step (about 230 reads/s per core on this workload): large enough that thread start-up
        # and the skew between the reference's static per-thread splits do not dominate (round 1: 300 reads per thread did)
        sample = args.cpu_sample or int(min(400_000, max(20_000, 2_300 * cores)))
        vals, secs = [], []
        for s in range(args.warmup + args.steps):
            if s < args.warmup and s > 0:
                continue  # one warm-up run is enough to page the index files in; each run is tens of seconds
            reads = gen_reads(pool, sample, GEN_SEED + 1000 + s)
            v, t, total, _ = run_reference_sample(fastas, idx_dir, reads, cores)
            if s >= args.warmup:
                vals.append(v); secs.append(t)
        v = float(np.mean(vals))
        desc = f"{sample} synthetic 150 bp reads per step vs the 8 databases, alignment loops only (index loading excluded), -threads {cores}"
        emit(({
            "metric": METRIC if args.db_dir else METRIC_SYNTHETIC, "value": v, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * float(np.mean(secs)), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int16/u8 (SSE2)", "data": "synthetic", "impl": "reference",
            "config": {"workload": f"10 M synthetic 150 bp Illumina reads vs {db_words(args)}, 1xB200",
                       "sampled": "each step is a bounded sample of that workload (reads_per_step reads, same generator)",
                       "reads_per_step": sample, "read_len": READ_LEN, "databases": 8, "database_files": db_source(args)},
            "cpu_baseline": {"value": v, "unit": "reads/s", "cores": cores, "kind": "reference", "sample": desc, "host": core_info,
                             "per_step": [float(x) for x in vals]},
            "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return

    import torch
    from sortmerna_b200 import api
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    t_setup = time.time()
    if world > 1:       # the databases and their indexes are made once (rank 0, in its directory), the other ranks wait and then only read them
        shared = [work]
        dist.broadcast_object_list(shared, src=0)
        work = shared[0]
        if rank == 0:
            load_databases(work, args.db_dir)
        dist.barrier()
    fastas, idx_dir, prefixes, refs, stats, built = load_databases(work, args.db_dir)
    n_job = args.reads
    n = max(1, n_job // args.steps)                   # reads per step (batch) per GPU
    ms = minimal_scores(stats, fastas, n_job * world)  # refstats totals stay GLOBAL across shards (SURVEY 8(e))
    al = api.Aligner(local_rank)
    prm = api.default_params()
    al.set_params(prm)
    t_idx = time.time()
    load_resident_index(al, args.index_source, fastas, prefixes, refs, ms, stats)
    index_resident_s = time.time() - t_idx
    info = al.index_info()
    pool = DbPool(refs)
    # reads are sharded by record: each rank owns its own reads; one distinct batch per step, in pinned host memory
    nb = args.steps
    pins, cats = [], []
    for s_i in range(nb):
        reads = gen_reads(pool, n, GEN_SEED + 7919 * rank + s_i)
        pin = torch.empty(n * READ_LEN, dtype=torch.uint8, pin_memory=True)
        c = pin.numpy(); c[:] = reads.reshape(-1)
        pins.append(pin); cats.append(c)
        if s_i == 0:
            first_reads = reads
    pin_off = torch.empty(n + 1, dtype=torch.int64, pin_memory=True)
    off = pin_off.numpy().view(np.uint64); off[:] = np.arange(n + 1, dtype=np.uint64) * READ_LEN
    setup_s = time.time() - t_setup

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- kernels only: each step's batch is uploaded first (untimed), then timed with CUDA events inside the C ABI ----
    al.upload(cats[0], off)
    for _ in range(args.warmup):
        al.run_resident()
    sampler = ClockSampler(local_rank); sampler.start()
    barrier()
    t0 = time.perf_counter()
    dev_ms, seed_ms, lis_ms, fin_ms, launches = [], [], [], [], 0
    csum = None
    for s_i in range(args.steps):
        if s_i > 0:
            al.upload(cats[s_i], off)
        al.run_resident()
        t = al.timings()
        dev_ms.append(t["total_ms"]); seed_ms.append(t["seed_ms"]); lis_ms.append(t["lis_ms"]); fin_ms.append(t["final_ms"]); launches += t["launches"]
        res = al.download()
        vec_s = np.array([res["counters"][k] for k in api.CNT_NAMES] + [int(x) for x in res["matched"]], dtype=np.int64)
        csum = vec_s if csum is None else csum + vec_s
    barrier()
    last_res = res
    wall_ms = (time.perf_counter() - t0) * 1000.0
    sampler.stop_flag = True; sampler.join(timeout=2)
    step_ms = float(np.sum(dev_ms))          # CUDA events on the library's stream, summed over the K steps
    # ---- the same K batches once more, UNTIMED, through the instrumented instantiations of the kernels (smr_set_instrumentation):
    #      the seed-side counters (windows, lists, entries) and the cycle shares of the candidate kernel's roles come from this pass;
    #      the timed passes above run the product's kernels, which carry neither ----
    csum_i, instr_lis_ms, instr_mismatch, instr_error = None, [], [], None
    try:
        al.set_instrumentation(True)
        for s_i in range(args.steps):
            al.upload(cats[s_i], off)
            al.run_resident()
            instr_lis_ms.append(al.timings()["lis_ms"])
            res = al.download()
            vec_s = np.array([res["counters"][k] for k in api.CNT_NAMES], dtype=np.int64)
            csum_i = vec_s if csum_i is None else csum_i + vec_s
        for k in ("num_aligned", "sw_calls", "sw_cells", "pos_entries", "lis_calls", "spec_calls"):   # what both instantiations count must agree
            i = api.CNT_NAMES.index(k)
            if int(csum[i]) != int(csum_i[i]):
                instr_mismatch.append({"counter": k, "product": int(csum[i]), "instrumented": int(csum_i[i])})
                print(f"[bench] instrumented and product kernels disagree on {k}: {int(csum_i[i])} vs {int(csum[i])}", file=sys.stderr)
        for k in INSTR_ONLY:
            i = api.CNT_NAMES.index(k)
            csum[i] = csum_i[i]
    except Exception as e:     # the bench line must not depend on the counter pass: the timed numbers above stand without it
        instr_error = str(e)[:300]
        print(f"[bench] instrumented pass failed: {instr_error}", file=sys.stderr)
    finally:
        try:
            al.set_instrumentation(False)
        except Exception:
            pass
    # ---- end to end through the public call: pinned host buffers in, host results out, every step ----
    # Two contexts on the GPU, one host thread each, batches alternate: the H2D copy of one batch and the D2H copy + host-side
    # result packing of another run under the kernels of a third (the library serialises the kernel sections of contexts that
    # share a device).  Every step still pays its own copies inside the timed region.
    from concurrent.futures import ThreadPoolExecutor
    al2 = api.Aligner(local_rank)
    al2.set_params(prm)
    load_resident_index(al2, args.index_source, fastas, prefixes, refs, ms, stats)
    als = [al, al2]
    for a in als:
        a.align(cats[0][: min(n, 1 << 16) * READ_LEN], off[: min(n, 1 << 16) + 1])  # warm the host path
        a.align(cats[0], off, reuse_outputs=True)                                     # first touch of the reusable result buffers
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    with ThreadPoolExecutor(2) as ex:
        def one(s_i):
            r = als[s_i % 2].align(cats[s_i], off, reuse_outputs=True)
            return r["slots"], int(r["cigar"].nbytes)
        res_all = list(ex.map(one, range(e2e_steps)))
    barrier()
    e2e_s = time.perf_counter() - t0
    h2d = int(cats[0].nbytes + off.nbytes)
    slots = res_all[-1][0]
    d2h = int(n * (28 + 4 + 2) + n * slots * 40 + res_all[-1][1] + 8 * 80)
    # ---- reductions over ranks (the path's only collective: one all-reduce of the counter vector) ----
    cnt_names = list(api.CNT_NAMES)
    vec = csum
    tm = np.array([step_ms, e2e_s * 1000.0, wall_ms], dtype=np.float64)
    from sortmerna_b200 import shard
    dev = torch.device("cuda", local_rank)
    vec = shard.allreduce_counters(vec, dev)       # the path's only collective (NCCL): Readstats counters, SUM
    tm = shard.allreduce_max(tm, dev)              # device-side timings: max over ranks
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    counters = dict(zip(cnt_names, (int(x) for x in vec[: len(cnt_names)])))
    total_reads_step = n * world
    total_reads_job = total_reads_step * args.steps
    value = total_reads_job / (tm[0] / 1000.0)
    e2e_value = total_reads_step * e2e_steps / (tm[1] / 1000.0)
    # ---- rooflines (DESIGN.md section 4) ----
    peak, peak_src = peaks()
    seed_s = float(np.sum(seed_ms)) / 1000.0        # counters are summed over the K steps and all ranks; times are this rank's
    lis_s = float(np.sum(lis_ms)) / 1000.0
    # seed kernel, HBM-bound: bytes it must stream = per window two 16-byte lookup records, per scanned list entry 8 bytes
    # (text + id), the read bases once per (strand, index part)
    alg_bytes = counters["windows"] * 32 + counters["bucket_entries"] * 8 + total_reads_job * READ_LEN * 16
    ach = alg_bytes / world / seed_s / 1e9 if seed_s > 0 else 0.0
    # candidate kernel (dominant), integer-issue bound: forward Smith-Waterman cell updates (refLen x readLen per ssw_align-
    # equivalent call, SURVEY 8(d)) against the measured dependent-free DPX rate / 3.5 DPX-class ALU instructions per cell
    dpx = al.dpx_peak()                              # 1e9 thread-ops/s, measured on this device now
    cells_per_rank = counters["sw_cells"] / world                                   # algorithmic: the calls the reference makes
    exec_cells_per_rank = counters["spec_cells"] / world                            # executed by the scorer warps (speculation included)
    sw_kernel_rate = cells_per_rank / lis_s / 1e12 if lis_s > 0 else 0.0            # whole kernel (votes, LIS, ... included)
    sw_exec_rate = exec_cells_per_rank / lis_s / 1e12 if lis_s > 0 else 0.0
    sw_peak = dpx / 3.5 / 1e3                        # Tcell-updates/s
    tr = {}
    try:
        cands = [os.path.join(ROOT, "profiles", f) for f in ("r2c_traffic.json", "r2b_traffic.json", "r2_traffic.json")]   # the newest committed capture
        tr = json.load(open(next(f for f in cands if os.path.exists(f))))
    except Exception:
        pass
    def _traffic(kernel):   # ncu DRAM bytes of the committed capture, scaled to the reads of one launch of this run
        if kernel in tr and tr.get("reads_in_captured_launch"):
            return int(tr[kernel]["dram_bytes"] * n / tr["reads_in_captured_launch"])
        return None
    roof_sw = {"bound": "integer (alu pipe, DPX)", "kernel": "lis_kernel (candidates + Smith-Waterman score pass)",
               "achieved": sw_kernel_rate, "peak": sw_peak, "unit": "Tcell-updates/s", "frac": sw_kernel_rate / sw_peak if sw_peak else None,
               "traffic": _traffic("lis_kernel"), "traffic_unit": "DRAM bytes per launch (ncu capture scaled by reads per launch)",
               "executed_incl_speculation": sw_exec_rate, "speculation_overhead": (exec_cells_per_rank / cells_per_rank - 1.0) if cells_per_rank else None,
               "planner_wait_share": counters["cyc_wait"] / max(1, counters["dbg_sum_read_cycles"]),
               "peak_source": f"measured now: {dpx:.0f} G dependent-free VIADDMNMX thread-ops/s (smr_debug_dpx_peak) / 3.5 such instructions per cell",
               "cells_per_step": int(cells_per_rank / args.steps), "kernel_ms_per_step": float(np.mean(lis_ms))}
    roof_seed = {"bound": "hbm", "kernel": "seed_kernel", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                 "traffic": _traffic("seed_kernel"), "traffic_unit": "DRAM bytes of ONE launch (index part 0 of 8; ncu capture scaled by reads per launch)",
                 "algorithmic_bytes_per_launch": int(alg_bytes / world / args.steps / max(1, info["parts"])),
                 "peak_source": peak_src, "algorithmic_bytes_per_step": int(alg_bytes / world / args.steps),
                 "kernel_ms_per_step": float(np.mean(seed_ms))}
    out = {
        "metric": METRIC if args.db_dir else METRIC_SYNTHETIC, "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tm[0] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int16x2 (DPX) / u8", "data": "synthetic",
        "config": {"workload": f"10 M synthetic 150 bp Illumina reads vs {db_words(args)}, 1xB200" if (n_job == 10_000_000 and world == 1) else
                   f"{n_job} synthetic 150 bp Illumina reads per GPU vs {db_words(args)}",
                   "reads_per_gpu_per_step": n, "reads_per_gpu_job": n * args.steps, "read_len": READ_LEN, "databases": 8,
                   "database_files": db_source(args), "index_hbm_bytes": info["hbm_bytes"],
                   "l2": "inputs larger than L2 (index 1.3 GB + reads 1.5 GB per pass)", "parallelism": f"reads sharded by record x{world}",
                   "hit_rate": counters["num_aligned"] / total_reads_job},
        "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "roofline": roof_sw,            # the dominant kernel of the step
        "roofline_seed": roof_seed,     # the HBM-bound kernel of the path
        "kernel_ms_per_step": {"seed": float(np.mean(seed_ms)), "candidates_sw": float(np.mean(lis_ms)), "finalize": float(np.mean(fin_ms))},
        "instrumentation": {"timed_region": "off (product kernels)", "counters_from": "one extra untimed pass over the same batches with smr_set_instrumentation(1)",
                            "candidates_sw_ms_per_step_instrumented": float(np.mean(instr_lis_ms)) if instr_lis_ms else None,
                            "instr_only_counters": list(INSTR_ONLY), "disagreements": instr_mismatch,   # counters both instantiations produce (must be empty)
                            "error": instr_error},
        "clocks": sampler.summary(),
        "counters": counters,
        "setup_s": setup_s, "index_build_s": built, "index_source": args.index_source, "index_resident_s": round(index_resident_s, 2),
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_res, (args.steps - 1) * n)
    if not args.no_cpu_baseline and world == 1 and not os.path.exists(stage_data.REF_BIN):
        out["cpu_baseline"] = {"unavailable": "the reference CPU build (oracle/_ref/sortmerna_ref) is not built"}
    elif not args.no_cpu_baseline and world == 1:   # reported baseline: rank 0 at N = 1 only
        sample = min(n, args.cpu_sample or int(min(400_000, max(20_000, 2_300 * cores))))
        v, t, total, _ = run_reference_sample(fastas, reference_index_dir(fastas, work), first_reads[:sample], cores)
        out["cpu_baseline"] = {"value": v, "unit": "reads/s", "cores": cores, "kind": "reference", "host": core_info,
                               "sample": f"first {sample} reads of the same synthetic workload vs the 8 databases, reference CPU build "
                                         f"(oracle/_ref/sortmerna_ref -threads {cores}), alignment loops {t:.1f} s (index loading excluded; "
                                         f"'Done alignment' incl. loading {total:.1f} s)"}
        # SURVEY 8(d)'s own numerator for the seed search -- what the reference's pruned trie walk touches, "on-disk-minimal, each
        # datum once per (read, strand, index part)" -- from the oracle's instrumented walk (the checker, CPU) on a small sample
        try:
            out["roofline_seed"]["survey_8d"] = survey_8d_seed(fastas, prefixes, refs, ms, stats, first_reads[:2000], cores, n,
                                                                float(np.mean(seed_ms)), peak)
        except Exception as e:     # the oracle library is test infrastructure: its absence must not cost the bench line
            out["roofline_seed"]["survey_8d"] = {"unavailable": str(e)[:200]}
    emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
