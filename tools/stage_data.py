#!/usr/bin/env python
"""Stage the bundled reference data for the benchmark configs under data_cache/ (git-ignored; it
travels to the GPU box with the gpurun snapshot, like the built .so files):

  data_cache/rRNA_databases/*.fasta   copies of /root/reference/data/rRNA_databases (inputs, not code)
  data_cache/sets/...                 the bundled read sets used by BASELINE.json configs 2 and 4
  data_cache/idx/                     the index of each database in the reference's on-disk format, built by
                                      smr_build_index (our builder; tests/test_index_builder.py proves the files equal the
                                      reference builder's up to the arbitrary id numbering)

`ensure_indexes()` is also what bench.py calls to index its databases in the temporary directory of a run
(bench.py --db-dir data_cache/rRNA_databases measures against the staged databases).
"""
import os
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CACHE = os.path.join(ROOT, "data_cache")
REF_DATA = "/root/reference/data"
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "sortmerna_ref")

# --ref order of the 8-database sweep (README.md of the reference; SURVEY 8(d))
DBS = ["silva-bac-16s-id90", "silva-bac-23s-id98", "silva-arc-16s-id95", "silva-arc-23s-id98",
       "silva-euk-18s-id95", "silva-euk-28s-id98", "rfam-5s-database-id98", "rfam-5.8s-database-id98"]
SETS = ["set2_environmental_study_550_amplicon.fasta", "set4_mate_pairs_metatranscriptomics_1.fastq",
        "set4_mate_pairs_metatranscriptomics_2.fastq", "set5_simulated_amplicon_silva_bac_16s.fasta",
        "silva-bac-16s-database-id85.fasta", "test_read.fasta", "test_ref.fasta",
        "set4_mate_pairs_metatranscriptomics_1.fastq.gz", "set4_mate_pairs_metatranscriptomics_2.fastq.gz"]   # BASELINE config 4 as written (.gz mates)


def db_path(name):
    return os.path.join(CACHE, "rRNA_databases", name + ".fasta")


def stage_inputs():
    os.makedirs(os.path.join(CACHE, "rRNA_databases"), exist_ok=True)
    os.makedirs(os.path.join(CACHE, "sets"), exist_ok=True)
    for n in DBS:
        dst = db_path(n)
        if not os.path.exists(dst):
            shutil.copy(os.path.join(REF_DATA, "rRNA_databases", n + ".fasta"), dst)
            os.chmod(dst, 0o644)
    for n in SETS:
        dst = os.path.join(CACHE, "sets", n)
        if not os.path.exists(dst):
            shutil.copy(os.path.join(REF_DATA, n), dst)
            os.chmod(dst, 0o644)


def _have_index(idx_dir, fasta):
    from sortmerna_b200 import hostio
    if not os.path.isdir(idx_dir):
        return False
    pre = hostio.find_index_prefixes(idx_dir).get(os.path.basename(fasta))
    return bool(pre) and all(os.path.exists(pre + s) and os.path.getsize(pre + s) > 0
                             for s in (".kmer_0.dat", ".bursttrie_0.dat", ".pos_0.dat", ".stats"))


def build_index_native(fasta, idx_dir, **kw):
    """smr_build_index (sortmerna_b200/csrc/smr_build.cpp): our own builder, same files as the reference's."""
    from sortmerna_b200 import api
    os.makedirs(idx_dir, exist_ok=True)
    t0 = time.time()
    api.build_index(fasta, os.path.join(idx_dir, os.path.splitext(os.path.basename(fasta))[0]), **kw)
    return time.time() - t0


def build_index(fasta, idx_dir, extra=()):
    """Run the reference's index builder (indexdb.cpp:1119-2095) for one database (tests / cross-checks only)."""
    os.makedirs(idx_dir, exist_ok=True)
    wd = tempfile.mkdtemp(prefix="smr_idx_work_")
    tiny = os.path.join(wd, "tiny.fa")
    with open(tiny, "w") as f:
        f.write(">r\nACGTACGTACGTACGTACGTACGTACGTACGT\n")
    t0 = time.time()
    p = subprocess.run([REF_BIN, "-ref", fasta, "-reads", tiny, "-workdir", os.path.join(wd, "run"), "-idx-dir", idx_dir,
                        "-index", "1", "-threads", "1", *extra], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if p.returncode != 0:
        raise RuntimeError(f"index build failed for {fasta}:\n{p.stdout[-2000:]}")
    shutil.rmtree(wd, ignore_errors=True)
    return time.time() - t0


def ensure_indexes(fastas, idx_dir=None, workers=8, extra=(), builder="native", **kw):
    """Build whatever is missing, databases in parallel.  builder="native": smr_build_index (kw: max_pos, interval, lnwin, max_mb);
    builder="reference": the unmodified reference binary with the CLI arguments in `extra` (cross-checks only)."""
    idx_dir = idx_dir or os.path.join(CACHE, "idx")
    todo = [f for f in fastas if not _have_index(idx_dir, f)]
    times = {}
    if todo:
        if builder == "reference":
            if not os.path.exists(REF_BIN):
                raise RuntimeError("oracle/_ref/sortmerna_ref is missing (build it with oracle/Makefile.ref where /root/reference exists)")
            fn = lambda f: build_index(f, idx_dir, extra)
        else:
            fn = lambda f: build_index_native(f, idx_dir, **kw)
        with ThreadPoolExecutor(max_workers=workers) as ex:
            for f, t in zip(todo, ex.map(fn, todo)):
                times[os.path.basename(f)] = round(t, 1)
    return idx_dir, times


if __name__ == "__main__":
    stage_inputs()
    t0 = time.time()
    d, times = ensure_indexes([db_path(n) for n in DBS])
    print("index dir", d, "built", times, "wall", round(time.time() - t0, 1), "s")
    ensure_indexes([os.path.join(CACHE, "sets", "silva-bac-16s-database-id85.fasta")], os.path.join(CACHE, "idx_set2"), max_pos=250)
    subprocess.run(["du", "-sh", os.path.join(CACHE, "idx"), CACHE])
