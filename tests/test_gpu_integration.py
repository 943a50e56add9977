"""The drop-in, end to end on the GPU: the unmodified reference host program linked with integration/align_gpu.cpp and the
PRODUCT library (oracle/_ref/sortmerna_gpu) writes the files the reference binary writes for the same command line.
The bundled-set cases run on stored samples (tests/golden/sets/: the first 100 records of both set4 mates and the sequences of
the databases they align to); where data_cache/ holds the full bundled data (tools/stage_data.py) they also run at full size,
with the known answers of scripts/test.jinja."""
import os
import shutil
import tempfile

import pytest

from conftest import GOLDEN
from helpers import ID85, SET4_SAMPLES, stored_databases, unpacked
from integration_common import REF_DIR, assert_same_outputs, run_host

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("extra", [[], ["-num_alignments", "3"]], ids=["default", "best3"])
def test_reference_host_with_gpu_library(extra):
    for b in ("sortmerna_ref", "sortmerna_gpu"):
        if not os.path.exists(os.path.join(REF_DIR, b)):
            pytest.skip(f"oracle/_ref/{b} not built (oracle/Makefile.ref)")
    d = tempfile.mkdtemp(prefix="smr_integ_gpu_")
    try:
        reads = [os.path.join(GOLDEN, "reads_mix.fq")]
        rep = ["-sam", "-blast", "1 cigar qcov qstrand", "-fastx", "-other"]
        ref, _ = run_host("sortmerna_ref", os.path.join(d, "ref"), reads, rep + extra)
        got, log = run_host("sortmerna_gpu", os.path.join(d, "got"), reads, rep + extra)
        assert "Starting alignment (libsmr_b200)" in log
        assert_same_outputs(got, ref)
    finally:
        shutil.rmtree(d, ignore_errors=True)


def test_reference_t9_golden_sam_rows_on_gpu():
    """scripts/test.jinja t9 (exact SAM rows, forward + reverse-complement reference) through the drop-in host program"""
    from test_integration_binding import T9_ROWS, run_t9
    if not os.path.exists(os.path.join(REF_DIR, "sortmerna_gpu")):
        pytest.skip("oracle/_ref/sortmerna_gpu not built")
    assert run_t9("sortmerna_gpu") == T9_ROWS


def _need_binaries():
    for b in ("sortmerna_ref", "sortmerna_gpu"):
        if not os.path.exists(os.path.join(REF_DIR, b)):
            pytest.skip(f"oracle/_ref/{b} not built (oracle/Makefile.ref)")


def test_reference_t5_mate_pairs_known_answer():
    """scripts/test.jinja t5: the two set4 mate files (paired feed, 5 threads) vs silva-bac-16s-id85 built with -max_pos 250; the
    drop-in host program on the GPU against the reference binary.  Stored sample: 2 x 100 mates vs the sequences of the database
    they align to; at full size 2 x 5000 mates vs the whole database: 10000 reads -> 6000 aligned / 4000 not."""
    from conftest import ROOT
    from tools import stage_data
    _need_binaries()
    d = tempfile.mkdtemp(prefix="smr_t5_")
    try:
        fasta = stored_databases(d, [ID85])[0]
        idx, _ = stage_data.ensure_indexes([fasta], os.path.join(d, "idx_ref"), extra=("-max_pos", "250"), builder="reference")
        _t5(fasta, unpacked(d, SET4_SAMPLES), idx, os.path.join(d, "sample"), None)
        cache = os.path.join(ROOT, "data_cache")
        fasta = os.path.join(cache, "sets", "silva-bac-16s-database-id85.fasta")
        reads = [os.path.join(cache, "sets", f"set4_mate_pairs_metatranscriptomics_{k}.fastq") for k in (1, 2)]
        if all(os.path.exists(p) for p in [fasta] + reads):
            idx, _ = stage_data.ensure_indexes([fasta], os.path.join(cache, "idx_set2_ref"), extra=("-max_pos", "250"), builder="reference")
            _t5(fasta, reads, idx, os.path.join(d, "full"), (6000, 4000))      # scripts/test.jinja:318-322
    finally:
        shutil.rmtree(d, ignore_errors=True)


def _t5(fasta, reads, idx, d, known):
    import subprocess
    outs = {}
    for b in ("sortmerna_ref", "sortmerna_gpu"):
        wd = os.path.join(d, b)
        cmd = [os.path.join(REF_DIR, b), "-ref", fasta, "-reads", reads[0], "-reads", reads[1], "-max_pos", "250", "-fastx", "-other", "-threads", "5",
               "-workdir", wd, "-idx-dir", idx, "-task", "4"]
        p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
        assert p.returncode == 0, p.stdout[-2000:]
        log = open(os.path.join(wd, "out", "aligned.log")).read()
        outs[b] = ([ln for ln in log.split("\n") if "E-value threshold" in ln],
                   {fn: open(os.path.join(wd, "out", fn)).read() for fn in os.listdir(os.path.join(wd, "out")) if fn.endswith(".fq")})
    assert outs["sortmerna_gpu"][0] == outs["sortmerna_ref"][0]
    if known:
        for b in outs:
            log = "\n".join(outs[b][0])
            assert f"passing E-value threshold = {known[0]}" in log and f"failing E-value threshold = {known[1]}" in log, b
    assert outs["sortmerna_gpu"][1] == outs["sortmerna_ref"][1]


def _run_binary(binary, fastas, reads, idx, wd, extra, threads=8, env=None):
    import subprocess
    cmd = [os.path.join(REF_DIR, binary)] + sum((["-ref", f] for f in fastas), []) + sum((["-reads", r] for r in reads), []) + \
          ["-workdir", wd, "-idx-dir", idx, "-threads", str(threads), "-task", "4"] + list(extra)
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=1800, env=env)
    assert p.returncode == 0, p.stdout[-3000:]
    out = os.path.join(wd, "out")
    files = {}
    import gzip
    for fn in sorted(os.listdir(out)):
        path = os.path.join(out, fn)
        text = gzip.open(path, "rt", errors="replace").read() if fn.endswith(".gz") else open(path, errors="replace").read()   # gz input -> gz reports
        lines = text.split("\n")
        fn = fn[:-3] if fn.endswith(".gz") else fn
        if fn.endswith(".sam"):
            lines = sorted(ln for ln in lines if ln and not ln.startswith("@"))   # several references: row order depends on the slot count (SURVEY 8(c))
        elif fn.endswith(".log"):
            lines = [ln for ln in lines if "E-value threshold" in ln or "Total reads =" in ln]
        files[fn] = lines
    return files, p.stdout


def _config4_sample(d):
    """The stored sample of BASELINE config 4: both set4 mates (2 x 100 reads, FASTQ.gz as stored) vs the sequences of the 8
    rRNA databases they align to -- (databases, reads, the reference builder's index)"""
    from tools import stage_data
    fastas = stored_databases(d, stage_data.DBS)
    idx, _ = stage_data.ensure_indexes(fastas, os.path.join(d, "idx_ref"), builder="reference")
    return fastas, list(SET4_SAMPLES), idx


def _config4_full():
    """BASELINE config 4 at full size where data_cache/ holds it, else None"""
    from conftest import ROOT
    from tools import stage_data
    cache = os.path.join(ROOT, "data_cache")
    reads = [os.path.join(cache, "sets", f"set4_mate_pairs_metatranscriptomics_{k}.fastq.gz") for k in (1, 2)]
    fastas = [stage_data.db_path(n) for n in stage_data.DBS]
    if not all(os.path.exists(p) for p in reads + fastas):
        return None
    idx, _ = stage_data.ensure_indexes(fastas, os.path.join(cache, "idx_ref"), builder="reference")
    return fastas, reads, idx


def test_baseline_config4_through_the_binary():
    """BASELINE config 4: set4 paired FASTQ.gz vs the 8 rRNA databases, -sam, through the CLI of the drop-in host program
    (gz inflate + paired feed + 8 resident indexes + report stage) against the unmodified reference binary: identical SAM rows /
    aligned / other reads, with the indexes read from the files and built on the GPU.  Stored sample always; at full size also
    the known answer 5944 / 4056 (scripts/test.jinja t17)."""
    _need_binaries()
    d = tempfile.mkdtemp(prefix="smr_cfg4_")
    try:
        _config4(*_config4_sample(d), os.path.join(d, "sample"), None)
        full = _config4_full()
        if full:
            _config4(*full, os.path.join(d, "full"), (5944, 4056))
    finally:
        shutil.rmtree(d, ignore_errors=True)


def _config4(fastas, reads, idx, d, known):
    extra = ["-sam", "-fastx", "-other", "-paired_in"]
    ref, _ = _run_binary("sortmerna_ref", fastas, reads, idx, os.path.join(d, "ref"), extra)
    got, log = _run_binary("sortmerna_gpu", fastas, reads, idx, os.path.join(d, "got"), extra)
    assert "Starting alignment (libsmr_b200)" in log
    if known:
        assert any(f"passing E-value threshold = {known[0]}" in ln for ln in got["aligned.log"])
        assert any(f"failing E-value threshold = {known[1]}" in ln for ln in got["aligned.log"])
    assert sorted(got) == sorted(ref)
    for fn in got:
        assert got[fn] == ref[fn], fn
    # the same with the 8 indexes built on the GPU from the FASTA files (smr_build_index_device) instead of read from the index files
    dev, log = _run_binary("sortmerna_gpu", fastas, reads, idx, os.path.join(d, "dev"), extra, env=dict(os.environ, SMR_INDEX_DEVICE="1"))
    assert "Starting alignment (libsmr_b200)" in log
    for fn in ref:
        assert dev[fn] == ref[fn], "device-built index: " + fn


def test_two_gpus_equal_one_gpu():
    """SMR_GPUS=2 (one context and one worker thread per GPU, batches in flight concurrently) writes what SMR_GPUS=1 writes, on
    the stored sample of BASELINE config 4.  Needs two devices; 200-read batches so that both GPUs get several."""
    from sortmerna_b200 import api
    if not os.path.exists(os.path.join(REF_DIR, "sortmerna_gpu")):
        pytest.skip("oracle/_ref/sortmerna_gpu not built (oracle/Makefile.ref)")
    if api.load_library().smr_device_count() < 2:
        pytest.skip("needs two GPUs")
    d = tempfile.mkdtemp(prefix="smr_2gpu_")
    try:
        fastas, reads, idx = _config4_sample(d)
        extra = ["-sam", "-fastx", "-other", "-paired_in"]
        one, _ = _run_binary("sortmerna_gpu", fastas, reads, idx, os.path.join(d, "g1"), extra, env=dict(os.environ, SMR_GPUS="1", SMR_BATCH_READS="200"))
        two, log = _run_binary("sortmerna_gpu", fastas, reads, idx, os.path.join(d, "g2"), extra, env=dict(os.environ, SMR_GPUS="2", SMR_BATCH_READS="200"))
        assert "resident on 2 GPU(s)" in log
        for fn in one:
            assert one[fn] == two[fn], fn
    finally:
        shutil.rmtree(d, ignore_errors=True)
