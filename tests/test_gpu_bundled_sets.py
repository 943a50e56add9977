"""Parity on the bundled read sets (BASELINE configs 2 and 4) and on the benchmark's workload: the GPU path against what the
unmodified reference binary prints for the same inputs -- every SAM row and the pass/fail totals.  The bundled-set cases run
on stored samples (the first 100 records of the read files and the sequences of the databases they align to, tests/golden/sets/
made by tests/golden/make_sets.py); where data_cache/ holds the full bundled data (tools/stage_data.py) they also run at full
size, with the known-answer counts of scripts/test.jinja (t3: 99999/1, t17: 5944/4056).  Where the reference build is absent,
its side comes from what it printed for the same inputs, recorded by this file's __main__ (tests/golden/sets_reference.json,
tests/golden/bench_workload_reference.json)."""
import hashlib
import json
import os
import tempfile

import numpy as np
import pytest

from helpers import ID85, SET2_SAMPLE, SET4_SAMPLES, stored_databases, unpacked
from sortmerna_b200 import api, hostio

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CACHE = os.path.join(ROOT, "data_cache")
GOLDEN_SETS = os.path.join(ROOT, "tests", "golden", "sets_reference.json")


def _have_full(*paths):
    from oracle import ora
    return ora.have_reference_binary() and all(os.path.exists(p) for p in paths)


def _record(log, sam):
    return {"minimal_score": log["minimal_score"], "passing": log["passing"], "failing": log["failing"], "rows": len(sam),
            "digest": hashlib.sha256("\n".join(sorted(sam)).encode()).hexdigest()}


def _check_against_reference(golden, fastas, read_files, ref_extra, d, **native_kw):
    """The GPU path on (fastas, read_files) against the reference: run here where its build exists (and `golden`, what it
    printed when recorded, checked against it), else against `golden`."""
    from oracle import ora
    sam = None
    if ora.have_reference_binary():
        log, sam = _run_reference(fastas, os.path.join(d, "idx_ref"), read_files, ref_extra, threads=os.cpu_count() or 8)
        assert _record(log, sam) == golden        # the recording still describes the reference
    rows, got, batch = _run_gpu(fastas, os.path.join(d, "idx"), read_files, golden["minimal_score"], **native_kw)
    assert int(got["res"]["is_hit"].sum()) == golden["passing"]
    assert golden["passing"] + golden["failing"] == batch.n
    if sam is not None:
        assert sorted(rows) == sorted(sam)
    assert (len(rows), hashlib.sha256("\n".join(sorted(rows)).encode()).hexdigest()) == (golden["rows"], golden["digest"])
    return got


def _set4_sample(d):
    from tools import stage_data
    return stored_databases(d, stage_data.DBS), unpacked(d, SET4_SAMPLES)


def _set2_sample(d):
    return stored_databases(d, [ID85]), unpacked(d, [SET2_SAMPLE])


def _run_reference(fastas, ref_idx_dir, read_files, ref_extra, threads):
    """The reference on the index ITS OWN builder makes: (parsed aligned.log, SAM rows)"""
    from oracle import ora
    from tools import stage_data
    ref_idx, _ = stage_data.ensure_indexes(fastas, ref_idx_dir, extra=tuple(ref_extra), builder="reference")   # index-build options (-max_pos) == run options here
    with tempfile.TemporaryDirectory(prefix="smr_sets_") as d:
        r = ora.run_reference(fastas, read_files, os.path.join(d, "w"), extra=["-sam", "-fastx", "-other"] + list(ref_extra), threads=threads, idx_dir=ref_idx)
        return ora.parse_log(r["log"]), ora.read_sam_rows(os.path.join(r["out_dir"], "aligned.sam"))


def _run_case(fastas, idx_dir, read_files, ref_extra, threads, **native_kw):
    """The reference runs on the index ITS OWN builder makes (<idx_dir>_ref); the GPU path runs on the index smr_build_index
    makes (<idx_dir>) -- so the comparison also covers the native index builder at full database size."""
    log, sam = _run_reference(fastas, idx_dir + "_ref", read_files, ref_extra, threads)
    rows, got, batch = _run_gpu(fastas, idx_dir, read_files, log["minimal_score"], **native_kw)
    return log, sam, rows, got, batch


def _run_gpu(fastas, idx_dir, read_files, minimal_score, **native_kw):
    from tools import stage_data
    idx_dir, _ = stage_data.ensure_indexes(fastas, idx_dir, **native_kw)
    pre = hostio.find_index_prefixes(idx_dir)
    refs = [hostio.load_references(f) for f in fastas]
    al = api.Aligner(0)
    al.set_params(api.default_params())
    for k, f in enumerate(fastas):
        p = pre[os.path.basename(f)]
        al.load_index_part(k, 0, p, refs[k], minimal_score[k], (18, 9, 3), hostio.parse_stats(p).lnwin)
    h, s, q = [], [], []
    for rf in read_files:
        hh, ss, qq = hostio.read_fastx(rf)
        h += hh; s += ss; q += qq
    batch = hostio.pack_reads(h, s, q)
    got = al.align(batch.cat, batch.off)
    rows = hostio.format_sam_rows(batch, refs, got["res"], got["alns"], got["cigar"], got["slots"])
    al.close()
    return rows, got, batch


def test_set4_paired_vs_8_databases(tmp_path):
    """BASELINE config 4 / t17: 2 x 100 mates vs the sequences of the 8 rRNA databases they align to; at full size 2 x 5000 mates
    vs the 8 databases."""
    from tools import stage_data
    fastas, reads = _set4_sample(str(tmp_path))
    got = _check_against_reference(json.load(open(GOLDEN_SETS))["set4_8db"], fastas, reads, [], str(tmp_path))
    assert int(got["res"]["is_hit"].sum()) > 100
    reads = [os.path.join(CACHE, "sets", f"set4_mate_pairs_metatranscriptomics_{k}.fastq") for k in (1, 2)]
    fastas = [stage_data.db_path(n) for n in stage_data.DBS]
    if not _have_full(*reads, *fastas):
        return
    log, sam, rows, got, batch = _run_case(fastas, os.path.join(CACHE, "idx"), reads, [], threads=os.cpu_count() or 8)
    assert (log["passing"], log["failing"]) == (5944, 4056)          # scripts/test.jinja:1186-1188
    assert int(got["res"]["is_hit"].sum()) == 5944
    assert sorted(rows) == sorted(sam)


def test_set2_amplicon_vs_bac16s_id85(tmp_path):
    """BASELINE config 2 / t3: 100 amplicon reads vs the sequences of silva-bac-16s-database-id85 they align to, built with
    -max_pos 250; at full size 100,000 reads vs the whole database."""
    fastas, reads = _set2_sample(str(tmp_path))
    got = _check_against_reference(json.load(open(GOLDEN_SETS))["set2_id85"], fastas, reads, ["-max_pos", "250"], str(tmp_path), max_pos=250)
    assert int(got["res"]["is_hit"].sum()) > 90
    reads = [os.path.join(CACHE, "sets", "set2_environmental_study_550_amplicon.fasta")]
    fastas = [os.path.join(CACHE, "sets", "silva-bac-16s-database-id85.fasta")]
    if not _have_full(*reads, *fastas):
        return
    log, sam, rows, got, batch = _run_case(fastas, os.path.join(CACHE, "idx_set2"), reads, ["-max_pos", "250"], threads=os.cpu_count() or 8, max_pos=250)
    assert (log["passing"], log["failing"]) == (99999, 1)            # scripts/t3.jinja:30-32
    assert int(got["res"]["is_hit"].sum()) == 99999
    assert sorted(rows) == sorted(sam)


GOLDEN_WORKLOAD = os.path.join(ROOT, "tests", "golden", "bench_workload_reference.json")


def _bench_workload(d):
    """The workload bench.py measures by default (BASELINE configs 3/5: 150 nt reads at 1 % / 10 % error + random, vs the 8
    synthetic databases of tools/synth_db.py), 20,000 reads of it from the numpy twin of bench.gen_reads (the same reads on
    every machine): (database FASTA files, FASTQ file) under d."""
    import bench
    from tools import synth_db
    fastas = synth_db.write_databases(os.path.join(d, "db"))
    reads = bench._gen_reads_numpy(bench.DbPool([hostio.load_references(f) for f in fastas]), 20000, bench.GEN_SEED + 4242)
    fq = os.path.join(d, "wl.fq")
    bench.write_fastq(fq, reads)
    return fastas, fq


def test_bench_workload_sample_vs_reference():
    """The benchmark's workload through the GPU path and through the unmodified reference -- every SAM row and the pass/fail
    totals identical."""
    golden = json.load(open(GOLDEN_WORKLOAD))
    with tempfile.TemporaryDirectory(prefix="smr_wl_") as d:
        fastas, fq = _bench_workload(d)
        _check_against_reference(golden, fastas, [fq], [], d)
    assert golden["passing"] + golden["failing"] == 20000
    assert 0.5 < golden["passing"] / 20000 < 0.8          # two thirds of the workload derive from the databases


def _recorded(fastas, read_files, ref_extra, d):
    return _record(*_run_reference(fastas, os.path.join(d, "idx_ref"), read_files, ref_extra, threads=os.cpu_count() or 8))


if __name__ == "__main__":   # record GOLDEN_SETS and GOLDEN_WORKLOAD from the reference build (oracle/_ref/sortmerna_ref); needs no GPU
    rec = {}
    with tempfile.TemporaryDirectory(prefix="smr_sets_rec_") as d:
        rec["set4_8db"] = _recorded(*_set4_sample(d), [], os.path.join(d, "set4"))
    with tempfile.TemporaryDirectory(prefix="smr_sets_rec_") as d:
        rec["set2_id85"] = _recorded(*_set2_sample(d), ["-max_pos", "250"], os.path.join(d, "set2"))
    with open(GOLDEN_SETS, "w") as f:
        json.dump(rec, f, indent=1)
    with tempfile.TemporaryDirectory(prefix="smr_wl_rec_") as d:
        fastas, fq = _bench_workload(d)
        wl = _recorded(fastas, [fq], [], d)
    with open(GOLDEN_WORKLOAD, "w") as f:
        json.dump(wl, f, indent=1)
    print(rec, wl)
