"""Differential fuzzing of the oracle against the UNMODIFIED reference binary: random database slices, damaged reads and
random option sets (scoring, -num_alignments, -no-best, -F/-R, -full_search, -num_seeds, -min_lis, -edges): identical SAM rows
and pass/fail totals.  (The GPU twin of this test, oracle vs kernels on the same generator, is tests/test_gpu_fuzz.py.)
Where the reference build is absent the reference's side comes from tests/golden/fuzz_reference.json, recorded from that build
by this file's __main__: its minimal scores, pass totals and a digest of its sorted SAM rows (sequence columns stripped)."""
import hashlib
import json
import os
import shutil
import tempfile

import pytest

from conftest import ROOT
from fuzz_common import make_case
from helpers import params_kwargs_from_args, strip_seq
from sortmerna_b200 import api, hostio

REF_BIN = os.path.join(ROOT, "oracle", "_ref", "sortmerna_ref")
GOLDEN_REF = os.path.join(ROOT, "tests", "golden", "fuzz_reference.json")


def rows_digest(rows):
    return hashlib.sha256("\n".join(sorted(rows)).encode()).hexdigest()


def run_reference(key, fastas, reads_p, workdir, extra):
    """The reference's side of one case: {"minimal_score", "passing", "rows", "digest"} and, when the binary is there, "sam"
    (the rows themselves); {"skip": reason} for a case the reference refuses."""
    from oracle import ora
    golden = json.load(open(GOLDEN_REF)).get(key) if os.path.exists(GOLDEN_REF) else None
    if not os.path.exists(REF_BIN):
        if golden is None:
            pytest.fail(f"{key}: no recorded reference output in {GOLDEN_REF} and no reference build")
        return golden
    try:
        r = ora.run_reference(fastas, reads_p, workdir, extra=extra, threads=1)
    except RuntimeError as e:
        if "Sls::error" in str(e) or "ALP" in str(e):
            got = {"skip": "scoring set outside the reference's Gumbel tables"}
        elif "[validate:" in str(e):
            got = {"skip": "option combination refused by the reference's own validation"}
        else:
            raise
    else:
        log = ora.parse_log(r["log"])
        sam = strip_seq(ora.read_sam_rows(os.path.join(r["out_dir"], "aligned.sam")))
        got = {"minimal_score": log["minimal_score"], "passing": log["passing"], "rows": len(sam), "digest": rows_digest(sam), "sam": sam}
    if golden is not None:      # the recording still describes the reference
        assert {k: v for k, v in got.items() if k != "sam"} == golden, key
    return got


def check_rows(rows, ref, what):
    if "sam" in ref:
        assert sorted(rows) == sorted(ref["sam"]), what
    assert (len(rows), rows_digest(rows)) == (ref["rows"], ref["digest"]), what


@pytest.mark.parametrize("seed", range(int(os.environ.get("SMR_FUZZ_SEEDS", "12"))))
def test_oracle_equals_reference_on_random_cases(seed):
    from oracle import ora
    d = tempfile.mkdtemp(prefix="smr_fz_")
    try:
        fastas, reads_p, args = make_case(seed, d)
        log = run_reference(f"random_{seed}", fastas, reads_p, os.path.join(d, "w"), ["-sam", "-fastx"] + args)
        if "skip" in log:
            pytest.skip(log["skip"])
        batch = hostio.load_reads(reads_p)
        refs = [hostio.load_references(f) for f in fastas]
        kw = params_kwargs_from_args(args)
        oix, prefixes = [], []
        for k, f in enumerate(fastas):
            p = os.path.join(d, f"idx{k}")
            api.build_index(f, p)                       # our builder (equal to the reference's: tests/test_index_builder.py)
            oix.append(ora.OracleIndex(p, 0, 18))
        out = ora.align(oix, [0, 1], [0, 0], 2, refs, log["minimal_score"], [18, 9, 3, 18, 9, 3], ora.default_params(**kw), batch, nthreads=2)
        rows = strip_seq(hostio.format_sam_rows(batch, refs, out["res"], out["alns"], out["cigar"], out["slots"]))
        check_rows(rows, log, args)
        assert int(out["res"]["is_hit"].sum()) == log["passing"], args
    finally:
        shutil.rmtree(d, ignore_errors=True)


INDEX_OPTS = [(["-max_pos", "2"], dict(max_pos=2)), (["-max_pos", "7"], dict(max_pos=7)), (["-interval", "2"], dict(interval=2)),
              (["-m", "0.4"], dict(max_mb=0.4)), (["-max_pos", "3", "-m", "0.25"], dict(max_pos=3, max_mb=0.25))]


@pytest.mark.parametrize("seed", range(int(os.environ.get("SMR_FUZZ_INDEX_SEEDS", "6"))))
def test_oracle_equals_reference_with_index_options(seed):
    """The same differential test with index-build options in play: truncated position lists (-max_pos), sparse (L+1)-mers
    (-interval) and indexes split into several parts (-m): the oracle runs on the files smr_build_index writes, the reference on
    the ones its own builder writes."""
    from oracle import ora
    d = tempfile.mkdtemp(prefix="smr_fzi_")
    try:
        fastas, reads_p, args = make_case(5000 + seed, d)
        ref_extra, kw_build = INDEX_OPTS[seed % len(INDEX_OPTS)]
        log = run_reference(f"index_options_{seed}", fastas, reads_p, os.path.join(d, "w"), ["-sam", "-fastx"] + args + ref_extra)
        if "skip" in log:
            pytest.skip(log["skip"])
        batch = hostio.load_reads(reads_p)
        kw = params_kwargs_from_args(args)
        oix, inum, parts, refs, ms, by_index = [], [], [], [], [], []
        for k, f in enumerate(fastas):
            p = os.path.join(d, f"idx{k}")
            api.build_index(f, p, **kw_build)
            st = hostio.parse_stats(p)
            pr = hostio.split_by_parts(hostio.load_references(f), st)
            by_index.append(pr)
            for part in range(st.num_parts):
                oix.append(ora.OracleIndex(p, part, 18)); inum.append(k); parts.append(part); refs.append(pr[part]); ms.append(log["minimal_score"][k])
        out = ora.align(oix, inum, parts, 2, refs, ms, [18, 9, 3] * len(oix), ora.default_params(**kw), batch, nthreads=2)
        rows = strip_seq(hostio.format_sam_rows(batch, by_index, out["res"], out["alns"], out["cigar"], out["slots"]))
        check_rows(rows, log, (args, ref_extra))
        assert int(out["res"]["is_hit"].sum()) == log["passing"]
    finally:
        shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":   # record tests/golden/fuzz_reference.json from the reference build (oracle/_ref/sortmerna_ref)
    if os.path.exists(GOLDEN_REF):
        os.remove(GOLDEN_REF)
    rec = {}
    for key, seed, extra in ([(f"random_{s}", s, []) for s in range(12)] +
                             [(f"index_options_{s}", 5000 + s, INDEX_OPTS[s % len(INDEX_OPTS)][0]) for s in range(6)]):
        with tempfile.TemporaryDirectory(prefix="smr_fz_") as d:
            fastas, reads_p, args = make_case(seed, d)
            got = run_reference(key, fastas, reads_p, os.path.join(d, "w"), ["-sam", "-fastx"] + args + extra)
            rec[key] = {k: v for k, v in got.items() if k != "sam"}
            print(key, rec[key])
    with open(GOLDEN_REF, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
