"""smr_build_index (sortmerna_b200/csrc/smr_build.cpp), the native stand-in for the reference's build_index
(indexdb.cpp:1119-2095): the files it writes must be the reference's index up to the arbitrary numbering of the unique L-mers
(tests/index_equiv_check.cpp: .kmer byte-identical, .bursttrie byte-identical except id words related by a bijection, position
lists equal under that bijection, .stats equal apart from the embedded path / struct padding), and the UNMODIFIED reference
binary must produce its golden output when it is handed these files instead of its own.  Where the reference build is absent,
its builder's side comes from tests/golden/index_reference.json, recorded from it by this file's __main__: a digest of the
numbering-free form of each index (index_equiv_check --canonical)."""
import hashlib
import json
import os
import shutil
import subprocess
import tempfile

import pytest

from conftest import GOLDEN, ROOT, load_case
from sortmerna_b200 import api, hostio

REF_BIN = os.path.join(ROOT, "oracle", "_ref", "sortmerna_ref")
need_ref = pytest.mark.skipif(not os.path.exists(REF_BIN), reason="oracle/_ref/sortmerna_ref not built")
GOLDEN_REF = os.path.join(GOLDEN, "index_reference.json")


@pytest.fixture(scope="module")
def checker():
    d = tempfile.mkdtemp(prefix="smr_chk_")
    exe = os.path.join(d, "index_equiv_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "index_equiv_check.cpp")], check=True)
    yield exe
    shutil.rmtree(d, ignore_errors=True)


def equiv(checker, a, b, lnwin=18):
    p = subprocess.run([checker, a, b, str(lnwin)], capture_output=True, text=True)
    assert p.returncode == 0 and p.stdout.startswith("OK"), p.stdout + p.stderr
    return p.stdout


def digest(checker, prefix, lnwin=18):
    """sha256 of the index's numbering-free form"""
    with tempfile.NamedTemporaryFile(prefix="smr_canon_") as f:
        p = subprocess.run([checker, "--canonical", prefix, str(lnwin), f.name], capture_output=True, text=True)
        assert p.returncode == 0 and p.stdout.startswith("OK"), p.stdout + p.stderr
        return hashlib.sha256(open(f.name, "rb").read()).hexdigest()


def equals_reference_builder(checker, key, fasta, ref_extra, prefix, lnwin=18):
    """the index at `prefix` against the reference builder's index of `fasta` with the CLI options ref_extra: built and compared
    directly where the reference build exists (and the recording checked against it), else against the recorded digest"""
    golden = json.load(open(GOLDEN_REF)).get(key) if os.path.exists(GOLDEN_REF) else None
    if os.path.exists(REF_BIN):
        with tempfile.TemporaryDirectory(prefix="smr_bi_ref_") as d:
            ref_prefix = reference_build(fasta, d, ref_extra)
            equiv(checker, ref_prefix, prefix, lnwin)
            want = digest(checker, ref_prefix, lnwin)
        if golden is not None:
            assert golden == want, key
        return want
    assert golden is not None, f"{key}: no recorded reference index in {GOLDEN_REF} and no reference build"
    assert digest(checker, prefix, lnwin) == golden, key
    return golden


def reference_build(fasta, idx_dir, extra=()):
    """the reference's own builder (sortmerna_ref -index 1); returns the index prefix it chose"""
    wd = tempfile.mkdtemp(prefix="smr_refidx_")
    tiny = os.path.join(wd, "tiny.fa")
    with open(tiny, "w") as f:
        f.write(">r\nACGTACGTACGTACGTACGTACGTACGTACGT\n")
    p = subprocess.run([REF_BIN, "-ref", fasta, "-reads", tiny, "-workdir", os.path.join(wd, "run"), "-idx-dir", idx_dir, "-index", "1",
                        "-threads", "1", *extra], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    shutil.rmtree(wd, ignore_errors=True)
    assert p.returncode == 0, p.stdout[-2000:]
    return hostio.find_index_prefixes(idx_dir)[os.path.basename(fasta)]


@pytest.mark.parametrize("db", ["db_arc.fasta", "db_bac.fasta"])
def test_native_index_equals_golden_reference_index(checker, golden, db):
    d = tempfile.mkdtemp(prefix="smr_bi_")
    try:
        rep = api.build_index(os.path.join(GOLDEN, db), os.path.join(d, "x"))
        ref_prefix = golden["prefixes"][["db_arc.fasta", "db_bac.fasta"].index(db)]
        out = equiv(checker, ref_prefix, os.path.join(d, "x"))
        assert f"ids={rep['unique_lmers']}" in out
        st = hostio.parse_stats(os.path.join(d, "x"))
        assert st.numseq == rep["numseq"] and st.num_parts == 1 and st.lnwin == 18
    finally:
        shutil.rmtree(d, ignore_errors=True)


def test_native_index_equals_golden_t0(checker, golden_t0):
    d = tempfile.mkdtemp(prefix="smr_bi_")
    try:
        api.build_index(os.path.join(GOLDEN, "t0", "db_t0.fasta"), os.path.join(d, "x"))
        equiv(checker, golden_t0["prefix"], os.path.join(d, "x"))
    finally:
        shutil.rmtree(d, ignore_errors=True)


OPTION_CASES = [
    ("max_pos", ("-max_pos", "3"), dict(max_pos=3)),
    ("all_pos", ("-max_pos", "0"), dict(max_pos=0)),
    ("interval", ("-interval", "2"), dict(interval=2)),
    ("parts", ("-m", "0.5"), dict(max_mb=0.5)),          # db_bac needs ~1.26 "MB" by the 9.5e-6 rule: 3 parts
    ("seed16", ("-L", "16"), dict(lnwin=16)),
]


@pytest.mark.parametrize("name,ref_extra,kw", OPTION_CASES)
def test_native_index_equals_reference_builder_with_options(checker, name, ref_extra, kw):
    d = tempfile.mkdtemp(prefix="smr_bi_")
    try:
        fasta = os.path.join(GOLDEN, "db_bac.fasta")
        rep = api.build_index(fasta, os.path.join(d, "x"), **kw)
        equals_reference_builder(checker, f"options_{name}", fasta, ref_extra, os.path.join(d, "x"), kw.get("lnwin", 18))
        if name == "parts":
            assert rep["parts"] == 3
    finally:
        shutil.rmtree(d, ignore_errors=True)


def test_builder_errors():
    d = tempfile.mkdtemp(prefix="smr_bi_")
    try:
        with pytest.raises(api.SmrError, match="Could not open"):
            api.build_index(os.path.join(d, "missing.fa"), os.path.join(d, "x"))
        short = os.path.join(d, "short.fa")
        with open(short, "w") as f:
            f.write(">a\nACGTACGTACGTACGTAC\n")          # 18 nt < seed length + 1 (indexdb.cpp:1259-1265)
        with pytest.raises(api.SmrError, match="shorter than the seed length 19"):
            api.build_index(short, os.path.join(d, "x"))
        bad = os.path.join(d, "bad.fa")
        with open(bad, "w") as f:
            f.write("ACGT\n")
        with pytest.raises(api.SmrError, match="must begin with '>'"):
            api.build_index(bad, os.path.join(d, "x"))
    finally:
        shutil.rmtree(d, ignore_errors=True)


@need_ref
def test_reference_binary_gives_golden_output_on_native_index():
    """Hand the unmodified reference our index files (under the prefix names it derives itself) and compare its SAM / BLAST rows
    and totals with the golden run that used its own index."""
    from oracle import ora
    d = tempfile.mkdtemp(prefix="smr_bi_")
    try:
        fastas = [os.path.join(GOLDEN, "db_arc.fasta"), os.path.join(GOLDEN, "db_bac.fasta")]
        idx = os.path.join(d, "idx")
        os.makedirs(idx)
        for f in fastas:
            pre = reference_build(f, idx)             # only to learn the prefix name; then overwrite every file
            for sfx in (".kmer_0.dat", ".bursttrie_0.dat", ".pos_0.dat", ".stats"):
                os.remove(pre + sfx)
            api.build_index(f, pre)
        r = ora.run_reference(fastas, os.path.join(GOLDEN, "reads_mix.fq"), os.path.join(d, "w"),
                              extra=["-sam", "-blast", "1 cigar qcov qstrand", "-fastx", "-other"], threads=1, idx_dir=idx)
        assert "Skipping indexing" in r["stdout"]
        exp = load_case("default")
        log = ora.parse_log(r["log"])
        assert (log["passing"], log["failing"], log["minimal_score"]) == (exp["log"]["passing"], exp["log"]["failing"], exp["log"]["minimal_score"])
        assert ora.read_sam_rows(os.path.join(r["out_dir"], "aligned.sam")) == exp["sam"]
        assert [ln.rstrip("\n") for ln in open(os.path.join(r["out_dir"], "aligned.blast"))] == exp["blast"]
    finally:
        shutil.rmtree(d, ignore_errors=True)


def fuzz_case(seed, d):
    """Random FASTA files (IUPAC / lower-case / odd letters, wrapped lines, blanks inside lines, repeats that fill buckets past
    the burst threshold, sequences of the minimum length 19, tabs and blanks in headers) written under d, and random build
    options: -> (fasta, the reference's CLI options, smr_build_index keywords, builder threads)"""
    import numpy as np
    rng = np.random.default_rng(1000 + seed)
    alpha = list("ACGT" * 12 + "NRYKMSWBDHVXacgtnu")
    nseq = int(rng.integers(1, 40))
    base = "".join(rng.choice(list("ACGT"), 400))
    recs = []
    for i in range(nseq):
        kind = rng.integers(0, 4)
        if kind == 0:
            s = "".join(rng.choice(alpha, int(rng.integers(19, 600))))
        elif kind == 1:   # near copies: many 19-mers share 9-mer prefixes -> buckets burst
            s = list(base[int(rng.integers(0, 50)):])
            for _ in range(int(rng.integers(0, 30))):
                s[int(rng.integers(len(s)))] = "ACGT"[int(rng.integers(4))]
            s = "".join(s)
        elif kind == 2:   # low complexity
            s = ("ACGT"[int(rng.integers(4))] * int(rng.integers(19, 200))) + "".join(rng.choice(list("AC"), int(rng.integers(0, 100))))
        else:
            s = "".join(rng.choice(list("ACGT"), 19))
        recs.append((f">s{i}\tdesc {i} x", s))
    wrap = int(rng.choice([0, 60, 7]))
    fasta = os.path.join(d, f"fz{seed}.fasta")
    with open(fasta, "w") as f:
        for h, s in recs:
            f.write(h + "\n")
            if wrap:
                f.write("\n".join(s[k:k + wrap] for k in range(0, len(s), wrap)) + "\n")
            else:
                f.write(s + "\n")
    opt = [dict(), dict(max_pos=2), dict(interval=3), dict(max_mb=0.002), dict(max_pos=0, interval=2)][int(rng.integers(5))]
    ref_extra = []
    for k, flag in (("max_pos", "-max_pos"), ("interval", "-interval"), ("max_mb", "-m")):
        if k in opt:
            ref_extra += [flag, str(opt[k])]
    return fasta, ref_extra, opt, int(rng.integers(1, 4))


@pytest.mark.parametrize("seed", range(12))
def test_native_index_fuzz_against_reference_builder(checker, seed):
    """smr_build_index == the reference's builder up to the id numbering on the random FASTA files and build options of
    fuzz_case."""
    d = tempfile.mkdtemp(prefix="smr_bi_fz_")
    try:
        fasta, ref_extra, opt, threads = fuzz_case(seed, d)
        api.build_index(fasta, os.path.join(d, "x"), threads=threads, **opt)
        equals_reference_builder(checker, f"fuzz_{seed}", fasta, ref_extra, os.path.join(d, "x"))
    finally:
        shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":   # record tests/golden/index_reference.json from the reference's builder (oracle/_ref/sortmerna_ref)
    d = tempfile.mkdtemp(prefix="smr_bi_rec_")
    try:
        exe = os.path.join(d, "index_equiv_check")
        subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "index_equiv_check.cpp")], check=True)
        rec = {}
        for name, ref_extra, kw in OPTION_CASES:
            w = os.path.join(d, "options_" + name)
            rec["options_" + name] = digest(exe, reference_build(os.path.join(GOLDEN, "db_bac.fasta"), w, ref_extra), kw.get("lnwin", 18))
        for seed in range(12):
            w = os.path.join(d, f"fuzz_{seed}")
            os.makedirs(w)
            fasta, ref_extra, _, _ = fuzz_case(seed, w)
            rec[f"fuzz_{seed}"] = digest(exe, reference_build(fasta, os.path.join(w, "ref"), ref_extra))
        with open(GOLDEN_REF, "w") as f:
            json.dump(rec, f, indent=1)
    finally:
        shutil.rmtree(d, ignore_errors=True)
