"""Shared helpers of the parity tests."""
import gzip
import os

import numpy as np

SETS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sets")
# the parity samples of the bundled read sets: the first 100 records of set2 and of both set4 mates (tests/golden/make_sets.py)
SET2_SAMPLE = os.path.join(SETS, "set2_environmental_study_550_amplicon.head100.fasta.gz")
SET4_SAMPLES = [os.path.join(SETS, f"set4_mate_pairs_metatranscriptomics_{k}.head100.fastq.gz") for k in (1, 2)]
ID85 = "silva-bac-16s-database-id85"


def stored_databases(workdir, names):
    """tests/golden/sets/<name>.hits.fasta.gz (the sequences of a bundled database the parity samples align to and its first
    three, made by tests/golden/make_sets.py) unpacked as <workdir>/<name>.fasta; returns the paths in the order of names"""
    out = []
    for n in names:
        p = os.path.join(workdir, n + ".fasta")
        with open(p, "wb") as f:
            f.write(gzip.decompress(open(os.path.join(SETS, n + ".hits.fasta.gz"), "rb").read()))
        out.append(p)
    return out


def unpacked(workdir, gz_paths):
    """the stored .gz read samples unpacked into workdir; returns the paths"""
    out = []
    for g in gz_paths:
        p = os.path.join(workdir, os.path.basename(g)[:-3])
        with open(p, "wb") as f:
            f.write(gzip.decompress(open(g, "rb").read()))
        out.append(p)
    return out


def params_kwargs_from_args(args):
    """Reference CLI arguments of a golden case -> parameter overrides (Runopts::validate, options.cpp:1566-1758)."""
    kw = {}
    i = 0
    while i < len(args):
        a = args[i].lstrip("-")
        if a == "num_alignments":
            kw["num_alignments"] = int(args[i + 1]); i += 2
        elif a == "no-best":
            kw["is_best"] = 0; i += 1
        elif a == "F":
            kw["is_forward"] = 1; kw["is_reverse"] = 0; i += 1
        elif a == "R":
            kw["is_forward"] = 0; kw["is_reverse"] = 1; i += 1
        elif a == "full_search":
            kw["is_full_search"] = 1; i += 1
        elif a in ("match", "mismatch", "gap_open", "gap_ext", "num_seeds", "min_lis"):
            kw[a] = int(args[i + 1]); i += 2
        elif a == "N":
            kw["score_N"] = int(args[i + 1]); i += 2
        elif a == "edges":
            v = args[i + 1]
            if v.endswith("%"):
                kw["edges"] = int(v[:-1]); kw["edges_is_percent"] = 1
            else:
                kw["edges"] = int(v)
            i += 2
        else:
            raise ValueError(f"unknown golden argument {args[i]}")
    if "mismatch" in kw and "score_N" not in kw:
        kw["score_N"] = kw["mismatch"]  # options.cpp:1707-1708
    return kw


def strip_seq(rows):
    return ["\t".join(f[:9] + ["*", "*"] + f[11:]) for f in (r.split("\t") for r in rows)]


def assert_same_results(a, b, what=""):
    """Field-by-field equality of two result dicts (res, alns, cigar) as returned by oracle.ora.align / api.Aligner.align."""
    ra, rb = a["res"], b["res"]
    for f in ra.dtype.names:
        bad = np.nonzero(ra[f] != rb[f])[0]
        assert bad.size == 0, f"{what}: result field {f} differs for reads {bad[:10].tolist()} ({ra[f][bad[:5]]} vs {rb[f][bad[:5]]})"
    slots = a["slots"]
    assert slots == b["slots"]
    for r in range(ra.size):
        for k in range(int(ra["n_align"][r])):
            x, y = a["alns"][r * slots + k], b["alns"][r * slots + k]
            for f in ("ref_num", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "readlen", "score1", "part", "index_num", "strand"):
                assert x[f] == y[f], f"{what}: read {r} alignment {k} field {f}: {x[f]} vs {y[f]}"
            cx = a["cigar"][int(x["cigar_off"]):int(x["cigar_off"]) + int(x["cigar_len"])]
            cy = b["cigar"][int(y["cigar_off"]):int(y["cigar_off"]) + int(y["cigar_len"])]
            assert np.array_equal(cx, cy), f"{what}: read {r} alignment {k} cigar {cx} vs {cy}"


def blast_rows(golden, exp, out, stats):
    """BLAST rows of a result dict the way the reference printed them for this golden case (report_blast.cpp:99-365)."""
    from sortmerna_b200 import hostio
    b = golden["batch"]
    tot = int(np.diff(b.off.astype(np.int64)).sum())
    gum = list(zip(exp["log"]["lambda_"], exp["log"]["K"]))
    evp = [hostio.evalue_params(st, k, tot, b.n) for st, (_, k) in zip(golden["stats"], gum)]
    return hostio.format_blast_rows(b, golden["refs"], out["res"], out["alns"], out["cigar"], out["slots"], stats, gum, evp)


def assert_blast_rows_equal(ours, theirs, evalue_rtol=1.2e-2):
    """Every column identical except the E-value (column 11), which the reference computes from the full-precision Gumbel
    lambda/K while the goldens only hold the 6 digits of aligned.log (exp(-lambda*S) moves by ~1e-4 relative) and prints with 3
    significant digits: tolerance = one unit of the last printed digit (1.2e-2 relative)."""
    a, b = sorted(ours), sorted(theirs)
    assert len(a) == len(b)
    for x, y in zip(a, b):
        fx, fy = x.split("\t"), y.split("\t")
        assert fx[:10] == fy[:10] and fx[11:] == fy[11:], (x, y)
        ex, ey = float(fx[10]), float(fy[10])
        assert abs(ex - ey) <= evalue_rtol * max(abs(ey), 1e-300) + 1e-300, (x, y)
