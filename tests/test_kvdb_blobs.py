"""smr_pack_kvdb_blobs (sortmerna_b200/csrc/smr_blob.cpp) against the UNMODIFIED reference's Read::toBinString():
oracle/_ref/blob_ref (oracle/blob_ref_main.cpp linked with the reference's own objects) serialises the same alignments through
the reference's classes; the bytes must be identical.  Where the reference build is absent the committed golden blobs
(tests/golden/kvdb_blobs.json, made by this file's __main__ from blob_ref) pin the writer."""
import hashlib
import json
import os
import struct
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, load_case, load_denovo
from helpers import params_kwargs_from_args
from sortmerna_b200 import api, hostio

BLOB_REF = os.path.join(ROOT, "oracle", "_ref", "blob_ref")
GOLD = os.path.join(GOLDEN, "kvdb_blobs.json")


def reference_blobs(out, num_alignments, denovo):
    res, alns, cig = out["res"], out["alns"], np.ascontiguousarray(out["cigar"], np.uint32)
    n, slots = res.shape[0], int(out["slots"])
    dn = np.ascontiguousarray(denovo, np.uint32) if denovo is not None else np.zeros((n, 4), np.uint32)
    payload = struct.pack("<IIiQ", n, slots, num_alignments, cig.size) + res.tobytes() + alns.tobytes() + cig.tobytes() + dn.tobytes()
    p = subprocess.run([BLOB_REF], input=payload, capture_output=True, check=True)
    blobs, o = [], 0
    for _ in range(n):
        (ln,) = struct.unpack_from("<Q", p.stdout, o); o += 8
        blobs.append(p.stdout[o:o + ln]); o += ln
    assert o == len(p.stdout)
    return blobs


def oracle_case(golden, case, denovo_case=None):
    from oracle import ora
    if denovo_case:
        dn = load_denovo()[denovo_case]
        args, ms = dn["args"], dn["minimal_score"]
    else:
        exp = load_case(case)
        args, ms = exp["args"], exp["log"]["minimal_score"]
    kw = params_kwargs_from_args(args)
    oix = [ora.OracleIndex(p, 0, s.lnwin) for p, s in zip(golden["prefixes"], golden["stats"])]
    out = ora.align(oix, [0, 1], [0, 0], 2, golden["refs"], ms, [18, 9, 3, 18, 9, 3], ora.default_params(**kw), golden["batch"], nthreads=2)
    denovo = None
    if denovo_case:
        st = hostio.host_aln_stats(golden["batch"], golden["refs"], out["res"], out["alns"], out["cigar"], out["slots"])
        denovo = hostio.denovo_classes(out["res"], out["alns"], out["slots"], st, dn["min_id"], dn["min_cov"])
    return out, kw.get("num_alignments", 1), denovo


CASES = [("default", None), ("best3", None), ("nobest2", None), (None, "best3")]


def ours(out, num_alignments, denovo):
    buf, off = api.pack_kvdb_blobs(out, num_alignments, denovo)
    return [bytes(buf[int(off[r]):int(off[r + 1])]) for r in range(out["res"].shape[0])]


@pytest.mark.parametrize("case,denovo_case", CASES)
def test_blobs_equal_reference_serializer(golden, case, denovo_case):
    if not os.path.exists(BLOB_REF):     # the reference serializer's bytes as recorded from it
        return test_blobs_equal_committed_golden(golden, case, denovo_case)
    out, na, denovo = oracle_case(golden, case, denovo_case)
    mine, ref = ours(out, na, denovo), reference_blobs(out, na, denovo)
    assert len(mine) == len(ref)
    for r, (a, b) in enumerate(zip(mine, ref)):
        assert a == b, f"read {r}: {a.hex()[:80]} vs {b.hex()[:80]}"
    assert sum(1 for b in mine if b) == int((out["res"]["n_align"] > 0).sum())


@pytest.mark.parametrize("case,denovo_case", CASES)
def test_blobs_equal_committed_golden(golden, case, denovo_case):
    out, na, denovo = oracle_case(golden, case, denovo_case)
    mine = ours(out, na, denovo)
    g = json.load(open(GOLD))[f"{case}|{denovo_case}"]
    assert len(mine) == g["n"] and sum(len(b) for b in mine) == g["total_bytes"]
    assert hashlib.sha256(b"".join(struct.pack("<Q", len(b)) + b for b in mine)).hexdigest() == g["sha256"]
    assert mine[g["first_nonempty"]].hex() == g["first_blob_hex"]


def test_blob_layout_round_trip(golden):
    """parse a blob back field by field (Read::load_db order, read.cpp:467-539)"""
    out, na, _ = oracle_case(golden, "best3")
    mine = ours(out, na, None)
    slots = out["slots"]
    for r in np.nonzero(out["res"]["n_align"] > 1)[0][:20]:
        b, res = mine[r], out["res"][r]
        li, lp, c0, c1, c2, c3, done, hit, nul, msw, nal, hs, asz = struct.unpack_from("<6I3BHiIQ", b, 0)
        assert (li, lp, done, hit, nul, msw, nal, hs) == (res["lastIndex"], res["lastPart"], res["is_done"], res["is_hit"], 0, res["max_SW_count"], 3, res["hit_seeds"])
        o = struct.calcsize("<6I3BHiIQ")
        assert asz == len(b) - o
        mn, mx, nv = struct.unpack_from("<IIQ", b, o); o += 16
        assert (mn, mx, nv) == (res["min_index"], res["max_index"], res["n_align"])
        for k in range(nv):
            al = out["alns"][r * slots + k]
            (sz, nc) = struct.unpack_from("<QQ", b, o); o += 16
            cig = np.frombuffer(b, "<u4", nc, o); o += 4 * nc
            assert np.array_equal(cig, out["cigar"][int(al["cigar_off"]):int(al["cigar_off"]) + nc])
            f = struct.unpack_from("<IiiiiIHHHB", b, o); o += struct.calcsize("<IiiiiIHHHB")
            assert f == tuple(int(al[x]) for x in ("ref_num", "ref_begin1", "ref_end1", "read_begin1", "read_end1", "readlen", "score1", "part", "index_num", "strand"))
            assert sz == 8 + 4 * nc + struct.calcsize("<IiiiiIHHHB")
        assert o == len(b)


if __name__ == "__main__":   # regenerate tests/golden/kvdb_blobs.json from the reference serializer (needs oracle/_ref/blob_ref)
    import sys
    sys.path.insert(0, ROOT)
    import conftest
    import tempfile, gzip, shutil
    d = tempfile.mkdtemp()
    for fn in os.listdir(os.path.join(GOLDEN, "idx")):
        src = os.path.join(GOLDEN, "idx", fn)
        if fn.endswith(".gz"):
            open(os.path.join(d, fn[:-3]), "wb").write(gzip.open(src).read())
        else:
            shutil.copy(src, d)
    refs = [hostio.load_references(os.path.join(GOLDEN, n)) for n in ("db_arc.fasta", "db_bac.fasta")]
    pre = hostio.find_index_prefixes(d)
    prefixes = [pre["db_arc.fasta"], pre["db_bac.fasta"]]
    golden = dict(refs=refs, prefixes=prefixes, stats=[hostio.parse_stats(p) for p in prefixes], batch=hostio.load_reads(os.path.join(GOLDEN, "reads_mix.fq")))
    res = {}
    for case, dc in CASES:
        out, na, denovo = oracle_case(golden, case, dc)
        ref = reference_blobs(out, na, denovo)
        first = next(i for i, b in enumerate(ref) if b)
        res[f"{case}|{dc}"] = dict(n=len(ref), total_bytes=sum(len(b) for b in ref), first_nonempty=first, first_blob_hex=ref[first].hex(),
                                   sha256=hashlib.sha256(b"".join(struct.pack("<Q", len(b)) + b for b in ref)).hexdigest())
        print(case, dc, res[f"{case}|{dc}"]["n"], res[f"{case}|{dc}"]["total_bytes"])
    json.dump(res, open(GOLD, "w"), indent=0)
