"""ora_ssw_align (the restated ssw_init + ssw_align, ssw.c:788-941) against the reference's OWN ssw.c,
compiled unmodified into oracle/_ref/libssw_ref.so by oracle/Makefile.ref.  Where that library is absent, the reference's
results come from tests/golden/ssw_reference.json, recorded from it by this file's __main__: a digest of every 100 cases."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import ora

GOLDEN_REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ssw_reference.json")
SCORES = [(2, -3, -3, 5, 2), (2, -4, -2, 6, 3), (1, -3, -3, 5, 2), (2, -7, -7, 3, 1),
          # the schemes tests/test_gpu_sw_scorer.py adds: gap_ext == gap_open, gap_ext == 0, score_N = 0, and the edges of the int8 matrix
          (2, -3, -3, 4, 4), (2, -3, -3, 5, 0), (2, -3, 0, 5, 2), (125, -128, -128, 255, 1), (126, -128, -128, 255, 1)]
BLOCK = 100


class SAlign(C.Structure):  # s_align, include/ssw.h:58-71
    _fields_ = [("cigar", C.POINTER(C.c_uint32)), ("ref_num", C.c_uint32), ("ref_begin1", C.c_int32), ("ref_end1", C.c_int32),
                ("read_begin1", C.c_int32), ("read_end1", C.c_int32), ("readlen", C.c_uint32), ("score1", C.c_uint16),
                ("part", C.c_uint16), ("index_num", C.c_uint16), ("cigarLen", C.c_uint16), ("strand", C.c_bool)]


def ref_ssw(lib, read, ref, mat, go, ge, filters):
    prof = lib.ssw_init(read.ctypes.data_as(C.c_void_p), len(read), mat.ctypes.data_as(C.c_void_p), 5, 2)
    r = lib.ssw_align(prof, ref.ctypes.data_as(C.c_void_p), len(ref), go, ge, 2, filters, 0, 0)
    a = r.contents
    out = (a.score1, a.ref_begin1, a.ref_end1, a.read_begin1, a.read_end1, [a.cigar[i] for i in range(a.cigarLen)])
    pp = C.c_void_p(prof)
    lib.init_destroy(C.byref(pp))
    return out


def make_pair(rng, qlen, tlen, err, nfrac=0.0):
    t = rng.integers(0, 4, tlen).astype(np.int8)
    p = int(rng.integers(0, max(1, tlen - qlen + 1)))
    q = []
    for c in t[p:p + qlen]:
        u = rng.random()
        if u < err / 3:
            continue
        if u < 2 * err / 3:
            q.append(rng.integers(0, 4))
        q.append(rng.integers(0, 4) if rng.random() < err else c)
    q = np.array(q[:qlen] if q else [0], dtype=np.int8)
    if nfrac:
        q[rng.random(q.size) < nfrac] = 4
        t = t.copy(); t[rng.random(t.size) < nfrac] = 4
    flank = rng.integers(0, 4, int(rng.integers(0, 8))).astype(np.int8)
    return np.concatenate([flank, q]), t


def reference_lib():
    lib = C.CDLL(ora.REF_SSW)
    lib.ssw_init.restype = C.c_void_p
    lib.ssw_init.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int8]
    lib.ssw_align.restype = C.POINTER(SAlign)
    lib.ssw_align.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_uint8, C.c_uint8, C.c_uint8, C.c_uint16, C.c_int32, C.c_int32]
    return lib


def cases(scores):
    """(q, t, filters) of the 1500 pairs of one scoring set"""
    match, mis, sn, go, ge = scores
    rng = np.random.default_rng(1234 + match * 7 + go)
    # the reference's word kernel saturates at 32767 (ssw.c:399-575) where the restatement keeps counting: with large match scores the
    # queries stay short enough (flank included) that no score gets there
    qmax = 32767 // match - 8
    for it in range(1500):
        qlen = int(rng.integers(20, 181)) if it % 10 else int(rng.integers(250, 500))
        qlen = min(qlen, qmax)
        tlen = qlen + int(rng.integers(-10, 40))
        q, t = make_pair(rng, qlen, max(20, tlen), float(rng.choice([0.0, 0.01, 0.05, 0.15])), nfrac=0.01 if it % 7 == 0 else 0.0)
        yield q, t, int(rng.integers(0, 60))


def pinned(score, ref_begin, ref_end, read_begin, read_end, cigar, filters):
    """what the comparison pins: score and end points always, begin points and CIGAR where the score passes the filter"""
    return [score, ref_end, read_end] + ([ref_begin, read_begin, cigar] if score >= filters else [])


def block_digests(rows):
    return [hashlib.sha256(json.dumps(rows[k:k + BLOCK]).encode()).hexdigest()[:16] for k in range(0, len(rows), BLOCK)]


def reference_results(scores):
    """[pinned(...) per case], word-path count -- from the reference's ssw.c"""
    lib = reference_lib()
    match, mis, sn, go, ge = scores
    mat = ora.score_matrix(match, mis, sn)
    rows, n_word = [], 0
    for q, t, filters in cases(scores):
        e = ref_ssw(lib, q, t, mat, go, ge, filters)
        rows.append(pinned(e[0], e[1], e[2], e[3], e[4], e[5], filters))
        n_word += e[0] >= 255 - abs(min(mis, sn))
    return rows, n_word


@pytest.mark.parametrize("scores", SCORES)
def test_ssw_restatement_matches_reference_ssw(scores):
    match, mis, sn, go, ge = scores
    mat = ora.score_matrix(match, mis, sn)
    rows = []
    for q, t, filters in cases(scores):
        rc, out, cig = ora.ssw_align(q, t, mat, go, ge, filters)
        assert rc == 0
        rows.append(pinned(int(out[0]), int(out[1]), int(out[2]), int(out[3]), int(out[4]), cig.tolist(), filters))
    golden = json.load(open(GOLDEN_REF))[str(scores)]
    if os.path.exists(ora.REF_SSW):
        exp, n_word = reference_results(scores)
        for it, (g, e) in enumerate(zip(rows, exp)):
            assert g == e, (it, g, e)
        assert {"blocks": block_digests(exp), "word_path_cases": int(n_word)} == golden    # the recording still describes the reference
    else:
        n_word = golden["word_path_cases"]
        for k, (g, e) in enumerate(zip(block_digests(rows), golden["blocks"])):
            assert g == e, f"cases {k * BLOCK}..{k * BLOCK + BLOCK - 1} differ from the reference's"
        assert len(rows) == BLOCK * len(golden["blocks"])
    assert n_word > 20  # the int16 (word) path of the reference was exercised too


if __name__ == "__main__":   # record tests/golden/ssw_reference.json from oracle/_ref/libssw_ref.so
    rec = {}
    for sc in SCORES:
        exp, n_word = reference_results(sc)
        rec[str(sc)] = {"blocks": block_digests(exp), "word_path_cases": int(n_word)}
    with open(GOLDEN_REF, "w") as f:
        json.dump(rec, f, indent=1)
