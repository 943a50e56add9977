"""Parity tests proper (need a B200): the CUDA hot path, called through the C ABI, against the
oracle on the same inputs, and against the committed golden output of the reference binary."""
import os

import numpy as np
import pytest

from conftest import case_names, load_case, load_denovo
from helpers import assert_blast_rows_equal, assert_same_results, blast_rows, params_kwargs_from_args, strip_seq
from sortmerna_b200 import api, hostio

pytestmark = pytest.mark.gpu


def _ora():
    from oracle import ora  # the checker; never imported by the product
    return ora


@pytest.fixture(scope="module")
def aligner(golden):
    a = api.Aligner(0)
    a.set_params(api.default_params())
    exp = load_case("default")
    for k in range(2):
        a.load_index_part(k, 0, golden["prefixes"][k], golden["refs"][k], exp["log"]["minimal_score"][k], (18, 9, 3), golden["stats"][k].lnwin)
    yield a
    a.close()


@pytest.fixture(scope="module")
def oracle_indexes(golden):
    ora = _ora()
    return [ora.OracleIndex(p, 0, s.lnwin) for p, s in zip(golden["prefixes"], golden["stats"])]


def test_index_resident(aligner, oracle_indexes):
    info = aligner.index_info()
    st = [ix.stats() for ix in oracle_indexes]
    assert info["parts"] == 2
    assert info["nodes"] == sum(s["nodes"] for s in st) and info["entries"] == sum(s["entries"] for s in st)
    assert info["ids"] == sum(s["ids"] for s in st) and info["positions"] == sum(s["positions"] for s in st)


def test_seed_windows_match_oracle(aligner, golden, oracle_indexes):
    """traversetrie_align: per-window id hits (order included) and the accept_zero_kmer flag."""
    b = golden["batch"]
    rng = np.random.default_rng(7)
    cat03 = np.where(b.cat > 3, 0, b.cat).astype(np.uint8)
    wr, wp = [], []
    for r in range(b.n):
        ln = int(b.off[r + 1] - b.off[r])
        if ln < 18:
            continue
        for p in range(0, ln - 18 + 1, 3):
            wr.append(r); wp.append(p)
    wr, wp = np.array(wr, np.uint32), np.array(wp, np.uint32)
    for slot, ix in enumerate(oracle_indexes):
      for fallback in (False, True):   # the cooperative search and the per-lane DFS it falls back to
        ids, counts, zero = aligner.debug_seed_windows(slot, cat03, b.off, wr, wp, cap=64, fallback_path=fallback)
        nz = 0
        for k in range(wr.size):
            seq = cat03[int(b.off[wr[k]]):int(b.off[wr[k] + 1])]
            eids, ez = ix.seed_window(seq, int(wp[k]))
            assert counts[k] == eids.size, (slot, k, counts[k], eids)
            assert ids[k, :eids.size].tolist() == eids.tolist(), (slot, k)
            assert bool(zero[k]) == ez
            nz += eids.size > 0
        assert nz > 500


@pytest.mark.parametrize("scores", [(2, -3, -3, 5, 2), (2, -4, -2, 6, 3), (2, -7, -7, 3, 1)])
def test_ssw_matches_oracle(aligner, scores):
    """ssw_align equivalents (score, end, begin, CIGAR) on random pairs, incl. long queries (row blocks) and N."""
    ora = _ora()
    match, mis, sn, go, ge = scores
    aligner.set_params(api.default_params(match=match, mismatch=mis, score_N=sn, gap_open=go, gap_ext=ge))
    mat = ora.score_matrix(match, mis, sn)
    rng = np.random.default_rng(99)
    qs, ts = [], []
    for it in range(600):
        qlen = int(rng.integers(18, 200)) if it % 12 else int(rng.integers(257, 700))
        t = rng.integers(0, 4, qlen + int(rng.integers(0, 30))).astype(np.uint8)
        p = int(rng.integers(0, t.size - qlen + 1))
        q = t[p:p + qlen].copy()
        err = float(rng.choice([0.0, 0.02, 0.1]))
        m = rng.random(q.size) < err
        q[m] = rng.integers(0, 4, int(m.sum()))
        if it % 5 == 0 and q.size > 40:  # an indel
            k = int(rng.integers(10, q.size - 10))
            q = np.concatenate([q[:k], q[k + int(rng.integers(1, 4)):]]) if it % 10 else np.concatenate([q[:k], rng.integers(0, 4, 2).astype(np.uint8), q[k:]])
        if it % 9 == 0:
            q[int(rng.integers(0, q.size))] = 4
            t[int(rng.integers(0, t.size))] = 4
        qs.append(q); ts.append(t)
    # queries shorter than 18, windows of 193..449 columns (both staged-window widths and the 448-column stage limit of the
    # score-only kernels) and windows shorter than the query
    rng2 = np.random.default_rng(199)
    for it in range(300):
        kind = it % 3
        qlen = int(rng2.integers(1, 18)) if kind == 0 else int(rng2.integers(18, 257))
        tlen = int(rng2.integers(193, 450)) if kind < 2 else int(rng2.integers(1, qlen + 1))
        q = rng2.integers(0, 4, qlen).astype(np.uint8)
        t = rng2.integers(0, 4, tlen).astype(np.uint8)
        k = min(qlen, tlen)
        p, o = int(rng2.integers(0, tlen - k + 1)), int(rng2.integers(0, qlen - k + 1))
        t[p:p + k] = q[o:o + k]
        m = rng2.random(tlen) < float(rng2.choice([0.0, 0.02, 0.1]))
        t[m] = rng2.integers(0, 4, int(m.sum()))
        if it % 7 == 0:
            q[int(rng2.integers(0, qlen))] = 4
        qs.append(q); ts.append(t)
    q_off = np.zeros(len(qs) + 1, np.uint64); np.cumsum([x.size for x in qs], out=q_off[1:])
    t_off = np.zeros(len(ts) + 1, np.uint64); np.cumsum([x.size for x in ts], out=t_off[1:])
    out, cig = aligner.debug_ssw(np.concatenate(qs), q_off, np.concatenate(ts), t_off, filters=30, cigar_cap=512)
    for k, (q, t) in enumerate(zip(qs, ts)):
        rc, eo, ec = ora.ssw_align(q.astype(np.int8), t.astype(np.int8), mat, go, ge, 30)
        assert rc == 0
        assert out[k, 0] == eo[0] and out[k, 2] == eo[2] and out[k, 4] == eo[4], (k, out[k], eo)
        if eo[0] >= 30:
            assert out[k, 1] == eo[1] and out[k, 3] == eo[3] and out[k, 5] == eo[5], (k, out[k], eo)
            assert cig[k, :eo[5]].tolist() == ec.tolist(), k
    aligner.set_params(api.default_params())


@pytest.mark.parametrize("case", case_names())
def test_align_matches_oracle_and_reference(aligner, golden, oracle_indexes, case):
    """End to end through smr_align_batch: identical per-read state, alignments and CIGARs to the oracle,
    and identical SAM rows / totals to what the reference binary printed."""
    ora = _ora()
    exp = load_case(case)
    kw = params_kwargs_from_args(exp["args"])
    aligner.set_params(api.default_params(**kw))
    for k in range(2):
        aligner.set_minimal_score(k, exp["log"]["minimal_score"][k])
    b = golden["batch"]
    got = aligner.align(b.cat, b.off)
    want = ora.align(oracle_indexes, [0, 1], [0, 0], 2, golden["refs"], exp["log"]["minimal_score"], [18, 9, 3, 18, 9, 3],
                     ora.default_params(**kw), b, nthreads=4)
    assert_same_results(got, want, case)
    assert got["matched"].tolist() == want["matched"].tolist()
    assert got["counters"]["num_aligned"] == want["counters"]["num_aligned"] == exp["log"]["passing"]
    assert got["counters"]["num_short"] == want["counters"]["num_short_last"]
    rows = hostio.format_sam_rows(b, golden["refs"], got["res"], got["alns"], got["cigar"], got["slots"])
    if case != "default":
        rows = strip_seq(rows)
    assert sorted(rows) == sorted(exp["sam"])
    aligner.set_params(api.default_params())


@pytest.mark.parametrize("case", ["default", "best3", "scores", "nobest2", "rev_only"])
def test_report_arithmetic_on_gpu(aligner, golden, case):
    """smr_aln_stats (calc_miss_gap_match computed by the traceback kernel) == the host restatement for every stored
    alignment, and the BLAST rows built from it == the rows the reference binary printed."""
    exp = load_case(case)
    kw = params_kwargs_from_args(exp["args"])
    aligner.set_params(api.default_params(**kw))
    for k in range(2):
        aligner.set_minimal_score(k, exp["log"]["minimal_score"][k])
    b = golden["batch"]
    got = aligner.align(b.cat, b.off, with_stats=True)
    want = hostio.host_aln_stats(b, golden["refs"], got["res"], got["alns"], got["cigar"], got["slots"])
    slots = got["slots"]
    live = np.zeros(b.n * slots, bool)
    for r in range(b.n):
        live[r * slots:r * slots + int(got["res"]["n_align"][r])] = True
    assert live.sum() > 0
    for f in ("n_miss", "n_gap", "n_match", "n_match_denovo"):
        assert np.array_equal(got["stats"][f][live], want[f][live]), f
    assert_blast_rows_equal(blast_rows(golden, exp, got, got["stats"]), exp["blast"])
    aligner.set_params(api.default_params())


@pytest.mark.parametrize("case", ["default", "best3", "rev_only", "loose"])
def test_denovo_classification_on_gpu(aligner, golden, case):
    """denovo_stats counters / aligned_denovo read set from the GPU's smr_aln_stats == what the reference binary reported."""
    dn = load_denovo()[case]
    aligner.set_params(api.default_params(**params_kwargs_from_args(dn["args"])))
    for k in range(2):
        aligner.set_minimal_score(k, dn["minimal_score"][k])
    b = golden["batch"]
    got = aligner.align(b.cat, b.off, with_stats=True)
    cls = hostio.denovo_classes(got["res"], got["alns"], got["slots"], got["stats"], dn["min_id"], dn["min_cov"])
    assert cls.sum(axis=0).tolist() == dn["counts"]
    ids = sorted(hostio.seq_id(b.headers[r]) for r in np.nonzero(hostio.is_denovo_read(cls))[0])
    assert ids == dn["denovo_reads"]
    aligner.set_params(api.default_params())


def test_batch_of_several_chunks(golden, monkeypatch):
    """A batch larger than the per-launch chunk (1 M reads in production; 200 here via SMR_CHUNK_READS): the chunk loop of
    run_impl must give the results of the single-chunk run."""
    exp = load_case("best3")
    b = golden["batch"]

    def run():
        al = api.Aligner(0)
        al.set_params(api.default_params(num_alignments=3))
        for k in range(2):
            al.load_index_part(k, 0, golden["prefixes"][k], golden["refs"][k], exp["log"]["minimal_score"][k], (18, 9, 3), golden["stats"][k].lnwin)
        out = al.align(b.cat, b.off, with_stats=True)
        al.close()
        return out

    one = run()
    monkeypatch.setenv("SMR_CHUNK_READS", "200")
    many = run()
    assert_same_results(many, one, "4 chunks vs 1")
    assert np.array_equal(many["stats"], one["stats"]) and many["matched"].tolist() == one["matched"].tolist()


def test_multipart_index(golden, golden_parts):
    """3 index parts per database resident at once: identical per-read state / alignments to the oracle's per-part loop and
    identical SAM rows to the reference's `-m 0.5` run (tests/golden/case_parts)."""
    ora = _ora()
    exp = load_case("parts")
    al = api.Aligner(0)
    al.set_params(api.default_params())
    oix, inum, parts, refs, ms = [], [], [], [], []
    for k, g in enumerate(golden_parts):
        for p in range(g["stats"].num_parts):
            al.load_index_part(k, p, g["prefix"], g["part_refs"][p], exp["log"]["minimal_score"][k], (18, 9, 3), g["stats"].lnwin)
            oix.append(ora.OracleIndex(g["prefix"], p, g["stats"].lnwin)); inum.append(k); parts.append(p)
            refs.append(g["part_refs"][p]); ms.append(exp["log"]["minimal_score"][k])
    b = golden["batch"]
    got = al.align(b.cat, b.off)
    want = ora.align(oix, inum, parts, 2, refs, ms, [18, 9, 3] * len(oix), ora.default_params(), b, nthreads=4)
    assert_same_results(got, want, "multipart")
    assert got["matched"].tolist() == want["matched"].tolist()
    by_index = [g["part_refs"] for g in golden_parts]
    rows = strip_seq(hostio.format_sam_rows(b, by_index, got["res"], got["alns"], got["cigar"], got["slots"]))
    assert sorted(rows) == sorted(exp["sam"])
    assert got["counters"]["num_aligned"] == exp["log"]["passing"]
    al.close()


def test_resident_path_equals_host_path(aligner, golden):
    exp = load_case("default")
    for k in range(2):
        aligner.set_minimal_score(k, exp["log"]["minimal_score"][k])
    b = golden["batch"]
    a = aligner.align(b.cat, b.off)
    aligner.upload(b.cat, b.off)
    aligner.run_resident()
    aligner.run_resident()  # idempotent: a second pass over the resident batch gives the same answer
    c = aligner.download()
    assert_same_results(a, c, "resident")
    t = aligner.timings()
    assert t["launches"] > 0 and t["total_ms"] > 0


def test_instrumented_kernels_give_the_same_results(aligner, golden):
    """smr_set_instrumentation: the instrumented instantiations of the seed and candidate kernels (what bench.py's counter pass runs)
    return what the product kernels return; only they fill the seed-side counters."""
    exp = load_case("default")
    for k in range(2):
        aligner.set_minimal_score(k, exp["log"]["minimal_score"][k])
    b = golden["batch"]
    a = aligner.align(b.cat, b.off)
    aligner.set_instrumentation(True)
    try:
        c = aligner.align(b.cat, b.off)
    finally:
        aligner.set_instrumentation(False)
    assert_same_results(a, c, "instrumented")
    for k in ("num_aligned", "num_short", "sw_calls", "sw_cells", "pos_entries", "lis_calls"):
        assert a["counters"][k] == c["counters"][k], k
    assert a["counters"]["windows"] == 0 and c["counters"]["windows"] > 0


def test_edge_batches(aligner, golden, oracle_indexes):
    """empty read, reads shorter than the seed, single read, all-N read, duplicate reads"""
    ora = _ora()
    seqs = [b"", b"ACGT", b"ACGTACGTACGTACGTAC", b"N" * 60, golden["batch"].seqs[0], golden["batch"].seqs[0], b"ACGTTGCA" * 40]
    batch = hostio.pack_reads([f"@r{i}" for i in range(len(seqs))], seqs)
    got = aligner.align(batch.cat, batch.off)
    want = ora.align(oracle_indexes, [0, 1], [0, 0], 2, golden["refs"], [37, 36], [18, 9, 3, 18, 9, 3], ora.default_params(), batch)
    assert_same_results(got, want, "edge")
    assert got["counters"]["num_short"] == want["counters"]["num_short_last"] == 2
    one = hostio.pack_reads(["@x"], [golden["batch"].seqs[3]])
    g1 = aligner.align(one.cat, one.off)
    w1 = ora.align(oracle_indexes, [0, 1], [0, 0], 2, golden["refs"], [37, 36], [18, 9, 3, 18, 9, 3], ora.default_params(), one)
    assert_same_results(g1, w1, "single")


def test_long_read_t0(golden_t0):
    """BASELINE config 1: a 1.5 kb read (several SW row blocks, score > 255) -- identical to the oracle and to the reference SAM row."""
    ora = _ora()
    g = golden_t0
    a = api.Aligner(0)
    a.set_params(api.default_params())
    a.load_index_part(0, 0, g["prefix"], g["refs"], g["exp"]["log"]["minimal_score"][0], (18, 9, 3), g["stats"].lnwin)
    got = a.align(g["batch"].cat, g["batch"].off)
    ix = ora.OracleIndex(g["prefix"], 0, g["stats"].lnwin)
    want = ora.align([ix], [0], [0], 1, [g["refs"]], g["exp"]["log"]["minimal_score"], [18, 9, 3], ora.default_params(), g["batch"])
    assert_same_results(got, want, "t0")
    rows = hostio.format_sam_rows(g["batch"], [g["refs"]], got["res"], got["alns"], got["cigar"], got["slots"])
    assert rows == g["exp"]["sam"]
    a.close()
