"""The candidate kernel's scorer -- the fetcher's staging, the packed 16-bit pass (sw_pair_warp, pair_profile, pair_sentinels,
the profile cache) and the s32 fallback -- called directly through smr_debug_sw_tasks, against an exact int32 Gotoh
(ora.ssw_align) on every shape, strand, buffer alignment and scoring scheme the scorer accepts.  A failure names the
(scheme, pair, task) that broke.

The CPU test at the end checks ora.ssw_align's score itself against a brute-force Gotoh written here, for every scheme used."""
import numpy as np
import pytest

from oracle import ora

# (match, mismatch, score_N, gap_open, gap_ext), all within the reference's int8 matrix and uint8 gaps
PACKED_SETS = [(2, -3, -3, 5, 2), (2, -4, -2, 6, 3), (1, -3, -3, 5, 2), (2, -7, -7, 3, 1),
               (2, -3, -3, 4, 4),          # gap_ext == gap_open
               (2, -3, -3, 5, 0),          # gap_ext == 0
               (125, -128, -128, 255, 1)]  # m = 256: an exact match scores exactly 32000, the packed pass's limit
FALLBACK_SETS = [(126, -128, -128, 255, 1),  # m >= 254: 126 * m > 32000
                 (2, -3, -3, 3, 4),          # gap_ext > gap_open
                 (2, -3, 0, 5, 2)]           # score_N = 0
ALL_SETS = PACKED_SETS + FALLBACK_SETS

M_SHAPES = [1, 2, 17, 31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128, 129, 159, 160, 161, 191, 192, 193, 224, 255, 256, 257, 300]
N_SHAPES = [1, 2, 31, 32, 33, 63, 64, 65, 150, 191, 192, 193, 300, 447, 448, 449, 600]
NO_TASK = -1


def sw_pair_ok(m, n, sc):
    """smr_sw.cuh sw_pair_ok: the shapes and schemes the packed 16-bit pass takes"""
    match, mis, sn, go, ge = sc
    return (m <= 256 and n <= 448 and -1024 < mis < 0 and 0 < go < 1024 and -1024 < sn < 0 and 0 <= ge <= go and match >= 0
            and m * match <= 32000)


def pair_rows(m):
    """smr_sw.cuh pair_rows: rows per lane of the packed pass"""
    for r, top in ((1, 32), (2, 64), (3, 96), (4, 128), (5, 160), (6, 192)):
        if m <= top:
            return r
    return 8


def comp(x):
    return np.where(x < 4, 3 - x, x).astype(np.uint8)


class Workload:
    """Query and reference buffers plus task records (ref_abs, q_abs, n, m, minus) and pairs, built the way the planner
    builds them: a query identity (q_abs, m, strand) may be shared by several tasks, each task has a window of its own."""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.q = []          # byte chunks of the query buffer
        self.qlen = 0
        self.t = []
        self.tlen = 0
        self.queries = []    # (q_abs, m, minus, bases as the strand reads them)
        self.tasks = []      # [ref_abs, q_abs, n, m, minus]
        self.expect_q = []   # index into self.queries (-1: empty task)
        self.windows = []
        self.pairs = []
        self.res = 0

    def _pad_to(self, chunks, cur, res):
        k = (res - cur) % 16
        chunks.append(self.rng.integers(0, 4, k).astype(np.uint8))
        return cur + k

    def seq(self, n, kind):
        if kind == "alln":
            return np.full(n, 4, np.uint8)
        s = self.rng.integers(0, 4, n).astype(np.uint8)
        if kind == "nrich":
            s[self.rng.random(n) < 0.3] = 4
        return s

    def add_query(self, m, minus, kind="random"):
        """stores a query of m rows; its first byte in the buffer lands on the next residue mod 16"""
        bases = self.seq(m, kind)
        seg = comp(bases[::-1]) if minus else bases
        self.res = (self.res + 1) % 16
        self.qlen = self._pad_to(self.q, self.qlen, self.res)
        start = self.qlen
        self.q.append(seg)
        self.qlen += m
        q_abs = start + m - 1 if minus and m else start
        self.queries.append((q_abs, m, minus, bases))
        return len(self.queries) - 1

    def add_twins(self, m):
        """two query identities with the same q_abs and m, one per strand: the plus one reads forwards from q_abs, the minus one
        backwards (they share only the byte at q_abs)"""
        seg = self.seq(2 * m - 1, "random")
        self.res = (self.res + 1) % 16
        self.qlen = self._pad_to(self.q, self.qlen, self.res)
        s = self.qlen + m - 1
        self.q.append(seg)
        self.qlen += seg.size
        self.queries.append((s, m, False, seg[m - 1:].copy()))
        self.queries.append((s, m, True, comp(seg[m - 1::-1])))
        return len(self.queries) - 2, len(self.queries) - 1

    def window_for(self, qi, n, kind):
        """a window of n columns for query qi: unrelated, a mutated copy of (part of) the query, or one whose best alignment ends on
        column 0, on column n-1 or on the query's last row"""
        bases = self.queries[qi][3]
        m = bases.size
        rng = self.rng
        w = self.seq(n, "nrich" if kind == "nrich" else "alln" if kind == "alln" else "random")
        if kind in ("random", "nrich", "alln") or m == 0:
            return w
        if kind == "col0":
            w[1:] = 4
            w[0] = bases[-1]
            return w
        if kind == "collast":
            k = min(n, m)
            w[n - k:] = bases[:k]
            return w
        if kind == "rowlast":
            k = min(n, m, int(rng.integers(1, 40)))
            p = int(rng.integers(0, n - k + 1))
            w[p:p + k] = bases[m - k:]
            return w
        # homolog: a copy of the query with substitutions (and for "indel" one gap of up to 40 in the query or the window)
        src = bases.copy()
        if kind == "indel" and m > 8:
            g = int(rng.integers(1, 41))
            k = int(rng.integers(1, m - 1))
            src = np.concatenate([src[:k], src[k + g:]]) if rng.random() < 0.5 else np.concatenate([src[:k], self.seq(g, "random"), src[k:]])
        rate = {"hom0": 0.0, "hom1": 0.01, "hom10": 0.1}.get(kind, 0.01)
        mut = rng.random(src.size) < rate
        src[mut] = (src[mut] + rng.integers(1, 4, int(mut.sum()))) % 4
        if src.size <= n:
            p = int(rng.integers(0, n - src.size + 1))
            w[p:p + src.size] = src
        else:
            p = int(rng.integers(0, src.size - n + 1))
            w[:] = src[p:p + n]
        return w

    def add_task(self, qi, n, kind="hom1"):
        w = self.window_for(qi, n, kind) if n else np.zeros(0, np.uint8)
        self.res = (self.res + 5) % 16
        self.tlen = self._pad_to(self.t, self.tlen, self.res)
        ref_abs = self.tlen
        self.t.append(w)
        self.tlen += n
        q_abs, m, minus, _ = self.queries[qi]
        self.tasks.append([ref_abs, q_abs, n, m, int(minus)])
        self.expect_q.append(qi)
        self.windows.append(w)
        return len(self.tasks) - 1

    def add_empty(self, m, n):
        """a task with no rows or no columns (what the planner emits for an empty query segment)"""
        qi = self.add_query(m, bool(self.rng.integers(0, 2)))
        return self.add_task(qi, n, "random")

    def buffers(self):
        return np.concatenate(self.q or [np.zeros(0, np.uint8)]), np.concatenate(self.t or [np.zeros(0, np.uint8)])

    def expected(self, sc):
        match, mis, sn, go, ge = sc
        mat = ora.score_matrix(match, mis, sn)
        out = np.zeros(len(self.tasks), np.int64)
        for i, (ref_abs, q_abs, n, m, minus) in enumerate(self.tasks):
            if m == 0 or n == 0:
                continue
            bases = self.queries[self.expect_q[i]][3]
            rc, res, _ = ora.ssw_align(bases.astype(np.int8), self.windows[i].astype(np.int8), mat, go, ge, 0)
            assert rc == 0
            out[i] = int(res[0])
        return out


KINDS = ["random", "hom0", "hom1", "hom10", "indel", "col0", "collast", "rowlast", "nrich", "alln"]
QKINDS = ["random"] * 8 + ["nrich", "alln"]


def build_workload(seed, a_shapes, m_cap, n_pairs_random):
    """Pairs in chain order.  A tasks: every (m, n, strand) of a_shapes, then n_pairs_random random ones.  B: a task of an independent
    shape, none, an empty task, a task sharing A's query (the shared-profile case), or the query of a recent pair (cache reuse / swap)."""
    W = Workload(seed)
    rng = W.rng
    ms = [m for m in M_SHAPES if m <= m_cap]
    shapes = list(a_shapes) + [(int(rng.choice(ms)), int(rng.choice(N_SHAPES)), bool(rng.integers(0, 2))) for _ in range(n_pairs_random)]
    order = rng.permutation(len(shapes))
    recent = []
    for j in order:
        m, n, minus = shapes[j]
        u = rng.random()
        if u < 0.08:   # B: the same q_abs and m on the other strand (the profile cache must tell them apart)
            qp, qm = W.add_twins(m)
            qa, qb = (qm, qp) if minus else (qp, qm)
        else:
            qa = W.add_query(m, minus, str(rng.choice(QKINDS)))
        ta = W.add_task(qa, n, str(rng.choice(KINDS)))
        if u < 0.08:
            tb = W.add_task(qb, int(rng.choice(N_SHAPES)), str(rng.choice(KINDS)))
        elif u < 0.35:
            qb = W.add_query(int(rng.choice(ms)), bool(rng.integers(0, 2)), str(rng.choice(QKINDS)))
            tb = W.add_task(qb, int(rng.choice(N_SHAPES)), str(rng.choice(KINDS)))
        elif u < 0.45:
            tb = NO_TASK
        elif u < 0.55:
            tb = W.add_empty(0, int(rng.choice(N_SHAPES))) if rng.random() < 0.5 else W.add_empty(int(rng.choice(ms)), 0)
        elif u < 0.75:
            tb = W.add_task(qa, int(rng.choice(N_SHAPES)), str(rng.choice(KINDS)))   # same query, another window
        else:
            qb = recent[int(rng.integers(0, len(recent)))] if recent else qa    # the query of a recent pair: a cached half reused or swapped
            tb = W.add_task(qb, int(rng.choice(N_SHAPES)), str(rng.choice(KINDS)))
        if rng.random() < 0.5:
            ta, tb = (tb, ta) if tb != NO_TASK else (ta, tb)
        W.pairs.append((ta, tb))
        recent = ([qa] + recent)[:3]
    # a query and a window that end on the last byte of their buffers, the query read on both strands
    qi = W.add_query(65, True, "random")
    tq = W.queries[qi]
    qj = len(W.queries)
    W.queries.append((tq[0] - 64, 65, False, comp(tq[3][::-1])))   # the same bytes read forwards: query element 0 = first byte
    ta = W.add_task(qj, 300, "hom1")
    tb = W.add_task(qi, 193, "hom1")   # the last window: it ends on the last byte of the reference buffer
    W.pairs.append((ta, tb))
    return W


def expected_paths(W, sc):
    out = []
    for ta, tb in W.pairs:
        _, _, na, ma, _ = W.tasks[ta]
        oka = ma > 0 and na > 0 and sw_pair_ok(ma, na, sc)
        if tb == NO_TASK:
            okb = True
        else:
            _, _, nb, mb, _ = W.tasks[tb]
            okb = mb == 0 or nb == 0 or sw_pair_ok(mb, nb, sc)
        out.append(oka and okb)
    return np.array(out, bool)


def run_and_check(aligner, W, sc, chain):
    from sortmerna_b200 import api
    match, mis, sn, go, ge = sc
    aligner.set_params(api.default_params(match=match, mismatch=mis, score_N=sn, gap_open=go, gap_ext=ge))
    qbuf, tbuf = W.buffers()
    # the last query and window end on the last byte of their buffers
    assert any(t[1] + 1 == qbuf.size and t[4] for t in W.tasks) and any(t[0] + t[2] == tbuf.size for t in W.tasks)
    got, path = aligner.debug_sw_tasks(qbuf, tbuf, np.array(W.tasks), np.array(W.pairs), chain=chain)
    want = W.expected(sc)
    want_path = expected_paths(W, sc)
    bad = np.nonzero(got != want)[0]
    if bad.size:
        msgs = []
        for i in bad[:10]:
            k = next(k for k, p in enumerate(W.pairs) if i in p)
            ref_abs, q_abs, n, m, minus = W.tasks[i]
            ta, tb = W.pairs[k]
            other = W.tasks[tb if ta == i else ta] if tb != NO_TASK else None
            msgs.append(f"task {i} (m={m} n={n} {'minus' if minus else 'plus'} ref_abs%16={ref_abs % 16}) of pair {k} "
                        f"[{'packed' if want_path[k] else 's32'}, other task {other}]: got {got[i]}, want {want[i]}")
        pytest.fail(f"scheme {sc}, chain {chain}: {bad.size} of {len(W.tasks)} task scores differ\n" + "\n".join(msgs))
    assert np.array_equal(path, want_path), (sc, np.nonzero(path != want_path)[0][:10])
    return path


def coverage(W, path):
    """(R, strand of A) and (R, sign of nA - nB) of the pairs the packed pass scored"""
    seen = set()
    for (ta, tb), packed in zip(W.pairs, path):
        if not packed or tb == NO_TASK:
            continue
        _, _, na, ma, minus = W.tasks[ta]
        _, _, nb, mb, _ = W.tasks[tb]
        r = pair_rows(max(ma, mb))
        seen.add((r, "minus" if minus else "plus"))
        if na != nb:
            seen.add((r, "nA<nB" if na < nb else "nA>nB"))
    return seen


@pytest.fixture(scope="module")
def aligner():
    from sortmerna_b200 import api
    a = api.Aligner(0)
    a.set_params(api.default_params())
    yield a
    a.close()


@pytest.mark.gpu
@pytest.mark.parametrize("chain", [1, 8])
def test_scorer_every_shape_default_scheme(aligner, chain):
    """Every (m, n, strand) as task A, B of an independent shape / none / empty / the same query; chains of 8 pairs keep the profile
    cache across R changes and s32 fallbacks, as one scorer warp does."""
    shapes = [(m, n, minus) for m in M_SHAPES for n in N_SHAPES for minus in (False, True)]
    W = build_workload(11 + chain, shapes, 300, 200)
    path = run_and_check(aligner, W, (2, -3, -3, 5, 2), chain)
    seen = coverage(W, path)
    for r in (1, 2, 3, 4, 5, 6, 8):
        for tag in ("plus", "minus", "nA<nB", "nA>nB"):
            assert (r, tag) in seen, (r, tag)
    assert path.sum() > 0.5 * path.size and (~path).sum() > 50


@pytest.mark.gpu
@pytest.mark.parametrize("scores", ALL_SETS[1:])
def test_scorer_other_schemes(aligner, scores):
    """The other schemes on random shapes; for match >= 125 queries stay short enough that no score leaves 15 bits on the
    reference's side (m <= 257 -- both sides of the packed pass's 32000 limit)."""
    m_cap = 257 if scores[0] >= 125 else 300
    shapes = []
    if scores[0] >= 125:   # an exact match at the packed pass's limit and just past it, both strands
        shapes = [(m, n, minus) for m in (253, 254, 255, 256, 257) for n in (256, 300) for minus in (False, True)]
    W = build_workload(1000 + sum(abs(x) * 7 ** k for k, x in enumerate(scores)), shapes, m_cap, 350)
    path = run_and_check(aligner, W, scores, 8)
    if scores in PACKED_SETS:
        assert path.sum() > 0.5 * path.size
    else:
        assert (~path).sum() > 0
    if scores[0] >= 125:
        # the exact-match ceiling itself: m = 256 on the packed path scores 125 * 256 = 32000
        W2 = Workload(5)
        qa = W2.add_query(256, False)
        ta = W2.add_task(qa, 256, "hom0")
        qb = W2.add_query(256, True)
        tb = W2.add_task(qb, 300, "hom0")
        W2.pairs = [(ta, tb)]
        run_and_check(aligner, W2, scores, 1)


@pytest.mark.gpu
def test_scorer_rejects_tasks_outside_the_buffers(aligner):
    from sortmerna_b200 import api
    q = np.zeros(100, np.uint8); t = np.zeros(200, np.uint8)
    ok = [[0, 0, 200, 100, 0]]
    aligner.debug_sw_tasks(q, t, ok, [[0, -1]])
    for bad in ([1, 0, 200, 10, 0], [0, 91, 10, 10, 0], [0, 100, 10, 1, 1], [0, 8, 10, 10, 1]):
        with pytest.raises(api.SmrError):
            aligner.debug_sw_tasks(q, t, [bad], [[0, -1]])
    with pytest.raises(api.SmrError):
        aligner.debug_sw_tasks(q, t, ok, [[0, 1]])


def gotoh_int64(q, t, mat, go, ge):
    """brute-force local Gotoh: H = max(0, diag + s, E, F), E / F = max(previous - ge, H - go) along a row / column"""
    m, n = q.size, t.size
    s = mat.reshape(5, 5).astype(np.int64)[t[None, :], q[:, None]]   # s[i, j] = mat[ref * 5 + read]
    H = np.zeros((m + 1, n + 1), np.int64)
    F = np.zeros((m + 1, n + 1), np.int64)
    best = 0
    for i in range(1, m + 1):
        F[i, 1:] = np.maximum(F[i - 1, 1:] - ge, H[i - 1, 1:] - go)
        e = 0
        for j in range(1, n + 1):
            h = max(0, H[i - 1, j - 1] + s[i - 1, j - 1], e, F[i, j])
            H[i, j] = h
            e = max(e - ge, h - go)
        best = max(best, int(H[i].max()))
    return best


@pytest.mark.parametrize("scores", ALL_SETS)
def test_oracle_score_matches_brute_force_gotoh(scores):
    """ora.ssw_align's score (the GPU tests' expected value) == an independent int64 Gotoh, on small cases of every scheme above"""
    match, mis, sn, go, ge = scores
    mat = ora.score_matrix(match, mis, sn)
    rng = np.random.default_rng(77 + match + go * 3 + ge)
    for it in range(300):
        m, n = int(rng.integers(1, 25)), int(rng.integers(1, 33))
        t = rng.integers(0, 4, n).astype(np.int8)
        if it % 3:
            p = int(rng.integers(0, n))
            q = np.concatenate([t[p:p + m], rng.integers(0, 4, max(0, m - (n - p))).astype(np.int8)])[:m].copy()
            q[rng.random(m) < 0.15] = rng.integers(0, 4)
            if it % 5 == 0 and m > 6:
                k = int(rng.integers(1, m - 2))
                q = np.concatenate([q[:k], q[k + 2:], rng.integers(0, 4, 2).astype(np.int8)])
        else:
            q = rng.integers(0, 4, m).astype(np.int8)
        if it % 4 == 0:
            q[rng.random(m) < 0.3] = 4
            t[rng.random(n) < 0.3] = 4
        rc, out, _ = ora.ssw_align(q, t, mat, go, ge, 0)
        assert rc == 0
        assert int(out[0]) == gotoh_int64(q, t, mat, go, ge), (scores, it, q.tolist(), t.tolist())
