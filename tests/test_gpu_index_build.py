"""Index build on the device (smr_build_index_device, SURVEY 8(f)(3): build_index, src/sortmerna/indexdb.cpp:1119-2095) against the
index smr_load_index_part makes from FILES: the reference builder's own files for the golden databases, and the files of the host
builder (smr_build_index, itself proven equal to the reference's in tests/test_index_builder.py) for the option variants.  Every
resident array must be equal up to the numbering of the L-mer ids, and alignment results must be identical."""
import os
import tempfile

import numpy as np
import pytest

from conftest import GOLDEN, load_case
from helpers import assert_same_results, strip_seq
from sortmerna_b200 import api, hostio

pytestmark = pytest.mark.gpu


def canon_ids(pos_off, pos):
    """id -> (seq << 32 | pos) of its first position: a name of the L-mer that does not depend on the numbering"""
    first = pos[pos_off[:-1].astype(np.int64)]
    return (first[:, 1].astype(np.uint64) << np.uint64(32)) | first[:, 0].astype(np.uint64)


def assert_same_part(a: api.Aligner, sa: int, b: api.Aligner, sb: int, what: str):
    la, lb = a.index_array(sa, "flookup"), b.index_array(sb, "flookup")
    assert np.array_equal(la[:, 1], lb[:, 1]) and np.array_equal(la[:, 3], lb[:, 3]), what + ": list lengths"
    for off, cnt in ((0, 1), (2, 3)):
        m = la[:, cnt] > 0
        assert np.array_equal(la[m, off], lb[m, off]), what + ": list offsets"
    fa, fb = a.index_array(sa, "flist"), b.index_array(sb, "flist")
    assert fa.shape == fb.shape, what
    assert np.array_equal(fa[:, 0], fb[:, 0]), what + ": entry texts / order"
    poa, pob = a.index_array(sa, "pos_off"), b.index_array(sb, "pos_off")
    pa, pb = a.index_array(sa, "pos"), b.index_array(sb, "pos")
    assert poa.shape == pob.shape and pa.shape == pb.shape, what + ": ids / positions"
    ca, cb = canon_ids(poa, pa), canon_ids(pob, pb)
    assert np.array_equal(ca[fa[:, 1]], cb[fb[:, 1]]), what + ": entry ids"
    oa, ob = np.argsort(ca), np.argsort(cb)
    assert np.array_equal(ca[oa], cb[ob]), what + ": L-mers"
    na, nb = np.diff(poa.astype(np.int64)), np.diff(pob.astype(np.int64))
    assert np.array_equal(na[oa], nb[ob]), what + ": position counts"

    def gathered(po, p, order, cnt):
        starts = po[:-1].astype(np.int64)[order]
        idx = np.repeat(starts - np.concatenate(([0], np.cumsum(cnt[order])[:-1])), cnt[order]) + np.arange(int(cnt.sum()))
        return p[idx]
    assert np.array_equal(gathered(poa, pa, oa, na), gathered(pob, pb, ob, nb)), what + ": position lists"
    assert np.array_equal(a.index_array(sa, "ref_off"), b.index_array(sb, "ref_off")), what + ": reference offsets"
    ra, rb = a.index_array(sa, "refseq"), b.index_array(sb, "refseq")
    n = int(a.index_array(sa, "ref_off")[-1])
    assert np.array_equal(ra[:n], rb[:n]), what + ": reference sequences"


def test_device_index_equals_reference_built_files(golden):
    exp = load_case("default")
    files, dev = api.Aligner(0), api.Aligner(0)
    for al in (files, dev):
        al.set_params(api.default_params())
    names = ("db_arc.fasta", "db_bac.fasta")
    for k in range(2):
        files.load_index_part(k, 0, golden["prefixes"][k], golden["refs"][k], exp["log"]["minimal_score"][k], (18, 9, 3), golden["stats"][k].lnwin)
        assert dev.build_index_device(k, os.path.join(GOLDEN, names[k]), golden["refs"][k], exp["log"]["minimal_score"][k]) == 1
        assert_same_part(files, k, dev, k, names[k])
    b = golden["batch"]
    want, got = files.align(b.cat, b.off), dev.align(b.cat, b.off)
    assert_same_results(got, want, "device-built vs file-loaded index")
    rows = hostio.format_sam_rows(b, golden["refs"], got["res"], got["alns"], got["cigar"], got["slots"])
    assert sorted(rows) == sorted(exp["sam"])          # what the reference binary printed
    assert got["counters"]["num_aligned"] == exp["log"]["passing"]
    files.close(); dev.close()


@pytest.mark.parametrize("name,kw", [("max_pos3", dict(max_pos=3)), ("max_pos0", dict(max_pos=0)), ("interval2", dict(interval=2)),
                                     ("parts", dict(max_mb=0.5)), ("L16", dict(lnwin=16)), ("L20", dict(lnwin=20))])
def test_device_index_equals_host_builder_with_options(golden, name, kw):
    with tempfile.TemporaryDirectory(prefix="smr_devidx_") as d:
        files, dev = api.Aligner(0), api.Aligner(0)
        lnwin = kw.get("lnwin", 18)
        skip = (lnwin, lnwin // 2, 3)
        slot = 0
        part_refs = []
        for k, fn in enumerate(("db_arc.fasta", "db_bac.fasta")):
            fasta, prefix = os.path.join(GOLDEN, fn), os.path.join(d, fn)
            api.build_index(fasta, prefix, **kw)
            st = hostio.parse_stats(prefix)
            prs = hostio.split_by_parts(golden["refs"][k], st)
            part_refs.append(prs)
            for p in range(st.num_parts):
                files.load_index_part(k, p, prefix, prs[p], 60, skip, lnwin)
            assert dev.build_index_device(k, fasta, prs, 60, skip, **kw) == st.num_parts
            for p in range(st.num_parts):
                assert_same_part(files, slot, dev, slot, f"{name} {fn} part {p}")
                slot += 1
        if name == "parts":
            assert slot == 6
        for al in (files, dev):
            al.set_params(api.default_params())
        b = golden["batch"]
        want, got = files.align(b.cat, b.off), dev.align(b.cat, b.off)
        assert_same_results(got, want, name)
        assert int(want["res"]["is_hit"].sum()) > 100
        files.close(); dev.close()


def test_device_index_bundled_database_and_time():
    """A database of the size of silva-arc-16s-id95 (tools/synth_db.py's stand-in: 3193 sequences of ~1.1 kb)."""
    import time
    from tools import synth_db
    with tempfile.TemporaryDirectory(prefix="smr_devidx_") as d:
        fasta = synth_db.write_databases(d, only=["silva-arc-16s-id95"])[0]
        prefix = os.path.join(d, "arc16s")
        t0 = time.time(); api.build_index(fasta, prefix); t_host = time.time() - t0
        refs = hostio.load_references(fasta)
        files, dev = api.Aligner(0), api.Aligner(0)
        t0 = time.time(); files.load_index_part(0, 0, prefix, refs, 60); t_load = time.time() - t0
        dev.build_index_device(0, fasta, refs, 60)       # first call pays the CUDA module load
        dev2 = api.Aligner(0)
        t0 = time.time(); dev2.build_index_device(0, fasta, refs, 60); t_dev = time.time() - t0
        assert_same_part(files, 0, dev2, 0, "silva-arc-16s-id95")
        print(f"silva-arc-16s-id95: host builder {t_host:.2f} s + load/flatten {t_load:.2f} s; device build (FASTA -> resident) {t_dev:.2f} s; {dev2.last_build_report}")
        for al in (files, dev, dev2):
            al.close()
