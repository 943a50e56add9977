"""Input decode on the device (smr_upload_fastx, SURVEY 8(f)(2)) against the host reader (hostio.read_fastx + encode_nt):
same records, same 0-4 codes, same header positions -- and the alignment results of the decoded batch equal those of the
host-parsed batch."""
import gzip
import os

import numpy as np
import pytest

from conftest import GOLDEN, load_case
from helpers import assert_same_results
from sortmerna_b200 import api, hostio

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def aligner(golden):
    al = api.Aligner(0)
    al.set_params(api.default_params())
    exp = load_case("default")
    for k in range(2):
        al.load_index_part(k, 0, golden["prefixes"][k], golden["refs"][k], exp["log"]["minimal_score"][k], (18, 9, 3), golden["stats"][k].lnwin)
    yield al
    al.close()


def check_text(al, text: bytes, path_for_host_reader: str):
    h, s, _ = hostio.read_fastx(path_for_host_reader)
    want = hostio.pack_reads(h, s)
    n = al.upload_fastx(text)
    assert n == want.n
    hdr, off, seq = al.resident_layout()
    assert np.array_equal(off, want.off)
    assert np.array_equal(seq, want.cat)
    for r in (0, n // 2, n - 1):
        o = int(hdr[r])
        line = text[o:text.index(b"\n", o) if b"\n" in text[o:] else len(text)].rstrip(b"\r")
        assert line.decode() == h[r]
    return want


def test_decode_golden_fastq(aligner):
    p = os.path.join(GOLDEN, "reads_mix.fq")
    check_text(aligner, open(p, "rb").read(), p)


def test_decode_fasta_variants(aligner, tmp_path):
    rng = np.random.default_rng(7)
    recs = []
    for i in range(300):
        ln = int(rng.integers(1, 400))
        recs.append((f">r{i} some description {i}", "".join(rng.choice(list("ACGTNacgtnURYKMSWBDHVX-"), ln))))
    variants = {
        "single_line": "".join(f"{h}\n{s}\n" for h, s in recs),
        "wrapped_60": "".join(h + "\n" + "\n".join(s[k:k + 60] for k in range(0, len(s), 60)) + "\n" for h, s in recs),
        "crlf_no_final_newline": "".join(h + "\r\n" + "\r\n".join(s[k:k + 70] for k in range(0, len(s), 70)) + "\r\n" for h, s in recs).rstrip("\r\n"),
        "trailing_blank_lines": "".join(f"{h}\n{s}\n" for h, s in recs) + "\n\n",
    }
    for name, text in variants.items():
        # the host reader wants single-line records: write the canonical form for it, feed the variant to the device
        canon = tmp_path / f"{name}.fa"
        canon.write_text("".join(f"{h}\n{s}\n" for h, s in recs))
        n = aligner.upload_fastx(text.encode())
        want = hostio.pack_reads(*hostio.read_fastx(str(canon))[:2])
        hdr, off, seq = aligner.resident_layout()
        assert n == want.n, name
        assert np.array_equal(off, want.off), name
        assert np.array_equal(seq, want.cat), name
        assert text.encode()[int(hdr[17]):].startswith(recs[17][0].encode()), name


def test_decode_fastq_edge_cases(aligner):
    text = b"@a desc\nACGTN\n+\nIIIII\n@b\nacgu\n+b\nIIII"          # lower case, U, repeated id on '+', no final newline
    n = aligner.upload_fastx(text)
    hdr, off, seq = aligner.resident_layout()
    assert n == 2 and off.tolist() == [0, 5, 9] and seq.tolist() == [0, 1, 2, 3, 4, 0, 1, 2, 3] and hdr.tolist() == [0, text.index(b"@b")]
    with pytest.raises(api.SmrError):
        aligner.upload_fastx(b"@a\nACGT\nIIII\n@b\n")          # separator line missing
    with pytest.raises(api.SmrError):
        aligner.upload_fastx(b"ACGT\n")
    assert aligner.upload_fastx(b"") == 0


def test_alignment_of_decoded_batch_equals_host_parsed(aligner, golden):
    b = golden["batch"]
    want = aligner.align(b.cat, b.off)
    n = aligner.upload_fastx(open(os.path.join(GOLDEN, "reads_mix.fq"), "rb").read())
    assert n == b.n
    aligner.run_resident()
    got = aligner.download()
    assert_same_results(got, want, "decoded vs host-parsed")
    assert got["counters"]["num_aligned"] == want["counters"]["num_aligned"]


def test_decode_bundled_set2_and_throughput(aligner, tmp_path):
    # the first 500 records of the bundled set2 amplicon study
    text = gzip.decompress(open(os.path.join(GOLDEN, "sets", "set2_environmental_study_550_amplicon.head500.fasta.gz"), "rb").read())
    p = tmp_path / "set2_head.fasta"
    p.write_bytes(text)
    want = check_text(aligner, text, str(p))
    assert want.n == 500
    # decode rate of a large text (the set repeated to ~0.5 GB), kernels only
    big = text * max(1, (1 << 29) // len(text))
    aligner.upload_fastx(big)      # first call sizes the device buffers
    aligner.upload_fastx(big)
    t = aligner.timings()
    print(f"decode {len(big) / 1e9:.2f} GB text: H2D {t['h2d_ms']:.1f} ms, kernels {t['decode_ms']:.1f} ms = {len(big) / t['decode_ms'] / 1e6:.0f} GB/s")
