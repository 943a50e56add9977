"""gzip inflate on the device (smr_upload_fastx_gz / smr_debug_inflate, SURVEY 8(f)(2): the gz half of the read feed,
src/sortmerna/readfeed.cpp:683-770) against zlib, and the decoded batch against the host-parsed one."""
import gzip
import os

import numpy as np
import pytest

import inflate_cases
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


def test_inflate_equals_zlib(aligner):
    most = 0
    for name, gz, want in inflate_cases.cases(6000):
        for chunk in (65536, 4096):
            got, info = aligner.debug_inflate(gz, chunk)
            assert got == want, (name, chunk, info)
            most = max(most, info["spans"])
    assert most > 20


def test_bad_input_is_refused(aligner):
    for name, gz in inflate_cases.bad_cases():
        with pytest.raises(api.SmrError):
            aligner.debug_inflate(gz, 4096)
    with pytest.raises(api.SmrError):
        aligner.upload_fastx_gz(b"\x1f\x8b")


def test_alignment_of_gz_batch_equals_host_parsed(aligner, golden):
    b = golden["batch"]
    want = aligner.align(b.cat, b.off)
    text = open(os.path.join(GOLDEN, "reads_mix.fq"), "rb").read()
    n = aligner.upload_fastx_gz(gzip.compress(text, 6))
    assert n == b.n
    assert aligner.resident_text() == text
    hdr, off, seq = aligner.resident_layout()
    assert np.array_equal(off, b.off) and np.array_equal(seq, b.cat)
    aligner.run_resident()
    got = aligner.download()
    assert_same_results(got, want, "gz-decoded vs host-parsed")


def test_bundled_gz_mates_and_throughput(aligner, tmp_path):
    raw = open(inflate_cases.SET4_HEAD, "rb").read()      # the first 500 records of the bundled set4 mate 1, gzip -9
    n = aligner.upload_fastx_gz(raw)
    p = tmp_path / "set4_head.fastq"
    p.write_bytes(gzip.decompress(raw))
    h, s, _ = hostio.read_fastx(str(p))
    want = hostio.pack_reads(h, s)
    assert n == want.n == 500
    _, off, seq = aligner.resident_layout()
    assert np.array_equal(off, want.off) and np.array_equal(seq, want.cat)
    # rate on a large file: ~100 MB of FASTQ text, gzip -6 (one member, a few thousand spans)
    txt = inflate_cases.fastq_text(40000, seed=5) * 8
    gz = gzip.compress(txt, 6)
    aligner.debug_inflate(gz, 0)      # first call sizes the buffers
    got, info = aligner.debug_inflate(gz, 0)
    assert got == txt
    print(f"inflate {len(gz) / 1e6:.1f} MB gz -> {len(txt) / 1e6:.1f} MB: {info['spans']} spans, device {info['device_us'] / 1e3:.1f} ms "
          f"= {len(txt) / max(1, info['device_us']) / 1e3:.2f} GB/s out, H2D {info['h2d_us'] / 1e3:.1f} ms")
