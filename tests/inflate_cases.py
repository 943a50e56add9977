"""gzip inputs shared by tests/test_inflate_host.py (the decode logic on the CPU) and tests/test_gpu_inflate.py (the kernels):
real gzip output at several levels, stored / fixed-Huffman streams, flush points, several members, header fields, long
back-references, plus corrupt and truncated files."""
import gzip
import io
import os
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def fastq_text(n: int, seed: int = 1) -> bytes:
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        ln = int(rng.integers(50, 152))
        seq = "".join(rng.choice(list("ACGT"), ln))
        if rng.random() < 0.2:
            k = int(rng.integers(0, ln))
            seq = seq[:k] + "N" + seq[k + 1:]
        qual = "".join(chr(c) for c in rng.integers(35, 74, ln))
        out.append(f"@read{i}/1 sample\n{seq}\n+\n{qual}\n")
    return "".join(out).encode()


def cases(n_reads: int = 6000):
    """-> list of (name, gz bytes, expected inflated bytes)"""
    txt = fastq_text(n_reads)
    out = []
    for lvl in (0, 1, 6, 9):
        out.append((f"level{lvl}", gzip.compress(txt, compresslevel=lvl), txt))
    third = len(txt) // 3
    multi = gzip.compress(b"@r\nACGT\n+\nIIII\n") + gzip.compress(txt[:third], 6) + gzip.compress(b"") + gzip.compress(txt[third:], 9)
    out.append(("multi_member", multi, b"@r\nACGT\n+\nIIII\n" + txt))
    out.append(("empty", gzip.compress(b""), b""))
    co = zlib.compressobj(6, zlib.DEFLATED, 31, 9, zlib.Z_FIXED)
    out.append(("fixed_huffman", co.compress(txt[:200000]) + co.flush(), txt[:200000]))
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    b = b""
    for i in range(0, 400000, 50000):
        b += co.compress(txt[i:i + 50000]) + co.flush(zlib.Z_SYNC_FLUSH if i % 100000 else zlib.Z_FULL_FLUSH)
    b += co.flush()
    out.append(("flush_points", b, txt[:400000]))
    rep = (b"ACGTACGTTTGACCA" * 7000 + txt[:5000]) * 5
    out.append(("long_matches", gzip.compress(rep, 9), rep))
    bio = io.BytesIO()
    with gzip.GzipFile(filename="reads_file.fq", mode="wb", fileobj=bio, mtime=123) as g:
        g.write(txt[:70000])
    out.append(("header_fname", bio.getvalue(), txt[:70000]))
    sampled = rrna_fastq_text(12000)
    out.append(("rrna_reads", gzip.compress(sampled, 6), sampled))
    raw = open(SET4_HEAD, "rb").read()
    out.append(("set4_head", raw, gzip.decompress(raw)))
    return out


SET4_HEAD = os.path.join(ROOT, "tests", "golden", "sets", "set4_mate_pairs_metatranscriptomics_1.head500.fastq.gz")


def rrna_fastq_text(n: int, seed: int = 11) -> bytes:
    """Reads of 100 nt cut from the golden rRNA slices with 1 % substitutions, Illumina-like headers and qualities: text that
    compresses like a real read file (long deflate streams of many blocks), made in memory."""
    rng = np.random.default_rng(seed)
    seqs = []
    for g in ("db_arc.fasta", "db_bac.fasta"):
        with open(os.path.join(ROOT, "tests", "golden", g), "rb") as f:
            seqs += [b"".join(rec.split(b"\n")[1:]) for rec in f.read().split(b">")[1:]]
    out = []
    for i in range(n):
        s = seqs[int(rng.integers(0, len(seqs)))]
        b = int(rng.integers(0, len(s) - 100))
        r = bytearray(s[b:b + 100])
        for k in np.flatnonzero(rng.random(100) < 0.01):
            r[k] = b"ACGT"[int(rng.integers(0, 4))]
        q = bytes((rng.integers(28, 41, 100) + 33 - (np.arange(100) > 80) * rng.integers(0, 20, 100)).astype(np.uint8))
        out.append(b"@sample.%09d/1 length=100 begin=%d\n%s\n+\n%s\n" % (i, b, bytes(r), q))
    return b"".join(out)


def bad_cases():
    txt = fastq_text(1500, seed=3)
    good = gzip.compress(txt, 6)
    flipped = bytearray(good)
    flipped[len(good) // 2] ^= 0x55
    return [("bit_flip", bytes(flipped)), ("truncated", good[:-2000]), ("not_gzip", b"@r\nACGT\n+\nIIII\n" * 4), ("wrong_isize", good[:-4] + b"\x01\x02\x03\x04")]
