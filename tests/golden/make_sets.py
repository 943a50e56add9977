#!/usr/bin/env python
"""Regenerates tests/golden/sets/ from the reference's bundled data (needs oracle/_ref/sortmerna_ref):

  set2_...head500.fasta.gz, set4_..._1.head500.fastq.gz       the first 500 records of the set2 amplicon reads and of set4
                                                              mate 1 (decode and inflate tests)
  set2_...head100.fasta.gz, set4_..._{1,2}.head100.fastq.gz   the first 100 records of the set2 reads and of both set4 mates
                                                              (parity samples of BASELINE configs 2 and 4, test.jinja t5)
  <database>.hits.fasta.gz                                    the sequences of each database that the reference aligns the
                                                              parity samples to (best alignment per read), plus its first
                                                              FIRST sequences, in database order: the 8 rRNA databases for
                                                              set4, silva-bac-16s-database-id85 for set2 and set4
                                                              (-max_pos 250)

  python tests/golden/make_sets.py <the reference's data directory>
"""
import gzip
import os
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
OUT = os.path.join(HERE, "sets")
HEAD = 500
SAMPLE = 100
FIRST = 3
SET2 = "set2_environmental_study_550_amplicon"
SET4 = "set4_mate_pairs_metatranscriptomics"
ID85 = "silva-bac-16s-database-id85"


def head_path(name, ext, n=HEAD):
    return os.path.join(OUT, f"{name}.head{n}.{ext}.gz")


def hits_path(db):
    return os.path.join(OUT, f"{db}.hits.fasta.gz")


def write_gz(path, data):
    with open(path, "wb") as f, gzip.GzipFile(filename=os.path.basename(path)[:-3], mode="wb", fileobj=f, mtime=0, compresslevel=9) as g:
        g.write(data)


def head(path, lines):
    with open(path, "rb") as f:
        return b"".join(f.readline() for _ in range(lines))


def hit_names(fastas, reads, workdir, extra, idx_dir):
    from oracle import ora
    from tools import stage_data
    idx, _ = stage_data.ensure_indexes(fastas, idx_dir, extra=tuple(extra), builder="reference")
    r = ora.run_reference(fastas, reads, workdir, extra=["-sam"] + list(extra), threads=os.cpu_count() or 8, idx_dir=idx)
    return {row.split("\t")[2] for row in ora.read_sam_rows(os.path.join(r["out_dir"], "aligned.sam"))}


def write_slice(fasta, names, dst):
    out, keep, seen = [], False, 0
    with open(fasta, "rb") as f:
        for ln in f:
            if ln.startswith(b">"):
                keep = ln[1:].split()[0].decode() in names or seen < FIRST
                seen += 1
            if keep:
                out.append(ln)
    write_gz(dst, b"".join(out))


def main(data):
    os.makedirs(OUT, exist_ok=True)
    write_gz(head_path(SET2, "fasta"), head(os.path.join(data, SET2 + ".fasta"), 2 * HEAD))
    write_gz(head_path(f"{SET4}_1", "fastq"), head(os.path.join(data, f"{SET4}_1.fastq"), 4 * HEAD))
    write_gz(head_path(SET2, "fasta", SAMPLE), head(os.path.join(data, SET2 + ".fasta"), 2 * SAMPLE))
    for k in (1, 2):
        write_gz(head_path(f"{SET4}_{k}", "fastq", SAMPLE), head(os.path.join(data, f"{SET4}_{k}.fastq"), 4 * SAMPLE))
    from tools import stage_data
    with tempfile.TemporaryDirectory(prefix="smr_sets_") as d:
        reads = {}
        for name, ext in ((SET2, "fasta"), (f"{SET4}_1", "fastq"), (f"{SET4}_2", "fastq")):
            reads[name] = os.path.join(d, f"{name}.{ext}")
            with open(reads[name], "wb") as f:
                f.write(gzip.decompress(open(head_path(name, ext, SAMPLE), "rb").read()))
        set4 = [reads[f"{SET4}_1"], reads[f"{SET4}_2"]]
        dbs = [os.path.join(data, "rRNA_databases", n + ".fasta") for n in stage_data.DBS]
        names = hit_names(dbs, set4, os.path.join(d, "set4"), [], os.path.join(d, "idx8"))
        for n, f in zip(stage_data.DBS, dbs):
            write_slice(f, names, hits_path(n))
        id85 = os.path.join(data, ID85 + ".fasta")
        names = set()
        for k, r in enumerate(([reads[SET2]], set4)):      # one read set per run: set2 is FASTA, set4 FASTQ
            names |= hit_names([id85], r, os.path.join(d, f"id85_{k}"), ["-max_pos", "250"], os.path.join(d, "idx85"))
        write_slice(id85, names, hits_path(ID85))
    for fn in sorted(os.listdir(OUT)):
        print(fn, os.path.getsize(os.path.join(OUT, fn)))


if __name__ == "__main__":
    main(sys.argv[1])
