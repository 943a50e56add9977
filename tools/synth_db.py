"""Synthetic stand-ins for the 8 rRNA databases the reference ships with (data/rRNA_databases), made from a seed in a few
seconds: same number of sequences and the same mean length per database, lower-case ACGT like the SILVA / Rfam files.
Sequences share conserved regions and come in families, clades and members with ragged ends, so that reads cut from them
hit many similar references, as they do in the real databases.  The benchmark aligns against these when no directory of
real database files is given."""
import os

import numpy as np

# (file name as the reference names it, sequences, mean length) of the databases of the reference's data/rRNA_databases
DBS = [("silva-bac-16s-id90", 12798, 1417), ("silva-bac-23s-id98", 4488, 2775), ("silva-arc-16s-id95", 3193, 1117),
       ("silva-arc-23s-id98", 251, 2894), ("silva-euk-18s-id95", 7348, 1702), ("silva-euk-28s-id98", 4935, 2926),
       ("rfam-5s-database-id98", 59513, 116), ("rfam-5.8s-database-id98", 13034, 153)]
SEED = 20261017
# one ancestor per database; families, clades of a family and members of a clade drift from it by substitutions at
# P_FAMILY / P_CLADE / P_MEMBER times the rate of the region (regions of ~SEGMENT nt, rates gamma-distributed with shape
# RATE_SHAPE, mean 1), members also by short indels.  Chosen so that the benchmark's reads meet about as many candidate
# references as in the real databases: per read ~44 Smith-Waterman calls and ~2300 position-list entries, against 43.6 and
# 2304 there (the oracle's counters on 2000 reads of the workload).
MEMBERS_PER_CLADE = 8
CLADES_PER_FAMILY = 5
RATE_SHAPE = 0.55
SEGMENT = 40
P_FAMILY, P_CLADE, P_MEMBER = 0.20, 0.08, 0.03


def _substitute(rng, s, p):
    s = s.copy()
    m = rng.random(s.size) < p
    s[m] = (s[m] + rng.integers(1, 4, int(m.sum()), dtype=np.uint8)) & 3
    return s


def _indels(rng, s, p):
    k = rng.random(s.size) < p
    if not k.any():
        return s
    pos = np.flatnonzero(k)
    ins = rng.random(pos.size) < 0.5
    keep = np.delete(np.arange(s.size), pos[~ins])
    return np.insert(s[keep], np.searchsorted(keep, pos[ins]), rng.integers(0, 4, int(ins.sum()), dtype=np.uint8))


def make_database(rng, nseq, mean_len):
    """-> list of uint8 arrays over 0..3"""
    L = int(mean_len * 1.04)
    ancestor = rng.integers(0, 4, L, dtype=np.uint8)
    seg = np.cumsum(rng.geometric(1.0 / SEGMENT, L))   # regions of ~SEGMENT nt, each conserved or variable as a whole
    seg_rate = np.minimum(rng.gamma(RATE_SHAPE, 1.0 / RATE_SHAPE, L), 1.0 / P_FAMILY)
    rate = seg_rate[np.searchsorted(seg, np.arange(L), side="right")]
    out = []
    while len(out) < nseq:
        founder = _substitute(rng, ancestor, P_FAMILY * rate)
        for _ in range(CLADES_PER_FAMILY):
            clade = _substitute(rng, founder, P_CLADE * rate)
            for _ in range(MEMBERS_PER_CLADE):
                m = _indels(rng, _substitute(rng, clade, P_MEMBER * rate), 0.002)
                a, b = rng.integers(0, max(1, mean_len // 25), 2)
                out.append(m[a:m.size - b])
                if len(out) == nseq:
                    return out
    return out


def write_databases(out_dir, seed=SEED, only=None):
    """Writes <out_dir>/<name>.fasta for the 8 databases (or those named in `only`) unless it is already there; returns their
    paths in the benchmark's --ref order."""
    os.makedirs(out_dir, exist_ok=True)
    lut = np.frombuffer(b"acgt", np.uint8)
    paths = []
    for k, (name, nseq, mean_len) in enumerate(DBS):
        if only is not None and name not in only:
            continue
        rng = np.random.default_rng([seed, k])
        p = os.path.join(out_dir, name + ".fasta")
        paths.append(p)
        if os.path.exists(p):
            continue
        with open(p + ".part", "wb") as f:
            for i, s in enumerate(make_database(rng, nseq, mean_len)):
                f.write(b">%s.%06d synthetic\n" % (name.encode(), i))
                f.write(lut[s].tobytes() + b"\n")
        os.replace(p + ".part", p)
    return paths
