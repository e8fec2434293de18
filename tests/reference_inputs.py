"""Inputs of the tests that compare with the reference's results stored under
tests/golden/reference_golden.* (written by tests/golden/make_reference_golden.py
from the reference's own sources). The tests and the generator both build their
inputs here, so a stored result always belongs to the input a test feeds."""
import numpy as np

from raven_b200 import seqio, synth

COMPLEXITY_K = (15, 19, 9, 4)
REGION_COVERAGES = (4, 1, 9, 30)


def synthetic_reads():
    return synth.make_reads(40_000, 150, 3000, seed=11)


def region_reads():
    """A deeper synthetic set for the pile regions of stage-1 piles."""
    return synth.make_reads(40_000, 300, 5000, seed=14)


def add_layers_overlaps():
    """(read id, read length, overlaps) of read 7 on both sides of the records."""
    rng = np.random.default_rng(3)
    length = 5000
    ovl = []
    for _ in range(300):
        b = int(rng.integers(0, length - 200))
        e = int(rng.integers(b + 100, min(length, b + 3000) + 1))
        side = rng.random() < 0.5
        rec = [7, b, e, 9, 16, 200, 100, 1] if side else [9, 16, 200, 7, b, e, 100, 0]
        ovl.append(rec)
    return 7, length, np.array(ovl, dtype=np.uint32)


def lowcomplexity_reads():
    rng = np.random.default_rng(17)
    seqs = [rng.integers(0, 4, 400, dtype=np.uint8)]
    seqs.append(np.repeat(rng.integers(0, 4, 60, dtype=np.uint8), rng.integers(1, 9, 60)))  # homopolymer runs
    seqs.append(np.tile(np.array([0, 1], np.uint8), 150))            # (AC)n
    seqs.append(np.tile(np.array([0, 1, 1, 0], np.uint8), 80))       # ACCA..
    seqs.append(np.tile(np.array([2, 0, 1], np.uint8), 100))         # (GAC)n
    seqs.append(np.concatenate([np.tile(np.array([3, 2], np.uint8), 40),
                                rng.integers(0, 4, 100, dtype=np.uint8)]))
    seqs.append(rng.integers(0, 4, 20, dtype=np.uint8))              # shorter than k near the end
    return seqio.pack_codes(seqs)


def lowcomplexity_positions():
    """The low-complexity reads and every third position of each."""
    rs = lowcomplexity_reads()
    idx, pos = [], []
    for r in range(rs.n):
        for p in range(0, int(rs.lens[r]), 3):
            idx.append(r); pos.append(p)
    return rs, idx, pos


def trim_rule_piles():
    """300 coverage histograms of five kinds; the list and the concatenation offsets."""
    rng = np.random.default_rng(1)
    piles, off = [], [0]
    for t in range(300):
        nb = int(rng.integers(1, 400))
        kind = t % 5
        if kind == 0:
            d = rng.integers(0, 10, nb)
        elif kind == 1:
            d = np.full(nb, 7)
        elif kind == 2:
            d = rng.integers(3, 40, nb)
            d[rng.integers(0, nb, max(1, nb // 50))] = 0
        elif kind == 3:
            d = rng.integers(4, 9, nb)
            if nb > 3:
                d[-1] = 0
                d[nb // 2] = 1
        else:
            d = rng.integers(0, 70000, nb).clip(0, 65535)
        piles.append(d.astype(np.uint16))
        off.append(off[-1] + nb)
    return piles, np.array(off, np.uint64)
