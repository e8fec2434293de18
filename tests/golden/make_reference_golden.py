"""Regenerate tests/golden/reference_golden.npz + reference_golden.json.

What the reference's own sources, compiled in place (oracle/_ref, built by
oracle/Makefile where the reference tree is present), return for the inputs
the comparison tests use: the stage-1 results of the lambda fixture and of a
synthetic set, AddLayers piles, the k-mer complexity rule, the pile trimming
rule on stored and on stage-1 piles, and the RavenTest.Assemble unitig before
and after polishing.  The tests compare the port and the device kernels
against these, so they run without the reference tree.  Large results are kept
as SHA-256 digests (the comparisons are exact), small ones as arrays.

    python tests/golden/make_reference_golden.py
"""
import hashlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_lib  # noqa: E402
import reference_inputs as inputs  # noqa: E402
from raven_b200 import seqio  # noqa: E402


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


if not oracle_lib.Reference.available():
    raise SystemExit("oracle/_ref/libraven_ref.so is missing: build it with `make -C oracle`")
R = oracle_lib.Reference()
O = oracle_lib.Oracle()
lam = seqio.ReadSet.load(os.path.join(HERE, "lambda_reads.npz"))
meta, arrays = {}, {}

for mh in (False, True):
    st = R.stage1(R.reads(lam), 15, 5, 0.001, 32, mh, 4)
    tag = "minhash" if mh else "plain"
    for k in ("overlaps", "ovl_off", "pile", "pile_off", "occurrences"):
        meta[f"stage1_{tag}_{k}_sha256"] = sha(st[k])

rs = inputs.synthetic_reads()
for kmax in (4, 32):
    st = R.stage1(R.reads(rs), 15, 5, 0.001, kmax, False, 4)
    for k in ("overlaps", "ovl_off", "pile", "pile_off"):
        meta[f"synthetic_kmax{kmax}_{k}_sha256"] = sha(st[k])

read_id, length, ovl = inputs.add_layers_overlaps()
arrays["add_layers_rounds2"] = R.pile_add_layers(read_id, length, ovl, rounds=2)
arrays["add_layers_rounds700"] = R.pile_add_layers(read_id, length, ovl, rounds=700)

rs, idx, pos = inputs.lowcomplexity_positions()
for k in inputs.COMPLEXITY_K:
    arrays[f"kmer_complexity_k{k}"] = R.kmer_complexity(R.reads(rs), idx, pos, k)

piles, off = inputs.trim_rule_piles()
got = oracle_lib.ref_pile_trim(R, np.concatenate(piles), off, 4)
for k in ("begin", "end", "median", "invalid", "data"):
    arrays[f"trim_rule_{k}"] = got[k]

# pile regions of the stage-1 piles (the device kernel's input); the piles
# themselves are the stage-1 result, checked against the reference above
for name, reads in (("lambda", lam), ("synthetic", inputs.region_reads())):
    st = R.stage1(R.reads(reads), 15, 5, 0.001, 32, False, 4)
    meta[f"regions_{name}_pile_sha256"] = sha(st["pile"])
    for cov in inputs.REGION_COVERAGES:
        got = oracle_lib.ref_pile_trim(R, st["pile"], st["pile_off"], cov)
        for k in ("begin", "end", "median", "invalid"):
            arrays[f"regions_{name}_cov{cov}_{k}"] = got[k]

# RavenTest.Assemble (raven_test.cpp:50-67): the unitig after layout and after the
# two polishing rounds of the test's configuration
for rounds in (0, 2):
    names, seqs = oracle_lib.ref_assemble(R, lam, True, rounds, 8)
    meta[f"assemble_rounds{rounds}_names"] = names
    for i, s in enumerate(seqs):
        arrays[f"assemble_rounds{rounds}_unitig{i}"] = np.frombuffer(s, np.uint8)

np.savez_compressed(os.path.join(HERE, "reference_golden.npz"), **arrays)
with open(os.path.join(HERE, "reference_golden.json"), "w") as f:
    json.dump(meta, f, indent=1, sort_keys=True)
print(json.dumps(meta, indent=1, sort_keys=True))
