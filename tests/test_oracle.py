"""CPU tests: the oracle against the committed golden vectors, against what the
reference's own sources return (stored by tests/golden/make_reference_golden.py),
and against independent numpy restatements of the small pieces."""
import hashlib
import json
import os

import numpy as np
import pytest

import reference_inputs as inputs
from raven_b200 import seqio, synth

HERE = os.path.dirname(os.path.abspath(__file__))
META = json.load(open(os.path.join(HERE, "golden", "lambda_golden.json")))
GOLD = np.load(os.path.join(HERE, "golden", "lambda_golden.npz"))
REF_META = json.load(open(os.path.join(HERE, "golden", "reference_golden.json")))
REF_GOLD = np.load(os.path.join(HERE, "golden", "reference_golden.npz"))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_fixture_is_the_reference_fixture(lambda_reads):
    # RavenTest/data/ERA476754.fastq.gz: 236 reads, 1,674,628 bases (SURVEY §4)
    assert lambda_reads.n == 236
    assert lambda_reads.bases == 1674628
    assert int(lambda_reads.lens.min()) == 443 and int(lambda_reads.lens.max()) == 11968


@pytest.mark.parametrize("minhash", [False, True])
def test_sketch_golden(oracle, lambda_reads, minhash):
    eng = oracle.engine(15, 5)
    sk = oracle.sketch(eng, oracle.reads(lambda_reads), 0, lambda_reads.n, minhash)
    tag = "micro" if minhash else "full"
    assert sk["value"].size == META[f"sketch_{tag}_n"]
    assert sha(sk["value"]) == META[f"sketch_{tag}_value_sha256"]
    assert sha(sk["origin"]) == META[f"sketch_{tag}_origin_sha256"]
    assert sha(sk["offsets"]) == META[f"sketch_{tag}_offsets_sha256"]


def test_survey_anchors(oracle, lambda_reads):
    """Counts measured independently by the survey (SURVEY.md App. C)."""
    eng = oracle.engine(15, 5, threads=4)
    reads = oracle.reads(lambda_reads)
    oracle.minimize(eng, reads, 0, lambda_reads.n, False)
    keys = oracle.keys(eng)
    assert keys["totals"].tolist() == [467532, 568395]
    assert int((keys["counts"] == 1).sum()) == 436140
    assert int(keys["counts"].max()) == 25
    assert oracle.filter(eng, 0.001) == 15
    m = oracle.map(eng, reads, 0, lambda_reads.n, True, True, True, True)
    assert m["match_group"].size == 68597 and m["overlaps"].shape[0] == 2407
    assert sha(m["overlaps"]) == META["map_micro_overlaps_sha256"]
    m = oracle.map(eng, reads, 0, lambda_reads.n, True, True, False, True)
    assert m["match_group"].size == 326834 and m["overlaps"].shape[0] == 3890
    assert sha(m["overlaps"]) == META["map_full_overlaps_sha256"]
    assert sha(m["filtered"]) == META["map_full_filtered_sha256"]


def test_filter_rejects_bad_frequency(oracle, lambda_reads):
    eng = oracle.engine(15, 5)
    oracle.minimize(eng, oracle.reads(lambda_reads), 0, 10, False)
    for f in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            oracle.filter(eng, f)
    assert oracle.filter(eng, 0) == 0xFFFFFFFF


@pytest.mark.parametrize("minhash", [False, True])
def test_stage1_golden(oracle, lambda_reads, minhash):
    tag = "minhash" if minhash else "plain"
    st = oracle.stage1(oracle.engine(15, 5, threads=4), oracle.reads(lambda_reads),
                       0.001, 32, minhash)
    for k in ("overlaps", "ovl_off", "pile", "pile_off"):
        assert np.array_equal(st[k], GOLD[f"stage1_{tag}_{k}"]), k
    assert int(st["num_mapped"][0]) == META[f"stage1_{tag}_num_mapped"]


@pytest.mark.parametrize("minhash", [False, True])
def test_stage1_port_equals_compiled_reference(oracle, lambda_reads, minhash):
    """construct.cc / pile.cc / overlap_utils.cc compiled in place (their stored
    results) vs the port."""
    tag = "minhash" if minhash else "plain"
    a = oracle.stage1(oracle.engine(15, 5, threads=4), oracle.reads(lambda_reads),
                      0.001, 32, minhash)
    for k in ("overlaps", "ovl_off", "pile", "pile_off", "occurrences"):
        assert sha(a[k]) == REF_META[f"stage1_{tag}_{k}_sha256"], k


def test_stage1_port_equals_compiled_reference_synthetic(oracle):
    rs = inputs.synthetic_reads()
    for kmax in (4, 32):
        a = oracle.stage1(oracle.engine(15, 5, threads=4), oracle.reads(rs), 0.001,
                          kmax, False)
        for k in ("overlaps", "ovl_off", "pile", "pile_off"):
            assert sha(a[k]) == REF_META[f"synthetic_kmax{kmax}_{k}_sha256"], (kmax, k)


def test_add_layers_equals_reference_pile(oracle):
    read_id, length, ovl = inputs.add_layers_overlaps()
    want = REF_GOLD["add_layers_rounds2"]
    got = np.zeros(length >> 4, np.uint16)
    got = oracle.pile_add_layers(read_id, got, ovl)
    got = oracle.pile_add_layers(read_id, got, ovl)
    assert np.array_equal(got, want)
    # saturation at 65535
    want = REF_GOLD["add_layers_rounds700"]
    got = np.zeros(length >> 4, np.uint16)
    for _ in range(700):
        got = oracle.pile_add_layers(read_id, got, ovl)
    assert np.array_equal(got, want) and got.max() == 65535


def test_multi_batch_schedule_is_exercised(oracle):
    """Small thresholds drive >1 index batch and >1 flush; the result must
    differ from the single-batch run only through the documented schedule."""
    rs = synth.make_reads(30_000, 100, 3000, seed=5)
    eng = oracle.engine(15, 5, threads=4)
    one = oracle.stage1(eng, oracle.reads(rs), 0.001, 8, False)
    many = oracle.stage1(oracle.engine(15, 5, threads=4), oracle.reads(rs), 0.001, 8,
                         False, index_batch_bases=100_000, query_batch_bases=40_000)
    assert len(many["occurrences"]) > 1
    assert np.array_equal(one["pile_off"], many["pile_off"])
    assert (np.diff(many["ovl_off"].astype(np.int64)) <= 8).all()


def _numpy_minimizers(codes, k, w):
    """Independent restatement: hash every k-mer, then the window rule."""
    n = len(codes)
    if n < k:
        return []
    mask = (1 << (2 * k)) - 1

    def h(key):
        key = (~key + (key << 21)) & mask
        key ^= key >> 24
        key = (key + (key << 3) + (key << 8)) & mask
        key ^= key >> 14
        key = (key + (key << 2) + (key << 4)) & mask
        key ^= key >> 28
        key = (key + (key << 31)) & mask
        return key

    vals, strands = [], []
    for p in range(n - k + 1):
        fw = rv = 0
        for i in range(k):
            fw = (fw << 2) | int(codes[p + i])
            rv |= (3 - int(codes[p + i])) << (2 * i)
        if fw < rv:
            vals.append(h(fw)); strands.append(0)
        elif fw > rv:
            vals.append(h(rv)); strands.append(1)
        else:
            vals.append(None); strands.append(0)
    L = len(vals)
    out = set()
    for s in range(0, L - w + 1):
        win = [(vals[q], q) for q in range(s, s + w) if vals[q] is not None]
        if not win:
            continue
        m = min(v for v, _ in win)
        out.update(q for v, q in win if v == m)
    return [(vals[q], (q << 1) | strands[q]) for q in sorted(out)]


def test_sketch_matches_naive_definition(oracle):
    rng = np.random.default_rng(9)
    seqs = [rng.integers(0, 4, n, dtype=np.uint8) for n in (14, 15, 18, 19, 20, 64, 300)]
    seqs.append(np.zeros(100, np.uint8))                      # homopolymer
    seqs.append(np.tile(np.array([0, 3], np.uint8), 60))      # ATAT.. (palindromes)
    seqs.append(np.tile(np.array([0, 1, 2, 3], np.uint8), 40))
    rs = seqio.pack_codes(seqs)
    for k, w in ((15, 5), (5, 3), (4, 1), (19, 10)):
        eng = oracle.engine(k, w)
        sk = oracle.sketch(eng, oracle.reads(rs), 0, rs.n, False)
        for i, s in enumerate(seqs):
            a, b = int(sk["offsets"][i]), int(sk["offsets"][i + 1])
            want = _numpy_minimizers(s, k, w)
            got = list(zip(sk["value"][a:b].tolist(),
                           (sk["origin"][a:b] & 0xFFFFFFFF).tolist()))
            assert got == want, (k, w, i)
            assert ((sk["origin"][a:b] >> 32) == i).all()


def test_edit_distance_oracle(oracle):
    assert oracle.edit_distance(b"kitten", b"sitting") == 3
    assert oracle.edit_distance(b"", b"ACGT") == 4
    assert oracle.edit_distance(b"ACGT", b"ACGT") == 0


def test_kmer_complexity_port_equals_reference_pile(oracle):
    rs, idx, pos = inputs.lowcomplexity_positions()
    for k in inputs.COMPLEXITY_K:
        a = oracle.kmer_complexity(oracle.reads(rs), idx, pos, k)
        assert np.array_equal(a, REF_GOLD[f"kmer_complexity_k{k}"]), k
        assert 0 < a.sum() < a.size


def _revcomp(s: bytes) -> bytes:
    return s.translate(bytes.maketrans(b"ACGT", b"TGCA"))[::-1]


def test_end_to_end_pin_against_reference_golden(oracle, lambda_reads):
    """RavenTest.Assemble (RavenTest/src/raven_test.cpp:50-67), the reference's ONLY
    golden value: the reference's own construct/assemble/polish/common sources
    (compiled in place) over the oracle restatements of ram, racon, spoa and the
    edlib path. Upstream expects 1137 and the restatement reproduces it exactly;
    what decides the last edits is edlib's Hirschberg split of alignments whose
    traceback data would exceed 1 MiB (oracle/nw_path.cpp) - without it the six
    fixed traceback preferences give 1131..1166.
    The unitig of the layout and the polished one come from that run (stored);
    here the oracle's racon::Polisher runs the two rounds raven::Polish
    (polish.cc:26-51) runs on the stored layout unitig and must give the stored
    polished unitig."""
    genome = seqio.ReadSet.load(os.path.join(HERE, "golden", "lambda_genome.npz")).ascii(0)
    names0 = REF_META["assemble_rounds0_names"]
    names = REF_META["assemble_rounds2_names"]
    assert len(names0) == 1 and names0[0].endswith("XO:i:0")   # linear: no rotation
    assert len(names) == 1 and names[0].startswith("Utg")
    unpolished = REF_GOLD["assemble_rounds0_unitig0"].tobytes()
    want = REF_GOLD["assemble_rounds2_unitig0"].tobytes()
    # the quality threshold raven passes: the mean over reads of the mean block quality
    bq, off = lambda_reads.block_quality.astype(np.float64), lambda_reads.bq_off.astype(np.int64)
    avg_q = np.mean([bq[off[i]:off[i + 1]].mean() for i in range(lambda_reads.n)])
    lut = np.zeros(256, np.uint8)
    lut[np.frombuffer(b"ACGT", np.uint8)] = np.arange(4, dtype=np.uint8)
    seq = unpolished
    for _ in range(2):
        target = seqio.pack_codes([lut[np.frombuffer(seq, np.uint8)]])
        _, (seq,), _ = oracle.polish(target, lambda_reads, q=avg_q, e=0.3, w=500, trim=True,
                                     m=3, n=-5, g=-4, threads=8)
    assert seq == want
    ed = oracle.edit_distance(_revcomp(seq), genome)
    assert ed == 1137                 # EXPECT_EQ(1137, ...) raven_test.cpp:66
    # unpolished assembly for scale
    assert oracle.edit_distance(_revcomp(unpolished), genome) > 5 * ed


def test_nw_path_is_optimal_and_deterministic(oracle):
    rng = np.random.default_rng(3)
    import ctypes as C
    oracle.lib.orc_nw_path.restype = C.c_int64
    oracle.lib.orc_nw_path.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_char_p]
    for _ in range(40):
        n = int(rng.integers(1, 300))
        a = bytes(rng.choice(list(b"ACGT"), n).tolist())
        b = bytes(synth.mutate(np.frombuffer(a, np.uint8) % 4, rng, 0.05, 0.05, 0.05).tolist())
        b = bytes(b"ACGT"[x] for x in b) or b"A"
        buf = C.create_string_buffer(len(a) + len(b) + 1)
        ln = oracle.lib.orc_nw_path(a, len(a), b, len(b), buf)
        path = buf.raw[:ln]
        assert path.count(b"M") + path.count(b"I") == len(a)
        assert path.count(b"M") + path.count(b"D") == len(b)
        # cost of the path == edit distance
        i = j = cost = 0
        for op in path:
            if op == ord("M"):
                cost += a[i] != b[j]; i += 1; j += 1
            elif op == ord("I"):
                cost += 1; i += 1
            else:
                cost += 1; j += 1
        assert cost == oracle.edit_distance(a, b)


def _host_edlib():
    """The PRODUCT's host edlib (raven_b200/host/edlib.cc) as a library of its own."""
    import ctypes as C
    import subprocess
    subprocess.run(["make", "-C", os.path.join(HERE, "cpp"), "host"], check=True,
                   stdout=subprocess.DEVNULL)
    lib = C.CDLL(os.path.join(HERE, "cpp", "_build", "libhost_edlib.so"))

    class Cfg(C.Structure):
        _fields_ = [("k", C.c_int), ("mode", C.c_int), ("task", C.c_int),
                    ("eq", C.c_void_p), ("n_eq", C.c_int)]

    class Res(C.Structure):
        _fields_ = [("status", C.c_int), ("editDistance", C.c_int),
                    ("endLocations", C.POINTER(C.c_int)), ("startLocations", C.POINTER(C.c_int)),
                    ("numLocations", C.c_int), ("alignment", C.POINTER(C.c_ubyte)),
                    ("alignmentLength", C.c_int), ("alphabetLength", C.c_int)]

    lib.edlibAlign.restype = Res
    lib.edlibAlign.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, Cfg]
    lib.edlibFreeAlignResult.argtypes = [Res]

    def align(a, b, task, k=-1):
        r = lib.edlibAlign(a, len(a), b, len(b), Cfg(k, 0, task, None, 0))
        assert r.status == 0
        path = bytes(r.alignment[i] for i in range(r.alignmentLength)) if task == 2 else b""
        d = r.editDistance
        lib.edlibFreeAlignResult(r)
        return d, path

    return align


def test_product_edlib_equals_oracle(oracle):
    """raven_b200/host/edlib.cc (bit-vector blocks, band doubling, traceback below
    1 MiB, Hirschberg split above) against the oracle's plain dynamic programmes:
    distance AND the one path upstream edlib would return, incl. 10 kb ONT pairs."""
    import ctypes as C
    align = _host_edlib()
    oracle.lib.orc_nw_path.restype = C.c_int64
    oracle.lib.orc_nw_path.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_char_p]
    rng = np.random.default_rng(11)
    letters = np.frombuffer(b"ACGT", np.uint8)
    cases = [(0, 0.1), (1, 0.1), (2, 0.5), (63, 0.1), (64, 0.1), (65, 0.2), (130, 0.0),
             (700, 0.3), (1500, 0.15), (3000, 0.1), (4100, 0.02), (6000, 0.12),
             (10000, 0.1), (12000, 0.01), (11000, 0.15)]
    cases += [(int(rng.integers(1, 900)), float(rng.uniform(0, 0.4))) for _ in range(30)]
    for n, err in cases:
        a = rng.integers(0, 4, n, dtype=np.uint8)
        b = synth.mutate(a, rng, err / 3, err / 3, err / 3) if n else a
        if n and rng.random() < 0.3:   # unequal ends
            b = np.concatenate([rng.integers(0, 4, int(rng.integers(0, 40)), dtype=np.uint8), b])
        sa, sb = letters[a].tobytes(), letters[np.asarray(b, dtype=np.uint8)].tobytes()
        d, path = align(sa, sb, 2)
        d0, _ = align(sa, sb, 0)
        assert d == d0
        if max(len(sa), len(sb)) <= 3000:
            assert d == oracle.edit_distance(sa, sb), (n, err)
        buf = C.create_string_buffer(len(sa) + len(sb) + 1)
        ln = oracle.lib.orc_nw_path(sa, len(sa), sb, len(sb), buf)
        want = buf.raw[:ln]
        got = path.translate(bytes.maketrans(bytes([0, 1, 2, 3]), b"MIDM"))
        assert got == want, (n, err)
        assert d == want.count(b"I") + want.count(b"D") + sum(
            1 for op in path if op == 3), (n, err)
        # bounded calls: k below the distance -> -1, k at the distance -> found
        if d > 0:
            assert align(sa, sb, 0, d - 1)[0] == -1
        assert align(sa, sb, 0, d)[0] == d


def test_oracle_spoa_simd_fill_equals_scalar(oracle):
    """The oracle's AVX2 int16 matrix fill (what upstream spoa's SIMD engine does;
    the CPU legs of bench.py time it) gives the same consensus, coverages, status
    and cell counts as the scalar int32 loops."""
    sets = [synth.make_windows(n_windows=10, backbone_len=500, layers=25, seed=21),
            synth.make_windows(n_windows=6, backbone_len=300, layers=12, seed=5,
                               with_quality=False, partial=1.0),
            synth.make_windows(n_windows=4, backbone_len=760, layers=10, seed=11),
            synth.make_windows(n_windows=8, backbone_len=200, layers=6, seed=7, min_layers=0)]
    for w in sets:
        for kw in (dict(), dict(m=5, n=-4, g=-8), dict(trim=False)):
            oracle.lib.orc_spoa_use_simd(0)
            a = oracle.poa_batch(w, threads=4, **kw)
            oracle.lib.orc_spoa_use_simd(1)
            try:
                b = oracle.poa_batch(w, threads=4, **kw)
            finally:
                oracle.lib.orc_spoa_use_simd(0)
            for k in ("consensus", "cons_off", "coverage", "status", "cells"):
                assert np.array_equal(a[k], b[k]), k


def test_reference_pile_trim_rule():
    """Pile::FindValidRegion + FindMedian of the compiled reference (pile.cc:122-172;
    its results stored) against the rule the device kernel implements (PileRegionsKernel):
    the first longest run of bins >= coverage that is FOLLOWED by a lower bin (a run that
    reaches the last bin is never recorded), valid from 1260 >> 4 bins on; the median is
    the element of rank size / 2. Pins the rule on CPU; the GPU test compares the kernel
    itself."""
    piles, off = inputs.trim_rule_piles()
    got = {k: REF_GOLD[f"trim_rule_{k}"] for k in ("begin", "end", "median", "invalid", "data")}
    for i, d in enumerate(piles):
        begin = end = 0
        run = -1
        for j, v in enumerate(d.tolist()):
            if run < 0:
                if v >= 4:
                    run = j
            elif v < 4:
                if end - begin < j - run:
                    begin, end = run, j
                run = -1
        invalid = begin >= end or end - begin < (1260 >> 4)
        if invalid:
            want = (0, len(d), 0, 1)
        else:
            want = (begin, end, int(np.sort(d[begin:end])[(end - begin) // 2]), 0)
        assert (int(got["begin"][i]), int(got["end"][i]), int(got["median"][i]),
                int(got["invalid"][i])) == want, i
        if not invalid:   # UpdateValidRegion zeroes the bins outside the region
            trimmed = got["data"][off[i]:off[i + 1]]
            assert not trimmed[:begin].any() and not trimmed[end:].any()
            assert np.array_equal(trimmed[begin:end], d[begin:end])
    assert (got["invalid"] == 0).sum() > 20
