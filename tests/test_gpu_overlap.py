"""GPU parity tests: every stage of the CUDA overlap path, called through the
C ABI, against the CPU oracle on the same inputs - bit exact."""
import json
import os

import numpy as np
import pytest

import reference_inputs as inputs
from raven_b200 import seqio, synth

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
META = json.load(open(os.path.join(HERE, "golden", "lambda_golden.json")))
GOLD = np.load(os.path.join(HERE, "golden", "lambda_golden.npz"))
REF_META = json.load(open(os.path.join(HERE, "golden", "reference_golden.json")))
REF_GOLD = np.load(os.path.join(HERE, "golden", "reference_golden.npz"))


def edge_reads():
    rng = np.random.default_rng(21)
    seqs = [rng.integers(0, 4, n, dtype=np.uint8)
            for n in (0, 1, 14, 15, 18, 19, 20, 31, 32, 33, 63, 64, 65, 2047, 2048,
                      2049, 2062, 2063, 2066, 4100, 9000)]
    seqs.append(np.zeros(500, np.uint8))                      # poly-A
    seqs.append(np.full(500, 3, np.uint8))                    # poly-T
    seqs.append(np.tile(np.array([0, 3], np.uint8), 300))     # palindromic k-mers
    seqs.append(np.tile(np.array([0, 1, 2, 3], np.uint8), 200))
    base = rng.integers(0, 4, 3000, dtype=np.uint8)
    seqs += [base.copy() for _ in range(6)]                   # identical reads
    seqs.append((3 - base[::-1]).astype(np.uint8))            # and a reverse complement
    return seqio.pack_codes(seqs)


@pytest.mark.parametrize("kw", [(15, 5), (19, 10), (5, 3), (4, 1), (31, 7), (11, 32)])
@pytest.mark.parametrize("minhash", [False, True])
def test_sketch_edge_cases(gpu_engine, oracle, kw, minhash):
    k, w = kw
    rs = edge_reads()
    gpu_engine.configure(k=k, w=w)
    gpu_engine.upload(rs)
    got = gpu_engine.sketch(0, rs.n, minhash)
    want = oracle.sketch(oracle.engine(k, w), oracle.reads(rs), 0, rs.n, minhash)
    assert np.array_equal(got["offsets"], want["offsets"])
    assert np.array_equal(got["value"], want["value"])
    assert np.array_equal(got["origin"], want["origin"])


@pytest.mark.parametrize("minhash", [False, True])
def test_sketch_lambda_golden(gpu_engine, oracle, lambda_reads, minhash):
    import hashlib
    gpu_engine.configure(k=15, w=5)
    gpu_engine.upload(lambda_reads)
    got = gpu_engine.sketch(0, lambda_reads.n, minhash)
    tag = "micro" if minhash else "full"
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
    assert got["value"].size == META[f"sketch_{tag}_n"]
    assert sha(got["value"]) == META[f"sketch_{tag}_value_sha256"]
    assert sha(got["origin"]) == META[f"sketch_{tag}_origin_sha256"]
    assert sha(got["offsets"]) == META[f"sketch_{tag}_offsets_sha256"]
    # a sub-range sketches identically
    sub = gpu_engine.sketch(17, 93, minhash)
    a, b = int(got["offsets"][17]), int(got["offsets"][93])
    assert np.array_equal(sub["value"], got["value"][a:b])
    assert np.array_equal(sub["origin"], got["origin"][a:b])


@pytest.mark.parametrize("minhash", [False, True])
def test_index_and_filter(gpu_engine, oracle, lambda_reads, minhash):
    gpu_engine.configure(k=15, w=5)
    gpu_engine.upload(lambda_reads)
    gpu_engine.minimize(0, lambda_reads.n, minhash)
    idx = gpu_engine.index_records()
    eng = oracle.engine(15, 5, threads=4)
    reads = oracle.reads(lambda_reads)
    oracle.minimize(eng, reads, 0, lambda_reads.n, minhash)
    keys = oracle.keys(eng)
    # sorted by value, postings of a key in (read, position) order
    v, o = idx["value"], idx["origin"]
    assert v.size == int(keys["totals"][1]) and idx["n_keys"] == int(keys["totals"][0])
    assert (np.diff(v.astype(np.int64)) >= 0).all() if v.max() < 2**62 else True
    same = v[1:] == v[:-1]
    assert (o[1:][same] > o[:-1][same]).all()
    uv, uc = np.unique(v, return_counts=True)
    assert np.array_equal(uv, keys["values"]) and np.array_equal(uc.astype(np.uint32), keys["counts"])
    for f in (0.001, 0.01, 0.5, 1.0, 1e-7, 0):
        assert gpu_engine.filter(f) == oracle.filter(eng, f), f
    for f in (-0.5, 1.01, float("nan")):
        with pytest.raises(ValueError):
            gpu_engine.filter(f)


def _check_map(gpu_engine, oracle, rs, k, w, freq, minhash_index, cases, **prm):
    gpu_engine.configure(k=k, w=w, **prm)
    gpu_engine.upload(rs)
    gpu_engine.set_option("keep_hits", 1)
    gpu_engine.minimize(0, rs.n, minhash_index)
    occ = gpu_engine.filter(freq)
    eng = oracle.engine(k, w, threads=4, **prm)
    reads = oracle.reads(rs)
    oracle.minimize(eng, reads, 0, rs.n, minhash_index)
    assert occ == oracle.filter(eng, freq)
    for (first, last, ae, asym, mh) in cases:
        got = gpu_engine.map(first, last, ae, asym, mh, want_filtered=True)
        hits = gpu_engine.map_hits(last - first)
        want = oracle.map(eng, reads, first, last, ae, asym, mh, want_matches=True)
        # hits: same multiset per query
        assert np.array_equal(hits["hit_off"], want["match_off"])
        for i in range(last - first):
            a, b = int(hits["hit_off"][i]), int(hits["hit_off"][i + 1])
            g = np.stack([hits["group"][a:b], hits["positions"][a:b]], 1)
            x = np.stack([want["match_group"][a:b], want["match_pos"][a:b]], 1)
            assert np.array_equal(g[np.lexsort((g[:, 1], g[:, 0]))],
                                  x[np.lexsort((x[:, 1], x[:, 0]))]), i
        assert np.array_equal(got["filt_off"], want["filt_off"])
        assert np.array_equal(got["filtered"], want["filtered"])
        assert np.array_equal(got["ovl_off"], want["ovl_off"])
        assert np.array_equal(got["overlaps"], want["overlaps"])
    gpu_engine.set_option("keep_hits", 0)


def test_map_lambda(gpu_engine, oracle, lambda_reads):
    n = lambda_reads.n
    _check_map(gpu_engine, oracle, lambda_reads, 15, 5, 0.001, False,
               [(0, n, True, True, True), (0, n, True, True, False),
                (10, 57, True, True, True), (0, n, False, False, False),
                (100, 101, True, False, True)])
    got = gpu_engine.map(0, n, True, True, True)
    assert np.array_equal(got["overlaps"], GOLD["map_micro_overlaps"])
    got = gpu_engine.map(0, n, True, True, False)
    assert np.array_equal(got["overlaps"], GOLD["map_full_overlaps"])


def test_map_minhash_index_and_params(gpu_engine, oracle, lambda_reads):
    n = lambda_reads.n
    _check_map(gpu_engine, oracle, lambda_reads, 15, 5, 0.001, True,
               [(0, n, True, True, True)])
    _check_map(gpu_engine, oracle, lambda_reads, 15, 5, 0.0, False,
               [(0, 60, True, True, True)])
    _check_map(gpu_engine, oracle, lambda_reads, 13, 7, 0.01, False,
               [(0, n, True, True, False)], bandwidth=200, chain=3, matches=60, gap=2000)


def test_map_edge_cases_and_repeats(gpu_engine, oracle):
    rs = edge_reads()
    _check_map(gpu_engine, oracle, rs, 15, 5, 0.001, False,
               [(0, rs.n, True, True, False), (0, rs.n, False, False, False),
                (0, rs.n, True, True, True)])
    # a repetitive genome: many hits per query, long bands, the global-memory path
    rng = np.random.default_rng(4)
    unit = rng.integers(0, 4, 400, dtype=np.uint8)
    genome = np.concatenate([unit] * 40 + [rng.integers(0, 4, 20000, dtype=np.uint8)])
    rs = synth.make_reads(n_reads=80, mean_len=6000, seed=8, genome=genome, sub=0.01,
                          ins=0.01, dele=0.01)
    _check_map(gpu_engine, oracle, rs, 15, 5, 0.0, False,
               [(0, rs.n, True, True, False)])


def test_map_external_read(gpu_engine, oracle, lambda_reads):
    """ram::MinimizerEngine::Map for a read outside the indexed/uploaded set
    (construct.cc:59-62 with several index batches; assemble.cc:757,780)."""
    n = lambda_reads.n
    n_idx = n - 6
    sub = lambda_reads.subset(range(n_idx))
    gpu_engine.configure(15, 5)
    gpu_engine.upload(sub)
    gpu_engine.minimize(0, n_idx, False)
    occ = gpu_engine.filter(0.001)
    eng = oracle.engine(15, 5, threads=4)
    reads = oracle.reads(lambda_reads)
    oracle.minimize(eng, reads, 0, n_idx, False)
    assert occ == oracle.filter(eng, 0.001)
    rs = lambda_reads
    for j in range(n_idx, n):
        w = rs.words[int(rs.word_off[j]):int(rs.word_off[j + 1])]
        for (ae, asym, mh) in ((True, True, True), (False, False, False), (True, False, True),
                               (True, True, False)):
            got = gpu_engine.map_external(w, int(rs.lens[j]), j, ae, asym, mh,
                                          want_filtered=True)
            want = oracle.map(eng, reads, j, j + 1, ae, asym, mh)
            assert np.array_equal(got["overlaps"], want["overlaps"]), (j, ae, asym, mh)
            assert np.array_equal(got["filtered"], want["filtered"]), (j, ae, asym, mh)
    # an id BELOW the indexed ids: avoid_symmetric keeps every posting
    j = n - 1
    w = rs.words[int(rs.word_off[j]):int(rs.word_off[j + 1])]
    got = gpu_engine.map_external(w, int(rs.lens[j]), j, False, False, True)
    assert got["overlaps"].shape[0] > 0
    # the uploaded set is intact afterwards
    again = gpu_engine.map(0, 20, True, True, True)
    want = oracle.map(eng, reads, 0, 20, True, True, True)
    assert np.array_equal(again["overlaps"], want["overlaps"])


def test_empty_inputs(gpu_engine, oracle):
    rs = seqio.pack_codes([])
    gpu_engine.configure(15, 5)
    gpu_engine.upload(rs)
    gpu_engine.minimize(0, 0, False)
    assert gpu_engine.filter(0.001) == 0xFFFFFFFF
    got = gpu_engine.map(0, 0)
    assert got["overlaps"].shape[0] == 0 and got["ovl_off"].tolist() == [0]
    st = gpu_engine.find_overlaps_and_create_piles()
    assert st["overlaps"].shape[0] == 0
    rs = synth.random_reads([5, 9, 3])
    gpu_engine.upload(rs)
    st = gpu_engine.find_overlaps_and_create_piles()
    assert st["overlaps"].shape[0] == 0 and st["pile"].size == 0
    with pytest.raises(RuntimeError):
        gpu_engine.configure(15, 5)
        gpu_engine.upload(rs)
        gpu_engine.map(0, 3)   # Map before Minimize


def test_pile_add_layers(gpu_engine, oracle):
    rng = np.random.default_rng(12)
    lens = rng.integers(200, 9000, 40)
    off = np.concatenate([[0], np.cumsum(lens >> 4)]).astype(np.uint64)
    ovl = []
    for _ in range(3000):
        a, b = rng.choice(40, 2, replace=False)
        def span(L):
            s = int(rng.integers(0, L - 150))
            return s, int(rng.integers(s + 100, L + 1))
        ab, ae = span(lens[a]); bb, be = span(lens[b])
        ovl.append([a, ab, ae, b, bb, be, 100, int(rng.integers(0, 2))])
    ovl = np.array(ovl, dtype=np.uint32)
    data = rng.integers(0, 3, int(off[-1])).astype(np.uint16)
    data[rng.integers(0, data.size, 50)] = 65530   # near saturation
    got = gpu_engine.pile_add_layers(data, off, ovl)
    got = gpu_engine.pile_add_layers(got, off, ovl)
    want = data.copy()
    for p in range(40):
        sl = slice(int(off[p]), int(off[p + 1]))
        d = oracle.pile_add_layers(p, want[sl], ovl)
        want[sl] = oracle.pile_add_layers(p, d, ovl)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("minhash", [False, True])
def test_stage1_lambda_golden(gpu_engine, lambda_reads, minhash):
    gpu_engine.configure(k=15, w=5)
    gpu_engine.upload(lambda_reads)
    got = gpu_engine.find_overlaps_and_create_piles(0.001, 32, minhash)
    tag = "minhash" if minhash else "plain"
    for k in ("overlaps", "ovl_off", "pile", "pile_off"):
        assert np.array_equal(got[k], GOLD[f"stage1_{tag}_{k}"]), k
    assert got["num_mapped"] == META[f"stage1_{tag}_num_mapped"]


@pytest.mark.parametrize("cfg", [
    dict(genome_len=80_000, n_reads=300, mean_len=4000, seed=2, kmax=32, ib=0, qb=0),
    dict(genome_len=30_000, n_reads=150, mean_len=3000, seed=3, kmax=8, ib=120_000, qb=50_000),
    dict(genome_len=30_000, n_reads=150, mean_len=3000, seed=4, kmax=4, ib=1 << 40, qb=70_000),
])
def test_stage1_synthetic_schedules(gpu_engine, oracle, cfg):
    rs = synth.make_reads(cfg["genome_len"], cfg["n_reads"], cfg["mean_len"], seed=cfg["seed"])
    gpu_engine.configure(k=15, w=5)
    gpu_engine.upload(rs)
    for minhash in (False, True):
        got = gpu_engine.find_overlaps_and_create_piles(0.001, cfg["kmax"], minhash,
                                                        cfg["ib"], cfg["qb"])
        want = oracle.stage1(oracle.engine(15, 5, threads=4), oracle.reads(rs), 0.001,
                             cfg["kmax"], minhash, cfg["ib"] or 1 << 32, cfg["qb"] or 1 << 30)
        for k in ("overlaps", "ovl_off", "pile", "pile_off"):
            assert np.array_equal(got[k], want[k]), (minhash, k)
        assert got["num_mapped"] == int(want["num_mapped"][0])


def test_stage1_tiered_index(gpu_engine, oracle, lambda_reads):
    """Stage 1 with the tiered index forced on small inputs (bench-size batches take
    it by default): records above the largest micromizer value are only counted for
    the occurrence threshold. Same result as the golden files / the oracle, incl.
    several index batches and a frequency that cuts deep."""
    gpu_engine.set_option("tier_min_records", 0)
    try:
        gpu_engine.configure(k=15, w=5)
        gpu_engine.upload(lambda_reads)
        got = gpu_engine.find_overlaps_and_create_piles(0.001, 32, False)
        for k in ("overlaps", "ovl_off", "pile", "pile_off"):
            assert np.array_equal(got[k], GOLD[f"stage1_plain_{k}"]), k
        assert got["num_mapped"] == META["stage1_plain_num_mapped"]
        rs = synth.make_reads(30_000, 150, 3000, seed=3)
        gpu_engine.upload(rs)
        for freq, ib, qb in ((0.001, 120_000, 50_000), (0.05, 0, 0), (0.3, 200_000, 0)):
            got = gpu_engine.find_overlaps_and_create_piles(freq, 8, False, ib, qb)
            want = oracle.stage1(oracle.engine(15, 5, threads=4), oracle.reads(rs), freq, 8,
                                 False, ib or 1 << 32, qb or 1 << 30)
            for k in ("overlaps", "ovl_off", "pile", "pile_off"):
                assert np.array_equal(got[k], want[k]), (freq, ib, k)
        # a map call with full sketches after a tiered stage 1 must not see the tiers
        gpu_engine.minimize(0, rs.n, False)
        gpu_engine.filter(0.001)
        a = gpu_engine.map(0, rs.n, True, True, False)
        eng = oracle.engine(15, 5, threads=4)
        reads = oracle.reads(rs)
        oracle.minimize(eng, reads, 0, rs.n, False)
        oracle.filter(eng, 0.001)
        assert np.array_equal(a["overlaps"], oracle.map(eng, reads, 0, rs.n, True, True, False)["overlaps"])
    finally:
        gpu_engine.set_option("tier_min_records", 1 << 18)


def test_stage1_probe_path_without_self_join(gpu_engine, oracle, lambda_reads):
    """By default the seed hits of a stage-1 flush inside the index batch come from the
    self-join over the sorted index (map.cu); with the option off every flush probes
    the table per micromizer like flushes outside the batch do. Same results, with
    repeats (low frequency cut), several index batches and flushes, both tier modes."""
    rs = synth.make_reads(30_000, 160, 3000, seed=9)
    for tiers in (0, 1 << 18):
        gpu_engine.set_option("tier_min_records", tiers)
        try:
            for join in (0, 1):
                gpu_engine.set_option("self_join", join)
                gpu_engine.configure(k=15, w=5)
                gpu_engine.upload(lambda_reads)
                got = gpu_engine.find_overlaps_and_create_piles(0.001, 32, False)
                for k in ("overlaps", "ovl_off", "pile", "pile_off"):
                    assert np.array_equal(got[k], GOLD[f"stage1_plain_{k}"]), (join, k)
                gpu_engine.upload(rs)
                for freq, ib, qb in ((0.001, 0, 0), (0.02, 150_000, 60_000), (0.3, 0, 100_000)):
                    got = gpu_engine.find_overlaps_and_create_piles(freq, 8, False, ib, qb)
                    want = oracle.stage1(oracle.engine(15, 5, threads=4), oracle.reads(rs), freq,
                                         8, False, ib or 1 << 32, qb or 1 << 30)
                    for k in ("overlaps", "ovl_off", "pile", "pile_off"):
                        assert np.array_equal(got[k], want[k]), (tiers, join, freq, ib, k)
                    assert got["num_mapped"] == int(want["num_mapped"][0])
        finally:
            gpu_engine.set_option("self_join", 1)
            gpu_engine.set_option("tier_min_records", 1 << 18)


def test_stage1_pile_regions_equal_reference(gpu_engine, lambda_reads):
    """rvn_stage1_pile_regions (Pile::FindValidRegion(4) + FindMedian on the piles stage 1
    left on the device, construct.cc:134-139) against the reference's own pile.cc compiled
    in place (its results on the reference's stage-1 piles stored): begin, end, median,
    invalid of every pile - the lambda reads, a deep synthetic set, other coverages; and
    the state check."""
    import hashlib
    for name, rs in (("lambda", lambda_reads), ("synthetic", inputs.region_reads())):
        gpu_engine.configure(15, 5)
        gpu_engine.upload(rs)
        res = gpu_engine.find_overlaps_and_create_piles(0.001, 32, False)
        assert (hashlib.sha256(np.ascontiguousarray(res["pile"]).tobytes()).hexdigest()
                == REF_META[f"regions_{name}_pile_sha256"])
        for cov in inputs.REGION_COVERAGES:
            got = gpu_engine.stage1_pile_regions(cov)
            for k in ("invalid", "begin", "end", "median"):
                assert np.array_equal(got[k], REF_GOLD[f"regions_{name}_cov{cov}_{k}"]), (cov, k)
        assert (got["invalid"] == 0).any() or rs is lambda_reads
    assert (gpu_engine.stage1_pile_regions(4)["invalid"] == 0).sum() > 100
    gpu_engine.upload(rs)
    with pytest.raises(RuntimeError):   # no stage-1 piles on the device any more
        gpu_engine.stage1_pile_regions(4)


def test_filter_with_very_long_runs(gpu_engine, oracle):
    """Keys that occur 65535 times or more fall out of the run-length histogram and are
    ranked by their exact lengths (CollectLongRuns) - in the tiered build this first
    finishes the sort of the upper tier's keys. 70 000 copies of one short read: its
    keys are that long. Stage 1 runs with a frequency that filters them (no hits); the
    thresholds of other frequencies are then asked of the SAME tiered index."""
    rng = np.random.default_rng(31)
    one = rng.integers(0, 4, 90, dtype=np.uint8)
    seqs = [one] * 70_000 + [rng.integers(0, 4, 400, dtype=np.uint8) for _ in range(50)]
    rs = seqio.pack_codes(seqs)
    eng = oracle.engine(15, 5, threads=8)
    reads = oracle.reads(rs)
    oracle.minimize(eng, reads, 0, rs.n, False)
    gpu_engine.configure(15, 5)
    gpu_engine.upload(rs)
    gpu_engine.set_option("tier_min_records", 0)
    try:
        gpu_engine.find_overlaps_and_create_piles(0.5, 8, False)
        assert gpu_engine.stats()["occurrence"] == oracle.filter(eng, 0.5)
        for freq in (0.0005, 0.002, 0.5, 0.001):   # the first ones rank the long runs
            assert gpu_engine.filter(freq) == oracle.filter(eng, freq), freq
    finally:
        gpu_engine.set_option("tier_min_records", 1 << 18)
    gpu_engine.minimize(0, rs.n, False)
    for freq in (0.0005, 0.5):
        assert gpu_engine.filter(freq) == oracle.filter(eng, freq), freq


def test_stage1_async_upload(gpu_engine, lambda_reads):
    """Option async_upload: the bases travel in chunks on a copy stream and the sketch
    kernel is launched piecewise behind them - same result, also when the upload is
    followed by a call that does not start with the sketch."""
    rs = synth.make_reads(200_000, 2400, 4000, seed=12)   # > 1024 reads: chunked
    gpu_engine.configure(k=15, w=5)
    gpu_engine.upload(rs)
    want = gpu_engine.find_overlaps_and_create_piles(0.001, 16, False)
    gpu_engine.set_option("async_upload", 1)
    try:
        for _ in range(2):
            gpu_engine.upload(rs)
            got = gpu_engine.find_overlaps_and_create_piles(0.001, 16, False)
            for k in ("overlaps", "ovl_off", "pile", "pile_off"):
                assert np.array_equal(got[k], want[k]), k
        gpu_engine.upload(rs)
        d = gpu_engine.edit_distance_batch([0], [0], [500], [0], [0], [500], [1])
        assert d.tolist() == [0]
        gpu_engine.upload(rs, resident=(100, 2000))
        a = gpu_engine.sketch(100, 2000, False)
        gpu_engine.set_option("async_upload", 0)
        gpu_engine.upload(rs, resident=(100, 2000))
        b = gpu_engine.sketch(100, 2000, False)
        assert all(np.array_equal(a[k], b[k]) for k in ("value", "origin", "offsets"))
    finally:
        gpu_engine.set_option("async_upload", 0)


def test_stage1_hifi_params(gpu_engine, oracle):
    rs = synth.make_reads(60_000, 120, 6000, seed=6, sub=0.002, ins=0.0015, dele=0.0015)
    gpu_engine.configure(k=19, w=10)
    gpu_engine.upload(rs)
    got = gpu_engine.find_overlaps_and_create_piles(0.001, 32, False)
    want = oracle.stage1(oracle.engine(19, 10, threads=4), oracle.reads(rs), 0.001, 32, False)
    for k in ("overlaps", "ovl_off", "pile", "pile_off"):
        assert np.array_equal(got[k], want[k]), k


def test_kmer_complexity(gpu_engine, oracle):
    """Pile::AddKmers' low-complexity rule on the positions Map reports as filtered."""
    rs = inputs.lowcomplexity_reads()
    gpu_engine.configure(15, 5)
    gpu_engine.upload(rs)
    idx, pos = [], []
    for r in range(rs.n):
        for p in range(0, int(rs.lens[r])):
            idx.append(r); pos.append(p)
    for k in (15, 19, 31, 9, 4, 1):
        got = gpu_engine.kmer_complexity(idx, pos, k)
        want = oracle.kmer_complexity(oracle.reads(rs), idx, pos, k)
        assert np.array_equal(got, want), k
    with pytest.raises(ValueError):
        gpu_engine.kmer_complexity([0], [0], 32)
    with pytest.raises(ValueError):
        gpu_engine.kmer_complexity([99], [0], 15)


def test_stage2_map_filtered_feeds_add_kmers(gpu_engine, oracle, lambda_reads):
    """Stage-2 semantics (construct.cc:363-383): full sketches, filtered positions,
    explicit ids after raven's re-sort of the sequences."""
    n = lambda_reads.n
    order = np.r_[np.arange(0, n, 2), np.arange(1, n, 2)]     # ids no longer == positions
    rs = lambda_reads.subset(order)
    lib = gpu_engine.lib
    import ctypes as C
    words = np.ascontiguousarray(rs.words); woff = np.ascontiguousarray(rs.word_off)
    lens = np.ascontiguousarray(rs.lens); ids = np.ascontiguousarray(order.astype(np.uint32))
    from raven_b200._lib import U64P, U32P
    gpu_engine.configure(15, 5)
    gpu_engine._check(lib.rvn_reads_upload_ids(gpu_engine.h, words.ctypes.data_as(U64P),
                                               woff.ctypes.data_as(U64P),
                                               lens.ctypes.data_as(U32P),
                                               ids.ctypes.data_as(U32P), rs.n))
    gpu_engine.n_reads = rs.n
    gpu_engine.minimize(0, 150, False)
    occ = gpu_engine.filter(0.001)
    got = gpu_engine.map(0, 150, True, True, False, want_filtered=True)
    # the oracle sees the same permuted set with the same ids
    eng = oracle.engine(15, 5, threads=4)
    reads = oracle.reads(rs)
    import oracle_lib
    # give the oracle's sequences the permuted ids
    oracle.lib.orc_reads_set_ids.argtypes = [C.c_void_p, oracle_lib._U32P]
    oracle.lib.orc_reads_set_ids(reads.h, ids.ctypes.data_as(oracle_lib._U32P))
    oracle.minimize(eng, reads, 0, 150, False)
    assert occ == oracle.filter(eng, 0.001)
    want = oracle.map(eng, reads, 0, 150, True, True, False)
    assert np.array_equal(got["overlaps"], want["overlaps"])
    assert np.array_equal(got["filtered"], want["filtered"])
    assert np.array_equal(got["filt_off"], want["filt_off"])
    # filtered positions -> AddKmers rule
    ri = np.repeat(np.arange(150), np.diff(got["filt_off"].astype(np.int64)))
    keep = gpu_engine.kmer_complexity(ri, got["filtered"], 15)
    assert np.array_equal(keep, oracle.kmer_complexity(reads, ri, got["filtered"], 15))
