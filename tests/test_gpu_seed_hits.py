"""Seed hits of the key-partitioned path (rvn_dist_hits_split) against the oracle's
ram::MinimizerEngine::Map matches, for every pair of avoid_equal / avoid_symmetric.

The multi-GPU schedule always asks for (1, 1); the other pairs take the filtered
probe or the whole-run path of the shared seed code (seed.cuh), so they are
called here through the C ABI directly."""
import ctypes as C

import numpy as np
import pytest
import torch

from raven_b200 import distributed, engine

pytestmark = pytest.mark.gpu

FREQ = 0.001


def _host(t, dtype):
    return distributed._as_torch(t).cpu().numpy().view(dtype)


def _hits_split(steps, qval, qorg, ae, asym, parts, n_query):
    g, p, l = C.c_void_p(), C.c_void_p(), C.c_void_p()
    cnt = (C.c_uint64 * parts)()
    steps.e._check(steps.lib.rvn_dist_hits_split(
        steps.h, steps._p(qval), steps._p(qorg), qval.numel(), ae, asym, parts, n_query,
        C.byref(g), C.byref(p), C.byref(l), cnt))
    cnt = [int(x) for x in cnt]
    n = sum(cnt)
    dev = distributed.DevArray
    return (_host(dev(g.value, (n,), torch.int64, steps.device), np.uint64),
            _host(dev(p.value, (n,), torch.int64, steps.device), np.uint64),
            _host(dev(l.value, (n,), torch.int32, steps.device), np.uint32), cnt)


def _by_read(lhs, grp, pos):
    order = np.lexsort((pos, grp, lhs))
    return np.stack([lhs.astype(np.uint64), grp, pos], 1)[order]


def test_dist_hits_every_flag_pair(oracle, lambda_reads):
    rs, n = lambda_reads, lambda_reads.n
    eng = engine.Engine(device=0)
    try:
        eng.configure(k=15, w=5)
        eng.upload(rs)
        steps = distributed.CudaSteps(eng, "cuda:0")
        # index of the full sketches, queries = micromizers in read order
        ival, iorg, _ = steps.sketch_split(0, n, 1, False)
        qval, qorg, _ = steps.sketch_split(0, n, 1, True)
        steps.build_index(ival, iorg, rs.bases)
        hist, n_keys = steps.histogram()
        occ = steps.set_occurrence(hist.cpu().numpy(), n_keys, FREQ)

        oeng = oracle.engine(15, 5, threads=4)
        reads = oracle.reads(rs)
        oracle.minimize(oeng, reads, 0, n, False)
        assert occ == oracle.filter(oeng, FREQ)

        for ae, asym in [(1, 1), (1, 0), (0, 1), (0, 0)]:
            want = oracle.map(oeng, reads, 0, n, ae, asym, True, want_matches=True)
            per_read = np.diff(want["match_off"]).astype(np.int64)
            w_lhs = np.repeat(np.arange(n, dtype=np.uint32), per_read)
            expect = _by_read(w_lhs, want["match_group"], want["match_pos"])
            assert expect.shape[0] > 0
            for parts in (1, 3):
                grp, pos, lhs, cnt = _hits_split(steps, qval, qorg, ae, asym, parts, n)
                assert sum(cnt) == grp.size == expect.shape[0], (ae, asym, parts)
                off = np.concatenate([[0], np.cumsum(cnt)])
                for d in range(parts):
                    assert np.all(lhs[off[d]:off[d + 1]] % parts == d), (ae, asym, parts, d)
                assert np.array_equal(_by_read(lhs, grp, pos), expect), (ae, asym, parts)
    finally:
        eng.close()
