#!/usr/bin/env python
"""bench.py — overlaps/s of the stage-1 all-vs-all overlap path on B200.

One "step" = one pass of raven::FindOverlapsAndCreatePiles (sketch, index,
filter, map/chain, pile coverage, truncation) over one synthetic read set.
Workload at N=1 = BASELINE.json configs[1]: 200k synthetic ONT reads ~10 kb
(~2 Gbp), k=15 w=5 f=0.001, overlap-only (-p 0).

  value   overlaps/s with the packed reads already resident in HBM
  e2e     the same through the C-ABI with HOST buffers: H2D of the packed
          reads and D2H of overlaps + piles inside the timed region
  --impl reference   the reference's own CPU code for the path (oracle/_ref:
          construct.cc/pile.cc/overlap_utils.cc compiled in place, over the
          restated ram engine) on a bounded sample, all host threads.

N>1 (torchrun): the SAME 200k-read set (strong scaling: total work fixed),
overlapped all-vs-all by all ranks together: reads sharded by id, index keys by
value, all-to-all of minimizer records, of seed hits and of overlaps
(raven_b200/distributed.py); value = all overlaps of the job / max-over-ranks
device time. (N x reads would not be N x work: with k=15 the random-match
part of the seed hits grows with the square of the read count - measured
350 M hits/GPU at 200k reads, 604 M at 2 x 200k on 2 GPUs.)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SEED = 20260924
K, W, FREQ, KMAX = 15, 5, 0.001, 32


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=200_000)
    ap.add_argument("--genome", type=int, default=50_000_000)
    ap.add_argument("--mean-len", type=int, default=10_000)
    ap.add_argument("--cpu-sample-reads", type=int, default=20_000)
    ap.add_argument("--index-batches", type=int, default=1,
                    help="C4-shaped run: cut the read set into this many index batches "
                         "(the reference starts a new batch every 2^32 bases, "
                         "construct.cc:35; here the batch size is total bases / K)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--poa-windows", type=int, default=8192,
                    help="windows of the POA sub-benchmark (0 = skip)")
    ap.add_argument("--c3-reads", type=int, default=20_000,
                    help="reads of the C3-shaped polishing run (0 = skip)")
    ap.add_argument("--c5-reads", type=int, default=30_000,
                    help="HiFi reads of the C5-shaped run: stage 1 + identity filter (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the stage-1 result of the last timed step to DIR/<name>.npy "
                         "(a fixed, seeded sample of the reads; at most 64 MB)")
    return ap.parse_args()


def workload_name(a):
    if a.index_batches > 1:
        return (f"C4-shaped: {a.reads} synthetic ONT reads ~{a.mean_len // 1000} kb over a "
                f"{a.genome / 1e6:.0f} Mbp genome (40x, 10% error) in {a.index_batches} index "
                f"batches (batch = total bases / {a.index_batches}; the reference's 2 M-read "
                f"run has 5 batches of 2^32 bases), k={K} w={W} f={FREQ} "
                f"kMaxNumOverlaps={KMAX}, stage-1 all-vs-all, -p 0")
    return (f"C2: {a.reads} synthetic ONT reads ~{a.mean_len // 1000} kb over a "
            f"{a.genome / 1e6:.0f} Mbp genome (40x, 10% error), k={K} w={W} f={FREQ} "
            f"kMaxNumOverlaps={KMAX}, stage-1 all-vs-all "
            "(FindOverlapsAndCreatePiles), -p 0")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []
        self.p = None
        try:
            self.p = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        self.t.join(timeout=2)
        sm = sorted(int(r[1]) for r in self.rows if len(r) > 8 and r[1].isdigit())
        mx = max([int(r[2]) for r in self.rows if len(r) > 8 and r[2].isdigit()] or [0])
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_sample(a):
    """Bounded sample of the same workload for the CPU legs: same read model and
    coverage (40x) over a proportionally smaller genome."""
    from bench import synth
    n = min(a.cpu_sample_reads, a.reads)
    g = max(int(a.genome * n / max(a.reads, 1)), 4 * a.mean_len)
    return synth.make_reads(SEED + 1, g, n, a.mean_len), n, g


def run_cpu(a, kind_pref="reference", threads=None):
    """One stage-1 pass of the CPU path on the bounded sample."""
    import oracle_lib
    threads = threads or os.cpu_count() or 1
    rs, n, g = cpu_sample(a)
    sample = (f"{n} reads / {g / 1e6:.1f} Mbp genome of the same 40x model "
              f"({rs.bases / 1e9:.3f} Gbp), one stage-1 pass")
    if kind_pref == "reference" and oracle_lib.Reference.available():
        R = oracle_lib.Reference()
        reads = R.reads(rs)

        def step():
            t = time.perf_counter()
            # stderr phase lines of the reference are silenced for the bench
            fd = os.dup(2)
            devnull = os.open(os.devnull, os.O_WRONLY)
            os.dup2(devnull, 2)
            try:
                res = R.stage1(reads, K, W, FREQ, KMAX, False, threads)
            finally:
                os.dup2(fd, 2)
                os.close(fd)
                os.close(devnull)
            dt = time.perf_counter() - t
            # overlaps returned by all Map calls = half the incidences before
            # truncation; the reference library does not expose it, so count
            # via the port's counter on the first call only
            return dt, res
        kind = "reference"
    else:
        O = oracle_lib.Oracle()
        reads = O.reads(rs)

        def step():
            t = time.perf_counter()
            res = O.stage1(O.engine(K, W, threads=threads), reads, FREQ, KMAX, False)
            return time.perf_counter() - t, res
        kind = "port"
    # number of mapped overlaps of the sample (identical for port and reference)
    O = oracle_lib.Oracle()
    n_mapped = int(O.stage1(O.engine(K, W, threads=threads), O.reads(rs), FREQ, KMAX,
                            False)["num_mapped"][0])
    return step, n_mapped, kind, threads, sample


def result_sha256(res):
    """One digest over the stage-1 result (kept overlaps, list offsets, piles)."""
    import hashlib
    import numpy as np
    h = hashlib.sha256()
    for k in ("overlaps", "ovl_off", "pile"):
        h.update(np.ascontiguousarray(res[k]).tobytes())
    return h.hexdigest()


def same_result(x, y):
    import numpy as np
    return all(np.array_equal(np.asarray(x[k]).reshape(-1), np.asarray(y[k]).reshape(-1))
               for k in ("overlaps", "ovl_off", "pile"))


DUMP_BYTES = 64 << 20
DUMP_MAX_READS = 4096


def gather_ranges(values, off, ids):
    """values[off[i]:off[i + 1]] of every read i in ids, concatenated, and their lengths."""
    import numpy as np
    o = off.astype(np.int64)
    cnt = o[ids + 1] - o[ids]
    idx = np.repeat(o[ids], cnt) + (np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt))
    return values[idx], cnt


def dump_outputs(path, res, budget, suffix=""):
    """The stage-1 result a caller receives (kept overlaps and pile of every read, the
    number of mapped overlaps) as float .npy files, for a fixed, seeded sample of the
    reads that fits `budget` bytes. float64 holds the uint32/uint64 fields exactly,
    float32 the uint16 pile bins. Files: read_ids, overlaps (one row of 8 fields per
    kept overlap of the sampled reads, in read order), overlaps_per_read, pile (the
    bins of the sampled reads), bins_per_read, num_mapped."""
    import numpy as np
    n = len(res["ovl_off"]) - 1
    per_read = (8 * 8 * np.diff(res["ovl_off"].astype(np.int64))
                + 4 * np.diff(res["pile_off"].astype(np.int64)) + 3 * 8)
    order = np.random.default_rng(SEED).permutation(n)
    fits = int(np.searchsorted(np.cumsum(per_read[order]), budget - 4096, side="right"))  # npy headers
    ids = np.sort(order[:min(fits, DUMP_MAX_READS)])
    ovl, n_ovl = gather_ranges(np.asarray(res["overlaps"]).reshape(-1, 8), res["ovl_off"], ids)
    pile, n_bins = gather_ranges(np.asarray(res["pile"]), res["pile_off"], ids)
    out = {"read_ids": ids.astype(np.float64), "overlaps": ovl.astype(np.float64),
           "overlaps_per_read": n_ovl.astype(np.float64), "pile": pile.astype(np.float32),
           "bins_per_read": n_bins.astype(np.float64),
           "num_mapped": np.array([res["num_mapped"]], dtype=np.float64)}
    os.makedirs(path, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(path, name + suffix + ".npy"), arr)


def share_of(res, rank, world):
    """The slice of a complete stage-1 result that rank `rank` owns (reads rank,
    rank + world, ...), in the layout of DistEngine's per-rank result."""
    import numpy as np
    n = len(res["ovl_off"]) - 1
    ids = np.arange(rank, n, world)
    out = {}
    for key, off in (("overlaps", "ovl_off"), ("pile", "pile_off")):
        out[key], cnt = gather_ranges(res[key], res[off], ids)
        out[off] = np.concatenate([[0], np.cumsum(cnt)]).astype(np.uint64)
    return out


def main_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    step, n_mapped, kind, threads, sample = run_cpu(a, "reference")
    for _ in range(a.warmup):
        step()
    ts = [step()[0] for _ in range(a.steps)]
    dt = sum(ts)
    v = n_mapped * a.steps / dt
    out = {
        "impl": "reference", "metric": "overlaps/s", "value": v, "unit": "overlaps/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": workload_name(a), "measured_on": sample,
                   "reference": "RavenLib construct.cc/pile.cc/overlap_utils.cc compiled "
                                "in place over the restated ram engine (ram is not "
                                "vendored upstream)" if kind == "reference" else
                                "oracle port (oracle/_ref absent)"},
        "cpu_baseline": {"value": v, "unit": "overlaps/s", "cores": threads, "kind": kind,
                         "sample": sample},
        "e2e": {"value": v, "unit": "overlaps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def main_ours(a):
    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from bench import synth
    from raven_b200 import distributed, engine

    # every rank holds the same read set (N>1: strong scaling of one job)
    rs = synth.make_reads(SEED, a.genome, a.reads, a.mean_len)
    # pinned host copies: the e2e leg uploads from these every step
    words = torch.from_numpy(rs.words.view(np.int64)).pin_memory()
    woff = torch.from_numpy(rs.word_off.view(np.int64)).pin_memory()
    lens = torch.from_numpy(rs.lens.view(np.int32)).pin_memory()

    class Pinned:
        pass

    prs = Pinned()
    prs.words = words.numpy().view(np.uint64)
    prs.word_off = woff.numpy().view(np.uint64)
    prs.lens = lens.numpy().view(np.uint32)
    prs.n = rs.n

    if world > 1:
        de = distributed.DistEngine(f"cuda:{local}", k=K, w=W)
        stream, eng = de.stream, de.engine
        eng.set_option("async_upload", 1)   # pinned host buffers that outlive every step
        de.upload(prs)
    else:
        stream = torch.cuda.current_stream()
        eng = engine.Engine(device=local, stream=stream.cuda_stream)
        eng.configure(K, W)
        eng.set_option("async_upload", 1)   # pinned host buffers that outlive every step
        eng.upload(prs)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def batch_bases(r):  # index batch size for --index-batches (0 = the reference's 2^32)
        if a.index_batches <= 1:
            return 0
        return -(-int(r.lens.astype(np.uint64).sum()) // a.index_batches)

    ib = batch_bases(prs)

    def step_resident():
        if world > 1:
            last.update(de.find_overlaps_and_create_piles(FREQ, KMAX, False, ib, fetch=False))
        else:
            eng.find_overlaps_and_create_piles(FREQ, KMAX, False, ib, fetch=False)

    def step_e2e():
        (de if world > 1 else eng).upload(prs)
        step_resident()
        # results are host-resident after the call (D2H inside the step)

    def timed(fn, steps):
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(steps):
            fn()
        ev1.record(stream)
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        barrier()
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(a.warmup):
        step_resident()
    sampler = ClockSampler(local) if rank == 0 else None
    eng.set_option("reset_stats", 1)
    ms_total = timed(step_resident, a.steps)
    st = eng.stats()          # counters of the LAST step (this rank's share)
    phases = eng.timings()    # device ms per phase of the LAST step
    launches_step = st["kernel_launches"]
    n_mapped = st["overlaps"]
    clocks = sampler.stop() if sampler else None
    if a.dump_outputs:        # the results of the LAST timed step (this rank's share)
        dump_outputs(a.dump_outputs,
                     distributed.CudaSteps(eng, f"cuda:{local}").stage1_results() if world > 1
                     else eng.stage1_results(),
                     DUMP_BYTES // world, f"_rank{rank}" if world > 1 else "")

    for _ in range(1):
        step_e2e()
    ms_e2e = timed(step_e2e, a.steps)

    tot = torch.tensor([float(n_mapped)], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    total_mapped = float(tot.item())

    # ---- parity on the CPU legs' sample, outside the timed region: the GPU path
    # (this rank's share at N>1) on the SAME reads the reference arm runs ----
    srs, s_n, s_g = cpu_sample(a)
    seng = engine.Engine(device=local)
    seng.configure(K, W)
    seng.upload(srs)
    s_ib = batch_bases(srs)
    s_single = seng.find_overlaps_and_create_piles(FREQ, KMAX, False, s_ib, fetch=True)
    parity = {"sample": f"{s_n} reads / {s_g / 1e6:.1f} Mbp genome ({srs.bases / 1e9:.3f} Gbp)",
              "sha256": result_sha256(s_single), "n_mapped": int(s_single["num_mapped"])}
    sample_ms = None
    if world > 1:
        de.upload(srs)
        s_share = de.find_overlaps_and_create_piles(FREQ, KMAX, False, s_ib, fetch=True)
        ok = same_result(s_share, share_of(s_single, rank, world))
        okt = torch.tensor([1 if ok else 0], device="cuda", dtype=torch.int32)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        parity["checked"] = (f"every rank's share of the {world}-GPU run ({de.exchange} exchange) "
                             "vs the single-GPU result on the sample")
        parity["identical"] = bool(okt.item())
        de.upload(prs)
    else:
        def sample_e2e():
            seng.upload(srs)
            seng.find_overlaps_and_create_piles(FREQ, KMAX, False, s_ib, fetch=True)
        for _ in range(2):
            sample_e2e()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            sample_e2e()
        sample_ms = 1e3 * (time.perf_counter() - t0) / a.steps
    seng.close()

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        # ---- roofline of the dominant kernel (by device time of the last step) ----
        own = {k: v for k, v in phases.items()}
        dom = max(own, key=own.get)
        alg = algorithmic_bytes(st)
        dom_bytes = alg.get(dom, 0.0)
        dom_ms = own[dom]
        achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        traffic = None
        prof = os.path.join(ROOT, "profiles", "traffic.json")
        tr = json.load(open(prof)) if os.path.exists(prof) else {}
        traffic = tr.get(dom)
        # the largest phase that is ONE kernel launch per step (the sort phase is a
        # partition + 6 radix passes + histograms) gets its own entry
        od = max((k for k in own if k != "index_sort"), key=own.get)
        od_ach = alg.get(od, 0.0) / (own[od] * 1e-3) / 1e9 if own[od] > 0 else 0.0
        own_roofline = {"kernel": od, "bound": "hbm", "achieved": od_ach, "peak": peak,
                        "unit": "GB/s", "frac": od_ach / peak,
                        "algorithmic_bytes_per_launch": alg.get(od, 0.0),
                        "ms_per_launch": own[od], "traffic": tr.get(od)}
        h2d = int(prs.words.nbytes + prs.word_off.nbytes + prs.lens.nbytes)
        if world > 1:  # bases of this rank's sketch range, lengths of all reads
            sb = distributed.sketch_bounds(prs.lens, world)
            h2d = int(8 * (prs.word_off[sb[1]] - prs.word_off[sb[0]])
                      + prs.word_off.nbytes + prs.lens.nbytes)
        if world > 1:
            res = distributed.CudaSteps(eng, f"cuda:{local}").stage1_results()  # this rank's share
            d2h = int(res["overlaps"].nbytes + res["ovl_off"].nbytes + res["pile"].nbytes)
        else:
            res = eng.find_overlaps_and_create_piles(FREQ, KMAX, False, ib, fetch=True)
            d2h = int(res["overlaps"].nbytes + res["ovl_off"].nbytes + res["pile"].nbytes
                      + n_mapped * 32)
        out = {
            "metric": "overlaps/s", "value": total_mapped * a.steps / (ms_total * 1e-3),
            "unit": "overlaps/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms_total / a.steps, "higher_is_better": True,
            "scaling": "strong",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload_name(a), "reads_per_gpu": rs.n // world,
                       "bases_per_gpu": int(rs.bases) // world,
                       "reads_total": rs.n, "overlaps_per_step": int(total_mapped),
                       "l2": "inputs (0.5 GB packed reads, 8.1 GB minimizer records) "
                             "exceed the 126 MB L2; no explicit flush",
                       "parallelism": "1 GPU" if world == 1 else
                       f"{world} ranks: reads sharded by id, index keys by value mod "
                       f"{world}, reads (queries, piles, lists) by id mod {world}; NCCL "
                       "all-to-all of minimizer records, of seed hits and of overlaps; "
                       "results stay sharded (d2h = this rank's share)",
                       "exchange": "-" if world == 1 else
                       f"{de.exchange} {getattr(de.comm, 'stats', '')}"},
            "clocks": clocks,
            "e2e": {"value": total_mapped * a.steps / (ms_e2e * 1e-3), "unit": "overlaps/s",
                    "ms_per_step": ms_e2e / a.steps, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches_step),
            "phases_ms": {k: round(v, 3) for k, v in sorted(phases.items())},
            "query_mbases_per_s": st["query_bases"] / 1e6 / (ms_total / a.steps * 1e-3),
            "index_mbases_per_s": st["index_bases"] / 1e6 / (ms_total / a.steps * 1e-3),
            "roofline": {"kernel": PHASE_KERNELS.get(dom, dom), "bound": "hbm",
                         "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)"
                         if peaks else "fallback 6650 GB/s (of fallback)",
                         "algorithmic_bytes_per_launch": dom_bytes, "ms_per_launch": dom_ms,
                         "traffic": traffic},
            "roofline_own": own_roofline,
            "phase_rooflines": {k: {"ms": round(own[k], 3),
                                    "algorithmic_gb": round(alg.get(k, 0.0) / 1e9, 3),
                                    "frac": round(alg.get(k, 0.0) / (own[k] * 1e-3) / 1e9 / peak, 4)
                                    if own[k] > 0 else None}
                                for k in sorted(own) if k in alg},
            "path_roofline": {"algorithmic_bytes": sum(alg.values()),
                              "achieved": sum(alg.values()) / (ms_total / a.steps * 1e-3) / 1e9,
                              "frac": sum(alg.values()) / (ms_total / a.steps * 1e-3) / 1e9 / peak},
        }
        if "trace_ms" in last:  # RVN_DIST_TRACE=1 (analysis run, not a bench value)
            out["dist_trace_ms"] = {k: round(v, 2) for k, v in last["trace_ms"].items()}
        if world == 1 and a.poa_windows > 0:
            out["poa"] = bench_poa(eng, a, peak, not a.no_cpu_baseline)
        if world == 1 and a.c3_reads > 0:
            out["poa"] = dict(out.get("poa", {}), c3=bench_c3(a, not a.no_cpu_baseline))
        if world == 1 and a.c5_reads > 0:
            out["c5"] = bench_c5(a, local, not a.no_cpu_baseline)
        if world == 1 and not a.no_cpu_baseline and a.index_batches <= 1:
            step, n_map_cpu, kind, threads, sample = run_cpu(a, "reference")
            dt, cpu_res = step()
            out["cpu_baseline"] = {"value": n_map_cpu / dt, "unit": "overlaps/s",
                                   "cores": threads, "kind": kind, "sample": sample,
                                   "seconds": dt}
            # same reads, same parameters: the GPU result must equal the CPU path's
            parity["checked"] = ("GPU stage-1 result (kept overlaps, list offsets, piles) vs "
                                 + ("oracle/_ref (reference construct.cc/pile.cc compiled in place)"
                                    if kind == "reference" else "oracle port")
                                 + " on the sample")
            parity["identical"] = bool(same_result(s_single, cpu_res)
                                       and int(s_single["num_mapped"]) == n_map_cpu)
            parity["cpu_sha256"] = result_sha256(cpu_res)
            gv = n_map_cpu / (sample_ms * 1e-3)
            out["same_config"] = {
                "workload": sample, "gpu_e2e_overlaps_per_s": gv,
                "gpu_e2e_ms": sample_ms, "cpu_overlaps_per_s": n_map_cpu / dt,
                "cpu_cores": threads, "ratio": gv / (n_map_cpu / dt),
                "note": "GPU (upload + stage 1 + results to host, wall clock) and the CPU "
                        "reference arm on the SAME reads; at 1/10 of C2 the GPU run is "
                        "dominated by fixed per-call costs"}
        out["parity"] = parity
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def poa_windows(n_windows):
    """C3-like consensus workload: 500-base windows, 30 ONT layers (10 % error) each,
    Phred block qualities; 512 distinct windows tiled to n_windows."""
    import numpy as np
    from raven_b200 import synth
    distinct = min(512, n_windows)
    w0 = synth.make_windows(n_windows=distinct, backbone_len=500, layers=30, seed=SEED % 1000)
    reps = max(1, n_windows // distinct)
    nseq, nb = int(w0["win_first"][-1]), int(w0["seq_off"][-1])
    w = dict(
        win_first=np.concatenate([w0["win_first"][:-1] + r * nseq for r in range(reps)]
                                 + [[reps * nseq]]).astype(np.uint32),
        seq_off=np.concatenate([w0["seq_off"][:-1] + np.uint64(r * nb) for r in range(reps)]
                               + [[reps * nb]]).astype(np.uint64),
        bases=np.tile(w0["bases"], reps), quals=np.tile(w0["quals"], reps),
        seq_begin=np.tile(w0["seq_begin"], reps), seq_end=np.tile(w0["seq_end"], reps))
    return w, w0, distinct * reps


def bench_poa(eng, a, peak, with_cpu):
    """POA windows/s (second headline of BASELINE.json): racon window consensus."""
    import torch
    w, w0, nw = poa_windows(a.poa_windows)
    for _ in range(2):
        eng.poa_batch(w, want_coverage=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    kernel_ms = 0.0
    cells = 0
    for _ in range(a.steps):
        r = eng.poa_batch(w, want_coverage=False)
        kernel_ms += eng.timings().get("poa", 0.0)
        cells = r["cells"]
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    bytes_in = int(w["bases"].nbytes + w["quals"].nbytes + w["seq_off"].nbytes
                   + w["seq_begin"].nbytes * 2 + w["win_first"].nbytes)
    out = {
        "metric": "POA windows/s", "unit": "windows/s",
        "workload": f"{nw} windows of 500 bases x 30 ONT layers (10% error), m=3 n=-5 g=-4, "
                    "trim, full (unbanded) DP like the reference's CPU path",
        "value": nw * a.steps / (kernel_ms * 1e-3) if kernel_ms else None,
        "e2e": {"value": nw * a.steps / dt, "unit": "windows/s",
                "h2d_bytes_per_step": bytes_in, "d2h_bytes_per_step": int(r["consensus"].nbytes)},
        "ms_per_step": 1e3 * dt / a.steps, "gcups": cells / (kernel_ms / a.steps * 1e-3) / 1e9
        if kernel_ms else None,
        "roofline": {"bound": "hbm", "achieved": bytes_in / (kernel_ms / a.steps * 1e-3) / 1e9
                     if kernel_ms else None, "peak": peak, "unit": "GB/s",
                     "note": "POA is latency/integer bound (graph surgery + DP in registers); "
                             "HBM fraction reported for completeness"},
    }
    if out["roofline"]["achieved"]:
        out["roofline"]["frac"] = out["roofline"]["achieved"] / peak
    if out["gcups"]:
        # SURVEY.md 8(d): integer-issue ceiling of a packed int16 DP on 148 SMs, ~10 TCUPS
        out["issue_bound"] = {"ceiling_gcups": 10000.0, "frac": out["gcups"] / 10000.0,
                              "ncu": "profiles/r01_poa_ncu.txt"}
    if with_cpu:
        import oracle_lib
        O = oracle_lib.Oracle()
        threads = os.cpu_count() or 1
        reps = max(1, (4 * threads) // 512 + 1)
        O.lib.orc_spoa_use_simd(1)  # AVX2 int16 rows + prefix-max, like upstream spoa's SIMD engine
        try:
            O.poa_batch(w0, threads=threads)
            t = time.perf_counter()
            for _ in range(reps):
                rc = O.poa_batch(w0, threads=threads)
            dtc = time.perf_counter() - t
        finally:
            O.lib.orc_spoa_use_simd(0)
        out["cpu_baseline"] = {"value": 512 * reps / dtc, "unit": "windows/s", "cores": threads,
                               "kind": "simd",
                               "sample": f"{512 * reps} of the same windows; restatement of "
                                         "racon::Window + spoa with an AVX2 int16 matrix fill "
                                         "(16 cells per instruction, prefix-max rows), one "
                                         "window per host thread",
                               "gcups": float(rc["cells"].sum()) * reps / dtc / 1e9}
    return out


def bench_c3(a, with_cpu):
    """C3-shaped polishing (BASELINE configs[2]: the C2 read model, one round, m=3 n=-5
    g=-4): windows cut by the REAL polisher - racon::Polisher facade: GPU mapping of
    the reads to draft contigs, host alignment paths + breaking points, GPU POA of
    every 500-base window - instead of synthetic windows."""
    from bench import synth
    from raven_b200 import polish
    n = min(a.c3_reads, a.reads)
    g = max(int(a.genome * n / max(a.reads, 1)), 8 * a.mean_len)
    reads = synth.make_reads(SEED + 1, g, n, a.mean_len)
    draft = synth.make_contigs(SEED + 1, g, contig_len=1_000_000)
    threads = os.cpu_count() or 1
    polish.polish(draft, reads, threads=threads)            # warm-up (allocations)
    _, st = polish.polish(draft, reads, threads=threads)
    out = {
        "workload": f"C3-shaped: {n} ONT reads (~{a.mean_len // 1000} kb, 40x) polished onto "
                    f"{draft.n} draft contigs ({g / 1e6:.1f} Mbp, ~1% error), one round, w=500 "
                    "m=3 n=-5 g=-4 trim, through the racon::Polisher facade",
        "windows": st["windows"], "polished_windows": st["polished_windows"],
        "value": st["polished_windows"] / st["poa_seconds"], "unit": "windows/s",
        "note": "value = polished windows / consensus phase (H2D of the window batch + POA "
                "kernels + D2H); e2e = the whole Polish call",
        "e2e": {"value": st["polished_windows"] / st["seconds"], "unit": "windows/s",
                "seconds": st["seconds"], "poa_seconds": st["poa_seconds"],
                "phases_s": {k: round(v, 3) for k, v in st["phases_s"].items()}},
    }
    if with_cpu:
        import oracle_lib
        O = oracle_lib.Oracle()
        ns = max(1, n // 8)  # bounded CPU sample: 1/8 of the reads over 1/8 of the genome
        gs = max(g // 8, 8 * a.mean_len)
        sreads = synth.make_reads(SEED + 2, gs, ns, a.mean_len)
        sdraft = synth.make_contigs(SEED + 2, gs, contig_len=1_000_000)
        O.lib.orc_spoa_use_simd(1)
        try:
            _, _, ost = O.polish(sdraft, sreads, threads=threads)
        finally:
            O.lib.orc_spoa_use_simd(0)
        _, gst = polish.polish(sdraft, sreads, threads=threads)
        out["cpu_baseline"] = {
            "value": float(ost[1]) / float(ost[2]), "unit": "windows/s (whole Polish call)",
            "cores": threads, "kind": "simd",
            "sample": f"{ns} reads / {gs / 1e6:.2f} Mbp of the same model; restatement of "
                      "racon/spoa/edlib with the AVX2 int16 POA fill, whole Polish call",
            "gpu_same_sample": {"value": gst["polished_windows"] / gst["seconds"],
                                "unit": "windows/s (whole Polish call)"}}
    return out


def bench_c5(a, local, with_cpu):
    """C5-shaped (BASELINE configs[4], one GPU's worth): PacBio HiFi reads ~15 kb,
    k=19 w=10 f=0.001 kMaxNumOverlaps=32, identity 0.95: stage 1
    (FindOverlapsAndCreatePiles) and the identity filter's edit distances
    (construct.cc:162-217) on the kept overlaps, batched on the device."""
    import numpy as np
    import torch
    from bench import synth
    from raven_b200 import engine
    n, mean = a.c5_reads, 15_000
    g = int(n * mean / 30)  # 30x
    rs = synth.make_reads(SEED + 5, g, n, mean, sub=0.002, ins=0.0015, dele=0.0015)
    eng = engine.Engine(device=local)
    eng.configure(19, 10)
    eng.upload(rs)
    for _ in range(2):
        eng.find_overlaps_and_create_piles(0.001, 32, False, fetch=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        eng.find_overlaps_and_create_piles(0.001, 32, False, fetch=False)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / a.steps
    st = eng.stats()
    res = eng.find_overlaps_and_create_piles(0.001, 32, False, fetch=True)
    o = res["overlaps"]
    o = o[o[:, 0] < o[:, 3]]  # each pair once (the lists hold both directions)
    ll, rl = o[:, 2] - o[:, 1], o[:, 5] - o[:, 4]
    longest = np.maximum(ll, rl).astype(np.float64)
    identity = 0.95
    limit = (np.floor((1 - identity) * longest) + 2).astype(np.int32)
    args = (o[:, 0], o[:, 1], ll, o[:, 3], o[:, 4], rl, o[:, 7], limit)
    eng.edit_distance_batch(*args)
    t0 = time.perf_counter()
    d = eng.edit_distance_batch(*args)
    dte = time.perf_counter() - t0
    score = 1.0 - d.astype(np.float64) / longest
    keep = (d >= 0) & ~(score < identity)
    out = {
        "workload": f"C5-shaped, one GPU: {n} synthetic HiFi reads ~15 kb over a "
                    f"{g / 1e6:.0f} Mbp genome (30x, 0.5% error), k=19 w=10 f=0.001 "
                    "kMaxNumOverlaps=32 identity=0.95",
        "stage1": {"value": st["overlaps"] / dt, "unit": "overlaps/s", "ms_per_step": 1e3 * dt,
                   "overlaps_per_step": int(st["overlaps"]),
                   "phases_ms": {k: round(v, 3) for k, v in sorted(eng.timings().items())}},
        "identity_filter": {"value": int(o.shape[0]) / dte, "unit": "alignments/s",
                            "pairs": int(o.shape[0]), "seconds": dte,
                            "mean_pair_bases": float(longest.mean()) if o.shape[0] else 0.0,
                            "kept_fraction": float(keep.mean()) if o.shape[0] else 0.0,
                            "gcups_equivalent": float((ll.astype(np.float64) * rl).sum()) / dte / 1e9},
    }
    if with_cpu and o.shape[0]:
        # host leg: the product's own edlib (raven_b200/host/edlib.cc, what the reference's
        # per-overlap edlibAlign call runs on), one thread, a bounded sample
        import ctypes as C
        import subprocess as sp
        sp.run(["make", "-C", os.path.join(ROOT, "tests", "cpp"), "host"], check=True,
               stdout=sp.DEVNULL)
        lib = C.CDLL(os.path.join(ROOT, "tests", "cpp", "_build", "libhost_edlib.so"))

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
        letters = np.frombuffer(b"ACGT", np.uint8)
        m = min(200, o.shape[0])
        pairs = []
        for x in o[:m]:
            a_ = rs.codes(int(x[0]))[int(x[1]):int(x[2])]
            b_ = rs.codes(int(x[3]))[int(x[4]):int(x[5])]
            if not x[7]:
                b_ = (3 - b_[::-1]).astype(np.uint8)
            pairs.append((letters[a_].tobytes(), letters[b_].tobytes()))
        t0 = time.perf_counter()
        same = True
        for i, (sa, sb) in enumerate(pairs):
            r = lib.edlibAlign(sa, len(sa), sb, len(sb), Cfg(-1, 0, 0, None, 0))
            if d[i] >= 0 and r.editDistance != d[i]:
                same = False
            if d[i] < 0 and r.editDistance <= limit[i]:
                same = False
            lib.edlibFreeAlignResult(r)
        dtc = time.perf_counter() - t0
        out["identity_filter"]["cpu_baseline"] = {
            "value": m / dtc, "unit": "alignments/s", "cores": 1, "kind": "port",
            "sample": f"the first {m} pairs, host bit-vector edlib (band doubling), exact "
                      "distance like edlibDefaultAlignConfig()"}
        out["identity_filter"]["parity"] = {"checked": f"{m} distances vs the host edlib",
                                            "identical": bool(same)}
    eng.close()
    return out


PHASE_KERNELS = {
    "index_sort": "index_sort (radix.cu: RadixHistogramKernel + OnesweepPass per digit; "
                  "index.cu: TierCount/TierScatter)",
    "sketch": "sketch (SketchFastKernel<5>)",
    "chain": "chain (SplitKernel + GroupChainKernel + PairChainKernel)",
    "probe": "probe (JoinProbeKernel: self-join over the sorted postings)",
}


def algorithmic_bytes(st, k=K):
    """SURVEY.md §8(d) / DESIGN.md §4: bytes each phase must move at minimum. A
    minimizer record is value + origin: 12 bytes while the value fits 32 bits
    (2k <= 30; §8(d) counted 16), 16 otherwise."""
    nb, nm, nk = st["index_bases"], st["index_records"], st["index_keys"]
    qb, qm, nh, no = st["query_bases"], st["query_records"], st["hits"], st["overlaps"]
    rec = 12.0 if 2 * k <= 30 else 16.0
    return {
        "sketch": 0.25 * nb + rec * nm,
        "micromize": rec * nm + rec * qm,
        "index_sort": 2 * rec * nm,
        "index_table": (rec - 8.0) * nm + 4.0 * nk,
        "filter": 4.0 * nk,
        "probe": rec * qm + rec * qm,
        "expand": 8.0 * nh + 16.0 * nh,
        "chain": 16.0 * nh + 32.0 * no,
        "pile": 2 * 2.0 * st["pile_bins"],
    }


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        main_reference(args)
    else:
        main_ours(args)
