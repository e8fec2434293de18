"""Host-side mirror of the reference's overlap interface over the C ABI.

``Engine`` keeps the names and argument meaning of the reference calls it
stands in for:

* ``minimize / filter / map``  ->  ``ram::MinimizerEngine::{Minimize,Filter,Map}``
  (call sites RavenLib/src/construct.cc:42-44,59-64,363,372,377-381)
* ``find_overlaps_and_create_piles``  ->  ``raven::FindOverlapsAndCreatePiles``
  (RavenLib/src/construct.cc:14-121; Python binding of the reference:
  PythonLib/src/ravenpy.cc:214-218)

Errors: the reference throws ``std::invalid_argument`` for a frequency outside
[0, 1]; here that is ``ValueError``.  Everything else the C ABI reports is a
``RuntimeError``.  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import OVLP, U16P, U32P, U64P, Overlap, Stats

_ERR = {-1: ValueError, -2: RuntimeError, -3: RuntimeError, -4: OverflowError}


def _arr(ptr, n, dtype):
    if n == 0:
        return np.zeros(0, dtype=dtype)
    addr = C.cast(ptr, C.c_void_p).value
    buf = (C.c_uint8 * (n * np.dtype(dtype).itemsize)).from_address(addr)
    return np.frombuffer(buf, dtype=dtype).copy()


class Engine:
    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.rvn_ctx_create(device, C.c_void_p(stream) if stream else None,
                                     C.byref(h))
        if rc != 0:
            raise RuntimeError(
                f"rvn_ctx_create failed ({rc}): no usable sm_100 CUDA device "
                "(raven_b200 has no CPU fallback)")
        self.h = h
        self.n_reads = 0
        self._keep = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.rvn_ctx_destroy(self.h)
            self.h = None

    __del__ = close

    def _check(self, rc):
        if rc != 0:
            msg = self.lib.rvn_last_error(self.h).decode()
            raise _ERR.get(rc, RuntimeError)(msg)

    # ---- ram::MinimizerEngine ----
    def configure(self, k=15, w=5, bandwidth=500, chain=4, matches=100, gap=10000):
        self._check(self.lib.rvn_engine_configure(self.h, k, w, bandwidth, chain,
                                                  matches, gap))

    def upload(self, rs, resident=None):
        """resident = (first, last): copy only the bases of those reads to the
        device (a rank of a partitioned run sketches its own range)."""
        words = np.ascontiguousarray(rs.words, dtype=np.uint64)
        woff = np.ascontiguousarray(rs.word_off, dtype=np.uint64)
        lens = np.ascontiguousarray(rs.lens, dtype=np.uint32)
        self._keep = (words, woff, lens)
        if resident is None:
            self._check(self.lib.rvn_reads_upload(
                self.h, words.ctypes.data_as(U64P), woff.ctypes.data_as(U64P),
                lens.ctypes.data_as(U32P), rs.n))
        else:
            self._check(self.lib.rvn_reads_upload_range(
                self.h, words.ctypes.data_as(U64P), woff.ctypes.data_as(U64P),
                lens.ctypes.data_as(U32P), rs.n, resident[0], resident[1]))
        self.n_reads = rs.n

    def minimize(self, first, last, minhash=False):
        self._check(self.lib.rvn_minimize(self.h, first, last, int(minhash)))

    def filter(self, frequency):
        occ = C.c_uint32(0)
        self._check(self.lib.rvn_filter(self.h, float(frequency), C.byref(occ)))
        return occ.value

    def map(self, first, last, avoid_equal=True, avoid_symmetric=True,
            minhash=False, want_filtered=False):
        self._check(self.lib.rvn_map(self.h, first, last, int(avoid_equal),
                                     int(avoid_symmetric), int(minhash),
                                     int(want_filtered)))
        o, off, n = OVLP(), U64P(), C.c_uint64(0)
        f, foff = U32P(), U64P()
        self._check(self.lib.rvn_map_results(self.h, C.byref(o), C.byref(off),
                                             C.byref(n), C.byref(f), C.byref(foff)))
        nr = last - first
        res = dict(overlaps=_arr(o, n.value * 8, np.uint32).reshape(-1, 8),
                   ovl_off=_arr(off, nr + 1, np.uint64))
        fo = _arr(foff, nr + 1, np.uint64)
        res["filt_off"] = fo
        res["filtered"] = _arr(f, int(fo[-1]) if want_filtered else 0, np.uint32)
        return res

    def map_external(self, words, length, read_id, avoid_equal=True, avoid_symmetric=True,
                     minhash=False, want_filtered=False):
        """Map one read that is not part of the uploaded set (construct.cc:59 with more
        than one index batch; assemble.cc:757,780) against the current index."""
        w = np.ascontiguousarray(words, dtype=np.uint64)
        self._check(self.lib.rvn_map_external(
            self.h, w.ctypes.data_as(U64P), int(length), int(read_id), int(avoid_equal),
            int(avoid_symmetric), int(minhash), int(want_filtered)))
        o, off, n = OVLP(), U64P(), C.c_uint64(0)
        f, foff = U32P(), U64P()
        self._check(self.lib.rvn_map_results(self.h, C.byref(o), C.byref(off),
                                             C.byref(n), C.byref(f), C.byref(foff)))
        fo = _arr(foff, 2, np.uint64)
        return dict(overlaps=_arr(o, n.value * 8, np.uint32).reshape(-1, 8),
                    filtered=_arr(f, int(fo[-1]) if want_filtered else 0, np.uint32))

    def map_hits(self, nr):
        g, p, off, n = U64P(), U64P(), U64P(), C.c_uint64(0)
        self._check(self.lib.rvn_map_hits(self.h, C.byref(g), C.byref(p),
                                          C.byref(off), C.byref(n)))
        return dict(group=_arr(g, n.value, np.uint64),
                    positions=_arr(p, n.value, np.uint64),
                    hit_off=_arr(off, nr + 1, np.uint64))

    def sketch(self, first, last, minhash=False):
        v, o, off, n = U64P(), U64P(), U64P(), C.c_uint64(0)
        self._check(self.lib.rvn_sketch(self.h, first, last, int(minhash),
                                        C.byref(v), C.byref(o), C.byref(off),
                                        C.byref(n)))
        return dict(value=_arr(v, n.value, np.uint64),
                    origin=_arr(o, n.value, np.uint64),
                    offsets=_arr(off, last - first + 1, np.uint64))

    def index_records(self):
        v, o, n, nk = U64P(), U64P(), C.c_uint64(0), C.c_uint64(0)
        self._check(self.lib.rvn_index_records(self.h, C.byref(v), C.byref(o),
                                               C.byref(n), C.byref(nk)))
        return dict(value=_arr(v, n.value, np.uint64),
                    origin=_arr(o, n.value, np.uint64), n_keys=nk.value)

    # ---- raven::Pile::AddLayers ----
    def pile_add_layers(self, data, bin_off, overlaps):
        d = np.ascontiguousarray(data, dtype=np.uint16).copy()
        off = np.ascontiguousarray(bin_off, dtype=np.uint64)
        o = np.ascontiguousarray(overlaps, dtype=np.uint32).reshape(-1, 8)
        self._check(self.lib.rvn_pile_add_layers(
            self.h, d.ctypes.data_as(U16P), off.ctypes.data_as(U64P), off.size - 1,
            C.cast(o.ctypes.data, OVLP), o.shape[0]))
        return d

    # ---- racon::Polisher consensus phase (racon::Window + spoa) ----
    def poa_batch(self, w, m=3, n=-5, g=-4, trim=True, tgs=True, want_coverage=True):
        """Consensus of a flat batch of windows (layout: synth.make_windows)."""
        wf = np.ascontiguousarray(w["win_first"], dtype=np.uint32)
        so = np.ascontiguousarray(w["seq_off"], dtype=np.uint64)
        ba = np.ascontiguousarray(w["bases"], dtype=np.uint8)
        qu = None if w.get("quals") is None else np.ascontiguousarray(w["quals"], dtype=np.uint8)
        sb = np.ascontiguousarray(w["seq_begin"], dtype=np.uint32)
        se = np.ascontiguousarray(w["seq_end"], dtype=np.uint32)
        nw = wf.size - 1
        self._check(self.lib.rvn_poa_batch(
            self.h, nw, wf.ctypes.data_as(U32P), so.ctypes.data_as(U64P),
            ba.ctypes.data_as(C.c_char_p),
            qu.ctypes.data_as(C.c_char_p) if qu is not None else None,
            sb.ctypes.data_as(U32P), se.ctypes.data_as(U32P), m, n, g, int(trim), int(tgs),
            int(want_coverage)))
        cons, off, st, cov = C.c_void_p(), U64P(), C.POINTER(C.c_uint8)(), U32P()
        cells = C.c_uint64(0)
        self._check(self.lib.rvn_poa_results(self.h, C.byref(cons), C.byref(off),
                                             C.byref(st), C.byref(cov), C.byref(cells)))
        cons_off = _arr(off, nw + 1, np.uint64)
        total = int(cons_off[-1]) if nw else 0
        return dict(consensus=_arr(cons, total, np.uint8), cons_off=cons_off,
                    status=_arr(st, nw, np.uint8),
                    coverage=_arr(cov, total if want_coverage else 0, np.uint32),
                    cells=cells.value)

    def kmer_complexity(self, read_index, positions, kmer_len):
        """Pile::AddKmers' low-complexity test (pile.cc:64-120): 1 = bin gets marked."""
        ri = np.ascontiguousarray(read_index, dtype=np.uint32)
        po = np.ascontiguousarray(positions, dtype=np.uint32)
        keep = np.zeros(ri.size, dtype=np.uint8)
        self._check(self.lib.rvn_kmer_complexity(
            self.h, ri.ctypes.data_as(U32P), po.ctypes.data_as(U32P), ri.size, kmer_len,
            keep.ctypes.data_as(C.POINTER(C.c_uint8))))
        return keep

    # ---- raven::FindOverlapsAndCreatePiles ----
    def find_overlaps_and_create_piles(self, freq=0.001, max_overlaps=32,
                                       use_minhash=False, index_batch_bases=0,
                                       query_batch_bases=0, fetch=True):
        self._check(self.lib.rvn_find_overlaps_and_create_piles(
            self.h, float(freq), max_overlaps, int(use_minhash), index_batch_bases,
            query_batch_bases))
        return self.stage1_results() if fetch else None

    def stage1_results(self):
        """Host copies of the last find_overlaps_and_create_piles call's results."""
        o, off, p, poff, nm = OVLP(), U64P(), U16P(), U64P(), C.c_uint64(0)
        self._check(self.lib.rvn_stage1_results(self.h, C.byref(o), C.byref(off),
                                                C.byref(p), C.byref(poff),
                                                C.byref(nm)))
        n = self.n_reads
        ovl_off = _arr(off, n + 1, np.uint64)
        pile_off = _arr(poff, n + 1, np.uint64)
        return dict(overlaps=_arr(o, int(ovl_off[-1]) * 8, np.uint32).reshape(-1, 8),
                    ovl_off=ovl_off, pile=_arr(p, int(pile_off[-1]), np.uint16),
                    pile_off=pile_off, num_mapped=nm.value)

    # ---- edlibAlign(..., edlibDefaultAlignConfig()) of the identity filter ----
    def edit_distance_batch(self, lhs_read, lhs_begin, lhs_len, rhs_read, rhs_begin, rhs_len,
                            strand, limit=None):
        """Global edit distances of substring pairs of the uploaded reads
        (construct.cc:176-199): -1 where the distance exceeds limit[i] >= 0."""
        a = [np.ascontiguousarray(x, dtype=np.uint32)
             for x in (lhs_read, lhs_begin, lhs_len, rhs_read, rhs_begin, rhs_len)]
        st = np.ascontiguousarray(strand, dtype=np.uint8)
        lim = None if limit is None else np.ascontiguousarray(limit, dtype=np.int32)
        out = np.zeros(a[0].size, dtype=np.int32)
        self._check(self.lib.rvn_edit_distance_batch(
            self.h, a[0].size, *[x.ctypes.data_as(U32P) for x in a],
            st.ctypes.data_as(C.POINTER(C.c_uint8)),
            None if lim is None else lim.ctypes.data_as(C.POINTER(C.c_int32)),
            out.ctypes.data_as(C.POINTER(C.c_int32))))
        return out

    def stage1_pile_regions(self, coverage=4):
        """Pile::FindValidRegion(coverage) + FindMedian (pile.cc:122-172) of the piles the
        last stage-1 call left on the device: begin, end (bins), median, invalid per read."""
        n = self.n_reads
        b, e = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
        m, inv = np.zeros(n, np.uint16), np.zeros(n, np.uint8)
        self._check(self.lib.rvn_stage1_pile_regions(
            self.h, coverage, b.ctypes.data_as(U32P), e.ctypes.data_as(U32P),
            m.ctypes.data_as(U16P), inv.ctypes.data_as(C.POINTER(C.c_uint8))))
        return dict(begin=b, end=e, median=m, invalid=inv)

    def align_breaking_points(self, q_read, q_begin, q_len, strand, t_read, t_begin, t_len,
                              window=500):
        """racon's read-to-target alignments + window cuts (polish.cc:43-51): distances,
        slot offsets (n + 1) and the breaking points, one row (first target, first
        query, last target + 1, last query + 1) per window a target substring touches."""
        a = [np.ascontiguousarray(x, dtype=np.uint32)
             for x in (q_read, q_begin, q_len, t_read, t_begin, t_len)]
        st = np.ascontiguousarray(strand, dtype=np.uint8)
        tb, tl = a[4].astype(np.int64), a[5].astype(np.int64)
        wins = np.where(tl > 0, (tb + tl - 1) // window - tb // window + 1, 0)
        off = np.concatenate([[0], np.cumsum(wins)]).astype(np.uint64)
        dist = np.zeros(a[0].size, dtype=np.int32)
        bp = np.zeros((int(off[-1]), 4), dtype=np.uint32)
        self._check(self.lib.rvn_align_breaking_points(
            self.h, a[0].size, a[0].ctypes.data_as(U32P), a[1].ctypes.data_as(U32P),
            a[2].ctypes.data_as(U32P), st.ctypes.data_as(C.POINTER(C.c_uint8)),
            a[3].ctypes.data_as(U32P), a[4].ctypes.data_as(U32P), a[5].ctypes.data_as(U32P),
            window, off.ctypes.data_as(U64P), dist.ctypes.data_as(C.POINTER(C.c_int32)),
            bp.ctypes.data_as(U32P)))
        return dist, off, bp

    def debug_sort_pairs(self, keys, vals=None, begin_bit=0, end_bit=None, descending=False):
        """The engine's stable radix sort (csrc/radix.cu) on host arrays; returns copies."""
        k = np.ascontiguousarray(keys).copy()
        v = None if vals is None else np.ascontiguousarray(vals).copy()
        end_bit = 8 * k.itemsize if end_bit is None else end_bit
        self._check(self.lib.rvn_debug_sort_pairs(
            self.h, k.itemsize, 0 if v is None else v.itemsize, k.ctypes.data_as(C.c_void_p),
            None if v is None else v.ctypes.data_as(C.c_void_p), k.size, begin_bit, end_bit,
            int(descending)))
        return k, v

    # ---- bookkeeping ----
    def set_option(self, name, value):
        self._check(self.lib.rvn_set_option(self.h, name.encode(), int(value)))

    def stats(self):
        s = Stats()
        self._check(self.lib.rvn_get_stats(self.h, C.byref(s)))
        return {n: getattr(s, n) for n, _ in Stats._fields_ if n != "reserved"}

    def timings(self):
        names = C.POINTER(C.c_char_p)()
        ms = C.POINTER(C.c_float)()
        n = C.c_uint32(0)
        self._check(self.lib.rvn_get_timings(self.h, C.byref(names), C.byref(ms),
                                             C.byref(n)))
        out = {}
        for i in range(n.value):
            out[names[i].decode()] = out.get(names[i].decode(), 0.0) + ms[i]
        return out
