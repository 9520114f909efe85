"""dbi_mg_search_unindexed_local: the unindexed search over a proteome sharded over several handles of one process.
Every rank digests its own shard, the candidates travel to the owners of their mass slices, and the union of the
ranks' hits must be the single-GPU answer: dbi_search_unindexed on one handle holding the whole proteome, the
oracle, and a sharded index built from the same shards.  The GPU cases put every rank on cuda:0, which runs every
kernel and exchange of the multi-GPU path on one device."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import dbindex_b200 as dbi
from dbindex_b200 import synth
from dbindex_b200.capi import DBI_ERANGE, DbiError, DbiHitBuffers, DbiHitCounts
from dbindex_b200.indexer import (DBIndexerException, DBIndexImpl, DBIndexSearchParams, DBIndexer, MassRange,
                                  _merge_hits, search_unindexed_chunked)
from oracle.oracle_py import Oracle

from .test_gpu_parity import _dup_proteome, check_sharded, hits_canonical
from .test_unindexed_search import EIGHT_SHIFTS_K4, _keys
from .util import PARAM_SETS

NCPU = os.cpu_count() or 1
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DBI_ENOTINIT, DBI_EALREADY, DBI_EINVAL = -1, -2, -3


def oracle(p, res, off):
    o = Oracle(p, threads=NCPU)
    o.add_proteins(res, off)
    assert o.build() == 0
    return o


# ---- CPU --------------------------------------------------------------------------------------------------

class ShardedStandIn:
    """search_unindexed of a stand-in sharded searcher: rank r answers for the oracle entries in its mass slice, and
    DBI_ERANGE names the largest per-rank count of entries inside the union of the batch's windows."""

    def __init__(self, o, world):
        self.o, self.mass = o, o.entries()["mass"]
        self.split = np.quantile(self.mass, np.arange(1, world) / world)
        self.world, self.calls = world, 0

    def search_unindexed(self, lo, hi, max_candidates=0):
        inside = np.zeros(len(self.mass), bool)
        for a, b in zip(lo, hi):
            inside |= (self.mass >= a) & (self.mass <= b)
        rank_of = np.searchsorted(self.split, self.mass, side="right")
        per_rank = np.bincount(rank_of[inside], minlength=self.world).astype(np.uint64)
        if max_candidates and per_rank.max() > max_candidates:
            e = DbiError(DBI_ERANGE, "over the cap", int(per_rank.max()))
            e.rank_candidates = per_rank
            raise e
        self.calls += 1
        parts = []
        for r in range(self.world):
            edges = np.concatenate(([-np.inf], self.split, [np.inf]))
            h = self.o.query_hits(np.maximum(lo, edges[r]), np.minimum(hi, np.nextafter(edges[r + 1], -np.inf)))
            n = len(h["mass"])
            h["hit_pep"] = np.arange(n, dtype=np.int64)
            h["counts"] = DbiHitCounts(len(lo), n, n, len(h["seq"]), len(h["prot_ids"]))
            parts.append((np.arange(len(lo)), h))
        return _merge_hits(parts, len(lo))


def test_chunked_search_over_a_sharded_searcher_answers_every_query_once_in_order():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = synth.synth_proteome(60, 8, median_len=300, min_len=5)
    o = oracle(p, res, off)
    _, _, lo, hi = synth.synth_queries(o.entries()["mass"], 400, 21, da_fraction=0.1, da_tol=0.5)
    lo[:5], hi[:5] = lo[10], hi[10]  # duplicates
    exp = o.query_hits(lo, hi)
    per_q = np.diff(exp["hit_off"].astype(np.int64))
    for world in (2, 3):
        for cap in (0, int(per_q.max()) * 3, int(per_q.max())):
            g = ShardedStandIn(o, world)
            got = search_unindexed_chunked(g, lo, hi, cap)
            assert g.calls >= (1 if cap == 0 else 2)
            assert np.array_equal(got["hit_off"], exp["hit_off"]), (world, cap)
            assert hits_canonical(got) == hits_canonical(exp), (world, cap)


def test_devices_need_unindexed_mode():
    p = dbi.default_params()
    with pytest.raises(DBIndexerException):
        DBIndexer(p, devices=[0, 0])
    assert DBIndexer(p, use_index=False, devices=[0, 0]).devices == [0, 0]


def test_java_downcall_matches_the_header():
    """DbiNative's descriptor of dbi_mg_search_unindexed_local against the C prototype (no JDK here)."""
    java = open(os.path.join(ROOT, "java/edu/scripps/yates/dbindex/gpu/DbiNative.java")).read()
    m = re.search(r'"dbi_mg_search_unindexed_local",\s*FunctionDescriptor\.of\(([^)]*)\)', java)
    assert m, "no downcall for dbi_mg_search_unindexed_local"
    kinds = [k.strip() for k in m.group(1).split(",")]
    hdr = open(os.path.join(ROOT, "include/dbindex_gpu.h")).read()
    proto = re.search(r"int dbi_mg_search_unindexed_local\(([^)]*)\);", hdr).group(1)
    to_java = lambda a: ("ADDRESS" if "*" in a else "JAVA_LONG" if "uint64_t" in a else "JAVA_INT")  # noqa: E731
    assert kinds == ["JAVA_INT"] + [to_java(a) for a in proto.split(",")]


# ---- GPU ------------------------------------------------------------------------------------------------

gpu = pytest.mark.gpu


def sharded(p, res, off, world):
    from dbindex_b200.multigpu import shard_proteins
    hs = []
    for r in range(world):
        g = dbi.GpuIndex(p)
        sres, soff, _ = shard_proteins(res, off, r, world)
        g.add_proteins(sres, soff)
        hs.append(g)
    return hs


def close_all(hs):
    for g in hs:
        g.close()


def search(hs, lo, hi, cap=0):
    from dbindex_b200.multigpu import search_unindexed_local
    return search_unindexed_local(hs, lo, hi, cap)


def raw_search(hs, lo, hi, cap=0):
    """dbi_mg_search_unindexed_local without the read: (status, counts[n], n_candidates[n])."""
    lib = dbi.load_library()
    lib.dbi_mg_search_unindexed_local.restype = C.c_int
    lib.dbi_mg_search_unindexed_local.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                                  C.c_void_p, C.c_void_p]
    lo = np.ascontiguousarray(lo, dtype=np.float64)
    hi = np.ascontiguousarray(hi, dtype=np.float64)
    n = len(hs)
    arr = (C.c_void_p * max(n, 1))(*[g._h if g is not None else None for g in hs])
    counts = (DbiHitCounts * max(n, 1))()
    n_cand = np.zeros(max(n, 1), dtype=np.uint64)
    rc = lib.dbi_mg_search_unindexed_local(arr, n, lo.ctypes.data, hi.ctypes.data, len(lo), cap, counts,
                                           n_cand.ctypes.data)
    return rc, counts, n_cand


def sum_stat(hs, k):
    return sum(g.stats()[k] for g in hs)


def check_equal(hs, g1, o, lo, hi):
    """sharded = dbi_search_unindexed on the whole proteome = oracle, with the candidate pipelines' totals equal"""
    got = search(hs, lo, hi)
    one = g1.search_unindexed(lo, hi)
    exp = o.query_hits(lo, hi)
    assert np.array_equal(got["hit_off"], exp["hit_off"]) and np.array_equal(one["hit_off"], exp["hit_off"])
    assert hits_canonical(got) == hits_canonical(one) == hits_canonical(exp)
    st1 = g1.stats()
    assert sum_stat(hs, "n_emitted") == st1["n_emitted"]
    assert sum_stat(hs, "n_entries") == st1["n_entries"]
    assert int(got["n_candidates"].sum()) == st1["n_emitted"]
    return got


def check_routed_build(p, res, off, world, lo, hi, got):
    """sharded search = dbi_mg_build_local + dbi_query_hits routed to the slice owners, on fresh handles"""
    from dbindex_b200.multigpu import build_local, route_queries, split_masses
    hs = sharded(p, res, off, world)
    try:
        build_local(hs)
        split = split_masses(hs[0], world)
        routed = [[] for _ in lo]
        for r, g in enumerate(hs):
            sel = route_queries(lo, hi, split, r, world)
            if len(sel):
                hc = hits_canonical(g.query_hits(lo[sel], hi[sel]))
                for k, q in enumerate(sel):
                    routed[q].extend(hc[k])
        assert [sorted(x) for x in routed] == hits_canonical(got)
    finally:
        close_all(hs)


@gpu
@pytest.mark.parametrize("name,world", [("cfg1_tryptic", 2), ("cfg2_mods", 2), ("cfg2_mods", 3), ("cfg2_mods", 4),
                                        ("cfg3_semi", 3), ("many_classes", 2), ("many_classes", 4),
                                        ("lysc_neg_mod", 3), ("mandatory_K_no_h2o", 4), ("filter_K2_mods", 2)])
def test_sharded_equals_single_gpu_and_oracle(name, world):
    p = dbi.default_params(**PARAM_SETS[name])
    res, off = _dup_proteome(600)
    o = oracle(p, res, off)
    _, _, lo, hi = synth.synth_queries(o.entries()["mass"], 300, 11, da_fraction=0.3)
    hs = sharded(p, res, off, world)
    try:
        with dbi.GpuIndex(p) as g1:
            g1.add_proteins(res, off)
            got = check_equal(hs, g1, o, lo, hi)
        assert got["counts"].n_hits > 0
    finally:
        close_all(hs)
    check_routed_build(p, res, off, world, lo, hi, got)


@gpu
@pytest.mark.parametrize("mods", ["cfg2_mods", "eight_shifts_k4"])
def test_zero_width_windows_at_entry_masses(mods):
    p = dbi.default_params(**(EIGHT_SHIFTS_K4 if mods == "eight_shifts_k4" else PARAM_SETS[mods]))
    res, off = _dup_proteome(150 if mods == "eight_shifts_k4" else 600)
    o = oracle(p, res, off)
    m = np.unique(o.entries()["mass"])
    if len(m) > 10_000:
        m = np.random.default_rng(5).choice(m, 10_000, replace=False)
    hs = sharded(p, res, off, 3)
    try:
        got = hits_canonical(search(hs, m, m))
    finally:
        close_all(hs)
    assert got == hits_canonical(o.query_hits(m, m))
    assert all(len(x) > 0 for x in got)


@gpu
def test_full_cfg2_equals_the_index():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = synth.config_proteome(2)
    with dbi.GpuIndex(p) as g:
        g.add_proteins(res, off)
        g.build()
        _, _, lo, hi = synth.synth_queries(np.zeros(0), 2000, 3)  # uniform masses ...
        _, _, lo2, hi2 = synth.synth_queries(g.fetch(0, g.stats()["n_entries"], with_ids=False)["mass"], 2000, 4)
        lo, hi = np.concatenate([lo, lo2]), np.concatenate([hi, hi2])  # ... and masses of the index
        ix = g.query_hits(lo, hi)
        n_entries = g.stats()["n_entries"]
    exp = hits_canonical(ix)
    for world in (2, 4):
        hs = sharded(p, res, off, world)
        try:
            got = search(hs, lo, hi)
            assert np.array_equal(got["hit_off"], ix["hit_off"]) and hits_canonical(got) == exp, world
            assert got["counts"].n_hits > 100_000
            assert sum_stat(hs, "n_entries") <= n_entries
        finally:
            close_all(hs)


@gpu
def test_batch_shapes():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = _dup_proteome(400)
    o = oracle(p, res, off)
    m = o.entries()["mass"]
    mid = float(np.median(m))
    hs = sharded(p, res, off, 3)
    g1 = dbi.GpuIndex(p)
    g1.add_proteins(res, off)
    try:
        empty = search(hs, np.zeros(0), np.zeros(0))
        assert empty["counts"].n_hits == 0 and empty["hit_off"].tolist() == [0]
        assert not empty["n_candidates"].any()
        misses = search(hs, np.array([10.0, 7000.0, 599.0]), np.array([20.0, 7999.0, 599.5]))
        assert misses["counts"].n_hits == 0 and not misses["n_candidates"].any()  # every rank has zero candidates
        inv = check_equal(hs, g1, o, np.array([mid + 1.0, 900.0]), np.array([mid - 1.0, 800.0]))
        assert inv["counts"].n_hits == 0 and not inv["n_candidates"].any()
        nan_lo, nan_hi = np.array([np.nan, 900.0, np.nan]), np.array([1000.0, np.nan, np.nan])
        nan = search(hs, nan_lo, nan_hi)
        assert hits_canonical(nan) == hits_canonical(g1.search_unindexed(nan_lo, nan_hi))
        lo = np.array([mid - 3.0, mid - 3.0, 0.0, 6500.0, 6100.0, m[0], m[-1], mid - 50.0, mid])
        hi = np.array([mid + 3.0, mid + 3.0, 700.0, 9000.0, 6200.0, m[0], m[-1], mid + 50.0, mid])
        check_equal(hs, g1, o, lo, hi)  # duplicates, lo = 0, above max_mass, the extreme entries
        check_equal(hs, g1, o, np.array([0.0]), np.array([8000.0]))  # every record is a candidate
        assert sum_stat(hs, "n_emitted") == o.counts()["n_emitted"]
        assert sum_stat(hs, "n_entries") == o.counts()["n_entries"]
    finally:
        close_all(hs + [g1])
    # a window that only one rank's slices reach: without mods every candidate of [m, m] has mass m
    p1 = dbi.default_params(**PARAM_SETS["cfg1_tryptic"])
    o1 = oracle(p1, res, off)
    m1 = o1.entries()["mass"]
    hs = sharded(p1, res, off, 3)
    try:
        for x in (m1[0], m1[len(m1) // 2], m1[-1]):
            one = search(hs, np.array([x]), np.array([x]))
            assert int((one["n_candidates"] > 0).sum()) == 1
            assert hits_canonical(one) == hits_canonical(o1.query_hits(np.array([x]), np.array([x])))
    finally:
        close_all(hs)


@gpu
def test_empty_shard_as_the_sharded_build():
    """A rank given no proteins: whatever dbi_mg_build_local does with it, the search does too."""
    from dbindex_b200.multigpu import build_local
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = _dup_proteome(300)
    n = len(off) - 1
    cut = n // 2

    def handles():
        parts = [(0, cut), (cut, cut), (cut, n)]  # rank 1 is empty
        hs = []
        for a, b in parts:
            g = dbi.GpuIndex(p)
            g.add_proteins(res[int(off[a]):int(off[b])], (off[a:b + 1] - off[a]).astype(np.uint64))
            hs.append(g)
        return hs

    o = oracle(p, res, off)
    _, _, lo, hi = synth.synth_queries(o.entries()["mass"], 200, 12, da_fraction=0.3)
    hs = handles()
    try:
        try:
            build_local(hs)
            build_rc = 0
        except DbiError as e:
            build_rc = e.code
    finally:
        close_all(hs)
    assert build_rc in (0, DBI_EINVAL)
    hs = handles()
    try:
        if build_rc == DBI_EINVAL:
            rc, _, _ = raw_search(hs, lo, hi)
            assert rc == DBI_EINVAL
        else:
            got = search(hs, lo, hi)
            assert hits_canonical(got) == hits_canonical(o.query_hits(lo, hi))
            assert hs[1].stats()["n_emitted"] == 0
    finally:
        close_all(hs)


@gpu
def test_candidate_cap():
    from dbindex_b200.multigpu import ShardedSearcher
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = _dup_proteome(400)
    o = oracle(p, res, off)
    _, _, lo, hi = synth.synth_queries(o.entries()["mass"], 300, 2, da_fraction=0.3)
    hs = sharded(p, res, off, 3)
    try:
        first = search(hs, lo, hi)
        per_rank = first["n_candidates"].copy()
        top = int(per_rank.max())
        assert top > 1
        with pytest.raises(DbiError) as ei:
            search(hs, lo, hi, top - 1)
        assert ei.value.code == DBI_ERANGE and ei.value.n_candidates == top
        assert np.array_equal(ei.value.rank_candidates, per_rank)
        for g in hs:  # no pending result on any handle
            with pytest.raises(DbiError) as ei:
                g.query_hits_read(DbiHitBuffers())
            assert ei.value.code == DBI_ENOTINIT
        again = search(hs, lo, hi, top)
        assert np.array_equal(again["n_candidates"], per_rank)
        exp = hits_canonical(o.query_hits(lo, hi))
        assert hits_canonical(again) == hits_canonical(first) == exp
        searcher = ShardedSearcher(hs)
        calls = []
        inner = searcher.search_unindexed
        searcher.search_unindexed = lambda *a, **k: calls.append(1) or inner(*a, **k)
        chunked = search_unindexed_chunked(searcher, lo, hi, max(2, top // 5))
        assert len(calls) > 2
        assert np.array_equal(chunked["hit_off"], first["hit_off"]) and hits_canonical(chunked) == exp
    finally:
        close_all(hs)


@gpu
def test_lifecycle():
    from dbindex_b200.multigpu import build_local, split_masses
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = _dup_proteome(400)
    o = oracle(p, res, off)
    _, _, lo, hi = synth.synth_queries(o.entries()["mass"], 200, 6, da_fraction=0.3)
    hs = sharded(p, res, off, 3)
    try:
        first = search(hs, lo, hi)
        assert all(g.stats()["algo_bytes"]["pack"] > 0 for g in hs)
        second = search(hs, lo, hi)
        assert all(g.stats()["algo_bytes"]["pack"] == 0 for g in hs), "the proteome was packed or pulled again"
        assert hits_canonical(first) == hits_canonical(second) == hits_canonical(o.query_hits(lo, hi))
        for g in hs:  # the handles stay unbuilt
            for call in (lambda: g.query_hits(lo, hi), lambda: g.lookup_peptides(["PEPTIDEK"])):
                with pytest.raises(DbiError) as ei:
                    call()
                assert ei.value.code == DBI_ENOTINIT
        # proteins added to the last rank are seen by the next search, with global ids after every other protein
        res2, off2 = synth.synth_proteome(40, 99, median_len=300, min_len=5)
        res2 = np.concatenate([res2, res[int(off[0]):int(off[1])]])  # a duplicate of protein 0 at the end
        off2 = np.append(off2, off2[-1] + (off[1] - off[0])).astype(np.uint64)
        hs[-1].add_proteins(res2, off2)
        o_all = oracle(p, np.concatenate([res, res2]), np.concatenate([off, off2[1:] + off[-1]]).astype(np.uint64))
        grown = search(hs, lo, hi)
        assert all(g.stats()["algo_bytes"]["pack"] > 0 for g in hs)
        assert hits_canonical(grown) == hits_canonical(o_all.query_hits(lo, hi))
        # a new call drops the pending results of the previous one
        rc, _, _ = raw_search(hs, lo[:50], hi[:50])
        assert rc == 0
        rc, counts, _ = raw_search(hs, lo[50:], hi[50:])
        assert rc == 0
        parts = [(np.arange(len(lo) - 50), g._read_hits(counts[r], None, None, True)) for r, g in enumerate(hs)]
        assert all(counts[r].nq == len(lo) - 50 for r in range(3))
        assert hits_canonical(_merge_hits(parts, len(lo) - 50)) == hits_canonical(o_all.query_hits(lo[50:], hi[50:]))
        for g in hs:
            with pytest.raises(DbiError) as ei:
                g.query_hits_read(DbiHitBuffers())
            assert ei.value.code == DBI_ENOTINIT
        # the normal sharded index after searches
        build_local(hs)
        check_sharded(hs, o_all, split_masses(hs[0], 3))
        rc, _, _ = raw_search(hs, lo, hi)
        assert rc == DBI_EALREADY
    finally:
        close_all(hs)


@gpu
def test_one_rank_and_bad_arguments():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = _dup_proteome(200)
    _, _, lo, hi = synth.synth_queries(np.zeros(0), 100, 7, da_fraction=0.5)
    with dbi.GpuIndex(p) as a, dbi.GpuIndex(p) as b:
        a.add_proteins(res, off)
        b.add_proteins(res, off)
        assert hits_canonical(search([a], lo, hi)) == hits_canonical(b.search_unindexed(lo, hi))
        assert a.stats()["n_emitted"] == b.stats()["n_emitted"]
        other = dbi.GpuIndex(dbi.default_params(**PARAM_SETS["cfg1_tryptic"]))
        try:
            for hs in ([a, a], [a, None], [a, other], []):
                rc, _, _ = raw_search(hs, lo, hi)
                assert rc == DBI_EINVAL, hs
            rc, _, _ = raw_search([a, b] * 9, lo, hi)  # more than DBI_MG_MAX_RANKS
            assert rc == DBI_EINVAL
        finally:
            other.close()


@gpu
@pytest.mark.parametrize("cap", [None, 40])
def test_mirror_sharded_unindexed_equals_indexed(cap):
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = _dup_proteome(150)
    seqs = [res[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(len(off) - 1)]
    defs = synth.deflines(len(seqs))
    idx = DBIndexImpl(DBIndexSearchParams(params=p, dataBaseName="idx.fasta"), proteins=(defs, seqs))
    un = DBIndexImpl(DBIndexSearchParams(params=p, dataBaseName="shidx.fasta", useIndex=False), proteins=(defs, seqs),
                     devices=[0, 0, 0])
    try:
        assert len(un.indexer.shards) == 3 and all(g.stats()["n_proteins"] > 0 for g in un.indexer.shards)
        for pid in (0, 1, len(seqs) // 2, len(seqs) - 1):
            assert un.getProteinSequenceById(pid) == seqs[pid]
        calls = []
        if cap is not None:
            un.indexer.max_candidates = cap
            inner = un.indexer._searcher.search_unindexed
            un.indexer._searcher.search_unindexed = lambda *a, **k: calls.append(1) or inner(*a, **k)
        exp = idx.indexer.index.fetch(0, idx.indexer.getNumberSequences(), with_ids=False)["mass"]
        picks = [float(exp[i]) for i in np.linspace(0, len(exp) - 1, 10).astype(int)]
        for m in picks + [1234.5678, 7990.0]:
            assert _keys(un.getSequences(m, 0.02)) == _keys(idx.getSequences(m, 0.02)), m
            assert _keys(un.indexer.getSequencesUsingPPMTolerance(m, 10.0)) == \
                _keys(idx.indexer.getSequencesUsingPPMTolerance(m, 10.0)), m
        rs = [MassRange(picks[3], 0.5), MassRange(picks[3] + 0.2, 0.5), MassRange(picks[7], 0.01)]
        assert _keys(un.getSequences(rs)) == _keys(idx.getSequences(rs))
        peps = [s.sequence for s in idx.getSequences(picks[5], 1.0) if not s.modPositions][:20]
        assert peps
        negatives = [peps[0][::-1], peps[0].lower(), peps[0][:-1], peps[0] + "K", "", "PEPTIDEXK"]
        for s in peps[:5] + negatives:
            assert un.getProteins(s) == idx.getProteins(s), s
        assert un.getProteins(peps + negatives) == idx.getProteins(peps + negatives)
        assert any(un.getProteins(peps))
        if cap is not None:
            assert len(calls) > 1
    finally:
        idx.close()
        un.close()
