"""Batches of spectra on a sharded index and in the sharded unindexed search: dbi_mg_query_spectra_local,
dbi_mg_search_unindexed_spectra_local and the rank-level dbi_mg_spectra_stops + dbi_mg_query_spectra.  For every
spectrum the union of the ranks' answers must be what dbi_query_spectra returns on one handle holding the whole
index.  The PPM walk is the new part: its probes are spread over the ranks by mass, rank r computes K_r (where its
share of the walk ends) and the walk ends at min_r K_r.  The GPU cases put every rank on cuda:0, as
test_sharded_unindexed.py does."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import dbindex_b200 as dbi
from dbindex_b200 import synth
from dbindex_b200.capi import DBI_ERANGE, DBI_TOL_DA, DBI_TOL_PPM, DbiError, DbiHitBuffers, DbiHitCounts
from dbindex_b200.indexer import (PRECISION, DBIndexer, MassRange, _merge_hits, search_unindexed_spectra_chunked,
                                  tolerance_in_dalton)
from dbindex_b200.multigpu import slice_owner

from .test_gpu_parity import _dup_proteome, hits_canonical
from .test_spectrum_batch import (ISO, StandIn, dalton_spectra, expected_intervals, flatten, host_probe_loop,
                                  out_of_buckets, per_spectrum, ppm_expected, short)
from .util import PARAM_SETS, pack

NCPU = os.cpu_count() or 1
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DBI_ENOTINIT, DBI_EALREADY, DBI_EINVAL = -1, -2, -3
U64_MAX = (1 << 64) - 1


# ---- CPU ------------------------------------------------------------------------------------------------------

def single_stop(entries, m, ppm, f):
    """K of the reference walk (spec_probe_kernel): the index of the first probe it does not take."""
    u, k = m + tolerance_in_dalton(m, ppm), 0
    while True:
        if not (u - tolerance_in_dalton(u, ppm) < m) or u < 0.0 or out_of_buckets(u, f) or u not in entries:
            return k
        nu = u + PRECISION
        if nu == u:
            return k + 1
        u, k = nu, k + 1


def rank_stop(local, split, rank, world, m, ppm, f):
    """K_r as K14s computes it (spec_stop_kernel), early end included."""
    n_slices = len(split) + 1
    mine = [int(slice_owner(s, n_slices, world)) == rank for s in range(n_slices)]
    p1 = ppm / 1e6 + 1.0
    bound = (m * p1) * (1.0 + 2.0 ** -40) if m > 0.0 and p1 > 0.0 else float("inf")
    u, k = m + tolerance_in_dalton(m, ppm), 0
    while True:
        if not (u - tolerance_in_dalton(u, ppm) < m) or u < 0.0 or out_of_buckets(u, f):
            return k
        sl = int(np.searchsorted(split, u, side="right"))
        if mine[sl]:
            if u not in local:
                return k
        else:
            nxt = [t for t in range(sl + 1, n_slices) if mine[t]]
            if not nxt or split[nxt[0] - 1] > bound:
                return U64_MAX
        nu = u + PRECISION
        if nu == u:
            return k + 1
        u, k = nu, k + 1


def probes(m, ppm, n):
    u = [m + tolerance_in_dalton(m, ppm)]
    for _ in range(n - 1):
        u.append(u[-1] + PRECISION)
    return u


def test_min_of_rank_stops_is_the_single_walk():
    """min_r K_r == K on random entry sets (runs of present probes with gaps), random contiguous and folded cuts,
    cuts placed on probe masses and between them."""
    rng = np.random.default_rng(17)
    checked = walked = 0
    for trial in range(300):
        ppm = float(rng.choice([5.0, 10.0, 50.0, -50.0, 300.0]))
        m = float(rng.uniform(500, 7900))
        f = int(rng.choice([0, 3, 8]))
        us = probes(m, ppm, 40)
        present = rng.random(40) < 0.85
        entries = set(u for u, keep in zip(us, present) if keep) | set(rng.uniform(400, 8000, 20).tolist())
        world = int(rng.integers(1, 6))
        n_slices = world * int(rng.choice([1, 2])) if world > 1 else 1
        cand = us[:20] + [(a + b) / 2 for a, b in zip(us[:20], us[1:21])] + rng.uniform(400, 8000, 5).tolist()
        split = np.sort(rng.choice(cand, n_slices - 1, replace=False)) if n_slices > 1 else np.zeros(0)
        ent = np.array(sorted(entries))
        sl = np.searchsorted(split, ent, side="right")
        owner = slice_owner(sl, n_slices, world)
        ks = [rank_stop(set(ent[owner == r].tolist()), split, r, world, m, ppm, f) for r in range(world)]
        k = single_stop(entries, m, ppm, f)
        assert min(ks) == k, (trial, ks, k)
        checked += 1
        walked += k > 1
    assert checked == 300 and walked > 50


def test_java_downcalls_match_the_header():
    """DbiNative's descriptors of the two _local spectrum calls against the C prototypes (no JDK here)."""
    java = open(os.path.join(ROOT, "java/edu/scripps/yates/dbindex/gpu/DbiNative.java")).read()
    hdr = open(os.path.join(ROOT, "include/dbindex_gpu.h")).read()
    to_java = lambda a: ("ADDRESS" if "*" in a else "JAVA_LONG" if "uint64_t" in a else "JAVA_INT")  # noqa: E731
    for name in ("dbi_mg_query_spectra_local", "dbi_mg_search_unindexed_spectra_local"):
        m = re.search(r'"%s",\s*FunctionDescriptor\.of\(([^)]*)\)' % name, java)
        assert m, f"no downcall for {name}"
        kinds = [k.strip() for k in m.group(1).split(",")]
        proto = re.search(r"int %s\(([^)]*)\);" % name, hdr).group(1)
        assert kinds == ["JAVA_INT"] + [to_java(a) for a in proto.split(",")], name


class ShardedSpectraStandIn(StandIn):
    """StandIn's answers, with the candidates spread over `world` ranks by mass: DBI_ERANGE names the largest
    per-rank count (10 per range) and carries the per-rank counts, as ShardedSearcher does."""

    def __init__(self, world):
        super().__init__()
        self.world = world

    def search_unindexed_spectra(self, mass, tol, range_off=None, tol_mode=0, index_factor=0, max_candidates=0):
        per_rank = np.bincount(np.minimum((np.asarray(mass) // 500).astype(np.int64) % self.world, self.world - 1),
                               minlength=self.world).astype(np.uint64) * 10
        if max_candidates and per_rank.max() > max_candidates:
            e = DbiError(DBI_ERANGE, "over the cap", int(per_rank.max()))
            e.rank_candidates = per_rank
            raise e
        return super().search_unindexed_spectra(mass, tol, range_off, tol_mode, index_factor, 0)


@pytest.mark.parametrize("mode", [DBI_TOL_DA, DBI_TOL_PPM])
def test_spectrum_chunker_over_a_sharded_searcher(mode):
    rng = np.random.default_rng(8)
    n = 60
    if mode == DBI_TOL_DA:
        off = np.concatenate(([0], np.cumsum(rng.integers(0, 6, n)))).astype(np.uint64)
        mass = rng.uniform(500, 3000, int(off[-1]))
    else:
        off, mass = None, rng.uniform(500, 3000, n)
    tol = np.full(len(mass), 0.01)
    stand = ShardedSpectraStandIn(3)
    got = search_unindexed_spectra_chunked(stand, mass, tol, off, mode, 8, 40)
    assert len(stand.calls) > 2
    whole = StandIn().search_unindexed_spectra(mass, tol, off, mode, 8, 0)
    assert np.array_equal(got["hit_off"], whole["hit_off"])
    assert np.array_equal(got["mass"].view(np.uint64), whole["mass"].view(np.uint64))
    assert sum(len(co) - 1 for _, co in stand.calls) == n


# ---- GPU ------------------------------------------------------------------------------------------------------

gpu = pytest.mark.gpu


def oracle(p, res, off):
    from oracle.oracle_py import Oracle
    o = Oracle(p, threads=NCPU)
    o.add_proteins(res, off)
    assert o.build() == 0
    return o


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
        if g is not None:
            g.close()


def raw_local(fn, hs, mass, tol, off, ns, mode, f, extra=()):
    """One of the two _local calls without the read: (status, counts[n], n_candidates[n])."""
    lib = dbi.load_library()
    n = len(hs)
    arr = (C.c_void_p * max(n, 1))(*[g._h if g is not None else None for g in hs])
    counts = (DbiHitCounts * max(n, 1))()
    n_cand = np.zeros(max(n, 1), dtype=np.uint64)
    ptr = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)  # noqa: E731
    f_ = getattr(lib, fn)
    f_.restype = C.c_int
    if fn == "dbi_mg_query_spectra_local":
        f_.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int,
                       C.c_void_p]
        rc = f_(arr, n, ptr(mass), ptr(tol), ptr(off), ns, mode, f, counts)
    else:
        f_.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int,
                       C.c_uint64, C.c_void_p, C.c_void_p]
        rc = f_(arr, n, ptr(mass), ptr(tol), ptr(off), ns, mode, f, int(extra[0]) if extra else 0, counts,
                n_cand.ctypes.data)
    return rc, counts, n_cand


def nothing_pending(hs):
    for g in hs:
        with pytest.raises(DbiError) as ei:
            g.query_hits_read(DbiHitBuffers())
        assert ei.value.code == DBI_ENOTINIT


def ppm_masses(rng, masses, split, p):
    """Entry masses, uniform masses, and masses at, next to and straddling every cut (window across a cut, u_0 at
    the cut)."""
    ms = list(rng.choice(masses, 150)) + list(rng.uniform(p.min_mass, p.max_mass, 50))
    for c in split:
        c = float(c)
        ms += [c, np.nextafter(c, -np.inf), np.nextafter(c, np.inf), c - 0.001, c + 0.001]
        ms += [c / (1 + 10e-6 / (1 + 10e-6)), c / (1 + 50e-6 / (1 + 50e-6))]  # u_0 ~ c at 10 / 50 ppm
        near = masses[np.searchsorted(masses, c) - 2:np.searchsorted(masses, c) + 2]
        ms += [float(x) for x in near]
    return np.array([m for m in ms if m > 0], np.float64)


@gpu
@pytest.mark.parametrize("name,world", [("cfg1_tryptic", 2), ("cfg2_mods", 2), ("cfg2_mods", 3), ("cfg2_mods", 4),
                                        ("cfg3_semi", 3), ("lysc_neg_mod", 3), ("mandatory_K_no_h2o", 4)])
def test_sharded_index_equals_one_handle_and_oracle(name, world):
    from dbindex_b200.multigpu import build_local, query_spectra_local, split_masses
    p = dbi.default_params(**PARAM_SETS[name])
    res, off = _dup_proteome(300)
    o = oracle(p, res, off)
    oe = o.entries()
    hs = sharded(p, res, off, world)
    try:
        build_local(hs)
        split = split_masses(hs[0], world)
        assert len(split) == (2 * world if p.n_mods else world) - 1
        with dbi.GpuIndex(p) as g1:
            g1.add_proteins(res, off)
            g1.build()
            masses = oe["mass"]
            rng = np.random.default_rng(world)
            spectra = dalton_spectra(rng, masses, p.max_mass, 200)
            mass, tol, roff = flatten(spectra)
            for f in (8, 0):
                got = hits_canonical(query_spectra_local(hs, mass, tol, roff, DBI_TOL_DA, f))
                assert got == hits_canonical(g1.query_spectra(mass, tol, roff, DBI_TOL_DA, f)), f
                lo, hi, sid = expected_intervals(spectra, f)
                assert got == per_spectrum(o.query_hits(lo, hi), sid, len(spectra)), f
            ms = ppm_masses(rng, masses, split, p)
            for ppm in (5.0, 10.0, 50.0):
                tl = np.full(len(ms), ppm)
                got = hits_canonical(query_spectra_local(hs, ms, tl, None, DBI_TOL_PPM, 8))
                assert got == hits_canonical(g1.query_spectra(ms, tl, None, DBI_TOL_PPM, 8)), ppm
                got0 = hits_canonical(query_spectra_local(hs, ms, tl, None, DBI_TOL_PPM, 0))
                assert short(got0) == [ppm_expected(o, oe, float(m), ppm) for m in ms], ppm
            assert any(len(x) for x in got0)
    finally:
        close_all(hs)


WALK_PPM = 50.0
EDGE = 7997.9999985 / (1 + tolerance_in_dalton(1.0, WALK_PPM))  # index factor 3: u_0, u_1 pass, u_2 fails
PLAN = {1000.0: 0, 1500.0: 1, 2000.0: 2, 4000.0: 5, 3000.0: -2, EDGE: 3}  # -2: u_0, u_1, gap, u_3
NEG = (5000.0, -50.0)  # inverted window: u_0 is a probe of its own (probe0), walk u_0, u_1, u_2


def walk_records():
    recs, walks = [], {}
    for m, k in PLAN.items():
        us = probes(m, WALK_PPM, 7)
        take = us[:k + 1] if k >= 0 else [us[0], us[1], us[3]]
        recs += take + [m]
        walks[m] = us
    us = probes(NEG[0], NEG[1], 4)
    recs += us[:3] + [NEG[0]]
    walks[NEG[0]] = us
    return np.array(recs, np.float64), walks


def from_records(p, seqs, recs, keep=None):
    """A handle indexing records recs[keep] (all: keep None); record i is the peptide at offset i % 16 of length
    2 + i % 5 whichever handle holds it, so that the ranks' records are the whole handle's records."""
    g = dbi.GpuIndex(p)
    g.add_proteins(*pack(seqs))
    i = np.arange(len(recs)) if keep is None else np.nonzero(keep)[0]
    n = len(i)
    mass = np.ascontiguousarray(recs[i], np.float64)
    prot = np.zeros(max(n, 1), np.uint32)
    off = np.zeros(max(n, 1), np.uint32)
    ln = np.full(max(n, 1), 2, np.uint16)
    off[:n] = i % 16
    ln[:n] += (i % 5).astype(np.uint16)
    rc = g.lib.dbi_build_from_records(g._h, mass.ctypes.data_as(C.c_void_p), prot.ctypes.data_as(C.c_void_p),
                                      off.ctypes.data_as(C.c_void_p), ln.ctypes.data_as(C.c_void_p), n)
    assert rc == 0, g.lib.dbi_last_error()
    return g


def walk_cases(walks):
    """(label, cuts, n_slices, world): every probe of a walk on another rank, a gap owned by a third rank, cuts
    exactly at probe masses, folded owners, the bucket-rule stop and the probe0 walk."""
    mid = lambda us, a, b: [(x + y) / 2 for x, y in zip(us[a:b], us[a + 1:b + 1])]  # noqa: E731
    cases = []
    for m, k in list(PLAN.items()) + [(NEG[0], 2)]:
        us = walks[m]
        between = mid(us, 0, max(abs(k), 1) + 1)  # u_0 | u_1 | ... | u_k | u_{k+1}
        if k == 0:
            between = [(m + us[0]) / 2, between[0]]  # the window entry, u_0 and u_1 on three ranks
        cases.append((f"between {m} ({k})", between, len(between) + 1, len(between) + 1))
        cases.append((f"at probes {m}", us[1:max(abs(k), 1) + 2], max(abs(k), 1) + 2, max(abs(k), 1) + 2))
    us = walks[4000.0]
    cases.append(("folded 4000", mid(us, 0, 5), 6, 3))
    cases.append(("folded 3000 gap", [walks[1500.0][0]] + mid(walks[3000.0], 0, 3) + [6000.0], 6, 3))
    cases.append(("one rank", [], 1, 1))
    return cases


@gpu
def test_walks_across_ranks_from_records():
    from dbindex_b200.multigpu import owned_mask
    p = dbi.default_params(min_mass=0.0, max_mass=8000.0)
    seqs = ["PEPTIDEK" * 3]
    recs, walks = walk_records()
    ms = np.array(list(PLAN) + [NEG[0]], np.float64)
    ppm = np.array([WALK_PPM] * len(PLAN) + [NEG[1]], np.float64)
    whole = from_records(p, seqs, recs)
    per_rank_fails = 0
    try:
        exp = {f: hits_canonical(whole.query_spectra(ms, ppm, None, DBI_TOL_PPM, f)) for f in (3, 0)}
        for f in (3, 0):
            assert exp[f] == [host_probe_loop(whole, float(m), float(q), f) for m, q in zip(ms, ppm)]
        # u_0 of the inverted window is a probe of its own (probe0)
        assert len(exp[0][-1]) == 3 and [len(x) for x in exp[0][:len(PLAN)]] == [2, 3, 4, 7, 3, 5]
        for label, cuts, n_slices, world in walk_cases(walks):
            split = np.array(cuts, np.float64)
            assert np.all(np.diff(split) > 0), label
            hs = [from_records(p, seqs, recs, owned_mask(recs, split, r, world)) for r in range(world)]
            try:
                for f in (3, 0):
                    stops = [g.mg_spectra_stops(ms, ppm, split, r, world, f) for r, g in enumerate(hs)]
                    kmin = np.minimum.reduce(stops)
                    assert not np.any(kmin == np.uint64(U64_MAX)), label
                    q = np.arange(len(ms))
                    got = _merge_hits([(q, g.mg_query_spectra(ms, ppm, None, DBI_TOL_PPM, f, stop=kmin))
                                       for g in hs], len(ms))
                    assert hits_canonical(got) == exp[f], (label, f)
                    # each rank alone with dbi_query_spectra: right only when no walk crosses a rank it does not own
                    alone = _merge_hits([(q, g.query_spectra(ms, ppm, None, DBI_TOL_PPM, f)) for g in hs], len(ms))
                    per_rank_fails += hits_canonical(alone) != exp[f]
            finally:
                close_all(hs)
    finally:
        whole.close()
    assert per_rank_fails > 0  # what the stops fix


@gpu
@pytest.mark.parametrize("world", [2, 3, 4])
def test_sharded_unindexed_spectra_equal_one_handle(world):
    from dbindex_b200.multigpu import ShardedSearcher, search_unindexed_spectra_local
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = _dup_proteome(300)
    hs = sharded(p, res, off, world)
    try:
        with dbi.GpuIndex(p) as g, dbi.GpuIndex(p) as u:
            g.add_proteins(res, off)
            u.add_proteins(res, off)
            g.build()
            masses = g.fetch(0, g.stats()["n_entries"])["mass"]
            rng = np.random.default_rng(10 + world)
            spectra = dalton_spectra(rng, masses, p.max_mass, 150)
            mass, tol, roff = flatten(spectra)
            exp = hits_canonical(g.query_spectra(mass, tol, roff, DBI_TOL_DA, 8))
            got = search_unindexed_spectra_local(hs, mass, tol, roff, DBI_TOL_DA, 8)
            assert hits_canonical(got) == exp
            assert hits_canonical(u.search_unindexed_spectra(mass, tol, roff, DBI_TOL_DA, 8)) == exp
            ms = np.concatenate((rng.choice(masses, 300), rng.uniform(p.min_mass, p.max_mass, 50)))
            for ppm in (10.0, 50.0):
                tl = np.full(len(ms), ppm)
                exp = hits_canonical(g.query_spectra(ms, tl, None, DBI_TOL_PPM, 8))
                got = search_unindexed_spectra_local(hs, ms, tl, None, DBI_TOL_PPM, 8)
                assert hits_canonical(got) == exp, ppm
                assert hits_canonical(u.search_unindexed_spectra(ms, tl, None, DBI_TOL_PPM, 8)) == exp
            assert any(len(x) for x in exp)
            # the cap: DBI_ERANGE with the per-rank counts, nothing pending anywhere, a retry at the largest count
            tl = np.full(len(ms), 10.0)
            per_rank = search_unindexed_spectra_local(hs, ms, tl, None, DBI_TOL_PPM, 8)["n_candidates"].copy()
            top = int(per_rank.max())
            assert top > 1
            with pytest.raises(DbiError) as ei:
                search_unindexed_spectra_local(hs, ms, tl, None, DBI_TOL_PPM, 8, top - 1)
            assert ei.value.code == DBI_ERANGE and ei.value.n_candidates == top
            assert np.array_equal(ei.value.rank_candidates, per_rank)
            nothing_pending(hs)
            again = search_unindexed_spectra_local(hs, ms, tl, None, DBI_TOL_PPM, 8, top)
            exp10 = hits_canonical(g.query_spectra(ms, tl, None, DBI_TOL_PPM, 8))
            assert hits_canonical(again) == exp10
            # the mirror's chunked search over the ranks with a small cap
            searcher = ShardedSearcher(hs)
            calls = []
            inner = searcher.search_unindexed_spectra
            searcher.search_unindexed_spectra = lambda *a, **k: calls.append(1) or inner(*a, **k)
            chunked = search_unindexed_spectra_chunked(searcher, ms, tl, None, DBI_TOL_PPM, 8, max(2, top // 4))
            assert len(calls) > 2 and hits_canonical(chunked) == exp10
            m5, t5, o5 = flatten(spectra[:150])  # lists of <= 31 ranges: no single spectrum over the cap
            top_da = int(search_unindexed_spectra_local(hs, m5, t5, o5, DBI_TOL_DA, 8)["n_candidates"].max())
            calls.clear()
            chunked = search_unindexed_spectra_chunked(searcher, m5, t5, o5, DBI_TOL_DA, 8, max(2, top_da // 3))
            assert len(calls) > 2
            assert hits_canonical(chunked) == hits_canonical(g.query_spectra(m5, t5, o5, DBI_TOL_DA, 8))
    finally:
        close_all(hs)


@gpu
def test_shapes_lifecycle_and_arguments():
    from dbindex_b200.multigpu import build_local, query_spectra_local, search_unindexed_spectra_local
    p = dbi.default_params(**PARAM_SETS["cfg1_tryptic"])
    res, off = _dup_proteome(300)
    hs = sharded(p, res, off, 3)
    un = sharded(p, res, off, 3)
    g1 = dbi.GpuIndex(p)
    try:
        g1.add_proteins(res, off)
        # unbuilt handles for the index call, and the wrong call for built ones
        empty = np.zeros(0)
        rc, _, _ = raw_local("dbi_mg_query_spectra_local", hs, empty, empty, np.zeros(1, np.uint64), 0, DBI_TOL_DA, 8)
        assert rc == DBI_ENOTINIT
        build_local(hs)
        g1.build()
        rc, _, _ = raw_local("dbi_mg_search_unindexed_spectra_local", hs, empty, empty, np.zeros(1, np.uint64), 0,
                             DBI_TOL_DA, 8)
        assert rc == DBI_EALREADY
        masses = g1.fetch(0, g1.stats()["n_entries"])["mass"]
        for call in (query_spectra_local, search_unindexed_spectra_local):
            hh = hs if call is query_spectra_local else un
            r = call(hh, empty, empty, np.zeros(1, np.uint64), DBI_TOL_DA, 8)
            assert r["counts"].nq == 0 and list(r["hit_off"]) == [0]
            r = call(hh, empty, empty, np.zeros(6, np.uint64), DBI_TOL_DA, 8)
            assert r["counts"].nq == 5 and r["counts"].n_hits == 0 and list(r["hit_off"]) == [0] * 6
            r = call(hh, empty, empty, None, DBI_TOL_PPM, 8)
            assert r["counts"].nq == 0
        # 10^5 spectra with duplicates
        rng = np.random.default_rng(4)
        ms = rng.choice(masses, 100000)
        ms[1::2] = ms[0::2]
        tl = np.full(len(ms), 10.0)
        big = query_spectra_local(hs, ms, tl, None, DBI_TOL_PPM, 8)
        ho = big["hit_off"].astype(np.int64)
        assert big["counts"].nq == 100000 and np.array_equal(np.diff(ho)[0::2], np.diff(ho)[1::2])
        assert hits_canonical(big) == hits_canonical(g1.query_spectra(ms, tl, None, DBI_TOL_PPM, 8))
        # all hits on one rank: the other ranks hold valid empty results
        x = float(masses[len(masses) // 2])
        sp = [[(x, 0.0)], [(x, 0.0), (x, 0.0)]]
        rc, counts, _ = raw_local("dbi_mg_query_spectra_local", hs, *flatten(sp), 2, DBI_TOL_DA, 0)
        assert rc == 0 and [counts[r].nq for r in range(3)] == [2, 2, 2]
        assert sorted(counts[r].n_hits > 0 for r in range(3)) == [False, False, True]
        parts = [(np.arange(2), g._read_hits(counts[r], None, None, True)) for r, g in enumerate(hs)]
        assert hits_canonical(_merge_hits(parts, 2)) == hits_canonical(g1.query_spectra(*flatten(sp), DBI_TOL_DA, 0))
        # a new call drops every pending result of the previous one
        rc, _, _ = raw_local("dbi_mg_query_spectra_local", hs, ms[:50], tl[:50], None, 50, DBI_TOL_PPM, 8)
        assert rc == 0
        rc, counts, _ = raw_local("dbi_mg_query_spectra_local", hs, ms[50:80], tl[50:80], None, 30, DBI_TOL_PPM, 8)
        assert rc == 0 and all(counts[r].nq == 30 for r in range(3))
        parts = [(np.arange(30), g._read_hits(counts[r], None, None, True)) for r, g in enumerate(hs)]
        assert hits_canonical(_merge_hits(parts, 30)) == hits_canonical(
            g1.query_spectra(ms[50:80], tl[50:80], None, DBI_TOL_PPM, 8))
        nothing_pending(hs)
        # bad handles: out of rank order, repeated, null, n out of range, a lone rank of a sharded index
        one = ms[:3].copy()
        for bad in ([hs[1], hs[0], hs[2]], [hs[0], hs[0], hs[2]], [hs[0], None, hs[2]], [], hs[:2], [hs[1]],
                    [hs[0], hs[1], hs[2]] * 6):
            rc, _, _ = raw_local("dbi_mg_query_spectra_local", bad, one, tl[:3], None, 3, DBI_TOL_PPM, 8)
            assert rc == DBI_EINVAL, len(bad)
        # check_spectra's errors, once for the whole call
        nan = np.array([1000.0, np.nan])
        rc, _, _ = raw_local("dbi_mg_query_spectra_local", hs, nan, tl[:2], None, 2, DBI_TOL_PPM, 8)
        assert rc == DBI_EINVAL and b"spectrum 1" in dbi.load_library().dbi_last_error()
        # the rank-level calls: PPM needs the stops, Dalton takes none
        with pytest.raises(DbiError) as ei:
            hs[0].mg_query_spectra(one, tl[:3], None, DBI_TOL_PPM, 8, stop=None)
        assert ei.value.code == DBI_EINVAL
        with pytest.raises(DbiError) as ei:
            hs[0].mg_query_spectra(*flatten([[(x, 0.1)]]), DBI_TOL_DA, 8, stop=np.zeros(1, np.uint64))
        assert ei.value.code == DBI_EINVAL
        with pytest.raises(DbiError) as ei:  # 5 slices for world 3
            hs[0].mg_spectra_stops(one, tl[:3], np.array([1000.0, 2000.0, 3000.0, 4000.0]), 0, 3)
        assert ei.value.code == DBI_EINVAL
        # n == 1 is dbi_query_spectra / dbi_search_unindexed_spectra
        assert hits_canonical(query_spectra_local([g1], ms[:200], tl[:200], None, DBI_TOL_PPM, 8)) == \
            hits_canonical(g1.query_spectra(ms[:200], tl[:200], None, DBI_TOL_PPM, 8))
        with dbi.GpuIndex(p) as u1:
            u1.add_proteins(res, off)
            assert hits_canonical(search_unindexed_spectra_local([u1], ms[:200], tl[:200], None, DBI_TOL_PPM, 8)) \
                == hits_canonical(g1.query_spectra(ms[:200], tl[:200], None, DBI_TOL_PPM, 8))
        # the unindexed call: repeated or null handles
        for bad in ([un[0], un[0]], [un[0], None]):
            rc, _, _ = raw_local("dbi_mg_search_unindexed_spectra_local", bad, one, tl[:3], None, 3, DBI_TOL_PPM, 8)
            assert rc == DBI_EINVAL
    finally:
        close_all(hs + un + [g1])


@gpu
def test_mirror_sharded_spectra_batches():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = _dup_proteome(150)
    seqs = [res[int(o0):int(o1)].tobytes().decode() for o0, o1 in zip(off[:-1], off[1:])]
    names = [f"P{i}" for i in range(len(seqs))]
    ref = DBIndexer(p, 8)
    ref.init()
    ref.run(proteins=(names, seqs))
    sh = DBIndexer(p, 8, use_index=False, devices=[0, 0, 0])
    sh.init()
    sh.run(proteins=(names, seqs))
    key = lambda lst: sorted((s.key(), tuple(s.proteinIds), s.sequenceOffset) for s in lst)  # noqa: E731
    try:
        rng = np.random.default_rng(6)
        masses = ref.index.fetch(0, ref.index.stats()["n_entries"])["mass"]
        spectra = [[MassRange(float(m) + k * ISO, 0.02) for k in range(-1, 4)] for m in rng.choice(masses, 30)]
        spectra += [[], [MassRange(float(masses[3]), 0.5)], [MassRange(8100.0, 1.0), MassRange(1000.0, 1.0)]]
        got = [key(x) for x in sh.getSequencesForSpectra(spectra)]
        assert any(got)
        assert got == [key(x) for x in ref.getSequencesForSpectra(spectra)]
        assert got == [key(sh.getSequences(sp)) for sp in spectra]
        ms = [float(m) for m in rng.choice(masses, 30)]
        pb = [key(x) for x in sh.getSequencesUsingPPMToleranceBatch(ms, 10.0)]
        assert pb == [key(x) for x in ref.getSequencesUsingPPMToleranceBatch(ms, 10.0)]
        assert pb == [key(ref._ppm_probe_loop(m, 10.0)) for m in ms]
        assert pb == [key(sh.getSequencesUsingPPMTolerance(m, 10.0)) for m in ms]
    finally:
        ref.close()
        sh.close()
