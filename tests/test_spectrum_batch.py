"""dbi_query_spectra / dbi_search_unindexed_spectra: a batch of spectra answered in one call, every spectrum as the
reference's per-spectrum call answers it -- getSequences(List<MassRange>) for Dalton range lists,
getSequencesUsingPPMTolerance for (mass, ppm) pairs."""
import ctypes as C
import os

import numpy as np
import pytest

import dbindex_b200 as dbi
from dbindex_b200 import synth
from dbindex_b200.capi import DBI_ERANGE, DBI_TOL_DA, DBI_TOL_PPM, DbiError, DbiHitCounts, expand_hits, ppm_probe_bound
from dbindex_b200.indexer import (PRECISION, DBIndexer, DBIndexImpl, DBIndexSearchParams, MassRange, merge_intervals,
                                  search_unindexed_spectra_chunked, tolerance_in_dalton)
from oracle.oracle_py import Oracle

from .test_gpu_parity import hits_canonical
from .util import PARAM_SETS, bits, pack

NCPU = os.cpu_count() or 1
ISO = 1.00335  # isotope spacing of the query kind (a)


def out_of_buckets(x, f):
    if f == 0:
        return False
    return int(x) // (8000 // f) > f - 1


def expected_intervals(spectra, f):
    """The mirror's getSequences(ranges): merge_intervals, and nothing when a merged interval fails the bucket rule."""
    lo, hi, sid = [], [], []
    for s, sp in enumerate(spectra):
        merged = merge_intervals([MassRange(m, t) for m, t in sp])
        if any(out_of_buckets(a, f) or out_of_buckets(b, f) for a, b in merged):
            continue
        for a, b in merged:
            lo.append(a)
            hi.append(b)
            sid.append(s)
    return np.array(lo, np.float64), np.array(hi, np.float64), np.array(sid, np.int64)


def per_spectrum(h, sid, n):
    """Canonical hits of a flat interval answer grouped by spectrum."""
    per_iv = hits_canonical(h)
    out = [[] for _ in range(n)]
    for i, s in enumerate(sid):
        out[s].extend(per_iv[i])
    return [sorted(x) for x in out]


def flatten(spectra):
    mass = np.array([m for sp in spectra for m, _ in sp], np.float64)
    tol = np.array([t for sp in spectra for _, t in sp], np.float64)
    off = np.zeros(len(spectra) + 1, np.uint64)
    np.cumsum([len(sp) for sp in spectra], out=off[1:])
    return mass, tol, off


def spectra_canonical(h):
    return hits_canonical(expand_hits(h) if "hit_pep" not in h else h)


# ---- CPU ----------------------------------------------------------------------------------------------------

def test_ppm_probe_bound_holds_every_probe():
    """hi_ext (K13b) is >= every probe the reference loop admits, whatever the entries: walk the guard alone."""
    rng = np.random.default_rng(7)
    ms = np.concatenate((rng.uniform(50, 8000, 300), [1e-3, 0.5, 7999.999, 1e4]))
    ppms = np.concatenate((rng.uniform(0.01, 300, 300), [5, 10, 50, 300]))
    for m, p in zip(ms.tolist(), ppms.tolist()):
        bound = ppm_probe_bound(m, p)
        u = m + tolerance_in_dalton(m, p)
        while u - tolerance_in_dalton(u, p) < m:
            assert u <= bound, (m, p, u, bound)
            nu = u + PRECISION
            if nu == u:
                break
            u = nu


class StandIn:
    """A handle that answers spectra with made-up hits and refuses a batch whose candidates exceed the cap:
    spectrum hits = one per range, mass = first mass of the spectrum + rank; N_c = 10 per range."""

    def __init__(self):
        self.calls = []

    def search_unindexed_spectra(self, mass, tol, range_off, tol_mode, index_factor, max_candidates):
        off = np.arange(len(mass) + 1, dtype=np.uint64) if range_off is None else range_off
        n = len(off) - 1
        n_c = 10 * int(off[-1])
        if max_candidates and n_c > max_candidates:
            raise DbiError(DBI_ERANGE, "over the cap", n_c)
        self.calls.append((mass.copy(), off.copy()))
        cnt = np.diff(off.astype(np.int64))
        H = int(cnt.sum())
        hm = np.concatenate([mass[int(off[s])] + np.arange(cnt[s]) for s in range(n) if cnt[s]] + [np.zeros(0)])
        return {"hit_off": off.astype(np.uint64), "modpat": np.arange(H, dtype=np.uint32),
                "mass": hm.astype(np.float64), "first_prot": np.zeros(H, np.uint32),
                "first_off": np.zeros(H, np.uint32), "len": np.ones(H, np.uint16),
                "hit_pep": np.arange(H, dtype=np.int64), "flanks": np.zeros(6 * H, np.uint8),
                "seq_off": np.arange(H + 1, dtype=np.uint64), "seq": np.full(H, 65, np.uint8),
                "prot_list_off": np.arange(H + 1, dtype=np.uint64), "prot_ids": np.arange(H, dtype=np.uint32),
                "counts": DbiHitCounts(n, H, H, H, H)}


@pytest.mark.parametrize("mode", [DBI_TOL_DA, DBI_TOL_PPM])
def test_spectrum_chunker_keeps_spectra_whole(mode):
    rng = np.random.default_rng(3)
    n = 40
    if mode == DBI_TOL_DA:
        lens = rng.integers(0, 6, n)
        off = np.concatenate(([0], np.cumsum(lens))).astype(np.uint64)
        mass = rng.uniform(500, 3000, int(off[-1]))
    else:
        off, lens = None, np.ones(n, np.int64)
        mass = rng.uniform(500, 3000, n)
    tol = np.full(len(mass), 0.01)
    stand = StandIn()
    got = search_unindexed_spectra_chunked(stand, mass, tol, off, mode, 8, 60)
    assert len(stand.calls) > 1  # the cap split the batch
    whole = StandIn().search_unindexed_spectra(mass, tol, off, mode, 8, 0)
    # a hit's mass is its spectrum's first mass + its rank there: equal only when every call got whole spectra
    assert np.array_equal(got["hit_off"], whole["hit_off"])
    assert np.array_equal(bits(got["mass"]), bits(whole["mass"]))
    assert sum(len(co) - 1 for _, co in stand.calls) == n
    with pytest.raises(DbiError):  # one spectrum over the cap cannot be split
        search_unindexed_spectra_chunked(StandIn(), mass[:1], tol[:1], np.array([0, 1], np.uint64)
                                         if mode == DBI_TOL_DA else None, mode, 8, 5)


# ---- GPU ----------------------------------------------------------------------------------------------------

def proteome(n, seed):
    res, off = synth.synth_proteome(n, seed, median_len=300, min_len=5)
    return [res[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(len(off) - 1)]


def built(name, seqs):
    p = dbi.default_params(**PARAM_SETS[name])
    g = dbi.GpuIndex(p)
    g.add_proteins(*pack(seqs))
    g.build()
    o = Oracle(p, threads=NCPU)
    o.add_proteins(*pack(seqs))
    assert o.build() == 0
    return p, g, o


def dalton_spectra(rng, masses, max_mass, n=300):
    """0..30 ranges: isotope offsets, overlapping, nested, duplicate, touching, lo clamped at 0, negative tolerances,
    and a range past the last bucket in a few spectra."""
    out = []
    for s in range(n):
        m = float(rng.choice(masses)) if rng.random() < 0.7 else float(rng.uniform(400, max_mass))
        k = int(rng.integers(0, 31))
        sp = []
        for j in range(k):
            kind = j % 7
            if kind == 0:
                sp.append((m + (j % 5 - 1) * ISO, m * 1e-5))
            elif kind == 1:
                sp.append((m, 0.5))
            elif kind == 2:
                sp.append((m + 0.1, 0.05))  # nested
            elif kind == 3:
                sp.append(sp[-1] if sp else (m, 0.01))  # duplicate
            elif kind == 4:
                a, b = sp[-1][0] - sp[-1][1], sp[-1][0] + sp[-1][1]
                sp.append((b + 0.25, 0.25))  # touching: lo == previous hi (up to rounding)
            elif kind == 5:
                sp.append((m - 0.3, -0.2))  # inverted
            else:
                sp.append((float(rng.uniform(0, 2)), 3.0))  # lo clamped at 0
        if s % 37 == 5:
            sp.append((8005.0, 1.0))  # past the last bucket: empties this spectrum only
        out.append(sp)
    out.append([(m0, 0.02) for m0 in np.linspace(800, 1500, 33)])
    out.append([(float(x), 0.003) for x in rng.choice(masses, 1000)])
    out.append([(900.0, 1.0), (901.0, 1.0), (899.5, -2.0), (903.0, 1.0)])  # touching and inverted between them
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(PARAM_SETS))
def test_dalton_lists_equal_merged_intervals(name):
    seqs = proteome(120, 11)
    p, g, o = built(name, seqs)
    with g:
        masses = g.fetch(0, g.stats()["n_entries"])["mass"]
        rng = np.random.default_rng(5)
        spectra = dalton_spectra(rng, masses, p.max_mass)
        mass, tol, off = flatten(spectra)
        for f in (8, 0):
            got = spectra_canonical(g.query_spectra(mass, tol, off, DBI_TOL_DA, f, per_hit=False))
            lo, hi, sid = expected_intervals(spectra, f)
            assert got == per_spectrum(o.query_hits(lo, hi), sid, len(spectra))
            assert got == per_spectrum(g.query_hits(lo, hi), sid, len(spectra))
        if f == 0:
            assert any(len(x) for x in got)


def ppm_expected(o, oe, m, ppm):
    idx, _ = o.query_ppm(m, ppm)
    return sorted((int(bits(oe["mass"][i:i + 1])[0]), int(oe["first_prot"][i]), int(oe["first_off"][i]),
                   int(oe["len"][i]), int(oe["modpat"][i])) for i in idx.astype(np.int64))


def short(per):
    return [sorted(t[:5] for t in x) for x in per]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg1_tryptic", "cfg2_mods", "wide_mass_mod4"])
def test_ppm_equals_oracle(name):
    seqs = proteome(150, 12)
    p, g, o = built(name, seqs)
    with g:
        oe = o.entries()
        masses = oe["mass"]
        rng = np.random.default_rng(9)
        ms = np.concatenate((rng.choice(masses, 200), rng.uniform(p.min_mass, p.max_mass, 100),
                             [p.max_mass - 1e-3, p.max_mass, masses[-1]]))
        for ppm in (5.0, 10.0, 50.0):
            got = short(spectra_canonical(g.query_spectra(ms, np.full(len(ms), ppm), None, DBI_TOL_PPM, 0,
                                                          per_hit=False)))
            assert got == [ppm_expected(o, oe, float(m), ppm) for m in ms]


def host_probe_loop(g, m, ppm, f):
    """The mirror's per-probe host loop through dbi_query_hits (window, then [u_k, u_k] until one is empty)."""
    def q(lo, hi):
        if out_of_buckets(lo, f) or out_of_buckets(hi, f):
            return []
        return hits_canonical(g.query_hits([lo], [hi]))[0]
    tol = tolerance_in_dalton(m, ppm)
    res = q(max(m - tol, 0.0), m + tol)
    have = set(res)
    u = m + tol
    while u - tolerance_in_dalton(u, ppm) < m:
        h = q(max(u, 0.0), u)
        if not h:
            break
        res += [x for x in h if x not in have]
        have.update(h)
        nu = u + PRECISION
        if nu == u:
            break
        u = nu
    return sorted(res)


@pytest.mark.gpu
def test_continuing_probe_walks():
    """Entries at exactly u_0, u_1, ... of chosen spectra: walks of 0, 1, 2 and 5 probes, a gap, the last bucket."""
    ppm = 50.0
    # index factor 3: buckets of 2666 Da, a bound fails from 7998 on; u_0, u_1 below it, u_2 above
    edge = 7997.9999985 / (1 + tolerance_in_dalton(1.0, ppm))
    plan = {1000.0: 0, 1500.0: 1, 2000.0: 2, 4000.0: 5, 3000.0: -2, edge: 3}  # -2: u_0, u_1, gap, u_3
    recs = []
    for m, k in plan.items():
        u = m + tolerance_in_dalton(m, ppm)
        us = [u]
        for _ in range(6):
            us.append(us[-1] + PRECISION)
        take = us[:k + 1] if k >= 0 else [us[0], us[1], us[3]]
        recs += take
        recs.append(m)  # an entry inside the window
    seqs = ["PEPTIDEK" * 3]
    p = dbi.default_params(min_mass=0.0, max_mass=8000.0)
    with dbi.GpuIndex(p) as g:
        g.add_proteins(*pack(seqs))
        n = len(recs)
        mass = np.array(recs, np.float64)
        prot = np.zeros(n, np.uint32)
        off = (np.arange(n) % 16).astype(np.uint32)
        ln = np.full(n, 2 + (np.arange(n) % 5), np.uint16)
        rc = g.lib.dbi_build_from_records(g._h, mass.ctypes.data_as(C.c_void_p), prot.ctypes.data_as(C.c_void_p),
                                          off.ctypes.data_as(C.c_void_p), ln.ctypes.data_as(C.c_void_p), n)
        assert rc == 0, g.lib.dbi_last_error()
        ms = np.array(list(plan), np.float64)
        for f in (3, 0):
            got = spectra_canonical(g.query_spectra(ms, np.full(len(ms), ppm), None, DBI_TOL_PPM, f, per_hit=False))
            exp = [host_probe_loop(g, float(m), ppm, f) for m in ms]
            assert got == exp
            # the window holds m and u_0; then the continuing probes k >= 1 (u_2 of the last one fails the bucket rule)
            assert [len(x) for x in got] == [2, 3, 4, 7, 3, 3 if f else 5]


@pytest.mark.gpu
def test_unindexed_equals_built():
    seqs = proteome(150, 13)
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    with dbi.GpuIndex(p) as g, dbi.GpuIndex(p) as u:
        g.add_proteins(*pack(seqs))
        u.add_proteins(*pack(seqs))
        g.build()
        masses = g.fetch(0, g.stats()["n_entries"])["mass"]
        rng = np.random.default_rng(2)
        spectra = dalton_spectra(rng, masses, p.max_mass, 200)
        mass, tol, off = flatten(spectra)
        exp = spectra_canonical(g.query_spectra(mass, tol, off, DBI_TOL_DA, 8, per_hit=False))
        assert spectra_canonical(u.search_unindexed_spectra(mass, tol, off, DBI_TOL_DA, 8, per_hit=False)) == exp
        # a mass whose u_0 is exactly an entry mass (searched among the ulps next to an entry)
        ms = list(rng.choice(masses, 200))
        for e in masses[100:140]:
            for m in (float(e) / (1 + 10e-6 / (1 + 10e-6)) + d for d in np.linspace(-3e-12, 3e-12, 61)):
                if m + tolerance_in_dalton(m, 10.0) == float(e):
                    ms.append(m)
                    break
        assert len(ms) > 200
        ms = np.array(ms)
        for ppm in (10.0, 50.0):
            exp = spectra_canonical(g.query_spectra(ms, np.full(len(ms), ppm), None, DBI_TOL_PPM, 8, per_hit=False))
            got = spectra_canonical(u.search_unindexed_spectra(ms, np.full(len(ms), ppm), None, DBI_TOL_PPM, 8,
                                                               per_hit=False))
            assert got == exp
        # the cap: DBI_ERANGE with N_c, no pending result, then a retry at N_c
        u.search_unindexed_spectra(ms, np.full(len(ms), 10.0), None, DBI_TOL_PPM, 8, 0, per_hit=False)
        n_c = u.last_candidates
        assert n_c > 1
        with pytest.raises(DbiError) as ei:
            u.search_unindexed_spectra(ms, np.full(len(ms), 10.0), None, DBI_TOL_PPM, 8, n_c - 1)
        assert ei.value.code == DBI_ERANGE and ei.value.n_candidates == n_c
        assert u.lib.dbi_query_hits_read(u._h, None) == -1  # DBI_ENOTINIT: nothing pending
        again = u.search_unindexed_spectra(ms, np.full(len(ms), 10.0), None, DBI_TOL_PPM, 8, n_c, per_hit=False)
        assert spectra_canonical(again) == spectra_canonical(
            g.query_spectra(ms, np.full(len(ms), 10.0), None, DBI_TOL_PPM, 8, per_hit=False))
        # the mirror's chunked search with a tiny cap
        ppm10 = np.full(len(ms), 10.0)
        chunked = search_unindexed_spectra_chunked(u, ms, ppm10, None, DBI_TOL_PPM, 8, max(1, n_c // 5))
        assert hits_canonical(chunked) == spectra_canonical(g.query_spectra(ms, ppm10, None, DBI_TOL_PPM, 8,
                                                                            per_hit=False))


@pytest.mark.gpu
def test_batch_shapes_and_lifecycle():
    seqs = proteome(100, 14)
    p = dbi.default_params(**PARAM_SETS["cfg1_tryptic"])
    with dbi.GpuIndex(p) as g:
        g.add_proteins(*pack(seqs))
        empty = np.zeros(0)
        with pytest.raises(DbiError) as ei:  # not built
            g.query_spectra(np.array([1000.0]), np.array([10.0]), None, DBI_TOL_PPM)
        assert ei.value.code == -1
        g.build()
        with pytest.raises(DbiError) as ei:  # built: no unindexed search
            g.search_unindexed_spectra(np.array([1000.0]), np.array([10.0]), None, DBI_TOL_PPM)
        assert ei.value.code == -2
        masses = g.fetch(0, g.stats()["n_entries"])["mass"]
        r = g.query_spectra(empty, empty, np.zeros(1, np.uint64), DBI_TOL_DA, 8)
        assert r["counts"].nq == 0 and list(r["hit_off"]) == [0]
        r = g.query_spectra(empty, empty, np.zeros(6, np.uint64), DBI_TOL_DA, 8)
        assert r["counts"].nq == 5 and r["counts"].n_hits == 0 and list(r["hit_off"]) == [0] * 6
        rng = np.random.default_rng(4)
        ms = rng.choice(masses, 100000)
        ms[1::2] = ms[0::2]  # duplicate spectra
        big = g.query_spectra(ms, np.full(len(ms), 10.0), None, DBI_TOL_PPM, 8, per_hit=False)
        assert big["counts"].nq == 100000
        ho = big["hit_off"].astype(np.int64)
        assert np.array_equal(np.diff(ho)[0::2], np.diff(ho)[1::2])
        one = [g.query_spectra(ms[i:i + 1], np.array([10.0]), None, DBI_TOL_PPM, 8, per_hit=False)
               for i in range(0, 100000, 9973)]
        allc = spectra_canonical(big)
        assert [spectra_canonical(x)[0] for x in one] == [allc[i] for i in range(0, 100000, 9973)]
        # bad arguments name the spectrum
        lib = g.lib
        cnt = DbiHitCounts()
        bad = np.array([1000.0, np.nan])
        tol = np.array([1.0, 1.0])
        rc = lib.dbi_query_spectra(g._h, bad.ctypes.data_as(C.c_void_p), tol.ctypes.data_as(C.c_void_p), None, 2,
                                   DBI_TOL_PPM, 8, C.byref(cnt))
        assert rc == -3 and b"spectrum 1" in lib.dbi_last_error()
        ro = np.array([0, 2, 1], np.uint64)
        rc = lib.dbi_query_spectra(g._h, tol.ctypes.data_as(C.c_void_p), tol.ctypes.data_as(C.c_void_p),
                                   ro.ctypes.data_as(C.c_void_p), 2, DBI_TOL_DA, 8, C.byref(cnt))
        assert rc == -3 and b"spectrum 1" in lib.dbi_last_error()
        rc = lib.dbi_query_spectra(g._h, tol.ctypes.data_as(C.c_void_p), tol.ctypes.data_as(C.c_void_p),
                                   ro.ctypes.data_as(C.c_void_p), 1, DBI_TOL_PPM, 8, C.byref(cnt))
        assert rc == -3
        # a pending result is replaced by the next call; the read equals dbi_query_hits_read of the same intervals
        g.query_hits([1.0], [2.0])
        sp = [[(float(masses[10]), 0.5), (float(masses[10]) + ISO, 0.01)]]
        a = g.query_spectra(*flatten(sp), DBI_TOL_DA, 0, per_hit=False)
        lo, hi, _ = expected_intervals(sp, 0)
        b = g.query_hits(lo, hi, per_hit=False)
        for k in ("modpat", "pep_hit_off", "mass", "first_prot", "first_off", "len", "flanks", "seq_off", "seq",
                  "prot_list_off", "prot_ids"):
            assert np.array_equal(a[k], b[k]), k
        assert list(a["hit_off"]) == [0, int(b["hit_off"][-1])]


def old_get_sequences(ref, ranges):
    """DBIndexer.getSequences(ranges) as the mirror answered it before the spectrum batches."""
    if len(ranges) == 1:
        return ref.getSequencesBatch([ranges[0].precMass], [ranges[0].tolerance])[0]
    merged = merge_intervals(ranges)
    if not merged or any(ref._out_of_buckets(a, b) for a, b in merged):
        return []
    return [x for lst in ref._materialise(np.array([a for a, _ in merged]), np.array([b for _, b in merged]))
            for x in lst]


@pytest.mark.gpu
@pytest.mark.parametrize("use_index", [True, False])
def test_mirror_batches_equal_single_calls(use_index):
    seqs = proteome(80, 15)
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    names = [f"P{i}" for i in range(len(seqs))]
    impl = DBIndexImpl(DBIndexSearchParams(params=p, dataBaseName=f"spectra_{use_index}", useIndex=use_index),
                       proteins=(names, seqs))
    ref = DBIndexer(p, 8)
    ref.init()
    ref.run(proteins=(names, seqs))
    try:
        rng = np.random.default_rng(6)
        masses = ref.index.fetch(0, ref.index.stats()["n_entries"])["mass"]
        spectra = [[MassRange(float(m) + k * ISO, 0.02) for k in range(-1, 4)] for m in rng.choice(masses, 30)]
        spectra += [[], [MassRange(float(masses[3]), 0.5)], [MassRange(8100.0, 1.0), MassRange(1000.0, 1.0)]]
        keys = [sorted(s.key() for s in lst) for lst in impl.getSequencesForSpectra(spectra)]
        assert any(keys)
        assert keys == [sorted(s.key() for s in impl.getSequences(sp)) for sp in spectra]
        assert keys == [sorted(s.key() for s in old_get_sequences(ref, sp)) for sp in spectra]
        ms = [float(m) for m in rng.choice(masses, 30)]
        pb = [sorted(s.key() for s in lst) for lst in impl.indexer.getSequencesUsingPPMToleranceBatch(ms, 10.0)]
        assert pb == [sorted(s.key() for s in ref._ppm_probe_loop(m, 10.0)) for m in ms]
        assert pb == [sorted(s.key() for s in impl.indexer.getSequencesUsingPPMTolerance(m, 10.0)) for m in ms]
    finally:
        impl.close()
        ref.close()
