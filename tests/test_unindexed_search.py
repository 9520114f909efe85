"""dbi_search_unindexed (the reference's SEARCH_UNINDEXED mode): the hits of a batch straight from the proteins,
through a digest that keeps only the records that can land in a window.  The answer must equal what dbi_build +
dbi_query_hits give on the same handle; the oracle is the reference restated on the CPU."""
import ctypes as C
import itertools
import os

import numpy as np
import pytest

import dbindex_b200 as dbi
from dbindex_b200 import synth
from dbindex_b200.capi import DBI_ERANGE, DbiError, DbiHitBuffers, DbiHitCounts
from dbindex_b200.indexer import (DBIndexImpl, DBIndexSearchParams, DBIndexStoreException, MassRange,
                                  search_unindexed_chunked)
from oracle.oracle_py import Oracle

from .test_gpu_parity import check_hits, hits_canonical
from .util import PARAM_SETS, assert_entries_equal, pack

NCPU = os.cpu_count() or 1
EPS = 1e-9  # kShiftEps of csrc/window.cu
# 8 distinct shifts, K = 4: 495 class multisets, more than the 64 interval slots (the band fallback)
EIGHT_SHIFTS_K4 = dict(diff_mods=[("M", 15.9949), ("S", 79.96633), ("K", 42.010565), ("N", 0.984016),
                                  ("W", 31.989829), ("P", 15.994915), ("R", 14.01565), ("Y", 79.956815)],
                       max_mods_per_peptide=4, max_missed=1)
MOD_SETS = {k: v for k, v in PARAM_SETS.items() if "diff_mods" in v}
MOD_SETS["eight_shifts_k4"] = EIGHT_SHIFTS_K4
LONG_MODDED = "G" * 70 + "MSTYMWSTK" + "G" * 12 + "MR"  # mod sites beyond residue 64 of a peptide


def proteome(n, seed):
    res, off = synth.synth_proteome(n, seed, median_len=300, min_len=5)
    seqs = [res[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(len(off) - 1)]
    return seqs + [seqs[0], LONG_MODDED, "A" * 66 + "SSTTYYMMWK"]


def oracle(p, seqs):
    o = Oracle(p, threads=NCPU)
    o.add_proteins(*pack(seqs))
    assert o.build() == 0
    return o


class Unindexed:
    """query_hits of an unbuilt handle answered by dbi_search_unindexed (for check_hits)."""

    def __init__(self, g, cap=0):
        self.g, self.cap = g, cap

    def query_hits(self, lo, hi, per_hit=True):
        return self.g.search_unindexed(lo, hi, self.cap, per_hit=per_hit)


# ---- CPU: the prefilter's shift table, restated ------------------------------------------------------------

def class_shifts(p):
    """Distinct shifts in residue-code order (upload_tables: DiffModification, last one wins)."""
    diff = {}
    for i in range(p.n_mods):
        diff[p.mods[i].residue] = p.mods[i].delta
    out = []
    for r in sorted(diff):
        if diff[r] not in out:
            out.append(diff[r])
    return out


def shift_table(p, cap=64):
    """Per k = 0..K the intervals of InWindows: distinct sums of k class shifts (ascending class order) +- EPS, or
    the band [k mod_lo - EPS, k mod_hi + EPS] for a k whose sums no longer fit."""
    cls = np.array(class_shifts(p), dtype=np.float64)
    K = p.max_mods_per_peptide if len(cls) else 0
    mod_lo, mod_hi = min(0.0, *cls) if len(cls) else 0.0, max(0.0, *cls) if len(cls) else 0.0
    sums, top = np.zeros(1), np.zeros(1, np.int64)
    table, used = [], 0
    for k in range(K + 1):
        if k:
            reps = len(cls) - top
            parent = np.repeat(np.arange(len(sums)), reps)
            c = np.concatenate([np.arange(t, len(cls)) for t in top])
            sums, top = sums[parent] + cls[c], c
        distinct = np.unique(sums)
        if used + len(distinct) + (K - k) <= cap:
            table.append(("sums", distinct))
            used += len(distinct)
        else:
            table.append(("band", np.array([k * mod_lo, k * mod_hi])))
            used += 1
    return table


def test_shift_table_against_brute_force():
    for name, kw in MOD_SETS.items():
        p = dbi.default_params(**kw)
        cls = class_shifts(p)
        table = shift_table(p)
        assert len(table) == p.max_mods_per_peptide + 1
        for k, (kind, v) in enumerate(table):
            brute = set()
            for ms in itertools.combinations_with_replacement(range(len(cls)), k):
                s = 0.0
                for c in ms:
                    s += cls[c]
                brute.add(s)
            if kind == "sums":
                assert set(v.tolist()) == brute, (name, k)
            else:
                assert v[0] <= min(brute) and max(brute) <= v[1], (name, k)
    t = shift_table(dbi.default_params(**EIGHT_SHIFTS_K4))
    assert [kind for kind, _ in t] == ["sums", "sums", "sums", "band", "band"]
    assert [len(v) for _, v in t[:3]] == [1, 8, 36]


@pytest.mark.parametrize("name", sorted(MOD_SETS))
def test_every_entry_lies_in_a_shift_interval(name):
    """Every index entry with k mods lies within EPS of (its base peptide's mass + some sum of k shifts): the
    prefilter keeps every base peptide that has a variant in a window."""
    p = dbi.default_params(**MOD_SETS[name])
    seqs = proteome(40 if name == "eight_shifts_k4" else 120, 300 + len(name))
    o = oracle(p, seqs)
    e = o.entries()
    res, off = pack(seqs)
    gpos = off[e["first_prot"].astype(np.int64)].astype(np.int64) + e["first_off"].astype(np.int64)
    ln = e["len"].astype(np.int64)
    rm = np.array(p.residue_mass[:], dtype=np.float64)
    base = np.zeros(len(ln))  # dbi_calculate_mass: same order as the digest
    if p.add_h2o_proton:
        base += p.h2o_proton
    base += p.cterm
    base += p.nterm
    for j in range(int(ln.max())):
        live = ln > j
        base[live] += rm[res[gpos[live] + j]]
    pat = e["modpat"].astype(np.uint64)
    k = sum(((pat >> np.uint64(8 * b)) & np.uint64(0xFF)) != 0 for b in range(4)).astype(np.int64)
    delta = e["mass"] - base
    table = shift_table(p)
    for kk in range(len(table)):
        sel = k == kk
        kind, v = table[kk]
        if kind == "sums":
            near = np.min(np.abs(delta[sel, None] - v[None, :]), axis=1) <= EPS
        else:
            near = (delta[sel] >= v[0] - EPS) & (delta[sel] <= v[1] + EPS)
        assert np.all(near), (name, kk, delta[sel][~near][:5])
    assert np.count_nonzero(k) > 0


# ---- CPU: the mirror's split-and-reassemble ------------------------------------------------------------

class CappedHandle:
    """search_unindexed of a stand-in handle: the oracle's hits, and DBI_ERANGE when the batch's candidates
    (here: entries inside the union of its windows) exceed the cap."""

    def __init__(self, o):
        self.o, self.mass = o, o.entries()["mass"]
        self.calls = []

    def search_unindexed(self, lo, hi, max_candidates=0):
        inside = np.zeros(len(self.mass), bool)
        for a, b in zip(lo, hi):
            inside |= (self.mass >= a) & (self.mass <= b)
        n_c = int(inside.sum())
        if max_candidates and n_c > max_candidates:
            raise DbiError(DBI_ERANGE, "over the cap", n_c)
        self.calls.append((np.array(lo), np.array(hi)))
        h = self.o.query_hits(lo, hi)
        n = len(h["mass"])
        h["hit_pep"] = np.arange(n, dtype=np.int64)
        h["counts"] = DbiHitCounts(len(lo), n, n, len(h["seq"]), len(h["prot_ids"]))
        return h


def test_chunked_search_answers_every_query_once_in_order():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    o = oracle(p, proteome(60, 8))
    _, _, lo, hi = synth.synth_queries(o.entries()["mass"], 400, 21, da_fraction=0.1, da_tol=0.5)
    lo[:5], hi[:5] = lo[10], hi[10]  # duplicates
    exp = o.query_hits(lo, hi)
    per_q = np.diff(exp["hit_off"].astype(np.int64))
    for cap in (0, 10 ** 9, int(per_q.max()) * 3, int(per_q.max())):
        g = CappedHandle(o)
        got = search_unindexed_chunked(g, lo, hi, cap)
        assert len(g.calls) >= (1 if cap == 0 or cap > per_q.sum() else 2)
        # every query answered by exactly one call
        asked = np.sort(np.concatenate([c[0] for c in g.calls]))
        assert np.array_equal(asked, np.sort(lo))
        assert got["counts"].nq == len(lo) and got["counts"].n_hits == per_q.sum()
        for k in ("hit_off", "mass", "first_prot", "first_off", "len", "modpat", "seq_off", "seq", "flanks",
                  "prot_list_off", "prot_ids"):
            assert np.array_equal(got[k], exp[k]), (cap, k)
    # one query over the cap cannot be split
    g = CappedHandle(o)
    q = int(np.argmax(per_q))
    with pytest.raises(DbiError) as ei:
        search_unindexed_chunked(g, lo[q:q + 1], hi[q:q + 1], int(per_q[q]) - 1)
    assert ei.value.code == DBI_ERANGE and ei.value.n_candidates == per_q[q]
    empty = search_unindexed_chunked(CappedHandle(o), np.zeros(0), np.zeros(0), 5)
    assert empty["hit_off"].tolist() == [0] and empty["counts"].n_hits == 0


# ---- GPU ------------------------------------------------------------------------------------------------

gpu = pytest.mark.gpu


def unbuilt(p, seqs):
    g = dbi.GpuIndex(p)
    g.add_proteins(*pack(seqs))
    return g


@gpu
@pytest.mark.parametrize("name", list(PARAM_SETS))
def test_unindexed_equals_oracle(name):
    p = dbi.default_params(**PARAM_SETS[name])
    seqs = proteome(120, 1000 + len(name))
    o = oracle(p, seqs)
    with unbuilt(p, seqs) as g:
        _, _, lo, hi = synth.synth_queries(o.entries()["mass"], 300, 11, da_fraction=0.3)
        check_hits(Unindexed(g), o, lo, hi)
        st = g.stats()
        assert 0 < st["n_emitted"] <= o.counts()["n_emitted"] and st["n_entries"] <= o.counts()["n_entries"]
        assert st["n_emitted"] == g.last_candidates


@gpu
@pytest.mark.parametrize("name", ["cfg2_mods", "lysc_neg_mod", "many_classes", "wide_mass_mod4", "eight_shifts_k4"])
def test_zero_width_windows_at_entry_masses(name):
    """[m, m] for the index's own masses: a variant's mass and the prefilter's m + s differ by a few ulps."""
    p = dbi.default_params(**MOD_SETS[name])
    seqs = proteome(40 if name == "eight_shifts_k4" else 120, 77 + len(name))
    o = oracle(p, seqs)
    m = np.unique(o.entries()["mass"])
    if len(m) > 10_000:
        m = np.random.default_rng(5).choice(m, 10_000, replace=False)
    with unbuilt(p, seqs) as g:
        un = hits_canonical(g.search_unindexed(m, m))
        g.build()
        ix = hits_canonical(g.query_hits(m, m))
    assert un == ix == hits_canonical(o.query_hits(m, m))
    assert all(len(x) > 0 for x in un)


@gpu
def test_full_cfg2_equals_the_index():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = synth.config_proteome(2)
    with dbi.GpuIndex(p) as g:
        g.add_proteins(res, off)
        _, _, lo, hi = synth.synth_queries(np.zeros(0), 2000, 3)  # uniform masses ...
        un0 = g.search_unindexed(lo, hi)
        g.build()
        _, _, lo2, hi2 = synth.synth_queries(g.fetch(0, g.stats()["n_entries"], with_ids=False)["mass"], 2000, 4)
        ix0, ix2 = g.query_hits(lo, hi), g.query_hits(lo2, hi2)
        g.reset_index()
        un2 = g.search_unindexed(lo2, hi2)  # ... and masses of the index
    assert np.array_equal(un0["hit_off"], ix0["hit_off"]) and hits_canonical(un0) == hits_canonical(ix0)
    assert np.array_equal(un2["hit_off"], ix2["hit_off"]) and hits_canonical(un2) == hits_canonical(ix2)
    assert un2["counts"].n_hits > 100_000


@gpu
def test_batch_shapes():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    seqs = proteome(150, 4242)
    o = oracle(p, seqs)
    m = o.entries()["mass"]
    mid = float(np.median(m))
    with unbuilt(p, seqs) as g:
        u = Unindexed(g)
        empty = g.search_unindexed(np.zeros(0), np.zeros(0), per_hit=False)
        assert empty["counts"].n_hits == 0 and empty["hit_off"].tolist() == [0] and empty["pep_off"].tolist() == [0]
        assert g.last_candidates == 0
        check_hits(u, o, np.array([10.0, 7000.0, 599.0]), np.array([20.0, 7999.0, 599.5]))  # misses only
        assert g.last_candidates == 0
        check_hits(u, o, np.array([mid + 1.0, 900.0]), np.array([mid - 1.0, 800.0]))  # inverted
        assert g.last_candidates == 0
        nan_lo, nan_hi = np.array([np.nan, 900.0, np.nan]), np.array([1000.0, np.nan, np.nan])
        nan_un = g.search_unindexed(nan_lo, nan_hi)
        lo = np.array([mid - 3.0, mid - 3.0, 0.0, 6500.0, 6100.0, m[0], m[-1], mid - 50.0, mid])
        hi = np.array([mid + 3.0, mid + 3.0, 700.0, 9000.0, 6200.0, m[0], m[-1], mid + 50.0, mid])
        check_hits(u, o, lo, hi)  # duplicates, lo = 0, above max_mass, the extreme entries
        check_hits(u, o, np.array([0.0]), np.array([8000.0]))  # every record is a candidate
        assert g.stats()["n_emitted"] == o.counts()["n_emitted"]
        assert g.stats()["n_entries"] == o.counts()["n_entries"]
        g.build()  # NaN bounds select what dbi_query_hits selects
        assert hits_canonical(nan_un) == hits_canonical(g.query_hits(nan_lo, nan_hi))
        assert nan_un["counts"].n_hits > 0
    with dbi.GpuIndex(p) as g:  # no proteins
        h = g.search_unindexed(np.array([600.0, 0.0]), np.array([700.0, 8000.0]))
        assert h["hit_off"].tolist() == [0, 0, 0] and g.last_candidates == 0


@gpu
def test_candidate_cap():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    seqs = proteome(120, 17)
    o = oracle(p, seqs)
    _, _, lo, hi = synth.synth_queries(o.entries()["mass"], 200, 2)
    with unbuilt(p, seqs) as g:
        first = g.search_unindexed(lo, hi)
        n_c = g.last_candidates
        assert n_c > 1
        with pytest.raises(DbiError) as ei:
            g.search_unindexed(lo, hi, n_c - 1)
        assert ei.value.code == DBI_ERANGE and ei.value.n_candidates == n_c
        with pytest.raises(DbiError) as ei:
            g.query_hits_read(DbiHitBuffers())  # no pending result
        assert ei.value.code == -1
        again = g.search_unindexed(lo, hi, n_c)
        assert g.last_candidates == n_c and g.stats()["n_emitted"] == n_c
        assert hits_canonical(again) == hits_canonical(first) == hits_canonical(o.query_hits(lo, hi))


@gpu
def test_lifecycle():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    seqs = proteome(120, 23)
    o = oracle(p, seqs)
    _, _, lo, hi = synth.synth_queries(o.entries()["mass"], 200, 6, da_fraction=0.3)
    half = len(seqs) // 2
    with dbi.GpuIndex(p) as g:
        g.add_proteins(*pack(seqs[:half]))
        o_half = oracle(p, seqs[:half])
        assert hits_canonical(g.search_unindexed(lo, hi)) == hits_canonical(o_half.query_hits(lo, hi))
        for call in (lambda: g.query_hits(lo, hi), lambda: g.lookup_peptides(["PEPTIDEK"])):
            with pytest.raises(DbiError) as ei:
                call()
            assert ei.value.code == -1  # the handle stays unbuilt
        res2, off2 = pack(seqs[half:])
        g.add_proteins(res2, off2)  # seen by the next search
        check_hits(Unindexed(g), o, lo, hi)
        # a second read finds nothing; a new search drops the pending result of the previous one
        g.search_unindexed_begin(lo[:50], hi[:50])
        cnt = g.search_unindexed_begin(lo[50:], hi[50:])
        raw = g._read_hits(cnt, None, None, False)
        assert raw["counts"].nq == len(lo) - 50
        assert hits_canonical(dbi.capi.expand_hits(raw)) == hits_canonical(o.query_hits(lo[50:], hi[50:]))
        with pytest.raises(DbiError) as ei:
            g.query_hits_read(DbiHitBuffers())
        assert ei.value.code == -1
        # the normal index after searches
        g.build()
        assert_entries_equal(g.fetch(0, g.stats()["n_entries"]), o.entries())
        with pytest.raises(DbiError) as ei:
            g.search_unindexed(lo, hi)
        assert ei.value.code == -2  # DBI_EALREADY: a built handle answers through dbi_query_hits
    with unbuilt(p, seqs) as g:
        assert g.lib.dbi_mg_begin(g._h, C.c_int(0), C.c_int(2)) == 0
        with pytest.raises(DbiError) as ei:
            g.search_unindexed(lo, hi)
        assert ei.value.code == -3  # DBI_EINVAL: multi-GPU unindexed search is not supported


def _keys(seqs_list):
    return sorted((s.key(), tuple(s.proteinIds), s.resLeft, s.resRight, s.sequenceOffset, s.sequenceLen)
                  for s in seqs_list)


@gpu
@pytest.mark.parametrize("cap", [None, 40])
def test_mirror_unindexed_equals_indexed(cap):
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    seqs = proteome(100, 61)
    defs = synth.deflines(len(seqs))
    idx = DBIndexImpl(DBIndexSearchParams(params=p, dataBaseName="idx.fasta"), proteins=(defs, seqs))
    un = DBIndexImpl(DBIndexSearchParams(params=p, dataBaseName="unidx.fasta", useIndex=False), proteins=(defs, seqs))
    try:
        assert idx.indexer.use_index and not un.indexer.use_index
        calls = []
        if cap is not None:
            un.indexer.max_candidates = cap
            inner = un.indexer.index.search_unindexed
            un.indexer.index.search_unindexed = lambda *a, **k: calls.append(1) or inner(*a, **k)
        exp = idx.indexer.index.fetch(0, idx.indexer.getNumberSequences(), with_ids=False)["mass"]
        picks = [float(exp[i]) for i in np.linspace(0, len(exp) - 1, 12).astype(int)]
        for m in picks + [1234.5678, 7990.0]:
            assert _keys(un.getSequences(m, 0.02)) == _keys(idx.getSequences(m, 0.02)), m
            assert _keys(un.indexer.getSequencesUsingPPMTolerance(m, 10.0)) == \
                _keys(idx.indexer.getSequencesUsingPPMTolerance(m, 10.0)), m
        rs = [MassRange(picks[3], 0.5), MassRange(picks[3] + 0.2, 0.5), MassRange(picks[7], 0.01)]
        assert _keys(un.getSequences(rs)) == _keys(idx.getSequences(rs))
        peps = [s.sequence for s in idx.getSequences(picks[5], 1.0) if not s.modPositions][:20]
        assert peps
        negatives = [peps[0][::-1], peps[0].lower(), peps[0][:-1], peps[0] + "K", "", "PEPTIDEXK"]
        for s in peps + negatives:
            assert un.getProteins(s) == idx.getProteins(s), s
        assert un.getProteins(peps + negatives) == idx.getProteins(peps + negatives)
        assert any(un.getProteins(peps))
        if cap is not None:
            assert len(calls) > 1
        for call in (un.indexer.getNumberSequences, un.indexer.getParentMasses):
            with pytest.raises(DBIndexStoreException):
                call()
    finally:
        idx.close()
        un.close()
