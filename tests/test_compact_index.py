"""Compact variant index: a single-GPU group-path index that keeps the sorted variant groups and expands the entries
a query returns (K6q) instead of writing every entry at build time.  It is chosen when the entries would reach
2^32; DBI_COMPACT_VARIANTS forces it on small proteomes so that both layouts can be compared answer by answer.

GPU: every query entry point of a compact index against the expanded index of the same proteome, byte for byte,
and an index of 4.35 x 10^9 entries on one GPU.  CPU: the block order of K6x and its inverse rank (the lookup's
entry number) restated in numpy against brute-force enumeration, and the dbi_stats field n_groups."""
import ctypes as C
import itertools
import os

import numpy as np
import pytest

import dbindex_b200 as dbi
from dbindex_b200 import synth
from dbindex_b200.capi import (DBI_ERANGE, DBI_TOL_DA, DBI_TOL_PPM, HIT_FIELDS, DbiError, DbiHitBuffers,
                                DbiHitCounts, DbiStats, _ptr, spectra_arrays)

from .util import PARAM_SETS, bits

ENV = "DBI_COMPACT_VARIANTS"
GROUP_SETS = ["cfg2_mods", "semi_nocut_mods", "lysc_neg_mod", "three_classes_k2", "five_classes_k2",
              "filter_K2_mods", "wide_mass_mod4"]
# peptides of 66 to 90 light residues between cuts: many groups belong to peptides longer than 64 residues (K6l)
LONG_PARAMS = dict(enzyme="K", diff_mods=[("S", 79.96633), ("M", 15.9949)], max_mods_per_peptide=3, max_missed=0)


# ---- CPU: block order and rank ----------------------------------------------------------------------------------
def block_order(k, masks):
    """The entries of one group in K6x's order (mods_grp.cu block_entry): tuples of site positions."""
    c = [sorted(m) for m in masks]
    if k == 0:
        return [()]
    if k == 1:
        return [(p,) for p in c[0]]
    out = []
    if k == 2:
        for p in c[0]:
            out += [(p, b) for b in c[1] if b > p]
        return out
    for p in c[1]:  # block = the second site
        left = [a for a in c[0] if a < p]
        if k == 3:
            out += [(a, p, b) for a in left for b in c[2] if b > p]
        else:
            pairs = [(i2, i3) for i2 in c[2] if i2 > p for i3 in c[3] if i3 > i2]
            out += [(a, p, i2, i3) for a in left for (i2, i3) in pairs]
    return out


def popc(m, lo, hi):
    """sites of mask m strictly between lo and hi"""
    return sum(1 for x in m if lo < x < hi)


def entry_rank(k, pos, masks):
    """numpy-free restatement of group_entry_rank (mods_common.cuh)"""
    c0, c1, c2, c3 = (list(masks) + [[]] * 4)[:4]
    if k == 0:
        return 0
    if k == 1:
        return popc(c0, -1, pos[0])
    pb = pos[0] if k == 2 else pos[1]
    sites = c0 if k == 2 else c1

    def size(p):
        if k == 2:
            return popc(c1, p, 99)
        nl = popc(c0, -1, p)
        if k == 3:
            return nl * popc(c2, p, 99)
        return nl * sum(popc(c3, y, 99) for y in c2 if y > p)

    r = sum(size(x) for x in sites if x < pb)
    if k == 2:
        return r + popc(c1, pos[0], pos[1])
    a = popc(c0, -1, pos[0])
    if k == 3:
        return r + a * popc(c2, pb, 99) + popc(c2, pb, pos[2])
    w2 = sum(popc(c3, y, 99) for y in c2 if y > pb)
    b = sum(popc(c3, y, 99) for y in c2 if pb < y < pos[2]) + popc(c3, pos[2], pos[3])
    return r + a * w2 + b


def long_rank(k, pos, cls_of, want):
    """group_rank's right-to-left count for peptides over 64 residues (lexicographic order of the site tuples)"""
    S = [0] * k + [1]
    rank = 0
    for x in range(len(cls_of) - 1, -1, -1):
        for j in range(k):
            if cls_of[x] != want[j]:
                continue
            if x < pos[j] and (j == 0 or x > pos[j - 1]):
                rank += S[j + 1]
            S[j] += S[j + 1]
    return rank


@pytest.mark.parametrize("k", [1, 2, 3, 4])
def test_block_order_rank_cpu(k):
    rng = np.random.default_rng(k)
    for trial in range(60):
        L = int(rng.integers(k, 40))
        n_cls = int(rng.integers(1, 3))
        cls_of = rng.integers(-1, n_cls, L)  # -1: no site
        seq = [int(x) for x in rng.integers(0, n_cls, k)]
        masks = [[i for i in range(L) if cls_of[i] == seq[j]] for j in range(k)]
        order = block_order(k, masks)
        # the block order lists every chain of the class sequence exactly once
        chains = [t for t in itertools.combinations(range(L), k) if all(cls_of[t[j]] == seq[j] for j in range(k))]
        assert sorted(order) == chains
        for r, t in enumerate(order):
            assert entry_rank(k, t, masks) == r
        for r, t in enumerate(chains):  # lexicographic: the order of K6l
            assert long_rank(k, t, list(cls_of), seq) == r


def test_stats_n_groups_layout():
    # n_groups takes the place of the u32 padding after exp_ms: size and every other offset unchanged
    assert DbiStats.n_groups.offset == DbiStats.exp_ms.offset + 4
    assert DbiStats.exp_bytes_per_launch.offset == DbiStats.n_groups.offset + 4
    assert DbiStats.n_groups.size == 4
    assert C.sizeof(DbiStats) == DbiStats.exp_bytes_per_launch.offset + 8
    hdr = open(os.path.join(os.path.dirname(__file__), "..", "include", "dbindex_gpu.h")).read()
    assert "uint32_t n_groups;" in hdr and "uint32_t _pad;" not in hdr


# ---- GPU ----------------------------------------------------------------------------------------------------------
def build(params, res, off, compact, monkeypatch):
    if compact:
        monkeypatch.setenv(ENV, "1")
    else:
        monkeypatch.delenv(ENV, raising=False)
    g = dbi.GpuIndex(params)
    g.add_proteins(res, off)
    g.build()
    monkeypatch.delenv(ENV, raising=False)
    return g


def raw_hits(g, call, *args, **kw):
    """every buffer of dbi_query_hits_read, as the library delivers them"""
    cnt = call(*args, **kw)
    out, bufs = {}, DbiHitBuffers()
    for name, (dt, size) in HIT_FIELDS.items():
        out[name] = np.empty(int(size(cnt)), dtype=dt)
        setattr(bufs, name, out[name].ctypes.data)
    g.query_hits_read(bufs)
    return (cnt.nq, cnt.n_hits, cnt.n_peps, cnt.n_seq_bytes, cnt.n_prot_ids), out


def spectra_begin(g, mass, tol, range_off, mode):
    mass, tol, range_off, n = spectra_arrays(mass, tol, range_off, mode)
    cnt = DbiHitCounts()
    g._check(g.lib.dbi_query_spectra(g._h, _ptr(mass), _ptr(tol), _ptr(range_off), n, mode, 0, C.byref(cnt)))
    return cnt


def assert_same_raw(a, b):
    assert a[0] == b[0], (a[0], b[0])
    for k in a[1]:
        assert np.array_equal(a[1][k].view(np.uint8), b[1][k].view(np.uint8)), f"{k} differs"


def long_proteome(n, seed):
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(b"GGAASSSMLV", np.uint8)
    prots = []
    for _ in range(n):
        segs = [rng.choice(alpha, int(rng.integers(66, 91) if rng.random() < 0.7 else rng.integers(8, 60)))
                for _ in range(int(rng.integers(2, 6)))]
        prots.append(b"K".join(s.tobytes() for s in segs) + b"K")
    off = np.zeros(n + 1, np.uint64)
    off[1:] = np.cumsum([len(p) for p in prots])
    return np.frombuffer(b"".join(prots), np.uint8).copy(), off


def proteome(name):
    if name == "long_peptides":
        return dbi.default_params(**LONG_PARAMS), *long_proteome(300, 7)
    n = 1500 if name == "cfg2_mods" else 300
    return dbi.default_params(**PARAM_SETS[name]), *synth.synth_proteome(n, 4242)


@pytest.mark.gpu
@pytest.mark.parametrize("name", GROUP_SETS + ["long_peptides"])
def test_compact_equals_expanded(name, monkeypatch, tmp_path):
    p, res, off = proteome(name)
    ge = build(p, res, off, False, monkeypatch)
    gc = build(p, res, off, True, monkeypatch)
    se, sc = ge.stats(), gc.stats()
    V = se["n_entries"]
    assert sc["n_entries"] == V and sc["n_unique"] == se["n_unique"] and V > 0
    assert se["n_groups"] == 0 and 0 < sc["n_groups"] <= V
    if name == "cfg2_mods":
        assert sc["device_bytes"] < se["device_bytes"]
    whole = ge.fetch(0, V)
    if name == "long_peptides":
        assert np.count_nonzero(whole["len"] > 64) > V // 10
    # fetch: the whole index and random ranges
    assert_fetch_equal(ge.fetch(0, V), gc.fetch(0, V))
    rng = np.random.default_rng(11)
    for _ in range(20):
        b = int(rng.integers(0, V))
        c = int(rng.integers(0, min(V - b, 5000) + 1))
        assert_fetch_equal(ge.fetch(b, c), gc.fetch(b, c))
    # hit batches: 10 ppm and +-3 Da, empty, all-miss, the whole index
    m = whole["mass"]
    _, _, lo, hi = synth.synth_queries(m, 3000, 5, da_fraction=0.3)
    batches = [(lo, hi), (lo[:0], hi[:0]), (np.full(7, 1.0), np.full(7, 2.0)),
               (np.array([0.0]), np.array([9000.0])), (np.array([m[0], m[-1]]), np.array([m[0], m[-1]]))]
    for lo_, hi_ in batches:
        assert_same_raw(raw_hits(ge, ge.query_hits_begin, lo_, hi_), raw_hits(gc, gc.query_hits_begin, lo_, hi_))
        be, ce = ge.query(lo_, hi_)
        bc, cc = gc.query(lo_, hi_)
        assert np.array_equal(be, bc) and np.array_equal(ce, cc)
    # spectra: Dalton lists and PPM
    sp = m[rng.integers(0, V, 400)]
    tol = np.full(len(sp), 0.5)
    ro = np.arange(0, len(sp) + 1, 2, dtype=np.uint64)
    assert_same_raw(raw_hits(ge, spectra_begin, ge, sp, tol, ro, DBI_TOL_DA),
                    raw_hits(gc, spectra_begin, gc, sp, tol, ro, DBI_TOL_DA))
    for ppm in (5.0, 10.0, 50.0):
        t = np.full(len(sp), ppm)
        assert_same_raw(raw_hits(ge, spectra_begin, ge, sp, t, None, DBI_TOL_PPM),
                        raw_hits(gc, spectra_begin, gc, sp, t, None, DBI_TOL_PPM))
    # entry keys
    assert np.array_equal(ge.entry_keys(), gc.entry_keys())
    # lookup: every entry (sampled on the larger sets) plus negatives
    idx = np.arange(V) if V <= 300_000 else np.sort(rng.choice(V, 300_000, replace=False))
    seqs, pats = lookup_rows(whole, res, off, idx)
    neg_pats = pats.copy()
    neg_pats[::3] = 0x01020304  # mostly malformed or absent
    for pt in (pats, neg_pats):
        le, lc = ge.lookup_peptides(seqs, pt), gc.lookup_peptides(seqs, pt)
        for k in le:
            assert np.array_equal(np.asarray(le[k]), np.asarray(lc[k])), f"lookup {k} differs"
    lf = ge.lookup_peptides(seqs, pats)
    assert np.all(lf["status"] == 1) and np.array_equal(lf["entry"], idx)
    # save / load
    path = str(tmp_path / "compact.idx")
    gc.save(path)
    gl = dbi.GpuIndex(p)
    gl.load(path)
    assert gl.stats()["n_groups"] == sc["n_groups"] and gl.stats()["n_entries"] == V
    assert_fetch_equal(ge.fetch(0, V), gl.fetch(0, V))
    assert_same_raw(raw_hits(ge, ge.query_hits_begin, lo, hi), raw_hits(gl, gl.query_hits_begin, lo, hi))
    ll = gl.lookup_peptides(seqs, pats)
    assert np.array_equal(ll["entry"], idx)
    # the unindexed search with a compact candidate index
    ue = dbi.GpuIndex(p)
    ue.add_proteins(res, off)
    uc = dbi.GpuIndex(p)
    uc.add_proteins(res, off)
    monkeypatch.delenv(ENV, raising=False)
    a = raw_hits(ue, ue.search_unindexed_begin, lo[:500], hi[:500])
    monkeypatch.setenv(ENV, "1")
    b = raw_hits(uc, uc.search_unindexed_begin, lo[:500], hi[:500])
    monkeypatch.delenv(ENV, raising=False)
    assert ue.stats()["n_groups"] == 0 and uc.stats()["n_groups"] > 0  # the candidate index took the compact layout
    assert_same_raw(a, b)
    for h in (ge, gc, gl, ue, uc):
        h.close()


def assert_fetch_equal(a, b):
    for k in a:
        assert np.array_equal(np.asarray(a[k]).view(np.uint8), np.asarray(b[k]).view(np.uint8)), f"fetch {k} differs"


def lookup_rows(f, res, off, idx):
    """(packed residues, offsets) and patterns of index entries idx, from a fetch of the whole index"""
    starts = off[f["first_prot"][idx].astype(np.int64)].astype(np.int64) + f["first_off"][idx].astype(np.int64)
    lens = f["len"][idx].astype(np.int64)
    qo = np.zeros(len(idx) + 1, np.uint64)
    qo[1:] = np.cumsum(lens)
    gather = np.repeat(starts - qo[:-1].astype(np.int64), lens) + np.arange(int(qo[-1]))
    return (res[gather], qo), f["modpat"][idx].astype(np.uint32)


@pytest.mark.gpu
def test_long_group_list_overflow(monkeypatch):
    """K6q lists the groups of peptides over 64 residues per (group, tile) in room for n_tiles + 1024 pairs and runs
    the tiles again with a larger list when they overflow it.  Here every peptide is a 70-mer with one site, so each
    contributes one 1-entry long group: the whole-index fetch has n_tiles = ceil(2 N / 512) tiles and N pairs."""
    rng = np.random.default_rng(31)
    N = 4000
    body = rng.choice(np.frombuffer(b"GALV", np.uint8), (N, 70))
    body[np.arange(N), rng.integers(0, 70, N)] = ord("S")
    prot = np.concatenate([body, np.full((N, 1), ord("K"), np.uint8)], axis=1)
    res, off = prot.reshape(-1).copy(), np.arange(0, 71 * (N + 1), 71, dtype=np.uint64)
    p = dbi.default_params(enzyme="K", max_missed=0, diff_mods=[("S", 79.96633)], max_mods_per_peptide=1,
                           max_mass=8000.0)
    ge = build(p, res, off, False, monkeypatch)
    gc = build(p, res, off, True, monkeypatch)
    V = ge.stats()["n_entries"]
    assert V == 2 * N and gc.stats()["n_groups"] == 2 * N
    assert N > -(-V // 512) + 1024  # more pairs than the first list holds
    assert_fetch_equal(ge.fetch(0, V), gc.fetch(0, V))
    lo, hi = np.array([0.0]), np.array([9000.0])
    assert_same_raw(raw_hits(ge, ge.query_hits_begin, lo, hi), raw_hits(gc, gc.query_hits_begin, lo, hi))
    whole = ge.fetch(0, V)
    seqs, pats = lookup_rows(whole, res, off, np.arange(V))
    assert np.array_equal(gc.lookup_peptides(seqs, pats)["entry"], np.arange(V))
    ge.close()
    gc.close()


# ---- GPU: beyond 2^32 entries on one GPU ----------------------------------------------------------------------
BIG_PARAMS = dict(enzyme="K", max_missed=0, diff_mods=[("ST", 79.966)], max_mods_per_peptide=4, max_mass=8000.0)
BIG_N = 8300
BIG_PER_PEP = sum(int(np.prod(range(61 - k, 61)) // np.prod(range(1, k + 1))) for k in range(5))  # 523 686


def big_proteome():
    rng = np.random.default_rng(2024)
    body = np.where(rng.random((BIG_N, 60)) < 0.5, ord("S"), ord("T")).astype(np.uint8)
    prot = np.concatenate([body, np.full((BIG_N, 1), ord("K"), np.uint8)], axis=1)
    off = np.arange(0, 61 * (BIG_N + 1), 61, dtype=np.uint64)
    return prot.reshape(-1), off, body


@pytest.mark.gpu
def test_beyond_2_32_entries(monkeypatch):
    monkeypatch.delenv(ENV, raising=False)
    p = dbi.default_params(**BIG_PARAMS)
    res, off, body = big_proteome()
    g = dbi.GpuIndex(p)
    g.add_proteins(res, off)
    g.build()
    st = g.stats()
    n_pep = st["n_unique"]
    assert n_pep == BIG_N  # distinct 60-mers
    assert BIG_PER_PEP == 523_686
    assert st["n_entries"] == n_pep * BIG_PER_PEP > 2 ** 32
    assert st["n_groups"] == 5 * n_pep
    # windows on every variant mass of the rarest S counts: every hit protein has that S count, and no other
    # (S count, mods) pair shares a mass
    n_s = (body == ord("S")).sum(axis=1)
    counts = np.bincount(n_s, minlength=61)
    rare = [int(s) for s in np.argsort(counts) if counts[s] > 0][:3]
    sub = np.nonzero(np.isin(n_s, rare))[0]
    gs = dbi.GpuIndex(p)
    gs.add_proteins(*pack_prots(res, off, sub))
    gs.build()
    assert gs.stats()["n_groups"] == 0
    ms = gs.fetch(0, gs.stats()["n_entries"])["mass"]
    centers = np.unique(ms)
    lo, hi = centers - 1e-6, centers + 1e-6  # distinct (S count, mods) masses lie > 1 Da apart
    a = dbi.capi.expand_hits(g.query_hits(lo, hi, per_hit=False))
    b = dbi.capi.expand_hits(gs.query_hits(lo, hi, per_hit=False))
    remap = sub.astype(np.uint32)
    assert np.array_equal(a["hit_off"], b["hit_off"])
    assert canon(a) == canon(b, remap)
    # fetch across entry 2^32, and lookups of 4-mod rows there
    b0 = 2 ** 32 - 3000
    f = g.fetch(b0, 6000)
    assert np.all(np.diff(f["mass"]) >= 0)
    four = np.nonzero([(x >> 24) != 0 for x in f["modpat"].tolist()])[0]
    assert len(four) > 0
    idx = np.arange(6000)
    seqs, pats = lookup_rows(f, res, off, idx)
    lk = g.lookup_peptides(seqs, pats)
    assert np.all(lk["status"] == 1)
    assert np.array_equal(lk["entry"], b0 + idx)
    assert np.any(lk["entry"][four] >= 2 ** 32)
    # a window over the whole index: more than 2^32 hits in one query
    with pytest.raises(DbiError) as e:
        g.query_hits(np.array([0.0]), np.array([9000.0]))
    assert e.value.code == DBI_ERANGE
    with pytest.raises(DbiError):
        g.query_hits_read(DbiHitBuffers())  # nothing pending
    g.close()
    gs.close()


def pack_prots(res, off, ids):
    parts = [res[int(off[i]):int(off[i + 1])] for i in ids]
    o = np.zeros(len(ids) + 1, np.uint64)
    o[1:] = np.cumsum([len(x) for x in parts])
    return np.concatenate(parts), o


def canon(h, remap=None):
    ho, so, po = (h[k].astype(np.int64) for k in ("hit_off", "seq_off", "prot_list_off"))
    out = []
    for q in range(len(ho) - 1):
        rows = []
        for i in range(ho[q], ho[q + 1]):
            fp = int(h["first_prot"][i])
            ids = h["prot_ids"][po[i]:po[i + 1]]
            if remap is not None:
                fp, ids = int(remap[fp]), remap[ids]
            rows.append((int(bits(h["mass"][i:i + 1])[0]), fp, int(h["first_off"][i]), int(h["modpat"][i]),
                         h["seq"][so[i]:so[i + 1]].tobytes(), tuple(int(x) for x in ids)))
        out.append(sorted(rows))
    return out
