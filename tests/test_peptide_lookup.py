"""Batched peptide lookup (dbi_lookup_peptides; getProteins(String) for a whole list) against the oracle's index.

The expectation is keyed independently of any GPU search logic: a dict from (peptide string cut from the
oracle's first occurrence, mod pattern) to (entry position, first occurrence, protein list)."""
import ctypes as C
import os

import numpy as np
import pytest

from dbindex_b200 import synth
from oracle.oracle_py import Oracle
from oracle.oracle_py import default_params as oracle_params

from .test_java_layout import JAVA, parse_layout
from .util import PARAM_SETS, bits

NCPU = os.cpu_count() or 1
ABSENT, FOUND, MALFORMED = 0, 1, 2
LONG_PROTEIN = "G" * 70 + "MSTYMWSTK" + "G" * 12 + "MR"  # peptides longer than 64 residues with mod sites


def proteome(seed, n_prot=120):
    res, off = synth.synth_proteome(n_prot, seed, median_len=300, min_len=5)
    seqs = [res[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(len(off) - 1)]
    seqs += [seqs[0], "AAGGLLKGGAALLKAAGGLLK", LONG_PROTEIN, "A" * 66 + "SSTTYYMMWK", seqs[3]]
    return seqs


def packed(seqs):
    residues = np.frombuffer("".join(seqs).encode("latin-1"), dtype=np.uint8)
    offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=offsets[1:])
    return residues, offsets


def oracle_entries(params, seqs):
    o = Oracle(params, threads=NCPU)
    o.add_proteins(*packed(seqs))
    assert o.build() == 0
    return o.entries()


def entry_peptides(seqs, e):
    return [seqs[p][f:f + n] for p, f, n in zip(e["first_prot"].tolist(), e["first_off"].tolist(), e["len"].tolist())]


def expectation(seqs, e):
    """(peptide, pattern) -> (entry position, first_prot, first_off, protein ids)"""
    plo = e["prot_list_off"].astype(np.int64)
    d = {}
    for i, (pep, pat) in enumerate(zip(entry_peptides(seqs, e), e["modpat"].tolist())):
        assert (pep, pat) not in d, (pep, pat)
        d[(pep, pat)] = (i, int(e["first_prot"][i]), int(e["first_off"][i]), tuple(e["prot_ids"][plo[i]:plo[i + 1]].tolist()))
    return d


def spec_mass(params, peps, pats):
    """The lookup mass restated in numpy float64: calculateMass (IndexUtil.java:198-207: h2o_proton if added, cterm,
    nterm, the residues left to right), then the diff-mod shift of every pattern position in pattern order."""
    table = np.array(params.residue_mass[:], dtype=np.float64)
    diff = np.zeros(256, np.float64)
    for k in range(params.n_mods):  # DiffModification: last one wins
        diff[params.mods[k].residue] = params.mods[k].delta
    n, lmax = len(peps), max(len(p) for p in peps)
    codes = np.zeros((n, lmax), np.uint8)
    for i, p in enumerate(peps):
        codes[i, :len(p)] = np.frombuffer(p.encode(), np.uint8)
    m = np.zeros(n, np.float64)
    if params.add_h2o_proton:
        m = m + params.h2o_proton
    m = m + params.cterm
    m = m + params.nterm
    masses = np.where(np.arange(lmax)[None, :] < np.array([len(p) for p in peps])[:, None], table[codes], 0.0)
    for k in range(lmax):  # x + 0.0 == x: the padding leaves the chain of a shorter peptide untouched
        m = m + masses[:, k]
    pats = np.asarray(pats, np.uint32)
    for k in range(4):
        b = ((pats >> np.uint32(8 * k)) & np.uint32(0xFF)).astype(np.int64)
        res = codes[np.arange(n), np.maximum(b - 1, 0)]
        m = m + np.where(b > 0, diff[res], 0.0)
    return m


# ---- CPU ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["cfg1_tryptic", "cfg2_mods", "lysc_neg_mod", "avg_no_h2o", "many_classes",
                                  "wide_mass_mod4", "semi_nocut_mods"])
def test_lookup_mass_spec_matches_every_indexed_mass(name):
    p = oracle_params(**PARAM_SETS[name])
    seqs = proteome(31 + len(name), n_prot=60)
    e = oracle_entries(p, seqs)
    got = spec_mass(p, entry_peptides(seqs, e), e["modpat"])
    assert np.array_equal(bits(got), bits(e["mass"])), np.nonzero(bits(got) != bits(e["mass"]))[0][:10]


def test_java_lookup_layouts_match_the_c_abi(tmp_path):
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    probe = tmp_path / "probe.c"
    probe.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "dbindex_gpu.h"
#define P(s, f) printf(#s "." #f " %zu\n", offsetof(s, f))
int main(void) {
  P(dbi_lookup_counts, n); P(dbi_lookup_counts, n_found); P(dbi_lookup_counts, n_prot_ids);
  printf("dbi_lookup_counts.sizeof %zu\n", sizeof(dbi_lookup_counts));
  P(dbi_lookup_buffers, status); P(dbi_lookup_buffers, mass); P(dbi_lookup_buffers, entry);
  P(dbi_lookup_buffers, first_prot); P(dbi_lookup_buffers, first_off); P(dbi_lookup_buffers, prot_list_off);
  P(dbi_lookup_buffers, prot_ids);
  printf("dbi_lookup_buffers.sizeof %zu\n", sizeof(dbi_lookup_buffers));
  return 0;
}
''')
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(root, "include"), str(probe), "-o", str(exe)])
    c = {k: int(v) for k, v in (line.split() for line in subprocess.check_output([str(exe)], text=True).split("\n") if line)}
    src = open(JAVA).read()
    for jname, cname in (("LOOKUP_COUNTS", "dbi_lookup_counts"), ("LOOKUP_BUFFERS", "dbi_lookup_buffers")):
        fields, size = parse_layout(src, jname, {})
        expect = {k.split(".", 1)[1]: v for k, v in c.items() if k.startswith(cname + ".") and not k.endswith(".sizeof")}
        assert fields == expect, (jname, fields, expect)
        assert size == c[cname + ".sizeof"], (jname, size)


# ---- GPU ---------------------------------------------------------------------------------------------------
def gpu_index(params, seqs):
    import dbindex_b200 as dbi
    g = dbi.GpuIndex(params)
    g.add_proteins(*packed(seqs))
    g.build()
    return g


def check_rows(g, r, rows, d, whole=None):
    """Every row's answer against the dict: status, entry (through the whole fetched index), first occurrence,
    protein list with duplicates in order."""
    plo = r["prot_list_off"].astype(np.int64)
    for i, (pep, pat) in enumerate(rows):
        exp = d.get((pep, pat))
        if exp is None:
            assert r["status"][i] in (ABSENT, MALFORMED), (i, pep, pat, r["status"][i])
            assert plo[i + 1] == plo[i] and r["entry"][i] == np.iinfo(np.uint64).max
            continue
        assert r["status"][i] == FOUND, (i, pep, pat)
        assert (int(r["first_prot"][i]), int(r["first_off"][i])) == exp[1:3], (i, pep)
        assert tuple(r["prot_ids"][plo[i]:plo[i + 1]].tolist()) == exp[3], (i, pep)
        if whole is not None:
            e = int(r["entry"][i])
            assert bits(whole["mass"][e:e + 1])[0] == bits(r["mass"][i:i + 1])[0]
            assert int(whole["modpat"][e]) == pat and int(whole["len"][e]) == len(pep)
            assert (int(whole["first_prot"][e]), int(whole["first_off"][e])) == exp[1:3]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg1_tryptic", "cfg2_mods", "many_classes", "lysc_neg_mod", "avg_no_h2o",
                                  "wide_mass_mod4", "semi_nocut_mods"])
def test_every_entry_is_found(name):
    import dbindex_b200 as dbi
    p = dbi.default_params(**PARAM_SETS[name])
    seqs = proteome(700 + len(name))
    e = oracle_entries(p, seqs)
    d = expectation(seqs, e)
    rows = list(d)
    g = gpu_index(p, seqs)
    try:
        r = g.lookup_peptides([k[0] for k in rows], [k[1] for k in rows])
        assert r["counts"].n_found == len(rows) and np.all(r["status"] == FOUND)
        assert np.array_equal(bits(r["mass"]), bits(e["mass"][[d[k][0] for k in rows]]))
        if p.n_mods:
            assert max(len(k[0]) for k in rows) > 64  # the long expansion path is among them
        check_rows(g, r, rows, d, g.fetch(0, g.stats()["n_entries"]))
    finally:
        g.close()


def negatives(peps):
    out = []
    for s in peps:
        sw = s.translate(str.maketrans("LI", "IL"))
        out += [sw, s[::-1], s[1:] + s[0], s[1:], s[:-1], s + "A", "K" + s, s.lower()]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg1_tryptic", "cfg2_mods", "lysc_neg_mod"])
def test_negatives_are_not_found(name):
    import dbindex_b200 as dbi
    p = dbi.default_params(**PARAM_SETS[name])
    seqs = proteome(900 + len(name))
    e = oracle_entries(p, seqs)
    d = expectation(seqs, e)
    base = [k[0] for k in d if k[1] == 0]
    rows = [(s, 0) for s in negatives(base[::7])]
    assert any(s != s.translate(str.maketrans("LI", "IL")) for s, _ in rows)
    if p.n_mods:
        # every single-site variant of the heaviest peptides: the ones whose shifted mass leaves [min, max] are
        # well formed and not indexed (status 0)
        diff = {p.mods[k].residue: p.mods[k].delta for k in range(p.n_mods)}
        heavy = [s for s, m in zip(entry_peptides(seqs, e), e["mass"]) if m > p.max_mass - 100 or m < p.min_mass + 20]
        for s in heavy:
            rows += [(s, j + 1) for j, ch in enumerate(s[:255]) if ord(ch) in diff]
    g = gpu_index(p, seqs)
    try:
        r = g.lookup_peptides([k[0] for k in rows], [k[1] for k in rows])
        check_rows(g, r, rows, d)
        assert not np.any(r["status"] == MALFORMED)
        exp_found = np.array([k in d for k in rows])
        assert np.array_equal(r["status"] == FOUND, exp_found)
        assert np.count_nonzero(~exp_found) > 0
        if p.n_mods:
            assert any(k[1] and k not in d for k in rows)  # variants excluded by the mass range were asked
    finally:
        g.close()


@pytest.mark.gpu
def test_malformed_rows_do_not_fail_the_batch():
    import dbindex_b200 as dbi
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    seqs = proteome(41)
    e = oracle_entries(p, seqs)
    d = expectation(seqs, e)
    good = [k for k in d if k[1]][:40] + [k for k in d if not k[1]][:40]
    sty = next(k[0] for k in d if sum(ch in "STY" for ch in k[0][:200]) >= 4)
    sites = [j + 1 for j, ch in enumerate(sty) if ch in "STY"][:4]
    a_pos = next(j + 1 for j, ch in enumerate(good[0][0]) if ch not in "MSTY")
    pep = good[0][0]
    bad = [("", 0), ("A" * 65536, 0),
           (sty, sites[1] | sites[0] << 8),              # not ascending
           (sty, sites[0] | sites[1] << 16),             # a nonzero byte after a zero byte
           (pep, len(pep) + 1),                          # position beyond the peptide
           (pep, a_pos),                                 # residue without a shift
           (sty, sites[0] | sites[1] << 8 | sites[2] << 16 | sites[3] << 24)]  # 4 mods > max_mods_per_peptide = 3
    rows = []
    for k, b in enumerate(bad):
        rows += [good[2 * k], b, good[2 * k + 1]]
    g = gpu_index(p, seqs)
    try:
        r = g.lookup_peptides([k[0] for k in rows], [k[1] for k in rows])
        assert np.array_equal(np.nonzero(r["status"] == MALFORMED)[0], np.arange(1, len(rows), 3))
        assert np.all(r["mass"][1::3] == 0.0)
        check_rows(g, r, rows, d)
    finally:
        g.close()
    # any pattern is malformed on an index without differential mods
    p1 = dbi.default_params()
    e1 = oracle_entries(p1, seqs)
    d1 = expectation(seqs, e1)
    pep1 = next(iter(d1))[0]
    g = gpu_index(p1, seqs)
    try:
        r = g.lookup_peptides([pep1, pep1, pep1], [0, 1, 0])
        assert r["status"].tolist() == [FOUND, MALFORMED, FOUND]
    finally:
        g.close()


@pytest.mark.gpu
def test_batch_shapes():
    import dbindex_b200 as dbi
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    seqs = proteome(43)
    e = oracle_entries(p, seqs)
    d = expectation(seqs, e)
    keys = list(d)
    g = gpu_index(p, seqs)
    try:
        r = g.lookup_peptides([])
        assert r["counts"].n == 0 and r["prot_list_off"].tolist() == [0] and len(r["prot_ids"]) == 0
        for rows in ([keys[5]], [keys[9]] * 1000,
                     [keys[i] for i in np.random.default_rng(3).integers(0, len(keys), 100_000)],
                     [k for k in keys if len(k[0]) > 64]):
            assert rows
            r = g.lookup_peptides([k[0] for k in rows], [k[1] for k in rows])
            assert r["counts"].n_found == len(rows)
            check_rows(g, r, rows, d)
        # all unmodified: modpat = None
        unmod = [k for k in keys if not k[1]][:500]
        r = g.lookup_peptides([k[0] for k in unmod])
        check_rows(g, r, unmod, d)
    finally:
        g.close()


@pytest.mark.gpu
def test_get_proteins_batch_equals_single_and_oracle():
    import dbindex_b200 as dbi
    from dbindex_b200.indexer import DBIndexImpl
    p = dbi.default_params()
    seqs = proteome(77, n_prot=60)
    defs = synth.deflines(len(seqs))
    e = oracle_entries(p, seqs)
    d = expectation(seqs, e)
    peps = [k[0] for k in d][::3]
    asked = peps + negatives(peps[:20]) + peps[:5]
    impl = DBIndexImpl(p, proteins=(defs, seqs))
    try:
        batch = impl.getProteins(asked)
        impl._proteins_by_seq.clear()
        single = [impl.getProteins(s) for s in asked]
        assert batch == single
        for s, got in zip(asked, batch):
            exp = d.get((s, 0))
            assert {q.id for q in got} == (set(exp[3]) if exp else set()), s
            assert all(q.accession == defs[q.id] for q in got)
        assert impl.getProteins(asked[0]) is impl.getProteins([asked[0]])[0]  # memoised
    finally:
        impl.close()


@pytest.mark.gpu
def test_lookup_lifecycle(tmp_path):
    import dbindex_b200 as dbi
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    seqs = proteome(45, n_prot=80)
    e = oracle_entries(p, seqs)
    d = expectation(seqs, e)
    rows = list(d)[::5]
    peps, pats = [k[0] for k in rows], [k[1] for k in rows]
    g = dbi.GpuIndex(p)
    try:
        with pytest.raises(dbi.DbiError) as ei:
            g.lookup_peptides(peps, pats)
        assert ei.value.code == -1
        g.add_proteins(*packed(seqs))
        g.build()
        with pytest.raises(dbi.DbiError) as ei:
            g.lookup_peptides_read(dbi.capi.DbiLookupCounts())
        assert ei.value.code == -1
        ref = g.lookup_peptides(peps, pats)
        check_rows(g, ref, rows, d)
        lo, hi = e["mass"][::50] - 0.01, e["mass"][::50] + 0.01
        hits_ref = g.query_hits(lo, hi, per_hit=False)

        def read_hits(cnt):
            out, bufs = {}, dbi.capi.DbiHitBuffers()
            for name, (dt, size) in dbi.capi.HIT_FIELDS.items():
                out[name] = a = np.empty(int(size(cnt)), dt)
                setattr(bufs, name, a.ctypes.data)
            g.query_hits_read(bufs)
            return out

        def same(a, b, names):
            return all(np.array_equal(a[k], b[k]) for k in names)

        # both pending at once, read in either order
        ch = g.query_hits_begin(lo, hi)
        cl = g.lookup_peptides_begin(peps, pats)
        assert same(g.lookup_peptides_read(cl), ref, dbi.capi.LOOKUP_FIELDS)
        assert same(read_hits(ch), hits_ref, dbi.capi.HIT_FIELDS)
        cl = g.lookup_peptides_begin(peps, pats)
        ch = g.query_hits_begin(lo, hi)
        assert same(read_hits(ch), hits_ref, dbi.capi.HIT_FIELDS)
        assert same(g.lookup_peptides_read(cl), ref, dbi.capi.LOOKUP_FIELDS)
        # a read consumes the result; reset_index drops a pending one
        with pytest.raises(dbi.DbiError) as ei:
            g.lookup_peptides_read(cl)
        assert ei.value.code == -1
        cl = g.lookup_peptides_begin(peps, pats)
        g.reset_index()
        with pytest.raises(dbi.DbiError) as ei:
            g.lookup_peptides_read(cl)
        assert ei.value.code == -1
        g.build()
        path = str(tmp_path / "index.gpuidx")
        g.save(path)
        g2 = dbi.GpuIndex(p)
        try:
            g2.load(path)
            assert same(g2.lookup_peptides(peps, pats), ref, dbi.capi.LOOKUP_FIELDS)
        finally:
            g2.close()
        lib = g.lib
        assert lib.dbi_lookup_peptides(g._h, None, None, None, 3, C.byref(dbi.capi.DbiLookupCounts())) == -3
    finally:
        g.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name,world", [("cfg1_tryptic", 2), ("cfg2_mods", 3)])
def test_sharded_lookup_in_one_process(name, world):
    import dbindex_b200 as dbi
    from dbindex_b200.multigpu import build_local, lookup_local, owned_mask, shard_proteins, split_masses

    from .test_gpu_parity import _dup_proteome
    p = dbi.default_params(**PARAM_SETS[name])
    res, off = _dup_proteome(600)
    seqs = [res[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(len(off) - 1)]
    e = oracle_entries(p, seqs)
    d = expectation(seqs, e)
    rows = list(d)
    rows += [(s, 0) for s in negatives([k[0] for k in rows if not k[1]][::40])]
    peps, pats = [k[0] for k in rows], [k[1] for k in rows]
    handles = []
    try:
        for r in range(world):
            g = dbi.GpuIndex(p)
            sres, soff, _ = shard_proteins(res, off, r, world)
            g.add_proteins(sres, soff)
            handles.append(g)
        build_local(handles)
        split = split_masses(handles[0], world)
        got = lookup_local(handles, peps, pats)
        check_rows(handles[0], got, rows, d)
        found = got["status"] == FOUND
        assert np.array_equal(found, [k in d for k in rows])
        for r in range(world):
            mine = got["rank"] == r
            assert np.array_equal(mine, found & owned_mask(got["mass"], split, r, world))
        if p.n_mods:  # variants that live on another rank than their unmodified peptide were resolved
            rank_of = {k: int(got["rank"][i]) for i, k in enumerate(rows) if found[i]}
            assert any(rank_of[k] != rank_of[(k[0], 0)] for k in rank_of if k[1])
        single = gpu_index(p, seqs)
        try:
            one = single.lookup_peptides(peps, pats)
        finally:
            single.close()
        for k in ("status", "mass", "first_prot", "first_off", "prot_list_off", "prot_ids"):
            assert np.array_equal(got[k], one[k]), k
    finally:
        for g in handles:
            g.close()
