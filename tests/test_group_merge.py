"""Group path on one GPU: K6g writes one sorted list per class sequence and K7m merges them in one pass.
The index must equal, position by position, the one built through the K7 radix sort of the peptide-major
group records (DBI_GROUP_RADIX), which is what the sharded build still uses."""
import os

import numpy as np
import pytest

import dbindex_b200 as dbi
from dbindex_b200 import synth

from .util import PARAM_SETS, bits, pack

pytestmark = pytest.mark.gpu

GROUP_SETS = ["cfg2_mods", "semi_nocut_mods", "lysc_neg_mod", "three_classes_k2", "five_classes_k2",
              "filter_K2_mods", "wide_mass_mod4"]
FIELDS = ("first_prot", "first_off", "len", "modpat", "prot_list_off")


def build(p, res, off, radix, monkeypatch):
    if radix:
        monkeypatch.setenv("DBI_GROUP_RADIX", "1")
    else:
        monkeypatch.delenv("DBI_GROUP_RADIX", raising=False)
    g = dbi.GpuIndex(p)
    g.add_proteins(res, off)
    g.build()
    monkeypatch.delenv("DBI_GROUP_RADIX", raising=False)
    return g


def assert_same_index(a, b, with_ids=True, chunk=8_000_000):
    n = a.stats()["n_entries"]
    assert b.stats()["n_entries"] == n
    for s in range(0, n, chunk):
        c = min(chunk, n - s)
        fa, fb = a.fetch(s, c, with_ids), b.fetch(s, c, with_ids)
        if not np.array_equal(bits(fa["mass"]), bits(fb["mass"])):
            bad = np.nonzero(bits(fa["mass"]) != bits(fb["mass"]))[0]
            raise AssertionError(f"mass differs at entry {s + bad[0]} ({len(bad)} in chunk)")
        for k in FIELDS:
            if not np.array_equal(fa[k], fb[k]):
                bad = np.nonzero(fa[k] != fb[k])[0]
                raise AssertionError(f"{k} differs at entry {s + bad[0]}: {fa[k][bad[0]]} vs {fb[k][bad[0]]}")
        if with_ids:
            assert np.array_equal(fa["prot_ids"], fb["prot_ids"]), "protein ids differ"
    return n


def compare(p, res, off, monkeypatch, with_ids=True):
    gm = build(p, res, off, False, monkeypatch)
    gr = build(p, res, off, True, monkeypatch)
    try:
        n = assert_same_index(gm, gr, with_ids)
        sm, sr = gm.stats(), gr.stats()
        assert sm["n_entries"] == sr["n_entries"] and sm["n_unique"] == sr["n_unique"]
        assert sm["sort_bits_var"] == 0 and sr["sort_bits_var"] > 0
        return n
    finally:
        gm.close()
        gr.close()


def proteome(n, seed):
    res, off = synth.synth_proteome(n, seed, median_len=300, min_len=5)
    seqs = [res[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(len(off) - 1)]
    # a duplicate protein and a peptide with mod sites beyond residue 64 (the long-peptide kernel)
    return seqs + [seqs[0], "G" * 70 + "MSTYMWSTK" + "G" * 12 + "MR"]


@pytest.mark.parametrize("name", GROUP_SETS)
def test_merge_equals_radix(name, monkeypatch):
    p = dbi.default_params(**PARAM_SETS[name])
    assert compare(p, *pack(proteome(400, 11)), monkeypatch) > 0


def test_merge_equals_radix_full_cfg2(monkeypatch):
    """The bench workload: 20 000 proteins, 69.3 M entries, compared chunk by chunk."""
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = synth.config_proteome(2, 20000)
    n = compare(p, res, off, monkeypatch, with_ids=False)
    assert n > 60_000_000


def test_merge_ties_across_lists(monkeypatch):
    """Shifts +16 and +32 (exact in binary) with K = 2: ((m + 16) + 16) and (m + 32) often have equal bits, so groups
    of different lists tie on the key; permuted isomers tie on the base mass inside list 0."""
    p = dbi.default_params(diff_mods=[("M", 16.0), ("W", 32.0)], max_mods_per_peptide=2, max_missed=2)
    rng = np.random.default_rng(5)
    aa = "ACDEFGHILMNPQSTVWY"
    seqs = []
    for _ in range(300):
        core = list("".join(rng.choice(list(aa), size=int(rng.integers(4, 14)))) + "MW")
        for _ in range(3):  # isomers: same residues, other orders
            rng.shuffle(core)
            seqs.append("".join(core) + "K" + "".join(rng.choice(list(aa), size=5)) + "R")
    res, off = pack(seqs)
    gm = build(p, res, off, False, monkeypatch)
    try:
        e = gm.fetch(0, gm.stats()["n_entries"], with_ids=False)
        m = bits(e["mass"])
        assert np.count_nonzero(m[1:] == m[:-1]) > 100  # the case is really exercised
    finally:
        gm.close()
    compare(p, res, off, monkeypatch)


def test_merge_tiny_and_empty_lists(monkeypatch):
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    # fewer groups than one merge tile
    compare(p, *pack(["MSTKAMYR", "PEPTIDEK"]), monkeypatch)
    # no M and no Y: every list of a class sequence with the M class is empty
    res, off = synth.synth_proteome(200, 3, median_len=200, min_len=5)
    s = res.tobytes().replace(b"M", b"L").replace(b"Y", b"F")
    compare(p, np.frombuffer(s, np.uint8).copy(), off, monkeypatch)
    # a single peptide without sites: only list 0
    compare(p, *pack(["AAGGLLK"]), monkeypatch)


def test_merge_stats(monkeypatch):
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    p.profile = 1
    res, off = pack(proteome(300, 21))
    gm = build(p, res, off, False, monkeypatch)
    gr = build(p, res, off, True, monkeypatch)
    try:
        sm, sr = gm.stats(), gr.stats()
        assert sm["n_entries"] == sr["n_entries"] > 0
        assert sm["sort_bits_var"] == 0 and sr["sort_bits_var"] > 0
        # the dominant-kernel probe brackets the base mass sort on the merge path
        assert sm["dom_kernel"] == 0 and sm["dom_launches"] > 0
        assert sm["dom_bytes_per_launch"] == sm["n_emitted"] * 24
        assert sr["dom_kernel"] == 1
    finally:
        gm.close()
        gr.close()
