"""The order of the entries inside a variant group, as the expansion kernels write it (K6x at build time, K6q when a
compact index expands at query time).  The compact index's peptide lookup turns a pattern into an entry number by
inverting this order (group_entry_rank), so it is part of the index: every group of a peptide of up to 64 residues
must list its patterns in exactly block_order(k, masks), and a group of a longer peptide (K6l) in lexicographic order.

The cases cover the tile edges of the expansion: groups that start before a tile, one group spanning several tiles,
tiles of up to 513 one-entry groups, and tiles whose site lists do not fit the shared list pool (those groups
un-rank their entries from the masks instead; the test asserts that such a tile exists)."""
import numpy as np
import pytest

import dbindex_b200 as dbi
from dbindex_b200 import synth

from .test_compact_index import LONG_PARAMS, assert_fetch_equal, block_order, build, long_proteome
from .util import PARAM_SETS, bits, pack

TILE = 512      # entries per expansion tile (kExpTile)
POOL = 3072     # bytes of site lists per tile (EP_POOL); byte 0 is reserved
MASK_LEN = 64   # peptides up to this length have site masks; longer ones are expanded in lexicographic order

# isomers of one S-rich 61-mer ending in ...MSK: the (M, S) group of each has 1 entry and 32 list bytes, and all of
# them share one mass, so hundreds sit side by side in the index.  The shifts are chosen so that the mass of (M, S),
# (base + dM) + dS, differs in its last bit from (base + dS) + dM: the 30-entry (S, M) groups do not fall in between.
POOL_PARAMS = dict(diff_mods=[("M", 15.99485), ("S", 79.96632)], max_mods_per_peptide=2, max_mass=8000.0,
                   max_missed=0)


def pool_proteome(n=600, seed=3):
    rng = np.random.default_rng(seed)
    body = list("S" * 30 + "GALVGALVGALVGALVGALVGALVGALV")
    seqs = set()
    while len(seqs) < n:
        rng.shuffle(body)
        seqs.add("".join(body) + "MSK")
    return pack(sorted(seqs))


def spanning_proteome():
    """cfg2's proteome on 100 proteins plus one peptide whose (S, S, S) group has C(30, 3) = 4060 entries"""
    res, off = synth.synth_proteome(100, 77)
    seqs = [res[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(len(off) - 1)]
    return pack(seqs + ["GA" + "SG" * 30 + "LK"])


def case(name):
    if name == "cfg2_500":
        return dbi.default_params(**PARAM_SETS["cfg2_mods"]), *synth.synth_proteome(500, 4242)
    if name == "wide_mass_mod4":
        return dbi.default_params(**PARAM_SETS["wide_mass_mod4"]), *synth.synth_proteome(300, 4242)
    if name == "long_peptides":
        return dbi.default_params(**LONG_PARAMS), *long_proteome(300, 7)
    if name == "spanning_group":
        return dbi.default_params(**PARAM_SETS["cfg2_mods"]), *spanning_proteome()
    return dbi.default_params(**POOL_PARAMS), *pool_proteome()


def residue_shift(diff_mods):
    """residue -> its shift; residues with equal shifts form one class"""
    out = {}
    for aas, d in diff_mods:
        for a in aas:
            out[ord(a)] = d
    return out


def groups_of(f, res, off, diff_mods):
    """Splits the fetched entries into groups (same mass bits, same peptide, same class sequence) and checks each
    group's patterns against the block order.  Returns (first entry, entries, list bytes, k, long) per group."""
    shift = residue_shift(diff_mods)
    V = len(f["mass"])
    mb = bits(f["mass"])
    prot, poff, plen, pat = f["first_prot"], f["first_off"], f["len"], f["modpat"]
    # runs of equal (mass, peptide); the class sequence splits them further below
    brk = np.ones(V, bool)
    brk[1:] = (mb[1:] != mb[:-1]) | (prot[1:] != prot[:-1]) | (poff[1:] != poff[:-1]) | (plen[1:] != plen[:-1])
    starts = np.flatnonzero(brk).tolist() + [V]
    out = []
    for a, b in zip(starts[:-1], starts[1:]):
        s0 = int(off[int(prot[a])]) + int(poff[a])
        pep = res[s0:s0 + int(plen[a])]
        by_seq, last = {}, None
        for e in range(a, b):
            p = int(pat[e])
            pos = tuple(((p >> (8 * j)) & 0xff) - 1 for j in range(4) if (p >> (8 * j)) & 0xff)
            seq = tuple(shift[int(pep[x])] for x in pos)
            if seq != last:
                assert seq not in by_seq, f"the group at entry {e} is not contiguous"
                by_seq[seq], last = (e, []), seq
            by_seq[seq][1].append(pos)
        for seq, (e, got) in by_seq.items():
            k = len(seq)
            masks = [[x for x in range(len(pep)) if shift.get(int(pep[x])) == d] for d in seq]
            order = block_order(k, masks)
            long = len(pep) > MASK_LEN
            if long:
                order = sorted(order)
            assert got == order, f"group at entry {e} (k = {k}, peptide length {len(pep)}) is out of order"
            # list bytes of the tile's pool: one list per distinct class of the sequence
            nbytes = 0 if long or k in (0, 4) else sum(len(masks[j]) for j in range(k) if seq[j] not in seq[:j])
            out.append((e, len(got), nbytes, k, long))
    assert sum(n for _, n, _, _, _ in out) == V
    return out


def tile_pool_demand(groups, V):
    """list bytes every tile of the expansion asks for: the groups that overlap it and start before its end"""
    n_tiles = -(-V // TILE)
    demand = np.zeros(n_tiles, np.int64)
    for e, n, nbytes, _, _ in groups:
        if nbytes:
            demand[e // TILE:(e + n - 1) // TILE + 1] += nbytes
    return demand


def fetch_in_pieces(g, V, cuts):
    """the whole index through dbi_fetch ranges that start at the given entries (mid-group for a compact index)"""
    edges = [0] + [c for c in cuts if 0 < c < V] + [V]
    parts = [g.fetch(a, b - a) for a, b in zip(edges[:-1], edges[1:])]
    return {k: np.concatenate([p[k] for p in parts]) for k in ("mass", "first_prot", "first_off", "len", "modpat")}


CASES = ["cfg2_500", "wide_mass_mod4", "long_peptides", "spanning_group", "pool_overflow"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_expand_order(name, monkeypatch):
    p, res, off = case(name)
    kw = {"cfg2_500": PARAM_SETS["cfg2_mods"], "wide_mass_mod4": PARAM_SETS["wide_mass_mod4"],
                 "long_peptides": LONG_PARAMS, "spanning_group": PARAM_SETS["cfg2_mods"]}.get(name, POOL_PARAMS)
    ge = build(p, res, off, False, monkeypatch)
    V = ge.stats()["n_entries"]
    f = ge.fetch(0, V, with_ids=False)
    groups = groups_of(f, res, off, kw["diff_mods"])
    ks = {k for _, _, _, k, _ in groups}
    if name == "wide_mass_mod4":
        assert 4 in ks
    if name == "long_peptides":
        assert any(lg for _, _, _, _, lg in groups)
    if name == "spanning_group":
        assert any((e + n - 1) // TILE - e // TILE >= 2 for e, n, _, _, _ in groups)
    if name == "pool_overflow":
        assert tile_pool_demand(groups, V).max() > POOL - 1, "no tile overflows the list pool"
    if name == "cfg2_500":
        assert ks == {0, 1, 2, 3}
    # the compact index expands the same entries from ranges that start inside groups and tiles
    gc = build(p, res, off, True, monkeypatch)
    assert gc.stats()["n_groups"] > 0
    rng = np.random.default_rng(5)
    cuts = sorted(set(int(x) for x in rng.integers(1, V, 6)) | {217, TILE + 1})
    fc = fetch_in_pieces(gc, V, cuts)
    assert_fetch_equal({k: f[k] for k in fc}, fc)
