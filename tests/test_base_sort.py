"""Order of the base records: the mass-only radix sort followed by the per-run ordering of records with
equal mass bits (K8r) must give exactly the order (mass bits, sequence hash masked to its width, arrival
index).  For a build without mods the entries are the unique tables, so their order is checked against a
numpy lexsort of the emitted records with the hash restated here.  The inputs are built to reach every
path of K8r: short runs sorted inside a tile, runs that cross tile edges or exceed the in-tile cap, runs
longer than one shared-memory pass of the second kernel (sorted chunks + merges), and bit-equal isomers."""
import numpy as np
import pytest

import dbindex_b200 as dbi
from dbindex_b200 import synth

from .test_gpu_parity import both, check_all
from .util import PARAM_SETS, bits, pack

pytestmark = pytest.mark.gpu

M32 = np.uint64(0xFFFFFFFF)


def _fmix32(h):
    h = h ^ (h >> np.uint64(16))
    h = (h * np.uint64(0x85EBCA6B)) & M32
    h = h ^ (h >> np.uint64(13))
    h = (h * np.uint64(0xC2B2AE35)) & M32
    return h ^ (h >> np.uint64(16))


def sequence_hash(residues, offsets, rec, hash_bits):
    """The seed-0 sequence hash of every emitted record, masked to hash_bits (a restatement of the kernel's)."""
    start = offsets[rec["prot"].astype(np.int64)].astype(np.int64) + rec["off"].astype(np.int64)
    ln = rec["len"].astype(np.uint64)
    h = np.full(len(start), 0x811C9DC5, np.uint64)
    h2 = np.full(len(start), 0x9747B28C, np.uint64)
    for k in range(int(ln.max()) if len(ln) else 0):
        act = ln > np.uint64(k)
        c = residues[np.where(act, start + k, 0)].astype(np.uint64)
        h = np.where(act, ((h ^ c) * np.uint64(16777619)) & M32, h)
        h2 = np.where(act, (((h2 + c + np.uint64(1)) * np.uint64(0x9E3779B1)) & M32) ^ (h2 >> np.uint64(15)), h2)
    lo = _fmix32(h ^ ((ln * np.uint64(0x9E3779B1)) & M32))
    if hash_bits <= 32:
        return lo
    full = (_fmix32(h2 ^ ln) << np.uint64(32)) | lo
    return full if hash_bits >= 64 else full & np.uint64((1 << hash_bits) - 1)


def expected_unique(residues, offsets, rec, hash_bits):
    """Emitted records in (mass bits, masked hash, arrival) order, merged by sequence: the first record of every
    sequence and the protein ids of all its records."""
    mb = bits(rec["mass"])
    hk = sequence_hash(residues, offsets, rec, hash_bits)
    order = np.lexsort((np.arange(len(mb)), hk, mb))
    start = offsets[rec["prot"].astype(np.int64)].astype(np.int64) + rec["off"].astype(np.int64)
    seq = [residues[start[i]:start[i] + int(rec["len"][i])].tobytes() for i in order]
    head = np.ones(len(order), bool)
    for j in range(1, len(order)):
        head[j] = not (mb[order[j]] == mb[order[j - 1]] and seq[j] == seq[j - 1])
    return order, head


def check_order(residues, offsets, hash_bits=32, params=None):
    p = (params or dbi.default_params()).copy()
    p.keep_emitted = 1
    with dbi.GpuIndex(p) as g:
        g.add_proteins(residues, offsets)
        g.build()
        st = g.stats()
        assert st["n_hash_retries"] == 0
        assert st["sort_bits_base"] >= hash_bits
        rec = g.debug_emitted()
        order, head = expected_unique(residues, offsets, rec, hash_bits)
        assert st["n_unique"] == st["n_entries"] == int(head.sum())
        got = g.fetch(0, st["n_entries"])
    first = order[head]
    assert np.array_equal(bits(got["mass"]), bits(rec["mass"][first]))
    assert np.array_equal(got["first_prot"], rec["prot"][first])
    assert np.array_equal(got["first_off"], rec["off"][first])
    assert np.array_equal(got["len"], rec["len"][first])
    assert np.array_equal(got["prot_list_off"], np.r_[np.flatnonzero(head), len(order)].astype(np.uint64))
    assert np.array_equal(got["prot_ids"], rec["prot"][order])
    return rec, order


def long_run_proteome():
    """A small proteome with repeated entries: one protein 3000 times (runs longer than one shared-memory
    pass), one 300 times and one 40 times, a short peptide-like entry 70 times, in interleaved order so
    that runs of every length start and end all over the tiles."""
    res, off = synth.synth_proteome(120, 4242, median_len=300)
    base = [res[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(len(off) - 1)]
    seqs = list(base)
    rng = np.random.default_rng(7)
    for i in range(3000):
        seqs.append(base[3])
        if i < 300:
            seqs.append(base[10])
        if i < 40:
            seqs.append(base[int(rng.integers(20, 120))])
        if i < 70:
            seqs.append("MAGGLLKPEPTIDEKRDESK")
    return pack(seqs)


def isomer_proteome():
    """Permutations of a few compositions as separate tryptic peptides: many distinct strings with bit-equal
    masses next to each other, plus copies of some of them."""
    rng = np.random.default_rng(11)
    seqs = []
    for comp in ("AAGGLLSVDEPT", "GGHHNQWYVTLA", "MMCCDDEEFFAS", "PPSSTTVVIILN"):
        letters = list(comp)
        for _ in range(200):
            rng.shuffle(letters)
            seqs.append("".join(letters) + "K")
    prots = []
    for i in range(0, len(seqs), 8):
        prots.append("".join(seqs[i:i + 8]))
    prots += prots[:30]
    return pack(prots)


def test_order_long_runs():
    res, off = long_run_proteome()
    rec, order = check_order(res, off)
    mb = bits(rec["mass"])[order]
    runs = np.diff(np.r_[np.flatnonzero(np.r_[True, mb[1:] != mb[:-1]]), len(mb)])
    assert runs.max() > 2048  # longer than one shared-memory pass of the second kernel
    assert ((runs > 64) & (runs <= 2048)).any() and ((runs >= 2) & (runs <= 64)).any()


def test_order_isomers():
    res, off = isomer_proteome()
    rec, order = check_order(res, off)
    mb = bits(rec["mass"])
    start = off[rec["prot"].astype(np.int64)].astype(np.int64) + rec["off"].astype(np.int64)
    # distinct strings share mass bits: the hash orders them
    by_mass = {}
    for i in range(len(mb)):
        by_mass.setdefault(int(mb[i]), set()).add(res[start[i]:start[i] + int(rec["len"][i])].tobytes())
    assert max(len(v) for v in by_mass.values()) > 10


def test_order_wide_hash(monkeypatch):
    monkeypatch.setenv("DBI_HASH_BITS", "44")
    res, off = long_run_proteome()
    check_order(res, off, hash_bits=44)
    res, off = isomer_proteome()
    check_order(res, off, hash_bits=44)


@pytest.mark.parametrize("inputs", ["long_runs", "isomers"])
def test_oracle_parity_cfg2(inputs):
    res, off = long_run_proteome() if inputs == "long_runs" else isomer_proteome()
    g, o = both(dbi.default_params(**PARAM_SETS["cfg2_mods"]), res, off)
    try:
        check_all(g, o)
    finally:
        g.close()
