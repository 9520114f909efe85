"""bench.py --dump-outputs without a device: dump_outputs reads the run-grouped answer of a handle; here the
handle is a stand-in that serves the oracle's hits grouped in runs the way dbi_query_hits_read delivers them."""
import ctypes as C
import os

import numpy as np

import bench
import dbindex_b200 as dbi
from dbindex_b200 import synth
from dbindex_b200.capi import HIT_FIELDS, DbiHitCounts, _expand_csr
from oracle.oracle_py import Oracle

from .test_gpu_parity import hits_canonical


class OracleHandle:
    """query_hits_read / stats / fetch of a built index, answered by the oracle."""

    def __init__(self, o, h, tie_rng=None):
        self.o, self.ent = o, o.entries()
        ho = h["hit_off"].astype(np.int64)
        idx = np.arange(ho[-1])
        if tie_rng is not None:  # another legal order: hits of one query that tie in mass permuted
            for q in range(len(ho) - 1):
                m = h["mass"][idx[ho[q]:ho[q + 1]]]
                for v in np.unique(m):
                    s = ho[q] + np.nonzero(m == v)[0]
                    idx[s] = idx[tie_rng.permutation(s)]
        key = np.stack([h[k][idx].astype(np.uint64) for k in ("first_prot", "first_off", "len")] +
                       [h["mass"][idx].view(np.uint64)])
        first = np.ones(len(idx), bool)  # a run starts at a new peptide / mass or at a new query
        first[1:] = np.any(key[:, 1:] != key[:, :-1], axis=0)
        first[ho[:-1][ho[:-1] < len(idx)]] = True
        start = np.nonzero(first)[0]
        runs = idx[start]
        self.raw = {"hit_off": ho, "pep_off": np.searchsorted(start, ho), "modpat": h["modpat"][idx],
                    "pep_hit_off": np.append(start, len(idx)), "flanks": h["flanks"].reshape(-1, 6)[runs]}
        for k in ("mass", "first_prot", "first_off", "len"):
            self.raw[k] = h[k][runs]
        self.raw["seq_off"], self.raw["seq"] = _expand_csr(h["seq_off"], h["seq"], runs)
        self.raw["prot_list_off"], self.raw["prot_ids"] = _expand_csr(h["prot_list_off"], h["prot_ids"], runs)
        self.counts = DbiHitCounts(len(ho) - 1, len(idx), len(runs), len(self.raw["seq"]), len(self.raw["prot_ids"]))

    def query_hits_read(self, bufs):
        for name, (dt, _) in HIT_FIELDS.items():
            a = np.ascontiguousarray(self.raw[name], dtype=dt)
            C.memmove(getattr(bufs, name), a.ctypes.data, a.nbytes)

    def stats(self):
        return self.o.counts()

    def fetch(self, begin, count, with_ids=True):
        return {"mass": self.ent["mass"][begin:begin + count]}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_holds_the_hits_in_canonical_order(tmp_path, monkeypatch):
    p = dbi.default_params(**bench.CFG2)
    res, off = synth.config_proteome(2, 150)
    o = Oracle(p, threads=os.cpu_count() or 1)
    o.add_proteins(res, off)
    assert o.build() == 0
    n_entries = o.counts()["n_entries"]
    _, _, lo, hi = synth.synth_queries(o.entries()["mass"], 200, 7)
    h = o.query_hits(lo, hi)
    g = OracleHandle(o, h)
    assert g.counts.n_peps < g.counts.n_hits  # the stand-in really groups hits in runs

    info = bench.dump_outputs(str(tmp_path / "a"), g, g.counts, n_entries)
    a = _load(tmp_path / "a")
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    assert info["bytes"] == sum(x.nbytes for x in a.values()) and info["queries"] == 200
    c = o.counts()
    assert a["counts"].tolist() == [c["n_emitted"], c["n_unique"], n_entries, g.counts.n_hits]
    assert np.array_equal(a["index_mass"], bench.sample_index_masses(g, n_entries))
    exp = hits_canonical(h)
    so, po = a["hit_seq_off"].astype(np.int64), a["hit_prot_list_off"].astype(np.int64)
    for j, q in enumerate(a["query"].astype(np.int64)):
        rows = np.nonzero(a["hit_query"] == q)[0]
        assert len(rows) == a["query_hits"][j]
        got = [(int(a["hit_mass"][i:i + 1].view(np.uint64)[0]), int(a["hit_first_prot"][i]), int(a["hit_first_off"][i]),
                int(a["hit_len"][i]), int(a["hit_modpat"][i]), a["hit_seq"][so[i]:so[i + 1]].astype(np.uint8).tobytes(),
                a["hit_flanks"][i].astype(np.uint8).tobytes(), tuple(a["hit_prot_ids"][po[i]:po[i + 1]].astype(int).tolist()))
               for i in rows]
        assert got == exp[q], q  # every hit, in canonical order

    # another legal tie order gives the same files
    g2 = OracleHandle(o, h, tie_rng=np.random.default_rng(3))
    bench.dump_outputs(str(tmp_path / "b"), g2, g2.counts, n_entries)
    b = _load(tmp_path / "b")
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)

    # a larger output: the longest prefix of the seeded query sample that fits the budget
    budget = a["index_mass"].nbytes + 200_000
    monkeypatch.setattr(bench, "DUMP_BYTES", budget)
    info = bench.dump_outputs(str(tmp_path / "c"), g, g.counts, n_entries)
    files = os.listdir(tmp_path / "c")
    assert 0 < info["queries"] < 200
    assert sum(os.path.getsize(tmp_path / "c" / f) for f in files) <= budget
    sample = _load(tmp_path / "c")["query"]
    assert set(sample.astype(int)) <= set(a["query"].astype(int))
