"""Compact variant index (the sorted groups kept, the entries a query returns expanded by K6q) measured on two
workloads.  Writes <out>/compact_bench.json (a part run alone is merged into an existing file).

(a) cfg2 (BASELINE.json configs[1]: 20 000 synthetic proteins, static C, variable M + STY, <= 3 per peptide) built
    expanded and compact (DBI_COMPACT_VARIANTS=1), the two layouts alternated, L2 flushed (256 MiB write) before
    every timed call, every shape warmed up, medians of --reps: the build, device_bytes, a 10^4-query batch at
    10 ppm (dbi_query_hits and dbi_query_hits_read timed apart) and a batch of 10^4 PPM spectra at 10 ppm
    (dbi_query_spectra and the read).  Parity: every buffer of both answers byte for byte.
(b) The --big proteome of scripts/unindexed_bench.py (synth.config_proteome(4, 2 x 10^6) with cfg2's parameters,
    about 6.9 G entries: more than the 2^32 an expanded index holds) built on one GPU without the environment
    variable, so the build keeps the compact layout.  Device memory in use sampled every 2 ms during the build
    (peak) and after it with the library's cache released (final); the build time; the 10^3 queries of
    unindexed_bench.py (b) answered by the compact index and by the chunked unindexed search, in groups of
    --group mass-sorted queries, both timed (L2 flushed before every group), with canonical parity of every hit.

    python scripts/compact_bench.py --out DIR [--parts a,b] [--reps 5] [--big 2000000]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from unindexed_bench import CFG2, gpu_identity, parity_failures  # noqa: E402

ENV = "DBI_COMPACT_VARIANTS"


class MemSampler:
    """Device memory in use (cudaMemGetInfo), sampled from a thread while a call runs."""

    def __init__(self, torch, period_s=0.002):
        self.torch, self.period_s, self.peak, self._stop = torch, period_s, 0, False

    def used(self):
        free, total = self.torch.cuda.mem_get_info()
        return total - free

    def __enter__(self):
        self.peak = self.used()
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def _run(self):
        while not self._stop:
            self.peak = max(self.peak, self.used())
            time.sleep(self.period_s)

    def __exit__(self, *a):
        self._stop = True
        self._t.join()
        self.peak = max(self.peak, self.used())


def raw_answer(g, cnt):
    return g._read_hits(cnt, None, None, False)


def same_bytes(a, b):
    ca, cb = a["counts"], b["counts"]
    if (ca.nq, ca.n_hits, ca.n_peps, ca.n_seq_bytes, ca.n_prot_ids) != (cb.nq, cb.n_hits, cb.n_peps, cb.n_seq_bytes,
                                                                        cb.n_prot_ids):
        return False
    return all(np.array_equal(np.asarray(a[k]).view(np.uint8), np.asarray(b[k]).view(np.uint8))
               for k in a if k != "counts")


def part_a(args, dbi, synth, torch, timed):
    from dbindex_b200.capi import DBI_TOL_PPM
    p = dbi.default_params(**CFG2)
    p.profile = 1
    res, off = synth.config_proteome(2, args.proteins)
    layouts = ("expanded", "compact")
    gs = {}

    def build(layout):
        if layout == "compact":
            os.environ[ENV] = "1"
        else:
            os.environ.pop(ENV, None)
        g = gs.get(layout)
        if g is None:
            g = gs[layout] = dbi.GpuIndex(p)
            g.add_proteins(res, off)
        g.build()
        os.environ.pop(ENV, None)
        return g

    for lay in layouts:
        build(lay)
    st = {lay: gs[lay].stats() for lay in layouts}
    assert st["expanded"]["n_groups"] == 0 and st["compact"]["n_groups"] > 0
    masses = gs["expanded"].fetch(0, st["expanded"]["n_entries"], with_ids=False)["mass"]
    _, _, lo, hi = synth.synth_queries(masses, 10_000, 20261022)
    rng = np.random.default_rng(20261023)
    sp = masses[rng.integers(0, len(masses), 10_000)] * (1 + rng.uniform(-5e-6, 5e-6, 10_000))
    ppm = np.full(len(sp), 10.0)
    del masses

    calls = {"query": lambda g: g.query_hits_begin(lo, hi),
             "spectra": lambda g: spectra_begin(g, sp, ppm, DBI_TOL_PPM)}
    rec = {f"{lay}_{k}": [] for lay in layouts for k in ("build_ms", "query_call_ms", "query_read_ms",
                                                          "spectra_call_ms", "spectra_read_ms", "device_bytes")}
    stage = {lay: [] for lay in layouts}
    for rep in range(args.reps + 2):  # two warm-up rounds
        for lay in layouts:
            gs[lay].reset_index()
            _, ms_b = timed(lambda: build(lay))
            g = gs[lay]
            s = g.stats()
            row = {"build_ms": ms_b, "device_bytes": s["device_bytes"]}
            for k, call in calls.items():
                cnt, ms = timed(lambda: call(g))
                t = time.perf_counter()
                g._read_hits(cnt, None, None, False)
                row[f"{k}_call_ms"], row[f"{k}_read_ms"] = ms, (time.perf_counter() - t) * 1e3
            if rep >= 2:
                for k, v in row.items():
                    rec[f"{lay}_{k}"].append(v)
                stage[lay].append(s["stage_ms"])
    answers = {lay: {k: raw_answer(gs[lay], call(gs[lay])) for k, call in calls.items()} for lay in layouts}
    parity = {k: same_bytes(answers["expanded"][k], answers["compact"][k]) for k in calls}
    hits = {k: int(answers["compact"][k]["counts"].n_hits) for k in calls}
    del answers
    med = {k: float(np.median(v)) for k, v in rec.items()}
    out = {"index": {"proteins": int(len(off) - 1), "residues": int(len(res)), "emitted": st["compact"]["n_emitted"],
                     "unique": st["compact"]["n_unique"], "entries": st["compact"]["n_entries"],
                     "groups": st["compact"]["n_groups"], "params": "cfg2 (static C, M + STY, <= 3)"},
           "l2": "flushed (256 MiB write) before every timed call; two warm-up rounds; layouts alternated",
           "reps": args.reps, "median": med, "all": rec,
           "build_stage_ms_median": {lay: {k: float(np.median([d[k] for d in stage[lay]])) for k in stage[lay][0]}
                                     for lay in layouts},
           "query_batch": {"queries": len(lo), "ppm": 10.0, "seed": 20261022, "hits": hits["query"]},
           "spectra_batch": {"spectra": len(sp), "ppm": 10.0, "seed": 20261023, "tol_mode": "DBI_TOL_PPM",
                             "masses": "index masses jittered +-5 ppm", "hits": hits["spectra"]},
           "byte_parity": parity}
    for g in gs.values():
        g.close()
    print(json.dumps({"a": {"median": med, "parity": parity, "hits": hits}}), flush=True)
    return out


def spectra_begin(g, mass, tol, mode):
    import ctypes as C

    from dbindex_b200.capi import DbiHitCounts, _ptr, spectra_arrays
    mass, tol, range_off, n = spectra_arrays(mass, tol, None, mode)
    cnt = DbiHitCounts()
    g._check(g.lib.dbi_query_spectra(g._h, _ptr(mass), _ptr(tol), _ptr(range_off), n, mode, 0, C.byref(cnt)))
    return cnt


def part_b(args, dbi, synth, torch, timed, save):
    from dbindex_b200.indexer import UNINDEXED_MAX_CANDIDATES, search_unindexed_chunked
    os.environ.pop(ENV, None)
    p = dbi.default_params(**CFG2)
    t = time.perf_counter()
    res, off = synth.config_proteome(4, args.big)
    t_gen = time.perf_counter() - t
    n_small = min(20_000, args.big)
    with dbi.GpuIndex(p) as small:  # the masses of half the queries (as unindexed_bench.py (b))
        small.add_proteins(res[:int(off[n_small])], off[:n_small + 1])
        small.build()
        m_small = small.fetch(0, small.stats()["n_entries"], with_ids=False)["mass"]
    _, _, lo, hi = synth.synth_queries(m_small, args.big_queries, 20261021)
    del m_small
    lib = dbi.load_library()
    lib.dbi_release_cached_memory(0)
    torch.cuda.synchronize()
    out = {"proteome": {"config": "synth.config_proteome(4, %d)" % args.big, "proteins": int(len(off) - 1),
                        "residues": int(len(res)), "params": "cfg2 (static C, M + STY, <= 3)",
                        "generate_s": round(t_gen, 1)}}
    g = dbi.GpuIndex(p)
    g.add_proteins(res, off)
    g.upload()
    sampler = MemSampler(torch)
    base = sampler.used()
    try:
        with sampler:
            t = time.perf_counter()
            g.build()
            build_s = time.perf_counter() - t
    except dbi.DbiError as e:  # report where the build stopped and how far memory got
        out["build"] = {"error": str(e), "peak_device_bytes_above_start": sampler.peak - base}
        print(json.dumps(out), flush=True)
        return out
    st = g.stats()
    lib.dbi_release_cached_memory(0)
    final = sampler.used() - base
    out["build"] = {"s": build_s, "n_emitted": st["n_emitted"], "n_unique": st["n_unique"],
                    "n_entries": st["n_entries"], "n_groups": st["n_groups"], "device_bytes": st["device_bytes"],
                    "peak_device_bytes_above_start": sampler.peak - base,
                    "final_device_bytes_above_start": final,
                    "memory": "cudaMemGetInfo sampled every 2 ms during dbi_build; final after the library's cache "
                              "was released; both above the level before the build (proteins already uploaded)",
                    "entry_arrays_of_an_expanded_index_bytes": st["n_entries"] * 16}
    print(json.dumps(out), flush=True)
    save(out)
    un = dbi.GpuIndex(p)
    un.add_proteins(res, off)
    un.upload()
    order = np.argsort(lo, kind="stable")
    groups = np.array_split(order, max(1, len(order) // args.group))
    rec = {"compact_call_ms": [], "compact_read_ms": [], "unindexed_ms": [], "hits": [], "parity_failed": []}
    for grp in groups:
        cnt, ms = timed(lambda: g.query_hits_begin(lo[grp], hi[grp]))
        t = time.perf_counter()
        a = g._read_hits(cnt, None, None, False)
        rec["compact_read_ms"].append((time.perf_counter() - t) * 1e3)
        rec["compact_call_ms"].append(ms)
        b, ms = timed(lambda: search_unindexed_chunked(un, lo[grp], hi[grp], UNINDEXED_MAX_CANDIDATES))
        rec["unindexed_ms"].append(ms)
        ea = dbi.capi.expand_hits(a)
        rec["hits"].append(int(a["counts"].n_hits))
        rec["parity_failed"].append(parity_failures(ea, b))
        del a, b, ea
        print(json.dumps({k: v[-1] for k, v in rec.items()}), flush=True)
        save({**out, "queries_so_far": {"groups": len(rec["hits"]), "per_group": rec}})
    t_c = sum(rec["compact_call_ms"]) + sum(rec["compact_read_ms"])
    t_u = sum(rec["unindexed_ms"])
    out["queries"] = {"n": len(lo), "ppm": 10.0, "seed": 20261021, "groups": len(groups),
                      "query_masses": "half from an index of the first 20 000 proteins jittered +-5 ppm, half uniform",
                      "l2": "flushed before every timed group",
                      "compact_ms": t_c, "compact_queries_per_s": len(lo) / (t_c / 1e3),
                      "unindexed_chunked_ms": t_u, "unindexed_queries_per_s": len(lo) / (t_u / 1e3),
                      "hits": sum(rec["hits"]), "parity_failed": sum(rec["parity_failed"]), "per_group": rec,
                      "compact_timing": "dbi_query_hits (call) + dbi_query_hits_read into numpy (read), per group",
                      "unindexed_timing": "indexer.search_unindexed_chunked (calls + reads), per group"}
    g.close()
    un.close()
    print(json.dumps({k: v for k, v in out["queries"].items() if k != "per_group"}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--parts", default="a,b")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--proteins", type=int, default=None, help="part (a): proteins of cfg2 (default 20 000)")
    ap.add_argument("--big", type=int, default=2_000_000, help="part (b): proteins of the cfg4 proteome")
    ap.add_argument("--big-queries", type=int, default=1000)
    ap.add_argument("--group", type=int, default=100, help="part (b): queries per timed group")
    args = ap.parse_args()
    import torch

    import dbindex_b200 as dbi
    from dbindex_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("compact_bench needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "compact_bench.json")
    out = json.load(open(path)) if os.path.exists(path) else {}
    out.update({"what": "compact variant index: (a) cfg2 compact against expanded; (b) a proteome whose expanded "
                        "index exceeds 2^32 entries, built compact on one GPU, against the chunked unindexed search"})
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(fn):
        flush.zero_()
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn()  # every call ends in a stream synchronise
        return r, (time.perf_counter() - t) * 1e3

    parts = args.parts.split(",")
    failed = 0
    if "a" in parts:
        out["a_cfg2"] = {**gpu_identity(), **part_a(args, dbi, synth, torch, timed)}
        failed += not all(out["a_cfg2"]["byte_parity"].values())
        with open(path, "w") as f:
            json.dump(out, f, indent=1)
    if "b" in parts:
        ident = gpu_identity()

        def save(part):  # after the build and after every query group: a run cut short keeps what it measured
            out["b_big_compact"] = {**ident, **part}
            with open(path, "w") as f:
                json.dump(out, f, indent=1)

        save(part_b(args, dbi, synth, torch, timed, save))
        failed += out["b_big_compact"].get("queries", {}).get("parity_failed", 1) != 0
    if failed:
        raise SystemExit(f"parity failed or the build did not finish ({failed})")


if __name__ == "__main__":
    main()
