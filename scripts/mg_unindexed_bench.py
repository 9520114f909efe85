"""Sharded unindexed search (dbi_mg_search_unindexed_local) against dbi_search_unindexed on one GPU.  Writes
<out>/mg_unindexed_bench.json.  Needs at least two visible GPUs: with fewer it says so and exits.

Every visible GPU holds one shard (multigpu.shard_proteins, residue-balanced, file order); GPU 0 also holds a handle
with the whole proteome for the single-GPU call.  The two paths alternate, L2 is flushed on every device (256 MiB
write each) before every timed call, every shape is warmed up twice, and the medians of --reps are reported.  The
device call (it ends synchronised) is timed apart from the read of the pending results.  Every call's canonical
answer (every hit, ties in canonical order) is compared with the other path's.

(a) cfg2 (BASELINE.json configs[1], static C, variable M + STY, <= 3 per peptide): seeded 10 ppm batches of 10^2,
    10^3 and 10^4 queries (synth.synth_queries: half jittered index masses, half uniform).  Per-rank stage times
    (params.profile) and candidate counts are recorded.
(b) The 2 x 10^6-protein proteome of unindexed_bench.py (b) (synth.config_proteome(4, ...), cfg2's parameters, never
    built): 10^3 queries at 10 ppm in 10 mass-sorted groups, each through the mirror's chunked search
    (UNINDEXED_MAX_CANDIDATES) on both paths.

    python scripts/mg_unindexed_bench.py --out DIR [--reps 5] [--big 2000000]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from unindexed_bench import CFG2, gpu_identity, parity_failures  # noqa: E402

BATCHES = (100, 1000, 10_000)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--big", type=int, default=2_000_000, help="part (b): proteins of the cfg4 proteome (0: skip)")
    ap.add_argument("--big-queries", type=int, default=1000)
    ap.add_argument("--groups", type=int, default=10)
    args = ap.parse_args()
    import torch

    n_gpu = torch.cuda.device_count()
    if n_gpu < 2:
        print(f"mg_unindexed_bench needs at least 2 GPUs, {n_gpu} visible: not measured")
        return

    import dbindex_b200 as dbi
    from dbindex_b200 import synth
    from dbindex_b200.capi import DbiHitCounts, expand_hits
    from dbindex_b200.indexer import UNINDEXED_MAX_CANDIDATES, _merge_hits, search_unindexed_chunked
    from dbindex_b200.multigpu import ShardedSearcher, shard_proteins

    os.makedirs(args.out, exist_ok=True)
    out = {"what": "dbi_mg_search_unindexed_local over every visible GPU against dbi_search_unindexed on one",
           "gpus": n_gpu, **gpu_identity(), "reps": args.reps,
           "l2": "flushed (256 MiB write on every device) before every timed call; every shape warmed up twice; "
                 "paths alternated"}
    flush = [torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{d}") for d in range(n_gpu)]

    def sync_all():
        for d in range(n_gpu):
            torch.cuda.synchronize(d)

    def timed(fn):
        for f in flush:
            f.zero_()
        sync_all()
        t = time.perf_counter()
        r = fn()  # every call ends in a stream synchronise of every handle it uses
        return r, (time.perf_counter() - t) * 1e3

    def handles(p, res, off):
        shards = []
        for r in range(n_gpu):
            q = p.copy()
            q.device = r
            g = dbi.GpuIndex(q)
            sres, soff, _ = shard_proteins(res, off, r, n_gpu)
            g.add_proteins(sres, soff)
            shards.append(g)
        one = dbi.GpuIndex(p)
        one.add_proteins(res, off)
        return shards, one

    lib = dbi.load_library()
    lib.dbi_mg_search_unindexed_local.restype = C.c_int
    lib.dbi_mg_search_unindexed_local.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64,
                                                  C.c_uint64, C.c_void_p, C.c_void_p]

    def mg_begin(shards, lo, hi):
        arr = (C.c_void_p * n_gpu)(*[g._h for g in shards])
        counts = (DbiHitCounts * n_gpu)()
        n_cand = np.zeros(n_gpu, dtype=np.uint64)
        rc = lib.dbi_mg_search_unindexed_local(arr, n_gpu, lo.ctypes.data, hi.ctypes.data, len(lo), 0, counts,
                                               n_cand.ctypes.data)
        shards[0]._check(rc)
        return counts

    # ---- (a) ----------------------------------------------------------------------------------------------
    p = dbi.default_params(**CFG2)
    p.profile = 1
    res, off = synth.config_proteome(2)
    shards, one = handles(p, res, off)
    with dbi.GpuIndex(p) as ix:
        ix.add_proteins(res, off)
        ix.build()
        masses = ix.fetch(0, ix.stats()["n_entries"], with_ids=False)["mass"]
    part_a = {"proteins": int(len(off) - 1), "residues": int(len(res)), "params": "cfg2 (static C, M + STY, <= 3)",
              "batches": {}}
    for nq in BATCHES:
        _, _, lo, hi = synth.synth_queries(masses, nq, 20261020 + nq)
        q = np.arange(nq)

        def read_mg(counts):
            t = time.perf_counter()
            raw = [g._read_hits(counts[r], None, None, False) for r, g in enumerate(shards)]
            return raw, (time.perf_counter() - t) * 1e3

        def read_one(cnt):
            t = time.perf_counter()
            raw = one._read_hits(cnt, None, None, False)
            return raw, (time.perf_counter() - t) * 1e3

        for _ in range(2):
            read_mg(mg_begin(shards, lo, hi))
            read_one(one.search_unindexed_begin(lo, hi))
        rec = {k: [] for k in ("sharded_call_ms", "sharded_read_ms", "single_call_ms", "single_read_ms")}
        rec.update({"rank_candidates": [], "rank_stage_ms": [], "parity_failed": []})
        for _ in range(args.reps):
            counts, ms = timed(lambda: mg_begin(shards, lo, hi))
            raw, rms = read_mg(counts)
            rec["sharded_call_ms"].append(ms)
            rec["sharded_read_ms"].append(rms)
            st = [g.stats() for g in shards]
            rec["rank_candidates"].append([s["n_emitted"] for s in st])
            rec["rank_stage_ms"].append([s["stage_ms"] for s in st])
            cnt, ms = timed(lambda: one.search_unindexed_begin(lo, hi))
            raw1, rms = read_one(cnt)
            rec["single_call_ms"].append(ms)
            rec["single_read_ms"].append(rms)
            got = _merge_hits([(q, expand_hits(x)) for x in raw], nq)
            rec["parity_failed"].append(parity_failures(got, expand_hits(raw1)))
        med = {k: float(np.median(v)) for k, v in rec.items() if k.endswith("_ms") and k != "rank_stage_ms"}
        part_a["batches"][str(nq)] = {"queries": nq, "ppm": 10.0, "seed": 20261020 + nq, "median_ms": med,
                                      "speedup_call": med["single_call_ms"] / med["sharded_call_ms"], "all": rec,
                                      "single_candidates": int(one.stats()["n_emitted"])}
        print(json.dumps({"nq": nq, **med, "parity_failed": rec["parity_failed"]}), flush=True)
    for g in shards + [one]:
        g.close()
    out["a_cfg2"] = part_a
    path = os.path.join(args.out, "mg_unindexed_bench.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)

    # ---- (b) ----------------------------------------------------------------------------------------------
    if args.big:
        p = dbi.default_params(**CFG2)
        res, off = synth.config_proteome(4, args.big)
        n_small = min(20_000, args.big)
        with dbi.GpuIndex(p) as small:  # the masses of half the queries
            small.add_proteins(res[:int(off[n_small])], off[:n_small + 1])
            small.build()
            m_small = small.fetch(0, small.stats()["n_entries"], with_ids=False)["mass"]
        _, _, lo, hi = synth.synth_queries(m_small, args.big_queries, 20261021)
        shards, one = handles(p, res, off)
        searcher = ShardedSearcher(shards)
        order = np.argsort(lo, kind="stable")
        groups = np.array_split(order, args.groups)
        for grp in groups[:1]:  # warm-up
            search_unindexed_chunked(searcher, lo[grp], hi[grp], UNINDEXED_MAX_CANDIDATES)
            search_unindexed_chunked(one, lo[grp], hi[grp], UNINDEXED_MAX_CANDIDATES)
        rec = {"sharded_ms": [], "single_ms": [], "hits": [], "parity_failed": []}
        for grp in groups:
            a, ms = timed(lambda: search_unindexed_chunked(searcher, lo[grp], hi[grp], UNINDEXED_MAX_CANDIDATES))
            rec["sharded_ms"].append(ms)
            b, ms = timed(lambda: search_unindexed_chunked(one, lo[grp], hi[grp], UNINDEXED_MAX_CANDIDATES))
            rec["single_ms"].append(ms)
            rec["hits"].append(int(b["counts"].n_hits))
            rec["parity_failed"].append(parity_failures(a, b))
            del a, b
            print(json.dumps({k: v[-1] for k, v in rec.items()}), flush=True)
        out["b_two_million_proteins"] = {
            "proteome": "synth.config_proteome(4, %d)" % args.big, "residues": int(len(res)),
            "queries": len(lo), "groups": len(groups), "ppm": 10.0, "seed": 20261021,
            "max_candidates": UNINDEXED_MAX_CANDIDATES, "what_is_timed": "the chunked search of a group, read included",
            "sharded_s": sum(rec["sharded_ms"]) / 1e3, "single_s": sum(rec["single_ms"]) / 1e3, "all": rec}
        for g in shards + [one]:
            g.close()

    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    failed = sum(sum(x != 0 for x in b["all"]["parity_failed"]) for b in out["a_cfg2"]["batches"].values())
    if "b_two_million_proteins" in out:
        failed += sum(x != 0 for x in out["b_two_million_proteins"]["all"]["parity_failed"])
    if failed:
        raise SystemExit(f"parity failed ({failed})")


if __name__ == "__main__":
    main()
