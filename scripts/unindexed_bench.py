"""Unindexed search (dbi_search_unindexed) measured on two workloads.  Writes <out>/unindexed_bench.json.

(a) cfg2, which fits one GPU (BASELINE.json configs[1]: 20 000 synthetic proteins, static C, variable M + STY, <= 3
    per peptide): seeded 10 ppm batches of 10^2, 10^3 and 10^4 queries (synth.synth_queries: half jittered index
    masses, half uniform).  Per batch three paths, alternated, L2 flushed (256 MiB write) before every timed call,
    every shape warmed up, medians of --reps: dbi_search_unindexed + read on an unbuilt handle; dbi_build +
    dbi_query_hits + read; dbi_query_hits + read alone on a prebuilt index.  Parity: the canonical answer of the
    whole batch (every hit, ties in canonical order) equals the indexed one.
(b) Beyond one GPU's index: --big proteins of synth.config_proteome(4, ...) with cfg2's parameters (about 10^9
    residues for 2 x 10^6 proteins; never built).  10^3 queries at 10 ppm, half masses of an index built on the first
    20 000 proteins jittered +-5 ppm, half uniform, through the mirror's chunked search.  Soundness on the whole
    answer: every hit's mass recomputed on the host in the index's summation order plus the shifts (bit-equal, and
    inside its window), every hit's residues equal to the proteome at its first occurrence.

    python scripts/unindexed_bench.py --out DIR [--reps 5] [--proteins N] [--big 2000000]
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CFG2 = dict(static_mods={"C": 57.02146}, diff_mods=[("M", 15.9949), ("STY", 79.96633)], max_mods_per_peptide=3)
BATCHES = (100, 1000, 10_000)


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.stdout.strip() else ""
    parts = [x.strip() for x in line.split(",")]
    return {"gpu": parts[0] if parts else None, "power_limit": parts[1] if len(parts) > 1 else None,
            "sm_max_clock": parts[2] if len(parts) > 2 else None, "nvidia_smi": line}


def canonical(h):
    """Per-hit arrays of a query_hits-style answer in canonical order: by query, then by every field (ties inside a
    query have no contractual order).  Variable-length parts (residues, protein lists) are ordered by a hash and then
    compared exactly."""
    ho = h["hit_off"].astype(np.int64)
    n = int(ho[-1])
    qid = np.repeat(np.arange(len(ho) - 1), np.diff(ho))
    so, po = h["seq_off"].astype(np.int64), h["prot_list_off"].astype(np.int64)

    def seg_hash(off, data, mult):
        sizes = np.diff(off)
        if len(data) == 0:
            return np.zeros(n, np.uint64)
        pos = np.arange(len(data), dtype=np.uint64) - np.repeat(off[:-1], sizes).astype(np.uint64)
        v = (data.astype(np.uint64) + np.uint64(1)) * (pos * np.uint64(mult) + np.uint64(0x9E3779B97F4A7C15))
        v ^= v >> np.uint64(29)
        out = np.zeros(n, np.uint64)
        nz = sizes > 0
        out[nz] = np.add.reduceat(v, off[:-1][nz])
        return out

    fl = h["flanks"].reshape(-1, 6).astype(np.uint64)
    flk = np.zeros(n, np.uint64)
    for j in range(6):
        flk |= fl[:, j] << np.uint64(8 * j)
    keys = [seg_hash(po, h["prot_ids"], 0xC2B2AE3D27D4EB4F), seg_hash(so, h["seq"], 0xFF51AFD7ED558CCD), flk,
            h["modpat"].astype(np.uint64), h["len"].astype(np.uint64), h["first_off"].astype(np.uint64),
            h["first_prot"].astype(np.uint64), h["mass"].view(np.uint64), qid.astype(np.uint64)]
    perm = np.lexsort(keys)
    from dbindex_b200.capi import _expand_csr
    out = {"q": qid[perm]}
    for k in ("mass", "first_prot", "first_off", "len", "modpat"):
        out[k] = h[k][perm]
    out["flanks"] = fl[perm]
    out["seq_off"], out["seq"] = _expand_csr(so, h["seq"], perm)
    out["prot_list_off"], out["prot_ids"] = _expand_csr(po, h["prot_ids"], perm)
    return out


def parity_failures(a, b):
    """0 when the two canonical answers are equal, else the number of differing hits (or -1 on a size mismatch)."""
    ca, cb = canonical(a), canonical(b)
    if len(ca["q"]) != len(cb["q"]):
        return -1
    bad = np.zeros(len(ca["q"]), bool)
    for k in ("q", "mass", "first_prot", "first_off", "len", "modpat"):
        bad |= ca[k].view(np.uint64) != cb[k].view(np.uint64) if k == "mass" else ca[k] != cb[k]
    bad |= np.any(ca["flanks"] != cb["flanks"], axis=1)
    for o, d in (("seq_off", "seq"), ("prot_list_off", "prot_ids")):
        if not (np.array_equal(ca[o], cb[o]) and np.array_equal(ca[d], cb[d])):
            bad |= True
    return int(np.count_nonzero(bad))


def soundness(p, res, off, lo, hi, h):
    """Failures of the whole answer h of [lo, hi] on the proteome (res, off): mass recomputed in the index's order
    (calculateMass, then the shift of every pattern position left to right) bit-equal and inside its window, residues
    equal to the proteome at the first occurrence."""
    rm = np.array(p.residue_mass[:], np.float64)
    diff = np.zeros(256, np.float64)
    for k in range(p.n_mods):
        diff[p.mods[k].residue] = p.mods[k].delta
    ho = h["hit_off"].astype(np.int64)
    qid = np.repeat(np.arange(len(ho) - 1), np.diff(ho))
    ln = h["len"].astype(np.int64)
    start = off[h["first_prot"].astype(np.int64)].astype(np.int64) + h["first_off"].astype(np.int64)
    # per run (hits of one run share the peptide): the base mass
    runs, first, inv = np.unique(h["hit_pep"], return_index=True, return_inverse=True)
    rs, rl = start[first], ln[first]
    base = np.zeros(len(runs), np.float64)
    if p.add_h2o_proton:
        base += p.h2o_proton
    base += p.cterm
    base += p.nterm
    for j in range(int(rl.max()) if len(rl) else 0):
        live = rl > j
        base[live] += rm[res[rs[live] + j]]
    m = base[inv]
    pat = h["modpat"].astype(np.int64)
    for k in range(4):
        b = (pat >> (8 * k)) & 0xFF
        sel = b > 0
        m[sel] += diff[res[start[sel] + b[sel] - 1]]
    bad = (m.view(np.uint64) != h["mass"].view(np.uint64)) | (h["mass"] < lo[qid]) | (h["mass"] > hi[qid])
    # residues at the first occurrence
    so = h["seq_off"].astype(np.int64)
    sizes = np.diff(so)
    pos = np.repeat(start, sizes) + (np.arange(int(so[-1])) - np.repeat(so[:-1], sizes))
    same = res[pos] == h["seq"]
    seq_bad = np.zeros(len(ln), bool)
    nz = sizes > 0
    seq_bad[nz] = np.minimum.reduceat(same.astype(np.uint8), so[:-1][nz]) == 0
    seq_bad |= sizes != ln
    return {"mass_or_window": int(np.count_nonzero(bad)), "residues": int(np.count_nonzero(seq_bad)),
            "hits": int(len(ln))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--proteins", type=int, default=None, help="part (a): proteins of cfg2 (default 20 000)")
    ap.add_argument("--big", type=int, default=2_000_000, help="part (b): proteins of the cfg4 proteome (0: skip)")
    ap.add_argument("--big-queries", type=int, default=1000)
    ap.add_argument("--group", type=int, default=100, help="part (b): queries per mirror call")
    args = ap.parse_args()
    import torch

    import dbindex_b200 as dbi
    from dbindex_b200 import synth
    from dbindex_b200.indexer import UNINDEXED_MAX_CANDIDATES, search_unindexed_chunked

    if not torch.cuda.is_available():
        raise SystemExit("unindexed_bench needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    out = {"what": "dbi_search_unindexed: (a) cfg2 against build + query and query alone; (b) a proteome whose "
                   "index does not fit one GPU", **gpu_identity()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(fn):
        flush.zero_()
        torch.cuda.synchronize()
        t = time.perf_counter()
        r = fn()  # every call ends in a stream synchronise
        return r, (time.perf_counter() - t) * 1e3

    # ---- (a) ----------------------------------------------------------------------------------------------
    p = dbi.default_params(**CFG2)
    p.profile = 1
    res, off = synth.config_proteome(2, args.proteins)
    un, ix, bq = dbi.GpuIndex(p), dbi.GpuIndex(p), dbi.GpuIndex(p)
    for g in (un, ix, bq):
        g.add_proteins(res, off)
    ix.build()
    st_ix = ix.stats()
    masses = ix.fetch(0, st_ix["n_entries"], with_ids=False)["mass"]
    part_a = {"index": {"proteins": int(len(off) - 1), "residues": int(len(res)), "emitted": st_ix["n_emitted"],
                        "unique": st_ix["n_unique"], "entries": st_ix["n_entries"],
                        "params": "cfg2 (static C, M + STY, <= 3)"},
              "l2": "flushed (256 MiB write) before every timed call; every shape warmed up twice; paths alternated",
              "reps": args.reps, "batches": {}}
    for nq in BATCHES:
        _, _, lo, hi = synth.synth_queries(masses, nq, 20261020 + nq)

        def read(g, cnt):  # dbi_query_hits_read into fresh numpy buffers: the same for every path
            t = time.perf_counter()
            g._read_hits(cnt, None, None, False)
            return (time.perf_counter() - t) * 1e3

        def rebuild():
            bq.reset_index()
            bq.build()

        paths = {"unindexed": (un, lambda: un.search_unindexed_begin(lo, hi)),
                 "build_query": (bq, lambda: (rebuild(), bq.query_hits_begin(lo, hi))[1]),
                 "query_only": (ix, lambda: ix.query_hits_begin(lo, hi))}
        for _ in range(2):
            for g, call in paths.values():
                read(g, call())
        rec = {f"{k}_{x}_ms": [] for k in paths for x in ("call", "read")}
        rec.update({"build_ms": [], "n_candidates": [], "unindexed_stage_ms": []})
        for _ in range(args.reps):
            for k, (g, call) in paths.items():
                cnt, ms = timed(call)
                rec[f"{k}_call_ms"].append(ms)
                rec[f"{k}_read_ms"].append(read(g, cnt))
                if k == "unindexed":
                    s = un.stats()
                    rec["n_candidates"].append(s["n_emitted"])
                    rec["unindexed_stage_ms"].append(s["stage_ms"])
            _, ms = timed(rebuild)
            rec["build_ms"].append(ms)
        su = un.stats()
        med = {k: float(np.median(v)) for k, v in rec.items() if k.endswith("_ms") and k != "unindexed_stage_ms"}
        stage_med = {k: float(np.median([d[k] for d in rec["unindexed_stage_ms"]])) for k in rec["unindexed_stage_ms"][0]}
        # the read is the same on every path: building pays off once k (unindexed call) > build + k (query call)
        gain = med["unindexed_call_ms"] - med["query_only_call_ms"]
        pays_off = math.floor(med["build_ms"] / gain) + 1 if gain > 0 else None
        ha = un.search_unindexed(lo, hi)
        hb = ix.query_hits(lo, hi)
        part_a["batches"][str(nq)] = {
            "queries": nq, "ppm": 10.0, "seed": 20261020 + nq, "median_ms": med, "all_ms": rec,
            "n_candidates": int(su["n_emitted"]), "candidate_unique": int(su["n_unique"]),
            "candidate_entries": int(su["n_entries"]),
            "candidate_fraction_of_emitted": su["n_emitted"] / st_ix["n_emitted"],
            "unindexed_stage_ms_median": stage_med,
            "hits": int(hb["counts"].n_hits),
            "batches_after_which_building_pays_off": pays_off,
            "parity": {"hits_checked": int(hb["counts"].n_hits), "failed": parity_failures(ha, hb)},
        }
        print(json.dumps({"nq": nq, **med, "n_candidates": int(su["n_emitted"]), "pays_off_after": pays_off,
                          "parity_failed": part_a["batches"][str(nq)]["parity"]["failed"]}), flush=True)
    for g in (un, ix, bq):
        g.close()
    del masses
    out["a_cfg2"] = part_a
    path = os.path.join(args.out, "unindexed_bench.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)

    # ---- (b) ----------------------------------------------------------------------------------------------
    if args.big:
        p = dbi.default_params(**CFG2)
        p.profile = 1
        t = time.perf_counter()
        res, off = synth.config_proteome(4, args.big)
        t_gen = time.perf_counter() - t
        print(json.dumps({"generated_residues": int(len(res)), "s": round(t_gen, 1)}), flush=True)
        n_small = min(20_000, args.big)
        with dbi.GpuIndex(p) as small:  # the masses of half the queries
            small.add_proteins(res[:int(off[n_small])], off[:n_small + 1])
            small.build()
            m_small = small.fetch(0, small.stats()["n_entries"], with_ids=False)["mass"]
        _, _, lo, hi = synth.synth_queries(m_small, args.big_queries, 20261021)
        del m_small
        g = dbi.GpuIndex(p)
        t = time.perf_counter()
        g.add_proteins(res, off)
        g.upload()
        t_add = time.perf_counter() - t
        calls = []
        inner = g.search_unindexed

        def counted(lo_, hi_, cap=0, **kw):
            t0 = time.perf_counter()
            try:
                r = inner(lo_, hi_, cap, **kw)
            except dbi.DbiError as e:
                calls.append({"queries": len(lo_), "n_candidates": e.n_candidates, "over_cap": True,
                              "ms": (time.perf_counter() - t0) * 1e3})
                raise
            s = g.stats()
            calls.append({"queries": len(lo_), "n_candidates": s["n_emitted"], "candidate_entries": s["n_entries"],
                          "hits": int(r["counts"].n_hits), "ms": (time.perf_counter() - t0) * 1e3,
                          "stage_ms": s["stage_ms"]})
            return r

        g.search_unindexed = counted
        # the whole answer is ~5 x 10^4 hits per query: the mass-sorted queries go through the chunked search in
        # groups, each checked and dropped before the next, so that the host holds one group's hits at a time
        order = np.argsort(lo, kind="stable")
        groups = np.array_split(order, max(1, len(order) // args.group))
        total_s, t_sound, n_hits = 0.0, 0.0, 0
        sound = {"mass_or_window": 0, "residues": 0, "hits": 0}
        for grp in groups:
            flush.zero_()
            torch.cuda.synchronize()
            t = time.perf_counter()
            h = search_unindexed_chunked(g, lo[grp], hi[grp], UNINDEXED_MAX_CANDIDATES)
            total_s += time.perf_counter() - t
            t = time.perf_counter()
            for k, v in soundness(p, res, off, lo[grp], hi[grp], h).items():
                sound[k] += v
            t_sound += time.perf_counter() - t
            n_hits += int(h["counts"].n_hits)
            del h
            print(json.dumps({"group_queries": len(grp), "calls": len(calls), "total_s": total_s, "hits": n_hits}),
                  flush=True)
        g.search_unindexed = inner
        out["b_beyond_one_gpu"] = {
            "proteome": {"config": "synth.config_proteome(4, %d)" % args.big, "proteins": int(len(off) - 1),
                         "residues": int(len(res)), "params": "cfg2 (static C, M + STY, <= 3)",
                         "index_built": False, "generate_s": round(t_gen, 1), "add_proteins_s": round(t_add, 2),
                         "index_entries": "not measured (extrapolated from the 3.46 G entries of 10^6 cfg4 proteins: "
                                          "about 6.9 G, above the 2^32 entries one handle holds)"},
            "queries": len(lo), "ppm": 10.0, "seed": 20261021, "query_masses": "half from an index of the first 20 000 "
                                                                           "proteins jittered +-5 ppm, half uniform",
            "max_candidates": UNINDEXED_MAX_CANDIDATES,
            "total_s": total_s, "queries_per_s": len(lo) / total_s,
            "query_groups": len(groups), "device_calls": len(calls),
            "chunks": sum(1 for c in calls if not c.get("over_cap")), "calls": calls,
            "hits": n_hits, "l2": "flushed before every query group",
            "soundness": {**sound, "failed": sound["mass_or_window"] + sound["residues"], "check_s": round(t_sound, 1)},
        }
        print(json.dumps({k: v for k, v in out["b_beyond_one_gpu"].items() if k != "calls"}), flush=True)
        g.close()

    path = os.path.join(args.out, "unindexed_bench.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    failed = sum(b["parity"]["failed"] != 0 for b in out["a_cfg2"]["batches"].values())
    if "b_beyond_one_gpu" in out:
        failed += out["b_beyond_one_gpu"]["soundness"]["failed"] != 0
    if failed:
        raise SystemExit(f"parity / soundness failed ({failed})")


if __name__ == "__main__":
    main()
