"""Batched spectrum queries on a sharded index against what sharded callers did before them.

Setup: the cfg2 index (20 000 synthetic proteins, static C, variable M + STY, <= 3 per peptide) sharded with
dbi_mg_build_local over every visible GPU, or over --world handles on one GPU when there is only one.  On one GPU
the numbers show the round trips the batch removes, not multi-GPU scaling: every record says which ("one_gpu").
Spectra (seeded, masses as in synth.synth_queries): 10^4 PPM spectra at 10 ppm and 10^4 isotope lists (5 windows
m + k * 1.00335 Da, k = -1..3, each 10 ppm of m in Da).
Paths, alternated, with a 256 MB write before every timed call so that L2 (126 MB) holds nothing of the previous
one, every shape warmed up, medians of --reps; every path ends with the hits of every rank read into host memory:
  batch   dbi_mg_query_spectra_local + dbi_query_hits_read on every rank;
  routed  the per-spectrum route, on the first --subset spectra (reported for that subset): host merge_intervals
          and one dbi_query_hits per spectrum on every rank owning a slice the spectrum's intervals touch; for PPM
          the routed window, then one routed dbi_query_hits per probe until one comes back empty on its owner.
Parity: the batch answer of the subset against the routed answer, hit by hit in canonical order; the number of
differing hits is reported (0 expected, -1: different hit counts).  Needs a GPU; card and power limit are read in
the same run.
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
sys.path.insert(0, os.path.join(ROOT, "scripts"))

ISO = 1.00335
PRECISION = 1e-6
FACTOR = 8


def out_of_buckets(x, f=FACTOR):
    return int(x) // (8000 // f) > f - 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--proteins", type=int, default=20000)
    ap.add_argument("--spectra", type=int, default=10000)
    ap.add_argument("--subset", type=int, default=1000)
    ap.add_argument("--world", type=int, default=3, help="handles on one GPU when only one is visible (2..4)")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("mg_spectra_bench needs a GPU")
    import dbindex_b200 as dbi
    from dbindex_b200 import synth
    from dbindex_b200.capi import DBI_TOL_DA, DBI_TOL_PPM, DbiHitCounts, _ptr, expand_hits
    from dbindex_b200.indexer import MassRange, _merge_hits, merge_intervals, tolerance_in_dalton
    from dbindex_b200.multigpu import build_local, route_queries, shard_proteins, split_masses
    from unindexed_bench import CFG2, gpu_identity, parity_failures

    n_gpu = torch.cuda.device_count()
    world = n_gpu if n_gpu > 1 else args.world
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    os.makedirs(args.out, exist_ok=True)
    out = {"identity": gpu_identity(), "proteins": args.proteins, "world": world, "gpus": n_gpu,
           "one_gpu": n_gpu == 1, "records": []}

    def save(rec):
        print(json.dumps({k: v for k, v in rec.items() if not k.endswith("_all")}), flush=True)
        with open(os.path.join(args.out, "mg_spectra_bench.json"), "w") as fh:
            json.dump(out, fh, indent=1)

    def timed(fn):
        flush_buf.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        for d in range(n_gpu):
            torch.cuda.synchronize(d)
        return time.perf_counter() - t0

    def measure(paths, rec):
        for f in paths.values():  # warm every shape
            f()
        times = {k: [] for k in paths}
        for _ in range(args.reps):
            for k, f in paths.items():
                times[k].append(timed(f))
                print(f"  {rec['kind']} {k}: {1e3 * times[k][-1]:.1f} ms", file=sys.stderr, flush=True)
        for k, v in times.items():
            rec[f"{k}_ms_median"] = 1e3 * float(np.median(v))
            rec[f"{k}_ms_all"] = [1e3 * x for x in v]

    p = dbi.default_params(**CFG2)
    res, off = synth.synth_proteome(args.proteins, 2024)
    hs = []
    for r in range(world):
        q = p.copy()
        q.device = r % n_gpu
        g = dbi.GpuIndex(q)
        sres, soff, _ = shard_proteins(res, off, r, world)
        g.add_proteins(sres, soff)
        hs.append(g)
    try:
        build_local(hs)
        split = split_masses(hs[0], world)
        entries = np.sort(np.concatenate([g.fetch(0, g.stats()["n_entries"], with_ids=False)["mass"] for g in hs]))
        out["n_entries"] = int(len(entries))
        lib = hs[0].lib
        lib.dbi_mg_query_spectra_local.restype = C.c_int
        lib.dbi_mg_query_spectra_local.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_uint64, C.c_int, C.c_int, C.POINTER(DbiHitCounts)]
        arr = (C.c_void_p * world)(*[g._h for g in hs])

        def batch(mass, tol, roff, mode, per_hit=False):
            counts = (DbiHitCounts * world)()
            ns = len(roff) - 1 if roff is not None else len(mass)
            rc = lib.dbi_mg_query_spectra_local(arr, world, _ptr(mass), _ptr(tol), _ptr(roff), ns, mode, FACTOR, counts)
            if rc != 0:
                raise RuntimeError(lib.dbi_last_error())
            return [g._read_hits(counts[r], None, None, per_hit) for r, g in enumerate(hs)]

        def routed_call(lo, hi, per_hit):
            """one dbi_query_hits per rank owning a slice [lo, hi] touches; the ranks' answers"""
            lo, hi = np.array([lo]), np.array([hi])
            return [g.query_hits(lo, hi, per_hit=per_hit) for r, g in enumerate(hs)
                    if len(route_queries(lo, hi, split, r, world))]

        def routed(kind, mass, tol, n, per_hit=False):
            parts = []
            for k in range(n):
                if kind == "isotopes_10ppm":
                    mg = merge_intervals([MassRange(float(mass[5 * k + j]), float(tol[5 * k + j])) for j in range(5)])
                    if not any(out_of_buckets(a) or out_of_buckets(b) for a, b in mg):
                        for a, b in mg:
                            parts += [(np.array([k]), h) for h in routed_call(a, b, per_hit)]
                    continue
                m, ppm = float(mass[k]), float(tol[k])  # getSequencesUsingPPMTolerance's loop (ppm > 0)
                t = tolerance_in_dalton(m, ppm)
                lo, hi = max(m - t, 0.0), m + t
                if out_of_buckets(lo) or out_of_buckets(hi):
                    continue
                parts += [(np.array([k]), h) for h in routed_call(lo, hi, per_hit)]
                u, first = hi, True
                while u - tolerance_in_dalton(u, ppm) < m and not out_of_buckets(u):
                    hh = routed_call(u, u, per_hit)
                    if sum(int(h["counts"].n_hits) for h in hh) == 0:
                        break
                    if not first:
                        parts += [(np.array([k]), h) for h in hh]
                    first = False
                    nu = u + PRECISION
                    if nu == u:
                        break
                    u = nu
            return parts

        n, sub = args.spectra, min(args.spectra, args.subset)
        m = np.ascontiguousarray(synth.synth_queries(entries, n, 77 + n)[0], np.float64)
        kinds = {
            "isotopes_10ppm": (np.repeat(m, 5) + np.tile(np.arange(-1, 4) * ISO, n), np.repeat(m * 1e-5, 5),
                               np.arange(0, 5 * n + 1, 5, dtype=np.uint64), DBI_TOL_DA),
            "ppm10": (m, np.full(n, 10.0), None, DBI_TOL_PPM),
        }
        for kind, (mass, tol, roff, mode) in kinds.items():
            rec = {"kind": kind, "n_spectra": n, "routed_subset_spectra": sub, "world": world, "one_gpu": n_gpu == 1}
            out["records"].append(rec)
            measure({"batch": lambda: batch(mass, tol, roff, mode),
                     "routed_subset": lambda: routed(kind, mass, tol, sub)}, rec)
            rec["n_hits"] = int(sum(h["counts"].n_hits for h in batch(mass, tol, roff, mode)))
            smass, stol = (mass[:5 * sub], tol[:5 * sub]) if roff is not None else (mass[:sub], tol[:sub])
            sroff = roff[:sub + 1] if roff is not None else None
            q = np.arange(sub)
            got = _merge_hits([(q, expand_hits(h)) for h in batch(smass, stol, sroff, mode)], sub)
            ref = _merge_hits(routed(kind, mass, tol, sub, per_hit=True), sub)
            rec["parity_checked_hits"] = int(ref["counts"].n_hits)
            rec["parity_diff_hits"] = parity_failures(got, ref)
            rec["batch_us_per_spectrum"] = 1e3 * rec["batch_ms_median"] / n
            rec["routed_us_per_spectrum"] = 1e3 * rec["routed_subset_ms_median"] / sub
            save(rec)
    finally:
        for g in hs:
            g.close()
    out["parity_diff_total"] = sum(abs(r["parity_diff_hits"]) for r in out["records"])
    save({"identity": out["identity"], "parity_diff_total": out["parity_diff_total"]})


if __name__ == "__main__":
    main()
