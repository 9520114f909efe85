"""Batched spectrum queries against the per-spectrum route, on one GPU.

Indexed, on the cfg2 index (20 000 synthetic proteins, static C, variable M + STY, <= 3 per peptide): 10^4 and 10^5
seeded spectra with masses as in synth.synth_queries (half an entry jittered by +-5 ppm, half uniform), three kinds:
  (a) 5 isotope windows m + k * 1.00335 Da, k = -1..3, each 10 ppm of m in Da (getSequences(List<MassRange>));
  (b) PPM at 10 ppm and (c) PPM at 50 ppm (getSequencesUsingPPMTolerance).
Paths, alternated, with a 256 MB write between timed passes so that L2 (126 MB) holds nothing of the previous one,
every shape warmed up, medians of 5; every path ends with the hits read into host memory (dbi_query_hits_read):
  batch   dbi_query_spectra + read;
  flat    (a) only: host merge_intervals + one dbi_query_hits over every merged interval of the batch + read;
  single  the per-spectrum route the mirror took before the batches, on the first 10^3 spectra (reported for that
          subset): host merge_intervals + one dbi_query_hits per spectrum; for PPM the window, then one
          dbi_query_hits per probe until one is empty.
Unindexed, on the same proteome: 10^3 PPM spectra (10 ppm) as one dbi_search_unindexed_spectra against the
per-spectrum route (window and probes, each a dbi_search_unindexed) on 10^2 of them.
Parity: the batch answer of the subset against the per-spectrum route, hit by hit in canonical order (mass bits,
first occurrence, length, mod pattern, flanks, residues, protein list); the number of differing hits is reported
(-1: different hit counts).  Needs a GPU; card and power limit are read in the same run.  Every record is printed
and the JSON rewritten as soon as it is measured.
"""
from __future__ import annotations

import argparse
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


def out_of_buckets(x, f=8):
    return int(x) // (8000 // f) > f - 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--proteins", type=int, default=20000)
    ap.add_argument("--sizes", default="10000,100000")
    ap.add_argument("--subset", type=int, default=1000)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("spectra_bench needs a GPU")
    import dbindex_b200 as dbi
    from dbindex_b200 import synth
    from dbindex_b200.capi import DBI_TOL_DA, DBI_TOL_PPM, expand_hits
    from dbindex_b200.indexer import MassRange, _merge_hits, merge_intervals, tolerance_in_dalton
    from unindexed_bench import CFG2, gpu_identity, parity_failures

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    os.makedirs(args.out, exist_ok=True)
    out = {"identity": gpu_identity(), "proteins": args.proteins, "indexed": [], "unindexed": None}

    def save(rec):
        print(json.dumps({k: v for k, v in rec.items() if not k.endswith("_all")}), flush=True)
        with open(os.path.join(args.out, "r06_spectra_bench.json"), "w") as fh:
            json.dump(out, fh, indent=1)

    def timed(fn):
        flush_buf.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    def measure(paths, rec):
        for f in paths.values():  # warm every shape
            f()
        times = {k: [] for k in paths}
        for _ in range(args.reps):
            for k, f in paths.items():
                times[k].append(timed(f))
                print(f"  {rec.get('kind', 'unindexed')} {k}: {1e3 * times[k][-1]:.1f} ms", file=sys.stderr, flush=True)
        for k, v in times.items():
            rec[f"{k}_ms_median"] = 1e3 * float(np.median(v))
            rec[f"{k}_ms_all"] = [1e3 * x for x in v]

    def da_single(call, mass, tol, r0, r1, k, parts):
        mg = merge_intervals([MassRange(float(mass[j]), float(tol[j])) for j in range(r0, r1)])
        if mg and not any(out_of_buckets(a) or out_of_buckets(b) for a, b in mg):
            parts.append((np.full(len(mg), k), call(np.array([a for a, _ in mg]), np.array([b for _, b in mg]))))

    def ppm_single(call, m, ppm, k, parts):
        """getSequencesUsingPPMTolerance's loop (ppm > 0): the window holds u_0, so probe hits count from u_1 on."""
        tol = tolerance_in_dalton(m, ppm)
        lo, hi = max(m - tol, 0.0), m + tol
        if out_of_buckets(lo) or out_of_buckets(hi):
            return
        parts.append((np.array([k]), call(np.array([lo]), np.array([hi]))))
        u, first = hi, True
        while u - tolerance_in_dalton(u, ppm) < m and not out_of_buckets(u):
            h = call(np.array([u]), np.array([u]))
            if h["counts"].n_hits == 0:
                break
            if not first:
                parts.append((np.array([k]), h))
            first = False
            nu = u + PRECISION
            if nu == u:
                break
            u = nu

    p = dbi.default_params(**CFG2)
    res, off = synth.synth_proteome(args.proteins, 2024)
    with dbi.GpuIndex(p) as g:
        g.add_proteins(res, off)
        g.build()
        entries = g.fetch(0, g.stats()["n_entries"])["mass"]
        out["n_entries"] = int(len(entries))
        raw = lambda lo, hi: g.query_hits(lo, hi, per_hit=False)  # noqa: E731
        exp = lambda lo, hi: g.query_hits(lo, hi)  # noqa: E731
        for n in [int(x) for x in args.sizes.split(",")]:
            m = np.ascontiguousarray(synth.synth_queries(entries, n, 77 + n)[0], np.float64)
            da_mass = np.repeat(m, 5) + np.tile(np.arange(-1, 4) * ISO, n)
            da_tol = np.repeat(m * 1e-5, 5)
            da_off = np.arange(0, 5 * n + 1, 5, dtype=np.uint64)
            sub = min(n, args.subset)

            def flat():
                lo, hi = [], []
                for s in range(n):
                    mg = merge_intervals([MassRange(float(da_mass[5 * s + j]), float(da_tol[5 * s + j]))
                                          for j in range(5)])
                    if not any(out_of_buckets(a) or out_of_buckets(b) for a, b in mg):
                        lo += [a for a, _ in mg]
                        hi += [b for _, b in mg]
                return raw(np.array(lo), np.array(hi))

            def run_singles(kind, call, k_end):
                parts = []
                for k in range(k_end):
                    if kind == "a":
                        da_single(call, da_mass, da_tol, 5 * k, 5 * k + 5, k, parts)
                    else:
                        ppm_single(call, float(m[k]), 10.0 if kind == "b" else 50.0, k, parts)
                return parts

            kinds = {
                "a": ("isotopes_10ppm", lambda s: g.query_spectra(da_mass[:5 * s], da_tol[:5 * s], da_off[:s + 1],
                                                                  DBI_TOL_DA, 8, per_hit=False)),
                "b": ("ppm10", lambda s: g.query_spectra(m[:s], np.full(s, 10.0), None, DBI_TOL_PPM, 8, per_hit=False)),
                "c": ("ppm50", lambda s: g.query_spectra(m[:s], np.full(s, 50.0), None, DBI_TOL_PPM, 8, per_hit=False)),
            }
            for kind, (name, batch) in kinds.items():
                rec = {"n_spectra": n, "kind": name, "single_subset_spectra": sub}
                out["indexed"].append(rec)
                paths = {"batch": lambda: batch(n), "single_subset": lambda: run_singles(kind, raw, sub)}
                if kind == "a":
                    paths["flat"] = flat
                measure(paths, rec)
                rec["n_hits"] = int(batch(n)["counts"].n_hits)
                got = expand_hits(batch(sub))
                ref = _merge_hits(run_singles(kind, exp, sub), sub)
                rec["parity_checked_hits"] = int(ref["counts"].n_hits)
                rec["parity_diff_hits"] = parity_failures(got, ref)
                rec["batch_us_per_spectrum"] = 1e3 * rec["batch_ms_median"] / n
                rec["single_us_per_spectrum"] = 1e3 * rec["single_subset_ms_median"] / sub
                save(rec)

    with dbi.GpuIndex(p) as u:  # unindexed: the proteins only
        u.add_proteins(res, off)
        m = np.ascontiguousarray(synth.synth_queries(entries, 1000, 4242)[0], np.float64)
        raw_u = lambda lo, hi: u.search_unindexed(lo, hi, per_hit=False)  # noqa: E731
        exp_u = lambda lo, hi: u.search_unindexed(lo, hi)  # noqa: E731
        batch = lambda s: u.search_unindexed_spectra(m[:s], np.full(s, 10.0), None, DBI_TOL_PPM, 8,  # noqa: E731
                                                     per_hit=False)

        def singles(call, k_end):
            parts = []
            for k in range(k_end):
                ppm_single(call, float(m[k]), 10.0, k, parts)
            return parts

        rec = {"batch_spectra": 1000, "single_spectra": 100, "ppm": 10.0}
        out["unindexed"] = rec
        measure({"batch": lambda: batch(1000), "single": lambda: singles(raw_u, 100)}, rec)
        rec["n_candidates_batch"] = int(u.last_candidates)
        got = expand_hits(batch(100))
        ref = _merge_hits(singles(exp_u, 100), 100)
        rec["parity_checked_hits"] = int(ref["counts"].n_hits)
        rec["parity_diff_hits"] = parity_failures(got, ref)
        save(rec)
    out["parity_diff_total"] = sum(abs(r["parity_diff_hits"]) for r in out["indexed"] + [out["unindexed"]])
    save({"identity": out["identity"], "parity_diff_total": out["parity_diff_total"]})


if __name__ == "__main__":
    main()
