"""Query views against one shared handle behind a lock, for the legacy per-spectrum call pattern of a search engine.
Writes <out>/views_bench.json.

Workload: the cfg2 index (BASELINE.json configs[1]: 20 000 synthetic proteins, static C, variable M + STY, <= 3 per
peptide) and 10^4 spectra at 10 ppm from synth.synth_queries.  Every spectrum is one getSequences(mass, tol) of the
reference: dbi_query_hits with nq = 1 and dbi_query_hits_read of every buffer, as GpuDBIndexStore.queryOn does.
T in --threads threads split the spectra round robin and call
  (a) lock:  one shared handle, each call pair under one process-wide lock (what a correct store does without views);
  (b) views: one view per thread (dbi_view_open), no lock.
The calls are raw ctypes calls into preallocated pinned buffers of each thread (dbi_host_alloc): ctypes releases the
GIL inside the foreign call, so the threads overlap in the library.  Reported per mode and T: calls/s over the wall
time of all threads, p50 / p99 latency of one call pair (lock wait included), and parity failures: every thread's
answer against the matching spectrum of one dbi_query_spectra batch of all 10^4 spectra (DBI_TOL_DA, one range per
spectrum), compared per spectrum as the multiset of (mass, first occurrence, length, mod patterns, residues, protein
ids).  That batch, timed with its read, is reported as the ceiling.  Each (mode, T) runs --reps times, alternating
the modes; the median run is reported.

    python scripts/views_bench.py --out DIR [--threads 1,2,4,8,16,32] [--reps 3]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from unindexed_bench import CFG2, gpu_identity  # noqa: E402

N_SPECTRA = 10_000


def run_key(h, s):
    """Per spectrum s of a raw (run-grouped) answer: the sorted multiset of its runs."""
    po, hp = h["pep_off"].astype(np.int64), h["pep_hit_off"].astype(np.int64)
    so, pl = h["seq_off"].astype(np.int64), h["prot_list_off"].astype(np.int64)
    out = []
    for p in range(po[s], po[s + 1]):
        out.append((int(h["mass"][p:p + 1].view(np.uint64)[0]), int(h["first_prot"][p]), int(h["first_off"][p]),
                    int(h["len"][p]), tuple(sorted(h["modpat"][hp[p]:hp[p + 1]].tolist())),
                    h["seq"][so[p]:so[p + 1]].tobytes(), tuple(h["prot_ids"][pl[p]:pl[p + 1]].tolist())))
    return sorted(out)


class Caller:
    """One thread's pinned buffers and its raw dbi_query_hits + dbi_query_hits_read pair."""

    def __init__(self, lib, cap, dbi):
        from dbindex_b200.capi import HIT_FIELDS, DbiHitBuffers, DbiHitCounts
        self.lib, self.blocks = lib, []
        self.fields = HIT_FIELDS
        self.io = self._pinned(np.float64, 2)
        self.cnt = DbiHitCounts()
        self.bufs = DbiHitBuffers()
        self.arr = {}
        for name, (dt, size) in HIT_FIELDS.items():
            self.arr[name] = a = self._pinned(dt, int(size(cap)) + 8)
            setattr(self.bufs, name, a.ctypes.data)

    def _pinned(self, dt, n):
        p = C.c_void_p()
        nbytes = max(1, n) * np.dtype(dt).itemsize
        rc = self.lib.dbi_host_alloc(nbytes, C.byref(p))
        assert rc == 0, rc
        self.blocks.append(p)
        return np.frombuffer((C.c_uint8 * nbytes).from_address(p.value), dtype=dt)

    def call(self, h, lo, hi):
        self.io[0], self.io[1] = lo, hi
        d = self.io.ctypes.data
        rc = self.lib.dbi_query_hits(h, d, d + 8, 1, C.byref(self.cnt))
        if rc == 0:
            rc = self.lib.dbi_query_hits_read(h, C.byref(self.bufs))
        assert rc == 0, (rc, self.lib.dbi_last_error())

    def snapshot(self):
        c = self.cnt
        return {name: np.array(self.arr[name][:int(size(c))]) for name, (dt, size) in self.fields.items()}

    def free(self):
        for p in self.blocks:
            self.lib.dbi_host_free(p)


def run_mode(g, lib, mode, T, lo, hi, cap, dbi, keep):
    callers = [Caller(lib, cap, dbi) for _ in range(T)]
    views = [g.view() for _ in range(T)] if mode == "views" else None
    lock = threading.Lock()
    lat = [[] for _ in range(T)]
    answers = [dict() for _ in range(T)]
    start = threading.Barrier(T + 1)

    def body(t):
        c, h = callers[t], (views[t]._h if views else g._h)
        my = range(t, len(lo), T)
        start.wait()
        for s in my:
            t0 = time.perf_counter()
            if views:
                c.call(h, lo[s], hi[s])
            else:
                with lock:
                    c.call(h, lo[s], hi[s])
            lat[t].append(time.perf_counter() - t0)
            if keep:
                answers[t][s] = c.snapshot()

    th = [threading.Thread(target=body, args=(t,)) for t in range(T)]
    for x in th:
        x.start()
    start.wait()
    t0 = time.perf_counter()
    for x in th:
        x.join()
    wall = time.perf_counter() - t0
    for c in callers:
        c.free()
    for v in views or []:
        v.close()
    ls = np.array([x for l_ in lat for x in l_])
    got = {}
    for a in answers:
        got.update(a)
    return {"wall_s": wall, "calls_per_s": len(lo) / wall, "p50_us": float(np.percentile(ls, 50) * 1e6),
            "p99_us": float(np.percentile(ls, 99) * 1e6), "mean_us": float(ls.mean() * 1e6)}, got


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--threads", default="1,2,4,8,16,32")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--proteins", type=int, default=20_000)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    import dbindex_b200 as dbi
    from dbindex_b200 import synth
    from dbindex_b200.capi import DBI_TOL_DA

    lib = dbi.load_library()
    p = dbi.default_params(**CFG2)
    res, off = synth.config_proteome(2, args.proteins)
    g = dbi.GpuIndex(p)
    g.add_proteins(res, off)
    g.build()
    masses = g.fetch(0, g.stats()["n_entries"], with_ids=False)["mass"]
    mass, tol, lo, hi = synth.synth_queries(masses, N_SPECTRA, 20240601 + 2, ppm=10.0)

    # the ceiling, and the reference answer of every spectrum
    range_off = np.arange(N_SPECTRA + 1, dtype=np.uint64)
    g.query_spectra(mass, tol, range_off, DBI_TOL_DA, per_hit=False)  # warm-up
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        batch = g.query_spectra(mass, tol, range_off, DBI_TOL_DA, per_hit=False)
        ts.append(time.perf_counter() - t0)
    t_batch = float(np.median(ts))
    ho, po = batch["hit_off"].astype(np.int64), batch["pep_off"].astype(np.int64)
    so, pl = batch["seq_off"].astype(np.int64), batch["prot_list_off"].astype(np.int64)
    per = [(int(ho[s + 1] - ho[s]), int(po[s + 1] - po[s]), int(so[po[s + 1]] - so[po[s]]),
            int(pl[po[s + 1]] - pl[po[s]])) for s in range(N_SPECTRA)]
    from dbindex_b200.capi import DbiHitCounts
    cap = DbiHitCounts(1, *[max(x[i] for x in per) for i in range(4)])
    want = [run_key(batch, s) for s in range(N_SPECTRA)]

    threads = [int(x) for x in args.threads.split(",")]
    result = {"gpu": gpu_identity(), "workload": {"index": "cfg2", "proteins": args.proteins,
                                                  "entries": int(g.stats()["n_entries"]), "spectra": N_SPECTRA,
                                                  "ppm": 10.0, "hits": int(ho[-1])},
              "ceiling_query_spectra": {"s": t_batch, "spectra_per_s": N_SPECTRA / t_batch}, "runs": []}
    run_mode(g, lib, "lock", 1, lo[:500], hi[:500], cap, dbi, False)  # warm-up of both modes
    run_mode(g, lib, "views", 1, lo[:500], hi[:500], cap, dbi, False)
    for T in threads:
        for mode in ("lock", "views"):
            result["runs"].append({"mode": mode, "threads": T, "reps": [], "parity_failures": None})
        for rep in range(args.reps):
            for mode in ("lock", "views"):
                keep = rep == 0
                r, got = run_mode(g, lib, mode, T, lo, hi, cap, dbi, keep)
                entry = next(x for x in result["runs"] if x["mode"] == mode and x["threads"] == T)
                entry["reps"].append(r)
                if keep:
                    entry["parity_failures"] = sum(run_key(got[s], 0) != want[s] for s in range(N_SPECTRA))
        for mode in ("lock", "views"):
            entry = next(x for x in result["runs"] if x["mode"] == mode and x["threads"] == T)
            med = sorted(entry["reps"], key=lambda r: r["calls_per_s"])[len(entry["reps"]) // 2]
            entry.update({k: v for k, v in med.items()})
            print(f"{mode:5s} T={T:2d}: {med['calls_per_s']:9.0f} calls/s  p50 {med['p50_us']:7.1f} us  "
                  f"p99 {med['p99_us']:8.1f} us  parity failures {entry['parity_failures']}", flush=True)
    g.close()
    single = {m: next(x for x in result["runs"] if x["mode"] == m and x["threads"] == 1)["mean_us"]
              for m in ("lock", "views")} if 1 in threads else None
    result["single_thread_us_per_call"] = single
    with open(os.path.join(args.out, "views_bench.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("gpu", "ceiling_query_spectra", "single_thread_us_per_call")}))


if __name__ == "__main__":
    main()
