"""Batched peptide lookup (dbi_lookup_peptides) on the cfg2 index, against the best way the library offered before:
one zero-tolerance dbi_query_hits over the same masses + dbi_query_hits_read + a host filter by string and pattern.

Workload: the cfg2 index (BASELINE.json configs[1]: 20 000 synthetic proteins, static C, variable M + STY, <= 3 per
peptide) and a seeded batch of 10^6 rows: 50 % unmodified indexed peptides, 30 % indexed variants with their
patterns, 20 % rows built to be absent (L<->I swap, one-residue substitution, substring).  The two paths alternate,
L2 flushed (256 MiB write) before every timed call; parity of the found sets and protein lists is checked on the
whole batch.  Writes <out>/lookup_bench.json.

    python scripts/lookup_bench.py --out DIR [--rows 1000000] [--reps 5]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
CFG2 = dict(static_mods={"C": 57.02146}, diff_mods=[("M", 15.9949), ("STY", 79.96633)], max_mods_per_peptide=3)
AA = np.frombuffer(b"ACDEFGHKLMNPQRSTVWY", np.uint8)


def gpu_identity():
    out = {}
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        h = pynvml.nvmlDeviceGetHandleByIndex(int(vis.split(",")[0]) if vis else 0)
        name = pynvml.nvmlDeviceGetName(h)
        out["gpu"] = name.decode() if isinstance(name, bytes) else name
        out["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
        out["sm_max_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    except Exception as e:  # noqa: BLE001
        out["nvml_error"] = str(e)
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
        out["nvidia_smi"] = q.stdout.strip()
    return out


def sample_entries(g, n_entries, n, rng):
    """n random index entries: (first_prot, first_off, len, modpat), fetched in chunks."""
    pos = np.sort(rng.choice(n_entries, size=n, replace=False))
    cols = {k: [] for k in ("first_prot", "first_off", "len", "modpat")}
    chunk = 8_000_000
    for s in range(0, n_entries, chunk):
        sel = pos[(pos >= s) & (pos < s + chunk)] - s
        if not len(sel):
            continue
        f = g.fetch(s, min(chunk, n_entries - s), with_ids=False)
        for k in cols:
            cols[k].append(f[k][sel])
    return {k: np.concatenate(v) for k, v in cols.items()}


def make_batch(g, res, off, n_rows, seed):
    rng = np.random.default_rng(seed)
    n_entries = g.stats()["n_entries"]
    ent = sample_entries(g, n_entries, min(n_entries, 4 * n_rows), rng)
    unmod = np.nonzero(ent["modpat"] == 0)[0]
    mod = np.nonzero(ent["modpat"] != 0)[0]
    n_un, n_mod = n_rows // 2, (3 * n_rows) // 10
    n_abs = n_rows - n_un - n_mod
    pick_un = rng.choice(unmod, n_un + n_abs, replace=len(unmod) < n_un + n_abs)
    pick_mod = rng.choice(mod, n_mod, replace=len(mod) < n_mod)

    def pep(i):
        a = int(off[ent["first_prot"][i]]) + int(ent["first_off"][i])
        return res[a:a + int(ent["len"][i])].tobytes()

    seqs = [pep(i) for i in pick_un[:n_un]] + [pep(i) for i in pick_mod]
    pats = [0] * n_un + ent["modpat"][pick_mod].tolist()
    kind = ["unmodified"] * n_un + ["modified"] * n_mod
    for j, i in enumerate(pick_un[n_un:]):
        s = bytearray(pep(i))
        k = j % 3
        if k == 0 and (b"L" in s or b"I" in s):  # equal mass, different string
            s = bytearray(bytes(s).translate(bytes.maketrans(b"LI", b"IL")))
            kind.append("swap_LI")
        elif k == 1 or k == 0:
            p = int(rng.integers(0, len(s)))
            s[p] = int(rng.choice(AA[AA != s[p]]))
            kind.append("substitution")
        else:
            s = s[1:] if len(s) > 1 else s + b"A"
            kind.append("substring")
        seqs.append(bytes(s))
        pats.append(0)
    order = rng.permutation(n_rows)
    return [seqs[i] for i in order], np.asarray(pats, np.uint32)[order], [kind[i] for i in order]


def host_masses(params, residues, offsets, pats):
    """The row masses on the host (calculateMass, then the shifts in pattern order), vectorised over rows."""
    table = np.array(params.residue_mass[:], np.float64)
    diff = np.zeros(256, np.float64)
    for k in range(params.n_mods):
        diff[params.mods[k].residue] = params.mods[k].delta
    lens = np.diff(offsets.astype(np.int64))
    n = len(lens)
    m = np.zeros(n, np.float64)
    if params.add_h2o_proton:
        m = m + params.h2o_proton
    m = m + params.cterm
    m = m + params.nterm
    start = offsets[:-1].astype(np.int64)
    for k in range(int(lens.max()) if n else 0):
        m = m + np.where(k < lens, table[residues[np.minimum(start + k, len(residues) - 1)]], 0.0)
    for k in range(4):
        b = ((pats >> np.uint32(8 * k)) & np.uint32(0xFF)).astype(np.int64)
        m = m + np.where(b > 0, diff[residues[np.minimum(start + np.maximum(b - 1, 0), len(residues) - 1)]], 0.0)
    return m


def filter_hits(h, residues, offsets, pats):
    """Host filter of the zero-tolerance answer by string and pattern: per row the run whose peptide equals the row
    and, inside it, the hit with the row's pattern.  -> (found bool[n], run index of the match or -1)."""
    n = len(offsets) - 1
    run_q = np.repeat(np.arange(n), np.diff(h["pep_off"].astype(np.int64)))
    so = h["seq_off"].astype(np.int64)
    rlen = np.diff(so)
    qs, ql = offsets[:-1].astype(np.int64), np.diff(offsets.astype(np.int64))
    cand = np.nonzero(rlen == ql[run_q])[0]
    # compare the residues column by column over the length-matching runs
    same = np.ones(len(cand), bool)
    L = int(rlen[cand].max()) if len(cand) else 0
    for k in range(L):
        live = k < rlen[cand]
        a = h["seq"][np.minimum(so[cand] + k, len(h["seq"]) - 1)]
        b = residues[np.minimum(qs[run_q[cand]] + k, len(residues) - 1)]
        same &= ~live | (a == b)
    runs = cand[same]
    # the pattern inside the run
    pho = h["pep_hit_off"].astype(np.int64)
    hit_run = np.repeat(np.arange(len(pho) - 1), np.diff(pho))
    is_match = np.zeros(len(pho) - 1, bool)
    is_match[runs] = True
    ok = is_match[hit_run] & (h["modpat"] == pats[run_q[hit_run]])
    match_run = np.full(n, -1, np.int64)
    match_run[run_q[hit_run[ok]]] = hit_run[ok]
    return match_run >= 0, match_run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rows", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--proteins", type=int, default=None)
    args = ap.parse_args()
    import torch

    import dbindex_b200 as dbi
    from dbindex_b200 import synth
    from dbindex_b200.capi import pack_peptides
    from dbindex_b200.indexer import DBIndexer

    if not torch.cuda.is_available():
        raise SystemExit("lookup_bench needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    ident = gpu_identity()
    p = dbi.default_params(**CFG2)
    p.profile = 1
    res, off = synth.config_proteome(2, args.proteins)
    stream = torch.cuda.Stream()
    g = dbi.GpuIndex(p)
    g.set_stream(stream.cuda_stream)
    g.add_proteins(res, off)
    g.build()
    n_entries = g.stats()["n_entries"]
    t0 = time.perf_counter()
    seqs, pats, kinds = make_batch(g, res, off, args.rows, 20261020)
    t_batch = time.perf_counter() - t0
    residues, offsets = pack_peptides(seqs)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]

    def timed(fn):
        flush.zero_()
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            ev[0].record(stream)
        t = time.perf_counter()
        out = fn()
        with torch.cuda.stream(stream):
            ev[1].record(stream)
        stream.synchronize()
        return out, ev[0].elapsed_time(ev[1]), (time.perf_counter() - t) * 1e3

    def new_path():
        cnt, ms_call, _ = timed(lambda: g.lookup_peptides_begin((residues, offsets), pats))
        r, ms_read, _ = timed(lambda: g.lookup_peptides_read(cnt))
        return r, ms_call, ms_read

    def old_path():
        t = time.perf_counter()
        m = host_masses(p, residues, offsets, pats)
        ms_mass = (time.perf_counter() - t) * 1e3
        h, ms_dev, _ = timed(lambda: g.query_hits(m, m, per_hit=False))
        t = time.perf_counter()
        found, match_run = filter_hits(h, residues, offsets, pats)
        ms_filter = (time.perf_counter() - t) * 1e3
        return (h, found, match_run), ms_mass, ms_dev, ms_filter

    for _ in range(2):  # warm-up of both paths (module load, allocator cache)
        new_path()
        old_path()
    rec = {"new_call_ms": [], "new_read_ms": [], "new_kernel_ms": [], "new_e2e_ms": [], "old_mass_ms": [],
           "old_hits_ms": [], "old_filter_ms": [], "old_e2e_ms": []}
    st0 = g.stats()
    for _ in range(args.reps):
        s0 = g.stats()
        t = time.perf_counter()
        r, a, b = new_path()
        rec["new_e2e_ms"].append((time.perf_counter() - t) * 1e3)
        s1 = g.stats()
        rec["new_call_ms"].append(a)
        rec["new_read_ms"].append(b)
        rec["new_kernel_ms"].append(sum(s1["stage_ms"][k] - s0["stage_ms"][k] for k in ("query", "fetch")))
        t = time.perf_counter()
        old, a, b, c = old_path()
        rec["old_e2e_ms"].append((time.perf_counter() - t) * 1e3)
        rec["old_mass_ms"].append(a)
        rec["old_hits_ms"].append(b)
        rec["old_filter_ms"].append(c)
    st1 = g.stats()
    # algorithmic bytes of the lookups only (the old path's query_hits also counts into query / fetch): from one call
    s0 = g.stats()
    g.lookup_peptides((residues, offsets), pats)
    s1 = g.stats()
    algo = sum(s1["algo_bytes"][k] - s0["algo_bytes"][k] for k in ("query", "fetch"))

    # parity on the whole batch: found sets and protein lists of the two paths
    h, found_old, match_run = old
    found_new = r["status"] == 1
    failed = int(np.count_nonzero(found_new != found_old))
    plo_new, plo_old = r["prot_list_off"].astype(np.int64), h["prot_list_off"].astype(np.int64)
    for q in np.nonzero(found_new & found_old)[0].tolist():
        run = match_run[q]
        if not np.array_equal(r["prot_ids"][plo_new[q]:plo_new[q + 1]], h["prot_ids"][plo_old[run]:plo_old[run + 1]]) \
                or r["first_prot"][q] != h["first_prot"][run] or r["first_off"][q] != h["first_off"][run]:
            failed += 1
    assert np.array_equal(r["mass"][r["status"] != 2].view(np.uint64),
                          host_masses(p, residues, offsets, pats)[r["status"] != 2].view(np.uint64))

    # one peptide per call on 10^3 rows: the new path, and the per-peptide path it replaces (host mass, zero-tolerance
    # dbi_query_hits, string filter)
    few = [s.decode() for s, pt in zip(seqs, pats) if pt == 0][:1000]
    mirror = DBIndexer(p)
    mirror.index, mirror.inited = g, True
    t = time.perf_counter()
    per_new = [mirror.getProteinsBatch([s])[0] for s in few]
    ms_per_new = (time.perf_counter() - t) * 1e3
    t = time.perf_counter()
    per_old = []
    for s in few:
        m = g.calculate_mass(s.encode())
        hh = g.query_hits(np.array([m]), np.array([m]))
        so = hh["seq_off"].astype(np.int64)
        po = hh["prot_list_off"].astype(np.int64)
        ids = set()
        for i in range(len(hh["mass"])):
            if hh["modpat"][i] == 0 and hh["seq"][so[i]:so[i + 1]].tobytes().decode() == s:
                ids |= set(hh["prot_ids"][po[i]:po[i + 1]].tolist())
        per_old.append(ids)
    ms_per_old = (time.perf_counter() - t) * 1e3
    per_failed = sum({q.id for q in a} != b for a, b in zip(per_new, per_old))
    mirror.index = None

    med = {k: float(np.median(v)) for k, v in rec.items()}
    n = args.rows
    bpr = algo / n
    out = {
        "what": "dbi_lookup_peptides vs zero-tolerance dbi_query_hits + host filter, cfg2 index",
        **ident,
        "index": {"proteins": int(len(off) - 1), "entries": int(n_entries), "params": "cfg2 (static C, M + STY, <= 3)"},
        "batch": {"rows": n, "kinds": {k: kinds.count(k) for k in sorted(set(kinds))}, "seed": 20261020,
                  "make_s": round(t_batch, 2), "found": int(np.count_nonzero(found_new)),
                  "malformed": int(np.count_nonzero(r["status"] == 2))},
        "l2": "flushed (256 MiB write) before every timed call; 2 warm-up rounds of both paths",
        "reps": args.reps, "median": med, "all": rec,
        "new": {"device_call_ms": med["new_call_ms"], "device_read_ms": med["new_read_ms"],
                "kernel_ms": med["new_kernel_ms"], "e2e_ms": med["new_e2e_ms"],
                "rows_per_s_call_plus_read": n / ((med["new_call_ms"] + med["new_read_ms"]) / 1e3),
                "rows_per_s_e2e": n / (med["new_e2e_ms"] / 1e3),
                "algo_bytes_per_row": bpr,
                "hbm_fraction_of_kernel_time": algo / (med["new_kernel_ms"] / 1e3) / HBM_BYTES_PER_S if med["new_kernel_ms"] else None},
        "query_hits_path": {"host_mass_ms": med["old_mass_ms"], "device_hits_plus_read_ms": med["old_hits_ms"],
                            "host_filter_ms": med["old_filter_ms"], "e2e_ms": med["old_e2e_ms"],
                            "rows_per_s_e2e": n / (med["old_e2e_ms"] / 1e3)},
        "speedup_e2e": med["old_e2e_ms"] / med["new_e2e_ms"],
        "speedup_device": med["old_hits_ms"] / (med["new_call_ms"] + med["new_read_ms"]),
        "per_peptide_1000_rows": {"new_one_row_per_call_ms": ms_per_new, "old_per_peptide_path_ms": ms_per_old,
                                  "failed": per_failed},
        "parity": {"checked": n, "failed": failed},
        "stats_delta_launches": {k: st1["stage_launches"][k] - st0["stage_launches"][k] for k in ("query", "fetch")},
    }
    path = os.path.join(args.out, "lookup_bench.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "power_limit_w", "new", "query_hits_path", "speedup_e2e", "parity")
                      if k in out}))
    g.close()
    if failed or per_failed:
        raise SystemExit(f"parity failed: {failed} rows, {per_failed} per-peptide rows")


if __name__ == "__main__":
    main()
