#!/usr/bin/env python
"""bench.py -- the hot path of dbIndex on B200: index build + precursor-mass queries.

One step = one pass of the hot path over one batch of synthetic input:
  dbi_build (pack -> digest -> sort -> merge -> mod expansion -> sort) on the device-resident
  residues of the workload, followed by one batch of precursor queries whose hits are materialised
  (what getSequences returns: mass, peptide sequence, flanks, protein ids, offset, mod pattern).
Workload at N = 1 (headline): BASELINE.json configs[1] -- the synthetic Swiss-Prot-sized FASTA (20 000
proteins, ~10 M residues, seed 20240601+1), trypsin, 2 missed cleavages, 600-6000 Da, static
carbamidomethyl-C, variable Met-oxidation + STY-phospho (<= 3 per peptide), 10 000 queries at 10 ppm.
The same JSON line carries the other single-GPU configs as `configs`: cfg1 (no mods), cfg3 (semi-tryptic,
200 000 proteins, full size) and a cfg5-style sweep of 10^6 queries (half 10 ppm, half +-3 Da) against
cfg3's index.  N > 1: ONE index over N x 20 000 proteins, FASTA sharded over the ranks (weak scaling),
with an in-run parity check against the oracle on every line.

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
  python bench.py --impl reference ...                    # CPU restatement of the reference (oracle/)
  python bench.py ... --dump-outputs DIR                  # + the last timed step's index and hits as DIR/*.npy

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = ("cfg2: synthetic Swiss-Prot-sized FASTA (20000 proteins, ~10M residues), trypsin, 2 missed cleavages, "
            "600-6000 Da, static C+57.02146, variable M+15.9949 / STY+79.96633, <=3 per peptide, "
            "index build + 10000 queries @ 10 ppm with every hit materialised")
CFG1 = dict()
CFG2 = dict(static_mods={"C": 57.02146}, diff_mods=[("M", 15.9949), ("STY", 79.96633)], max_mods_per_peptide=3)
CFG3 = dict(semi=1)
METRIC = "peptides_indexed_per_s"
UNIT = "peptides/s"
NOMINAL_HBM_GBS = 8000.0  # north_star's ~8 TB/s; the measured copy bandwidth is the roofline denominator


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(kernel: str, algo_bytes: float):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of a kernel from the
    committed ncu --set full capture (profiles/traffic.json: bytes measured on this workload next
    to the algorithmic bytes of that launch), scaled to this run's launch; None without a capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)[kernel]
        return float(t["dram_bytes_per_launch"]) * algo_bytes / float(t["algo_bytes_per_launch"])
    except Exception:
        return None


def roofline_of(st_sum: dict, build_ms_total: float):
    """The dominant kernel of the build = the one with the largest summed device time among the
    kernels bracketed by CUDA events inside the library (dbi_stats): the onesweep scatter passes of
    the largest radix sort, and the mod-expansion kernel."""
    peak, peak_src = measured_peak_gbs()
    cands = []
    if st_sum["dom_launches"]:
        name = "rs_onesweep_kernel<u64,u64>" if st_sum["dom_kernel"] == 1 else "rs_onesweep_kernel<u64,u32>"
        cands.append((name, st_sum["dom_ms"], st_sum["dom_launches"], st_sum["dom_bytes_per_launch"]))
    if st_sum["exp_launches"]:
        cands.append(("grp_expand_tab_kernel", st_sum["exp_ms"], st_sum["exp_launches"], st_sum["exp_bytes_per_launch"]))
    if not cands:
        return None
    out = []
    for name, ms, n, bytes_per in cands:
        avg_ms = ms / n
        achieved = (bytes_per / 1e9) / (avg_ms / 1e3)
        out.append({"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "frac_of_nominal_8TBs": achieved / NOMINAL_HBM_GBS,
                    "peak_source": peak_src, "bytes_per_launch": int(bytes_per),
                    "launches": int(n), "avg_launch_ms": avg_ms, "share_of_build": ms / max(build_ms_total, 1e-9),
                    "traffic": measured_traffic(name, bytes_per)})
    out.sort(key=lambda r: -r["share_of_build"])
    roof = out[0]
    roof["other_kernels"] = out[1:]
    return roof


class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every 5 ms from a thread, started at the
    first warm-up step (same load as the timed steps) and stopped right after the timed region."""

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = False
        self._thr = None

    def start(self):
        import threading
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except (ValueError, IndexError):
                    idx = self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            return
        names = {
            getattr(pynvml, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(pynvml, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(pynvml, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(pynvml, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }

        def loop():
            while not self._stop:
                try:
                    self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                    try:
                        r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                    except Exception:
                        r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                except Exception:
                    pass
                time.sleep(0.005)

        self._thr = threading.Thread(target=loop, daemon=True)
        self._thr.start()

    def stop(self) -> dict:
        self._stop = True
        if self._thr is not None:
            self._thr.join(timeout=2)
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples),
               "how": "NVML, 5 ms period, warm-up + timed steps"}
        if self.samples:
            out["sm_mhz"] = float(np.median(self.samples))
        return out


def sample_index_masses(g, n_entries: int, chunks: int = 64, chunk: int = 2048) -> np.ndarray:
    if n_entries == 0:
        return np.zeros(0)
    out = []
    for i in range(chunks):
        b = (n_entries - chunk) * i // max(1, chunks - 1) if n_entries > chunk else 0
        c = min(chunk, n_entries - b)
        out.append(g.fetch(b, c, with_ids=False)["mass"])
    return np.concatenate(out)


DUMP_BYTES = 64_000_000  # --dump-outputs: every file together
DUMP_SEED = 20240603


def dump_outputs(out_dir: str, g, cnt, n_entries: int):
    """--dump-outputs: what the last timed step computed, read from the handle after the timed region.

    counts.npy         n_emitted, n_unique, n_entries of the index, n_hits of the query batch
    index_mass.npy     the masses at 64 x 2048 fixed positions of the index
    query.npy          a seeded sample of the batch's queries (ascending): the longest prefix of one fixed
                       permutation whose hits fit in DUMP_BYTES
    query_hits.npy     the number of hits of each sampled query
    hit_*.npy          every hit of the sampled queries, one row per hit (the run-grouped answer expanded):
                       query, mass, first_prot, first_off, len, modpat, flanks [n, 6], the peptide residues
                       (hit_seq, CSR hit_seq_off) and the protein ids (hit_prot_ids, CSR hit_prot_list_off)
    The hits of one query are in canonical order (query, mass, first_prot, first_off, len, modpat): ties in
    mass have no contractual order, so two correct builds may deliver them differently.  Integers are
    stored as float64 (exact), residue and flank bytes as float32."""
    from dbindex_b200.capi import HIT_FIELDS, DbiHitBuffers, _expand_csr, expand_hits
    raw, bufs = {}, DbiHitBuffers()
    for name, (dt, size) in HIT_FIELDS.items():
        raw[name] = np.empty(int(size(cnt)), dtype=dt)
        setattr(bufs, name, raw[name].ctypes.data)
    g.query_hits_read(bufs)
    st = g.stats()
    out = {"counts": np.array([st["n_emitted"], st["n_unique"], n_entries, cnt.n_hits], np.float64),
           "index_mass": sample_index_masses(g, n_entries)}

    ho, po, pho = (raw[k].astype(np.int64) for k in ("hit_off", "pep_off", "pep_hit_off"))
    nq = len(ho) - 1
    run_hits = np.diff(pho)
    # bytes one query adds to the dump: 8 x (query, mass, first_prot, first_off, len, modpat, seq_off,
    # prot_list_off) + 4 x 6 flanks per hit, 4 per residue, 8 per protein id, 16 in query / query_hits
    run_bytes = run_hits * (8 * 8 + 4 * 6 + 4 * np.diff(raw["seq_off"].astype(np.int64)) +
                            8 * np.diff(raw["prot_list_off"].astype(np.int64)))
    cum = np.concatenate(([0], np.cumsum(run_bytes)))
    q_bytes = cum[po[1:]] - cum[po[:-1]] + 16
    perm = np.random.default_rng(DUMP_SEED).permutation(nq)
    room = DUMP_BYTES - sum(a.nbytes for a in out.values()) - 2 * 8 - 4096  # CSR terminators, .npy headers
    k = int(np.searchsorted(np.cumsum(q_bytes[perm]), room, side="right"))
    sel = np.sort(perm[:k])

    # the run-grouped answer restricted to the sampled queries, then one record per hit
    _, runs = _expand_csr(po, np.arange(len(run_hits), dtype=np.int64), sel)
    sub = {"mass": raw["mass"][runs], "first_prot": raw["first_prot"][runs], "first_off": raw["first_off"][runs],
           "len": raw["len"][runs], "flanks": raw["flanks"].reshape(-1, 6)[runs].reshape(-1)}
    sub["pep_hit_off"], sub["modpat"] = _expand_csr(pho, raw["modpat"], runs)
    sub["seq_off"], sub["seq"] = _expand_csr(raw["seq_off"], raw["seq"], runs)
    sub["prot_list_off"], sub["prot_ids"] = _expand_csr(raw["prot_list_off"], raw["prot_ids"], runs)
    h = expand_hits(sub)
    n_q = np.diff(ho)[sel]
    query = np.repeat(sel, n_q)
    order = np.lexsort((h["modpat"], h["len"], h["first_off"], h["first_prot"],
                        np.ascontiguousarray(h["mass"]).view(np.uint64), query))
    seq_off, seq = _expand_csr(h["seq_off"], h["seq"], order)
    prot_off, prot_ids = _expand_csr(h["prot_list_off"], h["prot_ids"], order)
    out.update({"query": sel, "query_hits": n_q, "hit_query": query[order], "hit_mass": h["mass"][order],
                "hit_first_prot": h["first_prot"][order], "hit_first_off": h["first_off"][order],
                "hit_len": h["len"][order], "hit_modpat": h["modpat"][order],
                "hit_flanks": h["flanks"].reshape(-1, 6)[order], "hit_seq": seq, "hit_seq_off": seq_off,
                "hit_prot_ids": prot_ids, "hit_prot_list_off": prot_off})
    out = {name: a.astype(np.float32 if name in ("hit_flanks", "hit_seq") else np.float64) for name, a in out.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {"dir": out_dir, "queries": int(k), "hits": int(len(order)), "bytes": int(sum(a.nbytes for a in out.values()))}


class PinnedHits:
    """Caller-owned, page-locked receive buffers for dbi_query_hits_read, sized once for the (deterministic)
    batch and reused by every end-to-end step."""

    def __init__(self, counts):
        import torch
        from dbindex_b200.capi import HIT_FIELDS, DbiHitBuffers
        self.bufs = DbiHitBuffers()
        self.tensors = {}
        self.nbytes = 0
        for name, (dt, size) in HIT_FIELDS.items():
            n = int(size(counts)) * np.dtype(dt).itemsize
            t = torch.empty(max(n, 1), dtype=torch.uint8).pin_memory()
            self.tensors[name] = t
            setattr(self.bufs, name, t.data_ptr())
            self.nbytes += n

    def field(self, name, dtype):
        return self.tensors[name].numpy().view(dtype)


def cpu_baseline(cfg: dict, n_proteins: int, nq: int, threads: int, seed_cfg: int = 2):
    """The oracle (CPU restatement of the reference algorithm) on the workload: build + one query batch with
    every hit materialised (parseAddPeptideInfo).  Uses liboracle.so only -- not the product library.  The
    queries are drawn exactly like the GPU arm's (same chunks of the index, same seed): equal indexes give
    equal batches, so the two arms answer the same questions."""
    from dbindex_b200 import synth  # pure numpy
    from oracle import oracle_py
    res, off = synth.config_proteome(seed_cfg, n_proteins)
    params = oracle_py.default_params(**cfg)
    t0 = time.perf_counter()
    o = oracle_py.Oracle(params, threads=threads)
    o.add_proteins(res, off)
    rc = o.build()
    t1 = time.perf_counter()
    assert rc == 0
    n = o.counts()["n_entries"]
    chunks, chunk = 64, 2048  # sample_index_masses
    m = np.concatenate([o.entries((n - chunk) * i // (chunks - 1) if n > chunk else 0,
                                  min(chunk, n - ((n - chunk) * i // (chunks - 1) if n > chunk else 0)))["mass"]
                        for i in range(chunks)]) if n else np.zeros(0)
    _, _, lo, hi = synth.synth_queries(m, nq, 20240602)
    t2 = time.perf_counter()
    h = o.query_hits(lo, hi)
    t3 = time.perf_counter()
    hits = int(h["hit_off"][-1])
    o.close()
    return {"entries": n, "build_s": t1 - t0, "query_s": t3 - t2, "nq": nq, "hits": hits}


def fasta_ingest_rate(n_proteins: int = 20000):
    """Side measurement (host only, not part of `value` / `e2e`): the synthetic FASTA of the workload
    written to a temp file and parsed by the native ingest (dbi_fasta_*) with every host thread."""
    from dbindex_b200 import synth
    from dbindex_b200.capi import parse_fasta
    res, off = synth.config_proteome(2, n_proteins)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "workload.fasta")
        synth.write_fasta(path, res, off)
        size = os.path.getsize(path)
        parse_fasta(path, raw_deflines=True)  # page cache warm
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            (dbuf, doff), r2, o2 = parse_fasta(path, raw_deflines=True)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    assert len(doff) == n_proteins + 1 and np.array_equal(r2, res) and np.array_equal(o2, off)
    return {"file_mb": size / 1e6, "ms": 1e3 * best, "mb_per_s": size / 1e6 / best, "threads": os.cpu_count() or 1,
            "what": "dbi_fasta_open + dbi_fasta_counts + dbi_fasta_read into packed buffers, page cache warm, best of 3; "
                    "outside the timed step"}


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's CPU implementation of the path.  The Java reference cannot
    be built here (no JDK, un-vendored utilities-1.6-SNAPSHOT), so this is the oracle port with every
    host thread, on the SAME workload as the GPU arm (full size); rank 0 alone runs it."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_prot = args.proteins if args.ref_proteins <= 0 else args.ref_proteins
    times, entries, qtimes, hits = [], 0, [], 0
    for i in range(args.warmup + args.steps):
        r = cpu_baseline(CFG2, n_prot, args.queries, threads)
        if i >= args.warmup:
            times.append(r["build_s"] + r["query_s"])
            qtimes.append(r["query_s"])
        entries, hits = r["entries"], r["hits"]
    total = sum(times)
    value = entries * len(times) / total
    total_prot = args.proteins * max(1, world)  # the GPU arm indexes proteins_per_gpu x world proteins in ONE index
    same = n_prot == total_prot
    sample = (f"the whole workload ({n_prot} proteins, {entries} index entries) + {args.queries} queries "
              f"({hits} hits materialised) per step") if same else \
        (f"first {n_prot} of the {total_prot} proteins ({entries} index entries) + {args.queries} queries "
         f"({hits} hits materialised) per step")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "proteins_per_gpu": n_prot, "queries": args.queries,
                   "same_workload_as_gpu_arm": same},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample +
                         "; oracle/ (C++ restatement, OpenMP; the Java reference cannot be built here)"},
        "queries": {"value": args.queries * len(qtimes) / max(sum(qtimes), 1e-12), "unit": "queries/s",
                    "hits_per_batch": hits},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- one single-GPU configuration: timed build + query batch ------------------------------------------
def time_config(dbi, torch, stream, params, res, off, nq, steps, warmup, flush, with_hits=True, query_seed=20240602,
                da_fraction=0.0):
    """Build + one query batch per step on device-resident residues.  Returns (result dict, handle, queries)."""
    from dbindex_b200 import synth
    g = dbi.GpuIndex(params)
    g.set_stream(stream.cuda_stream)
    g.add_proteins(res, off)
    g.upload()
    g.build()
    n_entries = g.stats()["n_entries"]
    masses = sample_index_masses(g, n_entries)
    qmass, qtol, lo, hi = synth.synth_queries(masses, nq, query_seed, da_fraction=da_fraction)
    d_lo, d_hi = torch.from_numpy(lo).cuda(), torch.from_numpy(hi).cuda()
    d_b = torch.empty(nq, dtype=torch.int64, device="cuda")
    d_c = torch.empty(nq, dtype=torch.int64, device="cuda")
    build_ms, query_ms = [], []
    probes = {"dom_ms": 0.0, "dom_launches": 0, "dom_bytes_per_launch": 0, "dom_kernel": 0, "exp_ms": 0.0,
              "exp_launches": 0, "exp_bytes_per_launch": 0}
    stage_ms = {}
    cnt = None
    launches0 = 0
    for i in range(warmup + steps):
        if i == warmup:
            torch.cuda.synchronize()
            launches0 = g.kernel_launches()
        g.reset_index()
        flush.zero_()  # flush L2 between iterations
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(stream)
        g.build()
        e1.record(stream)
        if with_hits:
            cnt = g.query_hits_device(d_lo.data_ptr(), d_hi.data_ptr(), nq)
        else:
            g.query_device(d_lo.data_ptr(), d_hi.data_ptr(), nq, d_b.data_ptr(), d_c.data_ptr())
        e2.record(stream)
        torch.cuda.synchronize()
        if i >= warmup:
            build_ms.append(e0.elapsed_time(e1))
            query_ms.append(e1.elapsed_time(e2))
            st = g.stats()
            for k in ("dom_ms", "dom_launches", "exp_ms", "exp_launches"):
                probes[k] += st[k]
            for k in ("dom_bytes_per_launch", "dom_kernel", "exp_bytes_per_launch"):
                probes[k] = st[k]
            for k, v in st["stage_ms"].items():
                stage_ms[k] = stage_ms.get(k, 0.0) + v
    torch.cuda.synchronize()
    n_launch = g.kernel_launches() - launches0
    st = g.stats()
    hits = int(cnt.n_hits) if with_hits else int(d_c.sum().item())
    tot = float(sum(build_ms) + sum(query_ms))
    r = {"value": n_entries * steps / (tot / 1e3), "unit": UNIT, "steps": steps, "ms_per_step": tot / steps,
         "build_ms": sum(build_ms) / steps, "query_ms": sum(query_ms) / steps,
         "queries_per_s": nq * steps / (sum(query_ms) / 1e3), "hits_per_batch": hits,
         "proteins": len(off) - 1, "residues": int(res.nbytes), "emitted": st["n_emitted"], "unique": st["n_unique"],
         "entries": n_entries, "queries": nq, "stage_ms": {k: v / steps for k, v in stage_ms.items() if v > 0},
         "roofline": roofline_of(probes, sum(build_ms)), "gpu_launches": int(n_launch),
         "sort_bits": [st["sort_bits_base"], st["sort_bits_var"]]}
    return r, g, (lo, hi, d_lo, d_hi, cnt)


def index_properties(g, n_entries: int, lo, hi, rng) -> dict:
    """Size-independent parity properties on the built index: sampled chunks sorted by exact mass; the
    (begin, count) of sampled queries are tight -- every hit inside [lo, hi], both neighbours outside."""
    checked = failed = 0
    chunk = 1 << 18
    for s in sorted(set([0, max(0, n_entries - chunk)] + [int(x) for x in rng.integers(0, max(1, n_entries - chunk), size=6)])):
        m = g.fetch(s, min(chunk, n_entries - s), with_ids=False)["mass"]
        checked += 1
        failed += 0 if np.all(np.diff(m) >= 0) else 1
    sel = rng.choice(len(lo), size=min(256, len(lo)), replace=False)
    b, c = g.query(lo[sel], hi[sel])
    for k in range(len(sel)):
        b0, c0 = int(b[k]), int(c[k])
        a = max(0, b0 - 1)
        m = g.fetch(a, min(n_entries - a, c0 + 2), with_ids=False)["mass"] if n_entries else np.zeros(0)
        inside = m[(b0 - a):(b0 - a) + c0]
        ok = np.all((inside >= lo[sel[k]]) & (inside <= hi[sel[k]]))
        if b0 > 0:
            ok = ok and m[0] < lo[sel[k]]
        if b0 + c0 < n_entries:
            ok = ok and m[(b0 - a) + c0] > hi[sel[k]]
        checked += 1
        failed += 0 if ok else 1
    return {"checked": int(checked), "failed": int(failed),
            "what": "sampled index chunks sorted by exact mass; sampled query ranges tight (hits inside, neighbours outside)"}


def query_sweep(torch, stream, g, n_entries, nq, masses):
    """cfg5-style sweep: nq precursor queries (half 10 ppm, half +-3 Da) against the built index, bounds
    only (the +-3 Da windows hold ~10^5 hits each).  Roofline per SURVEY 8(d): 32 B in/out + 2 x
    ceil(log2 V) dependent 32-byte sectors per query."""
    from dbindex_b200 import synth
    peak, peak_src = measured_peak_gbs()
    _, _, lo, hi = synth.synth_queries(masses, nq, 20240605, da_fraction=0.5)
    out = {}
    for tag, order in (("as_generated", None), ("sorted_by_mass", np.argsort(lo, kind="stable"))):
        l2, h2 = (lo, hi) if order is None else (lo[order], hi[order])
        d_lo, d_hi = torch.from_numpy(l2).cuda(), torch.from_numpy(h2).cuda()
        d_b = torch.empty(nq, dtype=torch.int64, device="cuda")
        d_c = torch.empty(nq, dtype=torch.int64, device="cuda")
        ms = []
        for i in range(4):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            g.query_device(d_lo.data_ptr(), d_hi.data_ptr(), nq, d_b.data_ptr(), d_c.data_ptr())
            b.record(stream)
            torch.cuda.synchronize()
            if i:
                ms.append(a.elapsed_time(b))
        t = float(np.mean(ms))
        depth = int(np.ceil(np.log2(max(2, n_entries))))
        algo = nq * (32 + 2 * depth * 32)
        out[tag] = {"ms": t, "queries_per_s": nq / (t / 1e3), "hits": int(d_c.sum().item()),
                    "roofline": {"bound": "hbm", "kernel": "query_kernel", "achieved": algo / 1e9 / (t / 1e3),
                                 "peak": peak, "unit": "GB/s", "frac": algo / 1e9 / (t / 1e3) / peak,
                                 "peak_source": peak_src, "bytes_per_launch": int(algo),
                                 "note": "dependent sector reads: latency-bound by construction, the fraction is reported "
                                         "for completeness"}}
    out["queries"] = nq
    out["what"] = "500k @ 10 ppm + 500k @ +-3 Da, masses half indexed (+-5 ppm jitter) / half uniform decoys; bounds only"
    return out, lo, hi


def run_ours(args, rank: int, local_rank: int, world: int):
    import torch
    import dbindex_b200 as dbi
    from dbindex_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                         "(use --impl reference for the CPU baseline)")
    if world > 1:
        return run_sharded(args, rank, local_rank, world)
    torch.cuda.set_device(local_rank)
    dbi.load_library()
    # a non-default stream: the legacy default stream serialises against every other stream
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    res, off = synth.config_proteome(2, args.proteins)
    params = dbi.default_params(**CFG2)
    params.device = local_rank
    params.profile = 1
    clocks = ClockSampler(local_rank)
    clocks.start()
    head, g, (lo, hi, d_lo, d_hi, cnt) = time_config(dbi, torch, stream, params, res, off, args.queries, args.steps,
                                                     args.warmup, flush)
    clk = clocks.stop()
    n_entries = head["entries"]
    dumped = dump_outputs(args.dump_outputs, g, cnt, n_entries) if args.dump_outputs else None
    parity = index_properties(g, n_entries, lo, hi, np.random.default_rng(1))

    # ---- e2e: the user-facing call sequence with HOST buffers, every copy inside the timed region ----
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()  # noqa: E731
    h_res, h_off, h_lo, h_hi = pin(res), pin(off.view(np.int64)), pin(lo), pin(hi)
    sink = PinnedHits(cnt)
    e2e_ms = []
    e2e_steps = max(1, min(args.steps, 5))
    E2E_WARM = 2  # fresh handles: the first ones fill the allocator caches
    for i in range(E2E_WARM + e2e_steps):
        flush.zero_()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        p2 = params.copy()
        p2.profile = 0
        g2 = dbi.GpuIndex(p2)
        g2.set_stream(stream.cuda_stream)
        g2.add_proteins(h_res.numpy(), h_off.numpy().view(np.uint64))
        g2.build()
        c2 = g2.query_hits_begin(h_lo.numpy(), h_hi.numpy())
        g2.query_hits_read(sink.bufs)
        b.record(stream)
        torch.cuda.synchronize()
        assert g2.stats()["n_entries"] == n_entries and c2.n_hits == cnt.n_hits
        assert int(sink.field("hit_off", np.uint64)[args.queries]) == cnt.n_hits
        g2.close()
        if i >= E2E_WARM:
            e2e_ms.append(a.elapsed_time(b))
    e2e_step_ms = float(sum(e2e_ms)) / len(e2e_ms)
    h2d = int(res.nbytes + off.nbytes + lo.nbytes + hi.nbytes + 4352 + 8)
    d2h = int(sink.nbytes + 7 * 8 + 4 * 4)

    base = None
    if not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        r = cpu_baseline(CFG2, args.proteins, args.queries, threads)
        base = {"value": r["entries"] / (r["build_s"] + r["query_s"]), "unit": UNIT, "cores": threads, "kind": "port",
                "sample": f"the whole workload once: {args.proteins} proteins ({r['entries']} index entries) + "
                          f"{args.queries} queries ({r['hits']} hits materialised), oracle/ (C++ restatement; the Java "
                          f"reference cannot be built here), build {r['build_s']:.2f} s, queries {r['query_s']:.3f} s",
                "queries_per_s": args.queries / max(r["query_s"], 1e-12)}
        assert r["entries"] == n_entries and r["hits"] == cnt.n_hits, "oracle and GPU disagree on the workload"
        parity["oracle_counts_equal"] = True
    g.close()

    # ---- the other single-GPU configurations (BASELINE.json configs[0], [2], [4]) ----
    configs = {}
    if not args.no_extra:
        try:
            configs = extra_configs(args, dbi, torch, stream, flush, local_rank)
        except Exception as e:  # never lose the headline to a side configuration
            configs = {"error": repr(e)[:300]}

    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "proteins_per_gpu": args.proteins, "residues_per_gpu": int(res.nbytes),
                   "emitted": head["emitted"], "unique": head["unique"], "entries_per_gpu": n_entries,
                   "queries": args.queries, "l2": "flushed between iterations (256 MiB write)", "parallelism": "1 GPU"},
        "queries": {"value": head["queries_per_s"], "unit": "queries/s", "hits_per_batch": head["hits_per_batch"],
                    "runs_per_batch": int(cnt.n_peps), "ms_per_batch": head["query_ms"],
                    "includes": "bounds + materialisation of every hit in HBM (grouped in runs of one peptide and mass)"},
        "build_ms": head["build_ms"], "stage_ms": head["stage_ms"], "sort_bits": head["sort_bits"],
        "roofline": head["roofline"], "cpu_baseline": base, "parity": parity,
        "e2e": {"value": n_entries / (e2e_step_ms / 1e3), "unit": UNIT, "ms_per_step": e2e_step_ms,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "hits_per_step": int(cnt.n_hits),
                "what": "dbi_create + dbi_add_proteins(pinned host) + dbi_build + dbi_query_hits(host bounds) + "
                        "dbi_query_hits_read(all 13 hit arrays into pinned host memory: peptide-level fields once per run of "
                        "same-peptide same-mass hits, mod pattern per hit) + dbi_destroy",
                "runs_per_step": int(cnt.n_peps)},
        "gpu_launches": head["gpu_launches"], "clocks": clk, "configs": configs,
    }
    if dumped:
        line["outputs"] = dumped
    try:
        line["fasta_ingest"] = fasta_ingest_rate(args.proteins)
    except Exception as e:  # a side measurement must never cost the bench line
        line["fasta_ingest"] = {"error": str(e)[:200]}
    print(json.dumps(line), flush=True)


def extra_configs(args, dbi, torch, stream, flush, local_rank):
    """cfg1, cfg3 (full size) and the cfg5-style sweep, each with its own roofline and parity properties."""
    from dbindex_b200 import synth
    out = {}
    # cfg1: same FASTA, no mods
    res, off = synth.config_proteome(1, args.proteins)
    p1 = dbi.default_params(**CFG1)
    p1.device, p1.profile = local_rank, 1
    r, g, (lo, hi, _, _, _) = time_config(dbi, torch, stream, p1, res, off, args.queries, 5, 3, flush)
    r["parity"] = index_properties(g, r["entries"], lo, hi, np.random.default_rng(2))
    r["workload"] = "cfg1: 20000 proteins, trypsin, 2 missed cleavages, 600-6000 Da, no mods, build + 10000 queries @ 10 ppm (hits materialised)"
    g.close()
    out["cfg1"] = r
    del res, off
    # cfg3: semi-tryptic, 200 000 proteins (full size): the largest single-GPU configuration
    res, off = synth.config_proteome(3, args.cfg3_proteins)
    p3 = dbi.default_params(**CFG3)
    p3.device, p3.profile = local_rank, 1
    r, g, (lo, hi, _, _, _) = time_config(dbi, torch, stream, p3, res, off, args.queries, 2, 1, flush)
    r["parity"] = index_properties(g, r["entries"], lo, hi, np.random.default_rng(3))
    r["workload"] = (f"cfg3: {args.cfg3_proteins} proteins (~{res.nbytes / 1e6:.0f}M residues), semi-tryptic, 2 missed cleavages, "
                     "600-6000 Da, no mods, build + 10000 queries @ 10 ppm (hits materialised)")
    out["cfg3"] = r
    # cfg5-style sweep against cfg3's index (the largest one a single GPU builds here)
    masses = sample_index_masses(g, r["entries"])
    sweep, slo, shi = query_sweep(torch, stream, g, r["entries"], args.sweep_queries, masses)
    sweep["parity"] = index_properties(g, r["entries"], slo, shi, np.random.default_rng(5))
    sweep["index"] = f"cfg3 ({r['entries']} entries)"
    out["cfg5_sweep"] = sweep
    g.close()
    dbi.load_library().dbi_release_cached_memory(local_rank)
    return out


# ---- N > 1 ---------------------------------------------------------------------------------------------
def sharded_parity(torch, dist, dbi, g, info, res, off, params, rank, world, n_sample=24, per_protein=16):
    """In-run check of the sharded index against the oracle (outside the timed region): every rank derives,
    with the oracle alone, the entries of the same sampled proteins, and each of them must be held by
    EXACTLY ONE rank -- zero-tolerance query, same peptide string, same mod pattern, the protein in the
    list; plus local sortedness and slices cut at the splitter masses."""
    from dbindex_b200.multigpu import owned_mask
    from oracle.oracle_py import Oracle
    srng = np.random.default_rng(5)
    P = len(off) - 1
    want_mass, want_seq, want_pat, want_pid = [], [], [], []
    for pid in np.sort(srng.choice(P, size=min(n_sample, P), replace=False)):
        r0, r1 = int(off[pid]), int(off[pid + 1])
        o = Oracle(params, threads=1)
        o.add_proteins(res[r0:r1], np.array([0, r1 - r0], dtype=np.uint64))
        assert o.build() == 0
        e = o.entries()
        o.close()
        if not len(e["mass"]):
            continue
        for i in srng.choice(len(e["mass"]), size=min(per_protein, len(e["mass"])), replace=False):
            want_mass.append(float(e["mass"][i]))
            want_seq.append(res[r0 + int(e["first_off"][i]):r0 + int(e["first_off"][i]) + int(e["len"][i])].tobytes())
            want_pat.append(int(e["modpat"][i]))
            want_pid.append(int(pid))
    m = np.array(want_mass)
    h = g.query_hits(m, m, fields=("hit_off", "modpat", "seq_off", "seq", "prot_list_off", "prot_ids"))
    ho, so, po = (h[k].astype(np.int64) for k in ("hit_off", "seq_off", "prot_list_off"))
    found = np.zeros(len(m), np.int64)
    for q in range(len(m)):
        for i in range(ho[q], ho[q + 1]):
            if int(h["modpat"][i]) == want_pat[q] and h["seq"][so[i]:so[i + 1]].tobytes() == want_seq[q] and \
                    want_pid[q] in h["prot_ids"][po[i]:po[i + 1]]:
                found[q] += 1
    tot = torch.from_numpy(found).cuda()
    dist.all_reduce(tot)
    failed = int((tot != 1).sum().item())
    # local order + cuts
    n = g.stats()["n_entries"]
    sm = info["split_mass"]
    chunk = 1 << 18
    rng = np.random.default_rng(11 + rank)
    bad = 0
    for s in sorted(set([0, max(0, n - chunk)] + [int(x) for x in rng.integers(0, max(1, n - chunk), size=4)])):
        mm = g.fetch(s, min(chunk, n - s), with_ids=False)["mass"]
        bad += 0 if np.all(np.diff(mm) >= 0) else 1
        bad += 0 if np.all(owned_mask(mm, sm, rank, world)) else 1  # every entry lies in a slice this rank holds
    t2 = torch.tensor([bad], device="cuda", dtype=torch.int64)
    dist.all_reduce(t2)
    return {"checked": int(len(m)) + 6 * world, "failed": failed + int(t2.item()),
            "what": f"{len(m)} oracle-derived entries of {n_sample} sampled proteins each held by exactly one rank (string, mod "
                    "pattern, protein list); every rank's entries sorted and inside the slices it holds"}


def run_sharded(args, rank: int, local_rank: int, world: int):
    """N > 1: ONE index over world x 20000 proteins (weak scaling): the FASTA is sharded over the ranks, the
    residues are replicated over NVLink, the records and the variant groups travel inside the two fused
    multisplit / peer-memory scatter kernels, queries are routed to the owning GPU."""
    import torch
    import torch.distributed as dist
    import dbindex_b200 as dbi
    from dbindex_b200 import synth
    from dbindex_b200.multigpu import GpuShardEngine, build_sharded, route_queries, shard_proteins, shard_sizes

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    lib = dbi.load_library()
    res, off = synth.config_proteome(2, args.proteins * world)  # generated on every rank; each keeps only its shard
    sres, soff, _ = shard_proteins(res, off, rank, world)
    sizes = shard_sizes(off, world)  # the host that cut the FASTA knows every shard's size: one collective less
    params = dbi.default_params(**CFG2)
    params.device = local_rank
    params.profile = 1
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    g = dbi.GpuIndex(params)
    g.set_stream(stream.cuda_stream)
    g.add_proteins(sres, soff)
    g.upload()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    nq = args.queries  # ONE batch for the whole index: hits per query grow with the index, so per-GPU work stays fixed
    info = build_sharded(GpuShardEngine(g, dev), sizes)  # also warms NCCL and the window mappings up
    n_mine = g.stats()["n_entries"]
    masses = sample_index_masses(g, n_mine)
    # the query masses follow the indexed mass density, exactly like the N = 1 batch (which samples the index
    # at evenly spaced ENTRY positions): every rank contributes samples of its slice in proportion to the
    # entries it holds
    counts = [None] * world
    dist.all_gather_object(counts, int(n_mine))
    k = max(1, int(round(16384 * n_mine / max(1, sum(counts)))))
    gathered = [None] * world
    dist.all_gather_object(gathered, masses[np.linspace(0, len(masses) - 1, k).astype(np.int64)].tolist() if len(masses) else [])
    allm = np.sort(np.concatenate([np.asarray(x) for x in gathered]))
    _, _, lo, hi = synth.synth_queries(allm, nq, 20240602)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    step_ms, query_ms, a2a_ms, a2a_bytes = [], [], 0.0, 0
    probes = {"dom_ms": 0.0, "dom_launches": 0, "dom_bytes_per_launch": 0, "dom_kernel": 0, "exp_ms": 0.0,
              "exp_launches": 0, "exp_bytes_per_launch": 0}
    clocks = ClockSampler(local_rank)
    launches0 = 0
    hits = 0
    clocks.start()
    for i in range(args.warmup + args.steps):
        if i == args.warmup:
            barrier()
            launches0 = lib.dbi_kernel_launches()
        g.reset_index()
        flush.zero_()
        barrier()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record(stream)
        info = build_sharded(GpuShardEngine(g, dev), sizes)
        e1.record(stream)
        sel = route_queries(lo, hi, info["split_mass"], rank, world)
        d_lo = torch.from_numpy(lo[sel]).cuda()
        d_hi = torch.from_numpy(hi[sel]).cuda()
        stream.synchronize()
        cnt = g.query_hits_device(d_lo.data_ptr(), d_hi.data_ptr(), len(sel))
        e2.record(stream)
        torch.cuda.synchronize()
        if i >= args.warmup:
            step_ms.append(e0.elapsed_time(e2))
            query_ms.append(e1.elapsed_time(e2))
            a2a_ms += info["a2a_ms"]
            a2a_bytes += info["a2a_bytes"]
            st = g.stats()
            for k in ("dom_ms", "dom_launches", "exp_ms", "exp_launches"):
                probes[k] += st[k]
            for k in ("dom_bytes_per_launch", "dom_kernel", "exp_bytes_per_launch"):
                probes[k] = st[k]
            hits = int(cnt.n_hits)
    barrier()
    n_launch = lib.dbi_kernel_launches() - launches0
    clk = clocks.stop()
    st = g.stats()
    n_entries = st["n_entries"]
    parity = sharded_parity(torch, dist, dbi, g, info, res, off, params, rank, world)

    # ---- e2e: fresh handle, host buffers, copies and routing inside the timed region ----
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()  # noqa: E731
    h_res, h_off = pin(sres), pin(soff.view(np.int64))
    sel0 = route_queries(lo, hi, info["split_mass"], rank, world)
    sink = PinnedHits(g.query_hits_begin(lo[sel0], hi[sel0]))
    e2e_ms = []
    E2E_WARM = 3  # fresh handles: the first ones fill the allocator and window caches on every rank
    for i in range(E2E_WARM + max(1, min(args.steps, 5))):
        flush.zero_()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        t0 = time.perf_counter()
        p2 = params.copy()
        p2.profile = 0
        g2 = dbi.GpuIndex(p2)
        g2.set_stream(stream.cuda_stream)
        g2.add_proteins(h_res.numpy(), h_off.numpy().view(np.uint64))
        t1 = time.perf_counter()
        inf2 = build_sharded(GpuShardEngine(g2, dev), sizes)
        t2 = time.perf_counter()
        sel = route_queries(lo, hi, inf2["split_mass"], rank, world)
        c2 = g2.query_hits_begin(lo[sel], hi[sel])
        t3 = time.perf_counter()
        g2.query_hits_read(sink.bufs)
        b.record(stream)
        torch.cuda.synchronize()
        t4 = time.perf_counter()
        e2e_host = {"create+add": 1e3 * (t1 - t0), "build": 1e3 * (t2 - t1), "route+query": 1e3 * (t3 - t2),
                    "read": 1e3 * (t4 - t3), **{"build." + k: v for k, v in inf2["t"].items()}}
        assert c2.n_hits == hits
        barrier()  # nobody releases its windows while another rank may still read them
        g2.close()
        if i >= E2E_WARM:
            e2e_ms.append(a.elapsed_time(b))

    e2e_all = [None] * world
    dist.all_gather_object(e2e_all, {"steps_ms": [round(float(x), 3) for x in e2e_ms],
                                     "last_step_host_ms": {k: round(v, 3) for k, v in e2e_host.items()
                                                           if not k.startswith("build.")}})
    per_rank = [None] * world
    dist.all_gather_object(per_rank, {"entries": int(n_entries), "records": int(info.get("recv0", 0)),
                                      "groups": int(info.get("recv1", 0)), "unique": int(st["n_unique"]),
                                      "hits": int(hits), "query_ms": round(sum(query_ms) / len(query_ms), 3),
                                      **{k: round(v, 3) for k, v in st["stage_ms"].items() if v > 0}})
    t = torch.tensor([float(sum(step_ms)), float(sum(query_ms)), float(sum(e2e_ms)) / len(e2e_ms), a2a_ms],
                     device="cuda", dtype=torch.float64)
    u = torch.tensor([float(n_entries), float(n_launch), float(hits), float(a2a_bytes), float(sink.nbytes),
                      float(sres.nbytes + soff.nbytes)], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(u, op=dist.ReduceOp.SUM)
    tot_ms, q_ms, e2e_step_ms, a2a_max_ms = t.tolist()
    entries_all, launches_all, hits_all, a2a_all, d2h_all, h2d_all = u.tolist()
    K = args.steps
    if rank == 0:
        roof = roofline_of(probes, sum(step_ms))
        if roof:
            roof["rank"] = 0
        line = {
            "metric": METRIC, "value": entries_all * K / (tot_ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": args.warmup, "ms_per_step": tot_ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD.replace("20000 proteins", f"{args.proteins} proteins per GPU"),
                       "proteins_total": args.proteins * world, "residues_total": int(res.nbytes),
                       "entries_total": int(entries_all), "unique_total": info["n_unique"],
                       "queries": nq, "l2": "flushed between iterations (256 MiB write)",
                       "parallelism": f"{world} GPUs: FASTA sharded by protein (each rank digests its shard while the "
                                      "others arrive over NVLink), fused multisplit + peer-memory scatter by mass slice "
                                      f"(records, then variant groups with their site masks; {info.get('n_slices', world)} "
                                      "folded slices, one light + one heavy per rank), routed queries"},
            "queries": {"value": nq * K / (q_ms / 1e3), "unit": "queries/s", "hits_per_batch": int(hits_all),
                        "ms_per_batch": q_ms / K,
                        "includes": "host routing + H2D of the routed bounds + materialisation of every hit in HBM"},
            "all_to_all": {"bytes_per_step_all_ranks": a2a_all / K, "ms_per_step_max_rank": a2a_max_ms / K,
                           "bus_gbs_per_gpu": (a2a_all / K / world / 1e9) / max(a2a_max_ms / K / 1e3, 1e-12),
                           "nvlink_ref_gbs": 770.0,
                           "what": "bytes leaving a GPU inside the two scatter kernels / kernel time (partition included)"},
            "roofline": roof,
            "cpu_baseline": None,
            "parity": parity,
            "e2e": {"value": entries_all / (e2e_step_ms / 1e3), "unit": UNIT, "ms_per_step": e2e_step_ms,
                    "h2d_bytes_per_step": int(h2d_all + 4360 * world + 16 * nq),
                    "d2h_bytes_per_step": int(d2h_all + 2 * (2 * 2 * 4096 * 8 + 400 * world) * world),
                    "what": "per rank: dbi_create + dbi_add_proteins(own FASTA shard, pinned host) + sharded build + routed "
                            "dbi_query_hits(host bounds) + dbi_query_hits_read(all hit arrays, pinned host) + dbi_destroy"},
            "gpu_launches": int(launches_all),
            "clocks": clk,
            "host_stage_ms_rank0_last_step": {k: round(v, 3) for k, v in info["t"].items()},
            "e2e_host_ms_rank0_last_step": {k: round(v, 3) for k, v in e2e_host.items()},
            "e2e_per_rank": e2e_all,
            "device_stage_ms_rank0_last_step": {k: round(v, 3) for k, v in st["stage_ms"].items() if v > 0},
            "per_rank_last_step": {k: [r.get(k, 0) for r in per_rank] for k in per_rank[0]},
            "split_mass": [float(x) for x in info["split_mass"]],
            "step_ms_rank0": [round(float(x), 3) for x in step_ms],
        }
        print(json.dumps(line), flush=True)
    barrier()
    g.close()
    dist.destroy_process_group()


def main():
    import gc
    gc.disable()  # no collector pauses inside timed regions (the steps allocate no cycles worth collecting)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--proteins", type=int, default=20000, help="proteins per GPU (BASELINE config: 20000)")
    ap.add_argument("--queries", type=int, default=10000)
    ap.add_argument("--ref-proteins", type=int, default=0,
                    help="--impl reference: proteins per step (0 = the whole workload, like the GPU arm)")
    ap.add_argument("--cfg3-proteins", type=int, default=200000)
    ap.add_argument("--sweep-queries", type=int, default=1000000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the cfg1 / cfg3 / cfg5 sub-results")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs writes the hits of the single-GPU path (--impl ours, one process)")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
