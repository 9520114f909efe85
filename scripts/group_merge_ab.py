"""A/B of the single-GPU group path: K6g's sorted lists + the one-pass K7m merge (default) against the K7 radix sort
of peptide-major group records (DBI_GROUP_RADIX=1), on the cfg2 build at full size, in one process.

The two paths alternate build by build on one handle, L2 flushed (256 MiB write) before every build.  Reports the
median and spread (min, max) of the device stage times sort_var, mod_count, mod_emit, expand_var and of the whole
build, and checks in the same run that both paths give the same index (every entry's mass bits, first occurrence,
length and mod pattern, compared chunk by chunk).  Writes <out>/group_merge_ab.json.

    python scripts/group_merge_ab.py --out DIR [--proteins 20000] [--rounds 7]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from lookup_bench import CFG2, gpu_identity  # noqa: E402

STAGES = ("sort_var", "mod_count", "mod_emit", "expand_var")
PATHS = ("merge", "radix")


def set_path(path):
    if path == "radix":
        os.environ["DBI_GROUP_RADIX"] = "1"
    else:
        os.environ.pop("DBI_GROUP_RADIX", None)


def index_digest(g, n, chunk=8_000_000):
    """Per-chunk SHA-1 of (mass bits, first_prot, first_off, len, modpat): equal digests = equal indexes."""
    import hashlib
    out = []
    for s in range(0, n, chunk):
        f = g.fetch(s, min(chunk, n - s), with_ids=False)
        h = hashlib.sha1()
        for k in ("mass", "first_prot", "first_off", "len", "modpat"):
            h.update(np.ascontiguousarray(f[k]).tobytes())
        out.append(h.hexdigest())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--proteins", type=int, default=20000)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch

    import dbindex_b200 as dbi
    from dbindex_b200 import synth

    if not torch.cuda.is_available():
        raise SystemExit("group_merge_ab.py: no CUDA device")
    dbi.load_library()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    res, off = synth.config_proteome(2, args.proteins)
    p = dbi.default_params(**CFG2)
    p.profile = 1
    g = dbi.GpuIndex(p)
    g.set_stream(stream.cuda_stream)
    g.add_proteins(res, off)
    g.upload()
    rec = {k: {"build_ms": [], **{s: [] for s in STAGES}} for k in PATHS}
    digests, stats = {}, {}
    for i in range(args.warmup + args.rounds):
        for path in (PATHS if i % 2 == 0 else PATHS[::-1]):
            set_path(path)
            g.reset_index()
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            g.build()
            b.record(stream)
            torch.cuda.synchronize()
            st = g.stats()
            if i < args.warmup:
                if path not in digests:
                    digests[path] = index_digest(g, st["n_entries"])
                    stats[path] = {k: st[k] for k in ("n_entries", "n_unique", "sort_bits_var", "dom_kernel")}
                continue
            rec[path]["build_ms"].append(a.elapsed_time(b))
            for s in STAGES:
                rec[path][s].append(st["stage_ms"][s])
    set_path("merge")
    g.close()

    def summ(x):
        x = np.asarray(x, dtype=np.float64)
        return {"median": round(float(np.median(x)), 4), "min": round(float(x.min()), 4), "max": round(float(x.max()), 4)}

    out = {
        "workload": f"cfg2 build, {args.proteins} proteins, {stats['merge']['n_entries']} entries; "
                    f"{args.rounds} rounds per path after {args.warmup} warm-up rounds, A B / B A alternating, "
                    "L2 flushed before every build",
        "device": gpu_identity(),
        "equal_index": digests["merge"] == digests["radix"],
        "stats": stats,
        **{path: {k: summ(v) for k, v in rec[path].items()} for path in PATHS},
        "raw": rec,
    }
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "group_merge_ab.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("equal_index", "stats", "merge", "radix", "device")}, indent=1))
    if not out["equal_index"]:
        raise SystemExit("the merge and radix paths built different indexes")


if __name__ == "__main__":
    main()
