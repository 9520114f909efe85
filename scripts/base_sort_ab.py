"""A/B of the base sort against another tree of this project (e.g. a checkout of the parent commit).

Two parts, in one call:
  identity  both trees build cfg1 and cfg2 at full size, cfg3 on 20 000 proteins, a proteome with long runs
            of repeated entries, and that proteome again under DBI_HASH_BITS=44; every index is written with
            dbi_save and the files must be equal byte for byte (the base order is a total order, so nothing
            is canonicalised).
  bench     bench.py --gpus 1 of the two trees alternated A B A B ..., the card's name, power limit and
            clocks read in the same call; then scripts/unindexed_bench.py part (a) of each tree.
Writes <out>/base_sort_ab.json (+ the raw bench lines).

    python scripts/base_sort_ab.py --other DIR --out DIR [--rounds 3] [--steps 10] [--warmup 3]
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CASES = ("cfg1", "cfg2", "cfg3_20k", "long_runs", "long_runs_hash44")


def long_run_proteome():
    """120 synthetic proteins, one of them repeated 3000 times, one 300 times, random ones 40 times and a
    short peptide-like entry 70 times, interleaved (the proteome of tests/test_base_sort.py)."""
    import numpy as np
    from dbindex_b200 import synth
    res, off = synth.synth_proteome(120, 4242, median_len=300)
    base = [res[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(len(off) - 1)]
    seqs = list(base)
    rng = np.random.default_rng(7)
    for i in range(3000):
        seqs.append(base[3])
        if i < 300:
            seqs.append(base[10])
        if i < 40:
            seqs.append(base[int(rng.integers(20, 120))])
        if i < 70:
            seqs.append("MAGGLLKPEPTIDEKRDESK")
    r = np.frombuffer("".join(seqs).encode("latin-1"), dtype=np.uint8)
    o = np.zeros(len(seqs) + 1, dtype=np.uint64)
    np.cumsum([len(s) for s in seqs], out=o[1:])
    return r, o


def save_cases(tree, out_dir):
    """Child process: build every case with the package of `tree` and dbi_save it under out_dir."""
    sys.path.insert(0, tree)
    import dbindex_b200 as dbi
    from dbindex_b200 import synth
    sys.path.insert(0, ROOT)
    from bench import CFG1, CFG2, CFG3
    os.makedirs(out_dir, exist_ok=True)
    info = {}
    for case in CASES:
        if case == "long_runs_hash44":
            os.environ["DBI_HASH_BITS"] = "44"
        else:
            os.environ.pop("DBI_HASH_BITS", None)
        cfg = {"cfg1": CFG1, "cfg2": CFG2, "cfg3_20k": CFG3}.get(case, {})
        if case.startswith("cfg"):
            res, off = synth.config_proteome(int(case[3]), 20000)
        else:
            res, off = long_run_proteome()
        with dbi.GpuIndex(dbi.default_params(**cfg)) as g:
            g.add_proteins(res, off)
            g.build()
            g.save(os.path.join(out_dir, case + ".dbi"))
            st = g.stats()
            info[case] = {k: st[k] for k in ("n_emitted", "n_unique", "n_entries", "n_hash_retries",
                                             "sort_bits_base", "device_bytes")}
    print(json.dumps(info))


def run(cmd, cwd, env=None):
    p = subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, text=True)
    if p.returncode:
        sys.stderr.write(p.stdout[-4000:] + p.stderr[-4000:])
        raise SystemExit(f"{cmd} in {cwd} failed ({p.returncode})")
    return p.stdout


def last_json(text):
    return json.loads([ln for ln in text.splitlines() if ln.startswith("{")][-1])


def pick(line):
    c = line.get("configs", {})
    return {"ms_per_step": line.get("ms_per_step"), "build_ms": line.get("build_ms"),
            "sort_base": line.get("stage_ms", {}).get("sort_base"), "dedup": line.get("stage_ms", {}).get("dedup"),
            **{name: {"ms_per_step": c.get(name, {}).get("ms_per_step"), "build_ms": c.get(name, {}).get("build_ms"),
                      "sort_base": c.get(name, {}).get("stage_ms", {}).get("sort_base"),
                      "dedup": c.get(name, {}).get("stage_ms", {}).get("dedup")} for name in ("cfg1", "cfg3")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--other", help="the tree to compare with (A); this tree is B")
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--save-cases", nargs=2, metavar=("TREE", "DIR"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.save_cases:
        return save_cases(*args.save_cases)
    trees = {"A": os.path.abspath(args.other), "B": ROOT}
    args.out = os.path.abspath(args.out)
    os.makedirs(args.out, exist_ok=True)
    result = {"gpu": run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem",
                          "--format=csv,noheader"], ROOT).strip()}
    # identity
    with tempfile.TemporaryDirectory() as tmp:
        info, digests = {}, {}
        for name, tree in trees.items():
            d = os.path.join(tmp, name)
            info[name] = last_json(run([sys.executable, os.path.abspath(__file__), "--save-cases", tree, d], ROOT))
            digests[name] = {c: hashlib.sha256(open(os.path.join(d, c + ".dbi"), "rb").read()).hexdigest()
                             for c in CASES}
        result["identity"] = {c: digests["A"][c] == digests["B"][c] for c in CASES}
        result["builds"] = info
    # bench, alternated
    result["bench"] = []
    env = dict(os.environ)
    env.pop("DBI_HASH_BITS", None)
    for r in range(args.rounds):
        for name, tree in trees.items():
            line = last_json(run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.steps),
                                  "--warmup", str(args.warmup)], tree, env))
            with open(os.path.join(args.out, f"bench_{name}{r}.json"), "w") as f:
                json.dump(line, f)
            result["bench"].append({"tree": name, "round": r, **pick(line)})
            print(json.dumps(result["bench"][-1]), flush=True)
    result["gpu_after"] = run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem",
                               "--format=csv,noheader"], ROOT).strip()
    # unindexed search at 10^2 .. 10^4 queries (part (a) of its benchmark)
    result["unindexed"] = {}
    for name, tree in trees.items():
        d = os.path.join(args.out, "unindexed_" + name)
        run([sys.executable, "scripts/unindexed_bench.py", "--out", d, "--big", "0"], tree, env)
        result["unindexed"][name] = d
    with open(os.path.join(args.out, "base_sort_ab.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("gpu", "identity", "builds")}))


if __name__ == "__main__":
    main()
