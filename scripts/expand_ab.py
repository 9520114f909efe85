"""A/B of the variant-group expansion (K6x, and K6q of the compact index) against another tree of this project (e.g.
a checkout of the parent commit).

In one call:
  identity  both trees build each case and dbi_save it; the files must be equal byte for byte (the entry order inside
            a group is part of the index, so nothing is canonicalised).  The compact-forced case is also fetched whole
            through dbi_fetch ranges that start mid-group (K6q) and hashed.  bench.py --dump-outputs of both trees
            must give identical .npy files.
  bench     bench.py --gpus 1 of the two trees alternated A B A B ..., the card's name, power limit and clocks read in
            the same call; then scripts/compact_bench.py --parts a (K6q at query time) and scripts/unindexed_bench.py
            --big 0 (K6x expands the candidate index) of each tree.
Writes <out>/expand_ab.json (+ the raw bench lines).

    python scripts/expand_ab.py --other DIR --out DIR [--rounds 3] [--steps 10] [--warmup 3]
"""
from __future__ import annotations

import argparse
import glob
import hashlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CASES = ("cfg2", "cfg2_compact", "wide_mass_mod4", "long_peptides", "pool_overflow", "three_classes_k2",
         "lysc_neg_mod")
SMI = ["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem", "--format=csv,noheader"]


def save_cases(tree, out_dir):
    """Child process: build every case with the package of `tree` and dbi_save it under out_dir."""
    sys.path.insert(0, tree)
    import numpy as np
    import dbindex_b200 as dbi
    from dbindex_b200 import synth
    sys.path.insert(0, ROOT)  # the proteomes and parameters of this tree's tests
    from bench import CFG2
    from tests.test_compact_index import LONG_PARAMS, long_proteome
    from tests.test_expand_order import POOL_PARAMS, pool_proteome
    from tests.util import PARAM_SETS
    os.makedirs(out_dir, exist_ok=True)
    info = {}
    for case in CASES:
        os.environ.pop("DBI_COMPACT_VARIANTS", None)
        if case.startswith("cfg2"):
            p, (res, off) = CFG2, synth.config_proteome(2, 20000)
        elif case == "long_peptides":
            p, (res, off) = LONG_PARAMS, long_proteome(300, 7)
        elif case == "pool_overflow":
            p, (res, off) = POOL_PARAMS, pool_proteome()
        else:
            p, (res, off) = PARAM_SETS[case], synth.synth_proteome(300, 4242)
        if case == "cfg2_compact":
            os.environ["DBI_COMPACT_VARIANTS"] = "1"
        with dbi.GpuIndex(dbi.default_params(**p)) as g:
            g.add_proteins(res, off)
            g.build()
            g.save(os.path.join(out_dir, case + ".dbi"))
            st = g.stats()
            info[case] = {k: st[k] for k in ("n_unique", "n_entries", "n_groups", "device_bytes")}
            if case == "cfg2_compact":  # K6q over ranges that start inside groups and tiles
                V, h, a = st["n_entries"], hashlib.sha256(), 0
                for b in sorted({int(x) for x in np.random.default_rng(1).integers(1, V, 40)} | {V}):
                    f = g.fetch(a, b - a, with_ids=False)
                    for k in ("mass", "first_prot", "first_off", "len", "modpat"):
                        h.update(np.ascontiguousarray(f[k]).tobytes())
                    a = b
                info[case]["fetch_sha256"] = h.hexdigest()
    os.environ.pop("DBI_COMPACT_VARIANTS", None)
    print(json.dumps(info))


def run(cmd, cwd, env=None):
    p = subprocess.run(cmd, cwd=cwd, env=env, capture_output=True, text=True)
    if p.returncode:
        sys.stderr.write(p.stdout[-4000:] + p.stderr[-4000:])
        raise SystemExit(f"{cmd} in {cwd} failed ({p.returncode})")
    return p.stdout


def last_json(text):
    return json.loads([ln for ln in text.splitlines() if ln.startswith("{")][-1])


def sha(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def pick(line):
    def one(d):
        roof = d.get("roofline") or {}
        exp = [r for r in [roof] + roof.get("other_kernels", []) if r.get("kernel") == "grp_expand_tab_kernel"]
        return {"ms_per_step": d.get("ms_per_step"), "build_ms": d.get("build_ms"),
                "expand_var": d.get("stage_ms", {}).get("expand_var"),
                "k6x_avg_launch_ms": exp[0]["avg_launch_ms"] if exp else None}
    c = line.get("configs", {})
    return {**one(line), **{name: one(c.get(name, {})) for name in ("cfg1", "cfg3")}}


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
    result = {"gpu": run(SMI, ROOT).strip()}
    env = dict(os.environ)
    env.pop("DBI_COMPACT_VARIANTS", None)
    # identity
    with tempfile.TemporaryDirectory() as tmp:
        info, digests, dumps = {}, {}, {}
        for name, tree in trees.items():
            d = os.path.join(tmp, name)
            info[name] = last_json(run([sys.executable, os.path.abspath(__file__), "--save-cases", tree, d], ROOT, env))
            digests[name] = {c: sha(os.path.join(d, c + ".dbi")) for c in CASES}
            dd = os.path.join(tmp, "dump_" + name)
            run([sys.executable, "bench.py", "--gpus", "1", "--steps", "1", "--warmup", "1", "--no-extra",
                 "--no-cpu-baseline", "--dump-outputs", dd], tree, env)
            dumps[name] = {os.path.basename(p): sha(p) for p in sorted(glob.glob(os.path.join(dd, "*.npy")))}
        result["identity"] = {c: digests["A"][c] == digests["B"][c] for c in CASES}
        result["identity"]["cfg2_compact_fetch"] = (info["A"]["cfg2_compact"]["fetch_sha256"] ==
                                                    info["B"]["cfg2_compact"]["fetch_sha256"])
        result["identity"]["bench_dump_npy"] = bool(dumps["A"]) and dumps["A"] == dumps["B"]
        result["builds"] = info
        result["bench_dump_files"] = sorted(dumps["B"])
    print(json.dumps({k: result[k] for k in ("gpu", "identity")}), flush=True)
    # bench, alternated
    result["bench"] = []
    for r in range(args.rounds):
        for name, tree in trees.items():
            line = last_json(run([sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.steps),
                                  "--warmup", str(args.warmup)], tree, env))
            with open(os.path.join(args.out, f"bench_{name}{r}.json"), "w") as f:
                json.dump(line, f)
            result["bench"].append({"tree": name, "round": r, **pick(line)})
            print(json.dumps(result["bench"][-1]), flush=True)
    result["gpu_after"] = run(SMI, ROOT).strip()
    # K6q at query time (compact index, cfg2) and the unindexed search, whose candidate index K6x expands
    result["compact_a"], result["unindexed"] = {}, {}
    for name, tree in trees.items():
        out = run([sys.executable, "scripts/compact_bench.py", "--out", os.path.join(args.out, "compact_" + name),
                   "--parts", "a"], tree, env)
        result["compact_a"][name] = next(json.loads(ln) for ln in out.splitlines() if ln.startswith('{"a"'))["a"]
        d = os.path.join(args.out, "unindexed_" + name)
        out = run([sys.executable, "scripts/unindexed_bench.py", "--out", d, "--big", "0"], tree, env)
        result["unindexed"][name] = [json.loads(ln) for ln in out.splitlines() if ln.startswith('{"nq"')]
        print(json.dumps({name: {"compact_a": result["compact_a"][name]["median"],
                                 "unindexed": result["unindexed"][name]}}), flush=True)
    with open(os.path.join(args.out, "expand_ab.json"), "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
