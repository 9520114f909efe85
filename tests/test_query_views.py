"""Query views (dbi_view_open): one built index answered from many host threads at once, each thread on a view with its
own stream, scratch and pending results.

GPU: every query entry point on views driven by 8 threads against the owner's single-threaded answers, byte for byte,
on a group-path index, an index without mods, a per-variant-path index and a compact index; pending results that stay
with the handle or view that made them; the refusals and the lifecycle (views pin the owner, outlive it); views of the
ranks of a sharded index; the stats of a view; the Python mirror from 8 threads.  The Java downcall of dbi_view_open
is checked against the header by tests/test_java_layout.py, which parses every downcall."""
import ctypes as C
import os
import re
import threading

import numpy as np
import pytest

import dbindex_b200 as dbi
from dbindex_b200 import synth
from dbindex_b200.capi import DBI_TOL_DA, DBI_TOL_PPM, LIB_PATH, DbiError, DbiHitBuffers

from .util import PARAM_SETS

gpu = pytest.mark.gpu
DBI_ENOTINIT, DBI_EINVAL = -1, -3
N_THREADS = 8
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INDEXES = {  # name: (parameter set, proteins, compact layout)
    "group_mods": ("cfg2_mods", 1500, False),
    "no_mods": ("cfg1_tryptic", 1500, False),
    "per_variant": ("many_classes", 400, False),  # 85 class sequences > 32
    "compact": ("cfg2_mods", 1500, True),
}


def build(params, res, off, compact=False):
    old = os.environ.pop("DBI_COMPACT_VARIANTS", None)
    if compact:
        os.environ["DBI_COMPACT_VARIANTS"] = "1"
    try:
        g = dbi.GpuIndex(params)
        g.add_proteins(res, off)
        g.build()
    finally:
        os.environ.pop("DBI_COMPACT_VARIANTS", None)
        if old is not None:
            os.environ["DBI_COMPACT_VARIANTS"] = old
    return g


def frozen(x):
    """A result as plain bytes, so that two answers compare byte for byte."""
    if isinstance(x, dict):
        return tuple((k, frozen(v)) for k, v in sorted(x.items()))
    if isinstance(x, (tuple, list)):
        return tuple(frozen(v) for v in x)
    if isinstance(x, np.ndarray):
        return (str(x.dtype), x.tobytes())
    if isinstance(x, C.Structure):
        return tuple((f, getattr(x, f)) for f, _ in x._fields_)
    return x


def make_batches(g, n_batches, seed):
    """Mixed work for the threads: ranges, Dalton spectra, PPM spectra, lookups (found and absent, with and without
    mods), an entry window."""
    n_entries = g.stats()["n_entries"]
    keys = g.entry_keys()
    masses = keys.astype(np.float64) / g.params.mass_group_factor
    rng = np.random.default_rng(seed)
    probe = g.query_hits(masses[:: max(1, len(masses) // 400)] - 0.01, masses[:: max(1, len(masses) // 400)] + 0.01)
    so = probe["seq_off"].astype(np.int64)
    seqs = [probe["seq"][so[i]:so[i + 1]].tobytes() for i in range(len(so) - 1)]
    pats = probe["modpat"]
    out = []
    for b in range(n_batches):
        nq = int(rng.integers(20, 120))
        m = rng.choice(masses, nq) * (1 + rng.uniform(-5e-6, 5e-6, nq))
        m[: nq // 4] = rng.uniform(g.params.min_mass, g.params.max_mass, nq // 4)
        tol = m * 10e-6
        ns = int(rng.integers(5, 40))
        lens = rng.integers(0, 4, ns)
        range_off = np.concatenate(([0], np.cumsum(lens))).astype(np.uint64)
        sm = rng.choice(masses, int(range_off[-1])) + rng.uniform(-0.02, 0.02, int(range_off[-1]))
        st = rng.uniform(0.001, 0.05, int(range_off[-1]))
        pm = rng.choice(masses, ns)
        pick = rng.integers(0, len(seqs), 60)
        lk = [seqs[i] for i in pick] + [b"PEPTIDEWXYZ", b"K" * 9]
        lk_pat = np.concatenate((pats[pick], [0, 0])).astype(np.uint32)
        lk_pat[::3] = 0  # unmodified rows of modified peptides too
        begin = int(rng.integers(0, max(1, n_entries - 300)))
        out.append(dict(lo=np.maximum(m - tol, 0), hi=m + tol, sm=sm, st=st, range_off=range_off, pm=pm,
                        lk=lk, lk_pat=lk_pat, begin=begin, count=min(300, n_entries - begin)))
    return out


def script(g, b):
    """One round of every query entry point on g: each answer as bytes."""
    return [
        frozen(g.query_hits(b["lo"], b["hi"], per_hit=False)),
        frozen(g.query_spectra(b["sm"], b["st"], b["range_off"], DBI_TOL_DA, per_hit=False)),
        frozen(g.query_spectra(b["pm"], np.full(len(b["pm"]), 5.0), None, DBI_TOL_PPM, per_hit=False)),
        frozen(g.query_spectra(b["pm"], np.full(len(b["pm"]), 50.0), None, DBI_TOL_PPM, per_hit=False)),
        frozen(g.lookup_peptides(b["lk"], b["lk_pat"])),
        frozen(g.query(b["lo"], b["hi"])),
        frozen(g.fetch(b["begin"], b["count"])),
        frozen(g.entry_keys()),
    ]


def run_threads(n, fn):
    errors = []

    def body(t):
        try:
            fn(t)
        except BaseException as e:  # noqa: BLE001 -- reported by the main thread
            errors.append((t, e))

    th = [threading.Thread(target=body, args=(t,)) for t in range(n)]
    for x in th:
        x.start()
    for x in th:
        x.join()
    if errors:
        raise errors[0][1]


@pytest.fixture(scope="module", params=list(INDEXES))
def index(request):
    name, n_prot, compact = INDEXES[request.param]
    p = dbi.default_params(**PARAM_SETS[name])
    res, off = synth.synth_proteome(n_prot, 777)
    g = build(p, res, off, compact)
    assert (g.stats()["n_groups"] > 0) == compact
    yield g, p, res, off
    g.close()


# ---- 1. parity under threads ------------------------------------------------------------------------------------
@gpu
def test_views_equal_owner_under_threads(index):
    g = index[0]
    batches = make_batches(g, 6, 11)
    expect = [script(g, b) for b in batches]
    rounds = 3

    def work(t):
        with g.view() as v:
            for r in range(rounds):
                for k in range(len(batches)):
                    i = (t + r + k) % len(batches)
                    got = script(v, batches[i])
                    for c, (a, e) in enumerate(zip(got, expect[i])):
                        assert a == e, f"thread {t} batch {i} call {c} differs from the owner"

    def owner_too(t):
        if t == N_THREADS:  # the owner keeps answering while its views run
            for r in range(rounds):
                for i, b in enumerate(batches):
                    assert script(g, b) == expect[i]
        else:
            work(t)

    run_threads(N_THREADS + 1, owner_too)


# ---- 2. pending results belong to their caller --------------------------------------------------------------------
@gpu
def test_pending_results_stay_with_their_handle(index):
    g = index[0]
    x, y = make_batches(g, 2, 23)
    exp_x = frozen(g.query_hits(x["lo"], x["hi"], per_hit=False))
    exp_y = frozen(g.query_hits(y["lo"], y["hi"], per_hit=False))
    exp_lx = frozen(g.lookup_peptides(x["lk"], x["lk_pat"]))
    exp_ly = frozen(g.lookup_peptides(y["lk"], y["lk_pat"]))
    with g.view() as a, g.view() as b:
        # the owner's own pending result survives its views' calls
        cg = g.query_hits_begin(x["lo"], x["hi"])
        lg = g.lookup_peptides_begin(x["lk"], x["lk_pat"])
        ca = a.query_hits_begin(x["lo"], x["hi"])
        la = a.lookup_peptides_begin(x["lk"], x["lk_pat"])
        assert frozen(b.query_hits(y["lo"], y["hi"], per_hit=False)) == exp_y
        assert frozen(b.lookup_peptides(y["lk"], y["lk_pat"])) == exp_ly
        assert frozen(a._read_hits(ca, None, None, False)) == exp_x
        assert frozen(a.lookup_peptides_read(la)) == exp_lx
        assert frozen(g._read_hits(cg, None, None, False)) == exp_x
        assert frozen(g.lookup_peptides_read(lg)) == exp_lx
        for h in (a, b, g):  # nothing left pending anywhere
            with pytest.raises(DbiError) as ei:
                h.query_hits_read(DbiHitBuffers())
            assert ei.value.code == DBI_ENOTINIT


# ---- 3. lifecycle and refusals ------------------------------------------------------------------------------------
def header_arity():
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "dbindex_gpu.h")).read(), flags=re.S)
    return {m.group(1): len(m.group(2).split(",")) if m.group(2).strip() else 0
            for m in re.finditer(r"\bint\s+(dbi_[a-z_0-9]+)\s*\(\s*dbi_handle\*\s*h\s*,?([^;]*?)\)\s*;", hdr, re.S)}


REFUSED = ["dbi_add_proteins", "dbi_upload", "dbi_reset_index", "dbi_build", "dbi_build_from_records", "dbi_save",
           "dbi_load", "dbi_search_unindexed", "dbi_search_unindexed_spectra", "dbi_mg_begin", "dbi_mg_set_shards",
           "dbi_mg_window_ensure", "dbi_mg_window_import", "dbi_mg_pull_proteome", "dbi_mg_digest", "dbi_mg_hist",
           "dbi_mg_count", "dbi_mg_scatter", "dbi_mg_index_base", "dbi_mg_unique_count", "dbi_mg_set_unique",
           "dbi_mg_groups", "dbi_mg_index_variants", "dbi_mg_finish", "dbi_mg_spectra_stops", "dbi_mg_query_spectra",
           "dbi_debug_emitted", "dbi_debug_radix_sort"]
LOCAL = ["dbi_mg_build_local", "dbi_mg_search_unindexed_local", "dbi_mg_search_unindexed_spectra_local",
         "dbi_mg_query_spectra_local"]


def raw_call(lib, name, h, n_args):
    """name(h, ...) with zeroed arguments and a valid scratch pointer wherever one is read before the handle check."""
    f = getattr(lib, name)
    f.restype = C.c_int
    scratch = (C.c_uint64 * 64)()
    f.argtypes = [C.c_void_p] * (n_args + 1)
    return f(h, *([C.addressof(scratch)] * n_args))


def local_call(lib, name, hs):
    arr = (C.c_void_p * len(hs))(*hs)
    scratch = (C.c_uint64 * 64)()
    f = getattr(lib, name)
    f.restype = C.c_int
    if name == "dbi_mg_build_local":
        f.argtypes = [C.c_void_p, C.c_int]
        return f(arr, len(hs))
    if name == "dbi_mg_search_unindexed_local":
        f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]
        return f(arr, len(hs), C.addressof(scratch), C.addressof(scratch), 1, 0, C.addressof(scratch),
                 C.addressof(scratch))
    off = np.array([0, 1], np.uint64)
    m = np.array([1000.0])
    if name == "dbi_mg_query_spectra_local":
        f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int,
                      C.c_void_p]
        return f(arr, len(hs), m.ctypes.data, m.ctypes.data, off.ctypes.data, 1, DBI_TOL_DA, 0, C.addressof(scratch))
    f.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_uint64,
                  C.c_void_p, C.c_void_p]
    return f(arr, len(hs), m.ctypes.data, m.ctypes.data, off.ctypes.data, 1, DBI_TOL_DA, 0, 0, C.addressof(scratch),
             C.addressof(scratch))


@gpu
def test_refusals_and_lifecycle():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = synth.synth_proteome(600, 31)
    lib = C.CDLL(LIB_PATH)  # its own function objects: the argument types set below stay local to this test
    lib.dbi_last_error.restype = C.c_char_p
    arity = header_arity()

    # a view needs a built owner: unbuilt, and a handle used for unindexed searches only
    with dbi.GpuIndex(p) as u:
        u.add_proteins(res, off)
        with pytest.raises(DbiError) as ei:
            u.view()
        assert ei.value.code == DBI_ENOTINIT
        u.search_unindexed(np.array([1000.0]), np.array([1010.0]))
        with pytest.raises(DbiError) as ei:
            u.view()
        assert ei.value.code == DBI_ENOTINIT

    g = build(p, res, off)
    (b,) = make_batches(g, 1, 5)
    expect = script(g, b)
    v = g.view()
    # every refused call on a view, a view of a view, the multi-handle calls with a view in them
    for name in REFUSED:
        assert raw_call(lib, name, v._h, arity[name]) == DBI_EINVAL, name
        assert "view" in lib.dbi_last_error().decode(), name
    with pytest.raises(DbiError) as ei:
        v.view()
    assert ei.value.code == DBI_EINVAL
    for name in LOCAL:
        assert local_call(lib, name, [v._h]) == DBI_EINVAL, name
    # the accepted host-side calls
    assert v.calculate_mass(b"PEPTIDEK") == g.calculate_mass(b"PEPTIDEK")
    assert v.get_protein(3) == g.get_protein(3) == res[int(off[3]):int(off[4])].tobytes()
    assert script(v, b) == expect

    # the owner is pinned while a view is open ...
    for name in ("dbi_add_proteins", "dbi_upload", "dbi_reset_index", "dbi_build", "dbi_load",
                 "dbi_search_unindexed", "dbi_mg_begin"):
        assert raw_call(lib, name, g._h, arity[name]) == DBI_EINVAL, name
        assert "1 views open" in lib.dbi_last_error().decode(), name
    assert local_call(lib, "dbi_mg_build_local", [g._h]) == DBI_EINVAL
    assert script(g, b) == expect  # ... and keeps answering
    v2 = g.view()
    v.close()
    assert raw_call(lib, "dbi_reset_index", g._h, 0) == DBI_EINVAL  # one view still open
    v2.close()
    # after the last view: the index may change again, and rebuilds to the same answers
    g.reset_index()
    g.build()
    assert script(g, b) == expect

    # the owner destroyed first: its views keep answering, then close cleanly
    views = [g.view() for _ in range(3)]
    g.close()

    def after_owner(t):
        for _ in range(2):
            assert script(views[t], b) == expect, f"view {t} after the owner was destroyed"

    run_threads(3, after_owner)
    assert views[0].get_protein(3) == res[int(off[3]):int(off[4])].tobytes()
    for x in views:
        x.close()


# ---- 4. ranks of a sharded index ---------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("world", [2, 3])
def test_views_of_sharded_ranks(world):
    from dbindex_b200.multigpu import build_local, shard_proteins
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = synth.synth_proteome(900, 41 + world)
    hs = []
    for r in range(world):
        g = dbi.GpuIndex(p)
        sres, soff, _ = shard_proteins(res, off, r, world)
        g.add_proteins(sres, soff)
        hs.append(g)
    try:
        build_local(hs)
        # lookups of every peptide of the proteome's first proteins: most base peptides live on another rank
        one = build(p, res, off)
        (b,) = make_batches(one, 1, 3)
        one.close()

        def calls(g):
            return [frozen(g.query_hits(b["lo"], b["hi"], per_hit=False)),
                    frozen(g.lookup_peptides(b["lk"], b["lk_pat"]))]

        expect = [calls(g) for g in hs]
        found = sum(int((hs[r].lookup_peptides(b["lk"], b["lk_pat"])["status"] == 1).sum()) for r in range(world))
        assert found > 0

        def work(t):
            r = t % world
            with hs[r].view() as v:
                for _ in range(4):
                    assert calls(v) == expect[r], f"rank {r}"

        run_threads(N_THREADS, work)
    finally:
        for g in hs:
            g.close()


# ---- 5. stats -----------------------------------------------------------------------------------------------------
@gpu
def test_view_stats():
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"], profile=1)
    res, off = synth.synth_proteome(600, 53)
    g = build(p, res, off)
    try:
        (b,) = make_batches(g, 1, 8)
        before = g.stats()
        with g.view() as v:
            s0 = v.stats()
            for k in ("n_proteins", "n_residues", "n_emitted", "n_unique", "n_entries", "device_bytes", "n_groups",
                      "sort_bits_base", "sort_bits_var"):
                assert s0[k] == before[k], k
            assert all(x == 0 for x in s0["stage_launches"].values())
            assert all(x == 0 for x in s0["algo_bytes"].values())
            v.query_hits(b["lo"], b["hi"])
            v.fetch(b["begin"], b["count"])
            s1 = v.stats()
            assert s1["stage_launches"]["query"] > 0 and s1["stage_launches"]["fetch"] > 0
            assert s1["algo_bytes"]["query"] > 0
            assert s1["stage_ms"]["query"] > 0
            after = g.stats()
            assert after["stage_launches"] == before["stage_launches"]
            assert after["algo_bytes"] == before["algo_bytes"]
            # the same call on the owner counts the same launches there
            g.query_hits(b["lo"], b["hi"])
            g.fetch(b["begin"], b["count"])
            own = g.stats()
            for st in ("query", "fetch"):
                assert own["stage_launches"][st] - before["stage_launches"][st] == s1["stage_launches"][st], st
    finally:
        g.close()


# ---- 6. the Python mirror -----------------------------------------------------------------------------------------
@gpu
def test_mirror_from_threads():
    from dbindex_b200.indexer import DBIndexer, MassRange
    p = dbi.default_params(**PARAM_SETS["cfg2_mods"])
    res, off = synth.synth_proteome(800, 61)
    seqs = [res[int(off[i]):int(off[i + 1])].tobytes().decode() for i in range(len(off) - 1)]
    ix = DBIndexer(p)
    ix.init()
    ix.run(proteins=(synth.deflines(len(seqs)), seqs))
    try:
        rng = np.random.default_rng(9)
        keys = ix.index.entry_keys().astype(np.float64) / p.mass_group_factor
        work = []
        for b in range(6):
            ms = rng.choice(keys, 30)
            spectra = [[MassRange(float(m), 0.02)] + [MassRange(float(m) + 1.00335, 0.02)] * int(k)
                       for m, k in zip(ms, rng.integers(0, 2, 30))]
            peps = [s.sequence for lst in ix.getSequencesBatch(ms[:8], [0.01] * 8) for s in lst][:20] + ["PEPTIDEK"]
            work.append((ms, spectra, peps))

        def answers(i):
            ms, spectra, peps = work[i]
            return (
                [ix.getSequencesUsingDaltonTolerance(float(m), 0.02) for m in ms[:5]],
                ix.getSequencesForSpectra(spectra),
                ix.getSequencesUsingPPMToleranceBatch(ms, 10.0),
                [sorted(x.id for x in st) for st in ix.getProteinsBatch(peps)],
            )

        expect = [answers(i) for i in range(len(work))]

        def run(t):
            for r in range(3):
                i = (t + r) % len(work)
                assert answers(i) == expect[i], f"thread {t} batch {i}"

        run_threads(N_THREADS, run)
        assert len(ix._views) == N_THREADS + 1  # the main thread's view, and one per worker

        # threads sharing one GpuIndex without views: the per-object lock keeps each begin / read pair together
        g = ix.index
        bs = make_batches(g, 4, 2)
        exp = [(frozen(g.query_hits(b["lo"], b["hi"], per_hit=False)), frozen(g.lookup_peptides(b["lk"], b["lk_pat"])),
                frozen(g.query_spectra(b["pm"], np.full(len(b["pm"]), 10.0), None, DBI_TOL_PPM, per_hit=False)))
               for b in bs]

        def shared(t):
            for r in range(6):
                i = (t + r) % len(bs)
                b = bs[i]
                got = (frozen(g.query_hits(b["lo"], b["hi"], per_hit=False)),
                       frozen(g.lookup_peptides(b["lk"], b["lk_pat"])),
                       frozen(g.query_spectra(b["pm"], np.full(len(b["pm"]), 10.0), None, DBI_TOL_PPM,
                                              per_hit=False)))
                assert got == exp[i], f"thread {t} batch {i}"

        run_threads(N_THREADS, shared)
    finally:
        ix.close()
