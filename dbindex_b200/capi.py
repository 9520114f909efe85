"""ctypes binding of include/dbindex_gpu.h (the drop-in C ABI).

The same calls a Java host makes through Panama FFM / JNI (INTEGRATION.md); used by
the tests and bench.py.  Nothing here computes: every method forwards to the CUDA
library and raises DbiError on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdbindex_gpu.so")

DBI_ABI_VERSION = 3
DBI_MAX_MODS = 16
DBI_N_STAGES = 12
STAGE_NAMES = [
    "pack", "digest_count", "digest_emit", "sort_base", "dedup", "mod_count",
    "mod_emit", "sort_var", "expand_var", "query", "fetch", "other",
]
ERR_NAMES = {
    0: "DBI_OK", -1: "DBI_ENOTINIT", -2: "DBI_EALREADY", -3: "DBI_EINVAL", -4: "DBI_ENOMEM",
    -5: "DBI_ECUDA", -6: "DBI_ENCCL", -7: "DBI_ERANGE",
}


class DbiMod(C.Structure):
    _fields_ = [("residue", C.c_uint8), ("_pad", C.c_uint8 * 7), ("delta", C.c_double)]


class DbiParams(C.Structure):
    """struct dbi_params (include/dbindex_gpu.h)."""

    _fields_ = [
        ("abi_version", C.c_uint32),
        ("device", C.c_int32),
        ("residue_mass", C.c_double * 256),
        ("h2o_proton", C.c_double),
        ("nterm", C.c_double),
        ("cterm", C.c_double),
        ("add_h2o_proton", C.c_int32),
        ("is_enzyme", C.c_uint8 * 256),
        ("is_nocut", C.c_uint8 * 256),
        ("max_missed", C.c_int32),
        ("semi", C.c_int32),
        ("min_len", C.c_int32),
        ("min_mass", C.c_double),
        ("max_mass", C.c_double),
        ("mass_group_factor", C.c_int32),
        ("n_mods", C.c_int32),
        ("max_mods_per_peptide", C.c_int32),
        ("mods", DbiMod * DBI_MAX_MODS),
        ("is_mandatory", C.c_uint8 * 256),
        ("has_mandatory", C.c_int32),
        ("filter_aa", C.c_int32),
        ("filter_max", C.c_int32),
        ("_pad_filters", C.c_int32),
        ("keep_emitted", C.c_int32),
        ("profile", C.c_int32),
        ("reserved", C.c_int32 * 6),
    ]

    def copy(self) -> "DbiParams":
        q = DbiParams()
        C.memmove(C.byref(q), C.byref(self), C.sizeof(DbiParams))
        return q


class DbiStats(C.Structure):
    _fields_ = [
        ("n_proteins", C.c_uint64),
        ("n_residues", C.c_uint64),
        ("n_emitted", C.c_uint64),
        ("n_unique", C.c_uint64),
        ("n_entries", C.c_uint64),
        ("n_hash_retries", C.c_uint64),
        ("device_bytes", C.c_uint64),
        ("algo_bytes", C.c_uint64 * DBI_N_STAGES),
        ("stage_ms", C.c_float * DBI_N_STAGES),
        ("stage_launches", C.c_uint32 * DBI_N_STAGES),
        ("sort_bits_base", C.c_uint32),
        ("sort_bits_var", C.c_uint32),
        ("dom_ms", C.c_float),
        ("dom_launches", C.c_uint32),
        ("dom_bytes_per_launch", C.c_uint64),
        ("dom_kernel", C.c_uint32),
        ("exp_launches", C.c_uint32),
        ("exp_ms", C.c_float),
        ("n_groups", C.c_uint32),
        ("exp_bytes_per_launch", C.c_uint64),
    ]


class DbiHitCounts(C.Structure):
    _fields_ = [("nq", C.c_uint64), ("n_hits", C.c_uint64), ("n_peps", C.c_uint64), ("n_seq_bytes", C.c_uint64),
                ("n_prot_ids", C.c_uint64)]


class DbiHitBuffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("hit_off", "pep_off", "modpat", "pep_hit_off", "mass", "first_prot", "first_off",
                                          "len", "flanks", "seq_off", "seq", "prot_list_off", "prot_ids")]


class DbiLookupCounts(C.Structure):
    _fields_ = [("n", C.c_uint64), ("n_found", C.c_uint64), ("n_prot_ids", C.c_uint64)]


class DbiLookupBuffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("status", "mass", "entry", "first_prot", "first_off", "prot_list_off",
                                          "prot_ids")]


LOOKUP_ABSENT, LOOKUP_FOUND, LOOKUP_MALFORMED = 0, 1, 2
LOOKUP_FIELDS = {  # dbi_lookup_buffers: name -> (dtype, size as a function of the counts)
    "status": (np.uint8, lambda c: c.n), "mass": (np.float64, lambda c: c.n), "entry": (np.uint64, lambda c: c.n),
    "first_prot": (np.uint32, lambda c: c.n), "first_off": (np.uint32, lambda c: c.n),
    "prot_list_off": (np.uint64, lambda c: c.n + 1), "prot_ids": (np.uint32, lambda c: c.n_prot_ids),
}


# dbi_hit_buffers: the hits of a batch grouped in RUNS (consecutive hits of one query that are variants of one
# peptide with one mass); per-run arrays have n_peps rows, only the mod pattern is per hit
HIT_FIELDS = {  # name -> (dtype, size as a function of the counts)
    "hit_off": (np.uint64, lambda c: c.nq + 1), "pep_off": (np.uint64, lambda c: c.nq + 1),
    "modpat": (np.uint32, lambda c: c.n_hits), "pep_hit_off": (np.uint64, lambda c: c.n_peps + 1),
    "mass": (np.float64, lambda c: c.n_peps),
    "first_prot": (np.uint32, lambda c: c.n_peps), "first_off": (np.uint32, lambda c: c.n_peps),
    "len": (np.uint16, lambda c: c.n_peps),
    "flanks": (np.uint8, lambda c: 6 * c.n_peps), "seq_off": (np.uint64, lambda c: c.n_peps + 1),
    "seq": (np.uint8, lambda c: c.n_seq_bytes), "prot_list_off": (np.uint64, lambda c: c.n_peps + 1),
    "prot_ids": (np.uint32, lambda c: c.n_prot_ids),
}


def _expand_csr(off_run: np.ndarray, data: np.ndarray, run_of_hit: np.ndarray):
    """Per-hit CSR (offsets, data) from a per-run CSR."""
    off_run = off_run.astype(np.int64)
    sizes = np.diff(off_run)[run_of_hit]
    off_hit = np.concatenate(([0], np.cumsum(sizes))).astype(np.int64)
    total = int(off_hit[-1])
    src = np.repeat(off_run[:-1][run_of_hit] - off_hit[:-1], sizes) + np.arange(total, dtype=np.int64)
    return off_hit.astype(np.uint64), data[src]


def expand_hits(raw: dict) -> dict:
    """One record per hit (the shape parseAddPeptideInfo produces and the oracle's query_hits returns) from
    the run-grouped answer of dbi_query_hits.  Host-side convenience for tests and the Python mirror."""
    run_of_hit = np.repeat(np.arange(len(raw["pep_hit_off"]) - 1, dtype=np.int64),
                           np.diff(raw["pep_hit_off"].astype(np.int64)))
    out = {k: raw[k] for k in ("counts", "hit_off", "modpat") if k in raw}
    out["hit_pep"] = run_of_hit
    for k in ("mass", "first_prot", "first_off", "len"):
        if k in raw:
            out[k] = raw[k][run_of_hit]
    if "flanks" in raw:
        out["flanks"] = np.ascontiguousarray(raw["flanks"].reshape(-1, 6)[run_of_hit]).reshape(-1)
    if "seq" in raw:
        out["seq_off"], out["seq"] = _expand_csr(raw["seq_off"], raw["seq"], run_of_hit)
    if "prot_ids" in raw:
        out["prot_list_off"], out["prot_ids"] = _expand_csr(raw["prot_list_off"], raw["prot_ids"], run_of_hit)
    return out


DBI_ERANGE = -7
DBI_TOL_DA = 0   # dbi_query_spectra: spectrum s = ranges [range_off[s], range_off[s+1]) of (mass, tol in Da)
DBI_TOL_PPM = 1  # dbi_query_spectra: spectrum s = mass[s] at tol[s] ppm


def spectra_arrays(mass, tol, range_off, tol_mode: int):
    """The contiguous arrays of a dbi_query_spectra batch and its number of spectra (range_off None: PPM only)."""
    mass = np.ascontiguousarray(mass, dtype=np.float64)
    tol = np.ascontiguousarray(tol, dtype=np.float64)
    if len(mass) != len(tol):
        raise ValueError(f"{len(mass)} masses and {len(tol)} tolerances")
    if range_off is None:
        if tol_mode == DBI_TOL_DA:
            raise ValueError("DBI_TOL_DA needs range_off")
        return mass, tol, None, len(mass)
    range_off = np.ascontiguousarray(range_off, dtype=np.uint64)
    if len(range_off) == 0 or (tol_mode == DBI_TOL_DA and int(range_off[-1]) > len(mass)):
        raise ValueError(f"range_off of {len(range_off)} offsets over {len(mass)} ranges")
    return mass, tol, range_off, len(range_off) - 1


def ppm_probe_bound(mass: float, ppm: float) -> float:
    """The upper end of the candidate window dbi_search_unindexed_spectra digests for one PPM spectrum: an upper
    bound of every probe u the walk of getSequencesUsingPPMTolerance admits (u - tol(u) < mass), computed as
    K13b computes it (spec_ppm_window_kernel)."""
    p1 = ppm / 1e6 + 1.0
    hi = mass + mass * (1 - 1 / p1)
    ext = (mass * p1) * (1.0 + 2.0 ** -40) if mass > 0.0 and p1 > 0.0 else float("inf")
    return max(ext, hi)


class DbiError(RuntimeError):
    """A non-zero status.  n_candidates: the candidate records of a dbi_search_unindexed that failed (DBI_ERANGE
    when they exceed the cap), else None."""

    def __init__(self, code: int, msg: str, n_candidates: Optional[int] = None):
        super().__init__(f"{ERR_NAMES.get(code, code)}: {msg}")
        self.code = code
        self.n_candidates = n_candidates


_lib = None


def load_library(path: Optional[str] = None) -> C.CDLL:
    """Load libdbindex_gpu.so.  Fails loudly when it has not been built: there is no
    pure-Python or CPU path to fall back to."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C dbindex_b200/csrc`). dbindex_b200 has no CPU fallback."
        )
    lib = C.CDLL(path)
    vp, u8p, u16p, u32p, i32p, u64p, dp = (
        C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint16), C.POINTER(C.c_uint32),
        C.POINTER(C.c_int32), C.POINTER(C.c_uint64), C.POINTER(C.c_double),
    )
    pp = C.POINTER(DbiParams)
    sigs = {
        "dbi_default_params": (None, [pp, C.c_int]),
        "dbi_params_add_static_mod": (None, [pp, C.c_uint8, C.c_double]),
        "dbi_params_set_enzyme": (None, [pp, C.c_char_p, C.c_char_p]),
        "dbi_params_add_diff_mod": (C.c_int, [pp, C.c_char_p, C.c_double]),
        "dbi_create": (C.c_int, [pp, C.POINTER(vp)]),
        "dbi_set_stream": (C.c_int, [vp, vp]),
        "dbi_add_proteins": (C.c_int, [vp, vp, vp, C.c_uint32]),
        "dbi_upload": (C.c_int, [vp]),
        "dbi_reset_index": (C.c_int, [vp]),
        "dbi_build": (C.c_int, [vp]),
        "dbi_stats_get": (C.c_int, [vp, C.POINTER(DbiStats)]),
        "dbi_save": (C.c_int, [vp, C.c_char_p]),
        "dbi_load": (C.c_int, [vp, C.c_char_p]),
        "dbi_query": (C.c_int, [vp, vp, vp, C.c_uint64, vp, vp]),
        "dbi_query_device": (C.c_int, [vp, vp, vp, C.c_uint64, vp, vp]),
        "dbi_fetch": (C.c_int, [vp, C.c_uint64, C.c_uint64, vp, vp, vp, vp, vp, vp, vp, C.c_uint64, u64p]),
        "dbi_query_hits": (C.c_int, [vp, vp, vp, C.c_uint64, C.POINTER(DbiHitCounts)]),
        "dbi_query_hits_device": (C.c_int, [vp, vp, vp, C.c_uint64, C.POINTER(DbiHitCounts)]),
        "dbi_query_hits_read": (C.c_int, [vp, C.POINTER(DbiHitBuffers)]),
        "dbi_search_unindexed": (C.c_int, [vp, vp, vp, C.c_uint64, C.c_uint64, C.POINTER(DbiHitCounts), u64p]),
        "dbi_query_spectra": (C.c_int, [vp, vp, vp, vp, C.c_uint64, C.c_int, C.c_int, C.POINTER(DbiHitCounts)]),
        "dbi_search_unindexed_spectra": (C.c_int, [vp, vp, vp, vp, C.c_uint64, C.c_int, C.c_int, C.c_uint64,
                                                   C.POINTER(DbiHitCounts), u64p]),
        "dbi_mg_spectra_stops": (C.c_int, [vp, vp, vp, C.c_uint64, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp]),
        "dbi_mg_query_spectra": (C.c_int, [vp, vp, vp, vp, C.c_uint64, C.c_int, C.c_int, vp,
                                           C.POINTER(DbiHitCounts)]),
        "dbi_lookup_peptides": (C.c_int, [vp, vp, vp, vp, C.c_uint64, C.POINTER(DbiLookupCounts)]),
        "dbi_lookup_peptides_read": (C.c_int, [vp, C.POINTER(DbiLookupBuffers)]),
        "dbi_host_alloc": (C.c_int, [C.c_uint64, C.POINTER(vp)]),
        "dbi_host_free": (C.c_int, [vp]),
        "dbi_get_protein": (C.c_int, [vp, C.c_uint32, C.POINTER(vp), u64p]),
        "dbi_fasta_open": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(vp)]),
        "dbi_fasta_counts": (C.c_int, [vp, u32p, u64p, u64p]),
        "dbi_fasta_read": (C.c_int, [vp, vp, vp, vp, vp]),
        "dbi_fasta_close": (None, [vp]),
        "dbi_calculate_mass": (C.c_int, [vp, C.c_char_p, C.c_uint64, dp]),
        "dbi_entry_keys": (C.c_int, [vp, vp, C.c_uint64, u64p]),
        "dbi_debug_emitted": (C.c_int, [vp, C.c_uint64, vp, vp, vp, vp, u64p]),
        "dbi_build_from_records": (C.c_int, [vp, vp, vp, vp, vp, C.c_uint64]),
        "dbi_debug_radix_sort": (C.c_int, [vp, vp, vp, C.c_uint64, C.c_int, C.c_int]),
        "dbi_destroy": (None, [vp]),
        "dbi_abi_sizes": (None, [u64p, u64p]),
        "dbi_release_cached_memory": (C.c_int, [C.c_int]),
        "dbi_last_error": (C.c_char_p, []),
        "dbi_kernel_launches": (C.c_uint64, []),
    }
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)  # AttributeError = the library does not export the ABI
        fn.restype = res
        fn.argtypes = args
    sp, ss = C.c_uint64(), C.c_uint64()
    lib.dbi_abi_sizes(C.byref(sp), C.byref(ss))
    if sp.value != C.sizeof(DbiParams) or ss.value != C.sizeof(DbiStats):
        raise ImportError(
            f"struct layout mismatch: dbi_params {sp.value} vs {C.sizeof(DbiParams)}, "
            f"dbi_stats {ss.value} vs {C.sizeof(DbiStats)}"
        )
    if path == LIB_PATH:
        _lib = lib
    return lib


ABI_SYMBOLS = [
    "dbi_default_params", "dbi_params_add_static_mod", "dbi_params_set_enzyme", "dbi_params_add_diff_mod",
    "dbi_create", "dbi_set_stream", "dbi_add_proteins", "dbi_upload", "dbi_reset_index", "dbi_build",
    "dbi_stats_get", "dbi_save", "dbi_load", "dbi_query", "dbi_query_device", "dbi_fetch", "dbi_query_hits", "dbi_query_hits_device", "dbi_query_hits_read",
    "dbi_search_unindexed", "dbi_query_spectra", "dbi_search_unindexed_spectra",
    "dbi_lookup_peptides", "dbi_lookup_peptides_read", "dbi_host_alloc", "dbi_host_free", "dbi_get_protein", "dbi_calculate_mass",
    "dbi_entry_keys", "dbi_debug_emitted", "dbi_build_from_records", "dbi_debug_radix_sort", "dbi_destroy",
    "dbi_abi_sizes", "dbi_release_cached_memory",
    "dbi_last_error", "dbi_kernel_launches",
    "dbi_fasta_open", "dbi_fasta_counts", "dbi_fasta_read", "dbi_fasta_close",
    # sharded build, bound in dbindex_b200/multigpu.py
    "dbi_mg_begin", "dbi_mg_set_shards", "dbi_mg_window_ensure", "dbi_mg_window_import", "dbi_mg_layout_bytes",
    "dbi_mg_side_classes", "dbi_mg_pull_proteome", "dbi_mg_digest", "dbi_mg_hist", "dbi_mg_plan", "dbi_mg_default_cost", "dbi_mg_count", "dbi_mg_scatter",
    "dbi_mg_index_base", "dbi_mg_unique_count", "dbi_mg_set_unique", "dbi_mg_groups", "dbi_mg_index_variants",
    "dbi_mg_finish", "dbi_mg_split_masses", "dbi_mg_slices", "dbi_mg_plan_matrix", "dbi_mg_build_local",
    "dbi_mg_search_unindexed_local", "dbi_mg_spectra_stops", "dbi_mg_query_spectra", "dbi_mg_query_spectra_local",
    "dbi_mg_search_unindexed_spectra_local",
]


def default_params(mono: bool = True, _lib=None, **overrides) -> DbiParams:
    """dbi_default_params + keyword overrides.

    Extra keywords: enzyme="KR", nocut="", static_mods={"C": 57.02146},
    diff_mods=[("M", 15.9949), ("STY", 79.96633)], mandatory_internal="K", peptide_filter=("K", 2)."""
    lib = _lib if _lib is not None else load_library()  # _lib: any library exporting the dbi_params_* helpers
    p = DbiParams()
    lib.dbi_default_params(C.byref(p), 1 if mono else 0)
    enzyme = overrides.pop("enzyme", None)
    nocut = overrides.pop("nocut", None)
    if enzyme is not None or nocut is not None:
        lib.dbi_params_set_enzyme(C.byref(p), (enzyme if enzyme is not None else "KR").encode(), (nocut or "").encode())
    for res, delta in (overrides.pop("static_mods", None) or {}).items():
        lib.dbi_params_add_static_mod(C.byref(p), ord(res), float(delta))
    for residues, delta in overrides.pop("diff_mods", None) or []:
        rc = lib.dbi_params_add_diff_mod(C.byref(p), residues.encode(), float(delta))
        if rc != 0:
            raise DbiError(rc, "too many differential mods")
    mandatory = overrides.pop("mandatory_internal", None)  # sparam.getMandatoryInternalAAs()
    if mandatory is not None:
        p.has_mandatory = 1
        for ch in mandatory:
            p.is_mandatory[ord(ch)] = 1
    pep_filter = overrides.pop("peptide_filter", None)      # PeptideFilterByMaxOccurrencies("K", 2) -> ("K", 2)
    if pep_filter is not None:
        p.filter_aa, p.filter_max = ord(pep_filter[0]), int(pep_filter[1])
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise TypeError(f"unknown dbi_params field {k!r}")
        setattr(p, k, v)
    return p


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def parse_fasta(path: str, threads: int = 0, raw_deflines: bool = False):
    """FASTA file -> (deflines list[str], residues uint8[R], offsets uint64[n + 1]) through the native
    multi-threaded parser (dbi_fasta_*, csrc/fasta.cpp): the packed layout `add_proteins` takes.
    raw_deflines: return the deflines as (bytes buffer uint8[], offsets uint64[n + 1]) instead of strings."""
    lib = load_library()
    f = C.c_void_p()
    rc = lib.dbi_fasta_open(os.fsencode(path), int(threads), C.byref(f))
    if rc != 0:
        raise DbiError(rc, (lib.dbi_last_error() or b"").decode(errors="replace"))
    try:
        n, r, d = C.c_uint32(), C.c_uint64(), C.c_uint64()
        lib.dbi_fasta_counts(f, C.byref(n), C.byref(r), C.byref(d))
        residues = np.empty(r.value, dtype=np.uint8)
        offsets = np.empty(n.value + 1, dtype=np.uint64)
        dbuf = np.empty(d.value, dtype=np.uint8)
        doff = np.empty(n.value + 1, dtype=np.uint64)
        rc = lib.dbi_fasta_read(f, residues.ctypes.data if r.value else None, offsets.ctypes.data,
                                dbuf.ctypes.data if d.value else None, doff.ctypes.data)
        if rc != 0:
            raise DbiError(rc, (lib.dbi_last_error() or b"").decode(errors="replace"))
    finally:
        lib.dbi_fasta_close(f)
    if raw_deflines:
        return (dbuf, doff), residues, offsets
    raw = dbuf.tobytes()
    deflines = [raw[int(doff[i]):int(doff[i + 1])].decode("latin-1") for i in range(n.value)]
    return deflines, residues, offsets


def pack_peptides(seqs):
    """Peptides -> the packed (residues uint8[R], offsets uint64[n + 1]) layout of the C ABI: a list of str / bytes,
    or such a pair already."""
    if isinstance(seqs, tuple) and len(seqs) == 2 and isinstance(seqs[0], np.ndarray):
        return np.ascontiguousarray(seqs[0], dtype=np.uint8), np.ascontiguousarray(seqs[1], dtype=np.uint64)
    bs = [s.encode("latin-1") if isinstance(s, str) else bytes(s) for s in seqs]
    offsets = np.zeros(len(bs) + 1, dtype=np.uint64)
    if bs:
        np.cumsum(np.fromiter((len(b) for b in bs), dtype=np.uint64, count=len(bs)), out=offsets[1:])
    return np.frombuffer(b"".join(bs), dtype=np.uint8), offsets


class GpuIndex:
    """One dbi_handle: a peptide index in the HBM of one GPU."""

    def __init__(self, params: DbiParams):
        self.lib = load_library()
        self.params = params.copy()
        h = C.c_void_p()
        rc = self.lib.dbi_create(C.byref(self.params), C.byref(h))
        self._h = h if rc == 0 else None
        self._check(rc)

    def _check(self, rc: int):
        if rc != 0:
            raise DbiError(rc, (self.lib.dbi_last_error() or b"").decode(errors="replace"))

    def close(self):
        if getattr(self, "_h", None):
            self.lib.dbi_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- build ---------------------------------------------------------------------
    def set_stream(self, cuda_stream_ptr: int):
        self._check(self.lib.dbi_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    def add_proteins(self, residues: np.ndarray, offsets: np.ndarray):
        residues = np.ascontiguousarray(residues, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        self._check(self.lib.dbi_add_proteins(self._h, _ptr(residues), _ptr(offsets), len(offsets) - 1))

    def upload(self):
        self._check(self.lib.dbi_upload(self._h))

    def reset_index(self):
        self._check(self.lib.dbi_reset_index(self._h))

    def build(self):
        self._check(self.lib.dbi_build(self._h))

    def build_from_records(self, mass, prot, off, length):
        mass = np.ascontiguousarray(mass, dtype=np.float64)
        prot = np.ascontiguousarray(prot, dtype=np.uint32)
        off = np.ascontiguousarray(off, dtype=np.uint32)
        length = np.ascontiguousarray(length, dtype=np.uint16)
        self._check(self.lib.dbi_build_from_records(self._h, _ptr(mass), _ptr(prot), _ptr(off), _ptr(length), len(mass)))

    def save(self, path: str):
        self._check(self.lib.dbi_save(self._h, os.fsencode(path)))

    def load(self, path: str):
        self._check(self.lib.dbi_load(self._h, os.fsencode(path)))

    def stats(self) -> dict:
        st = DbiStats()
        self._check(self.lib.dbi_stats_get(self._h, C.byref(st)))
        d = {k: getattr(st, k) for k in ("n_proteins", "n_residues", "n_emitted", "n_unique", "n_entries",
                                         "n_hash_retries", "device_bytes", "sort_bits_base", "sort_bits_var",
                                         "dom_ms", "dom_launches", "dom_bytes_per_launch", "dom_kernel",
                                         "exp_ms", "exp_launches", "exp_bytes_per_launch", "n_groups")}
        d["algo_bytes"] = dict(zip(STAGE_NAMES, list(st.algo_bytes)))
        d["stage_ms"] = dict(zip(STAGE_NAMES, [float(x) for x in st.stage_ms]))
        d["stage_launches"] = dict(zip(STAGE_NAMES, list(st.stage_launches)))
        return d

    # ---- query ---------------------------------------------------------------------
    def query(self, lo: np.ndarray, hi: np.ndarray, out_begin=None, out_count=None):
        lo = np.ascontiguousarray(lo, dtype=np.float64)
        hi = np.ascontiguousarray(hi, dtype=np.float64)
        nq = len(lo)
        begin = out_begin if out_begin is not None else np.empty(nq, dtype=np.uint64)
        count = out_count if out_count is not None else np.empty(nq, dtype=np.uint64)
        self._check(self.lib.dbi_query(self._h, _ptr(lo), _ptr(hi), nq, _ptr(begin), _ptr(count)))
        return begin, count

    def query_device(self, d_lo: int, d_hi: int, nq: int, d_begin: int, d_count: int):
        self._check(self.lib.dbi_query_device(self._h, C.c_void_p(d_lo), C.c_void_p(d_hi), nq,
                                              C.c_void_p(d_begin), C.c_void_p(d_count)))

    def fetch(self, begin: int, count: int, with_ids: bool = True) -> dict:
        count = int(count)
        out = {
            "mass": np.empty(count, dtype=np.float64),
            "first_prot": np.empty(count, dtype=np.uint32),
            "first_off": np.empty(count, dtype=np.uint32),
            "len": np.empty(count, dtype=np.uint16),
            "modpat": np.empty(count, dtype=np.uint32),
            "prot_list_off": np.zeros(count + 1, dtype=np.uint64),
        }
        n_ids = C.c_uint64(0)
        if with_ids:  # sizing call
            self._check(self.lib.dbi_fetch(self._h, int(begin), count, None, None, None, None, None, None, None, 0,
                                           C.byref(n_ids)))
        ids = np.empty(n_ids.value, dtype=np.uint32) if with_ids else None
        self._check(self.lib.dbi_fetch(self._h, int(begin), count, _ptr(out["mass"]), _ptr(out["first_prot"]),
                                       _ptr(out["first_off"]), _ptr(out["len"]), _ptr(out["modpat"]),
                                       _ptr(out["prot_list_off"]), _ptr(ids), n_ids.value, C.byref(n_ids)))
        out["prot_ids"] = ids
        return out

    def query_hits_begin(self, lo: np.ndarray, hi: np.ndarray) -> DbiHitCounts:
        """dbi_query_hits alone (host bounds): the hits stay in HBM until query_hits_read / the next call."""
        lo = np.ascontiguousarray(lo, dtype=np.float64)
        hi = np.ascontiguousarray(hi, dtype=np.float64)
        cnt = DbiHitCounts()
        self._check(self.lib.dbi_query_hits(self._h, _ptr(lo), _ptr(hi), len(lo), C.byref(cnt)))
        return cnt

    def query_hits_device(self, d_lo: int, d_hi: int, nq: int) -> DbiHitCounts:
        """dbi_query_hits_device: bounds resident in HBM; the hits stay in HBM until query_hits_read / the next call."""
        cnt = DbiHitCounts()
        self._check(self.lib.dbi_query_hits_device(self._h, C.c_void_p(d_lo), C.c_void_p(d_hi), nq, C.byref(cnt)))
        return cnt

    def query_hits_read(self, bufs: "DbiHitBuffers"):
        self._check(self.lib.dbi_query_hits_read(self._h, C.byref(bufs)))

    def query_hits(self, lo: np.ndarray, hi: np.ndarray, fields=None, alloc=None, per_hit: bool = True) -> dict:
        """dbi_query_hits + dbi_query_hits_read: every hit of every [lo[i], hi[i]] materialised (mass, first
        occurrence, peptide residues, flanks, mod pattern, protein ids).  per_hit = False returns the buffers as
        the library delivers them (grouped in runs, see HIT_FIELDS); per_hit = True expands them on the host to
        one record per hit.  `fields`: subset to read back (default all); `alloc(name, dtype, n)`: buffer
        factory (e.g. pinned memory), default numpy."""
        lo = np.ascontiguousarray(lo, dtype=np.float64)
        hi = np.ascontiguousarray(hi, dtype=np.float64)
        cnt = DbiHitCounts()
        self._check(self.lib.dbi_query_hits(self._h, _ptr(lo), _ptr(hi), len(lo), C.byref(cnt)))
        return self._read_hits(cnt, fields, alloc, per_hit)

    def search_unindexed_begin(self, lo: np.ndarray, hi: np.ndarray, max_candidates: int = 0) -> DbiHitCounts:
        """dbi_search_unindexed alone: the hits stay in HBM until query_hits_read / the next call.  Raises DbiError
        (code DBI_ERANGE, n_candidates set) when the candidate records exceed max_candidates (0 = no cap)."""
        lo = np.ascontiguousarray(lo, dtype=np.float64)
        hi = np.ascontiguousarray(hi, dtype=np.float64)
        if len(lo) != len(hi):
            raise ValueError(f"{len(lo)} lower and {len(hi)} upper bounds")
        cnt, n_cand = DbiHitCounts(), C.c_uint64(0)
        rc = self.lib.dbi_search_unindexed(self._h, _ptr(lo), _ptr(hi), len(lo), int(max_candidates), C.byref(cnt),
                                           C.byref(n_cand))
        self.last_candidates = n_cand.value
        if rc != 0:
            raise DbiError(rc, (self.lib.dbi_last_error() or b"").decode(errors="replace"), n_cand.value)
        return cnt

    def search_unindexed(self, lo: np.ndarray, hi: np.ndarray, max_candidates: int = 0, fields=None, alloc=None,
                         per_hit: bool = True) -> dict:
        """dbi_search_unindexed + dbi_query_hits_read: what query_hits returns for these ranges, answered from the
        proteins added so far without a built index (the handle stays unbuilt).  The candidate records of the
        call are in self.last_candidates."""
        return self._read_hits(self.search_unindexed_begin(lo, hi, max_candidates), fields, alloc, per_hit)

    def query_spectra(self, mass, tol, range_off=None, tol_mode: int = DBI_TOL_DA, index_factor: int = 0,
                      fields=None, alloc=None, per_hit: bool = True) -> dict:
        """dbi_query_spectra + dbi_query_hits_read: the answer of every spectrum of a batch as one query of a
        query_hits-style dict.  DBI_TOL_DA: spectrum s = the (mass, tol in Da) ranges [range_off[s], range_off[s+1])
        answered as getSequences(List<MassRange>); DBI_TOL_PPM (range_off None): mass[s] at tol[s] ppm answered as
        getSequencesUsingPPMTolerance.  index_factor: the bucket rule of the reference (0 = off)."""
        mass, tol, range_off, n = spectra_arrays(mass, tol, range_off, tol_mode)
        cnt = DbiHitCounts()
        self._check(self.lib.dbi_query_spectra(self._h, _ptr(mass), _ptr(tol), _ptr(range_off), n, int(tol_mode),
                                               int(index_factor), C.byref(cnt)))
        return self._read_hits(cnt, fields, alloc, per_hit)

    def search_unindexed_spectra(self, mass, tol, range_off=None, tol_mode: int = DBI_TOL_DA, index_factor: int = 0,
                                 max_candidates: int = 0, fields=None, alloc=None, per_hit: bool = True) -> dict:
        """dbi_search_unindexed_spectra + dbi_query_hits_read: query_spectra answered from the proteins added so far
        without a built index.  DbiError (DBI_ERANGE, n_candidates set) above max_candidates (0 = no cap); the
        candidate records of the call are in self.last_candidates."""
        mass, tol, range_off, n = spectra_arrays(mass, tol, range_off, tol_mode)
        cnt, n_cand = DbiHitCounts(), C.c_uint64(0)
        rc = self.lib.dbi_search_unindexed_spectra(self._h, _ptr(mass), _ptr(tol), _ptr(range_off), n, int(tol_mode),
                                                   int(index_factor), int(max_candidates), C.byref(cnt),
                                                   C.byref(n_cand))
        self.last_candidates = n_cand.value
        if rc != 0:
            raise DbiError(rc, (self.lib.dbi_last_error() or b"").decode(errors="replace"), n_cand.value)
        return self._read_hits(cnt, fields, alloc, per_hit)

    def mg_spectra_stops(self, mass, ppm, split_mass, rank: int, world: int, index_factor: int = 0) -> np.ndarray:
        """dbi_mg_spectra_stops: K_r of every PPM spectrum (mass[s] at ppm[s]) on this built handle as rank `rank` of
        `world` under the cuts split_mass (world or 2 * world slices): the probe at which this rank's share of the
        walk ends, UINT64_MAX where it cannot end here.  The walk ends at the minimum over the ranks."""
        mass, ppm, _, n = spectra_arrays(mass, ppm, None, DBI_TOL_PPM)
        split = np.ascontiguousarray(split_mass, dtype=np.float64)
        stop = np.zeros(n, dtype=np.uint64)
        self._check(self.lib.dbi_mg_spectra_stops(self._h, _ptr(mass), _ptr(ppm), n, int(index_factor), _ptr(split),
                                                  len(split) + 1, int(rank), int(world), _ptr(stop)))
        return stop

    def mg_query_spectra(self, mass, tol, range_off=None, tol_mode: int = DBI_TOL_DA, index_factor: int = 0,
                         stop=None, fields=None, alloc=None, per_hit: bool = True) -> dict:
        """dbi_mg_query_spectra + dbi_query_hits_read: this rank's share of query_spectra on a sharded index;
        DBI_TOL_PPM needs `stop`, the minimum over the ranks of mg_spectra_stops."""
        mass, tol, range_off, n = spectra_arrays(mass, tol, range_off, tol_mode)
        stop = None if stop is None else np.ascontiguousarray(stop, dtype=np.uint64)
        cnt = DbiHitCounts()
        self._check(self.lib.dbi_mg_query_spectra(self._h, _ptr(mass), _ptr(tol), _ptr(range_off), n, int(tol_mode),
                                                  int(index_factor), _ptr(stop), C.byref(cnt)))
        return self._read_hits(cnt, fields, alloc, per_hit)

    def _read_hits(self, cnt: DbiHitCounts, fields, alloc, per_hit: bool) -> dict:
        out, bufs = {"counts": cnt}, DbiHitBuffers()
        want = None if fields is None else set(fields)
        if want is not None and per_hit:
            want |= {"hit_off", "pep_hit_off"}
            want |= {"seq_off"} if "seq" in want else set()
            want |= {"prot_list_off"} if "prot_ids" in want else set()
        for name, (dt, size) in HIT_FIELDS.items():
            if want is not None and name not in want:
                continue
            a = alloc(name, dt, int(size(cnt))) if alloc else np.empty(int(size(cnt)), dtype=dt)
            out[name] = a
            setattr(bufs, name, a.ctypes.data)
        self._check(self.lib.dbi_query_hits_read(self._h, C.byref(bufs)))
        return expand_hits(out) if per_hit else out

    def lookup_peptides_begin(self, seqs, modpat=None) -> DbiLookupCounts:
        """dbi_lookup_peptides alone: the answer stays in HBM until lookup_peptides_read / the next call."""
        residues, offsets = pack_peptides(seqs)
        pat = None if modpat is None else np.ascontiguousarray(modpat, dtype=np.uint32)
        if pat is not None and len(pat) != len(offsets) - 1:
            raise ValueError(f"{len(pat)} mod patterns for {len(offsets) - 1} peptides")
        cnt = DbiLookupCounts()
        self._check(self.lib.dbi_lookup_peptides(self._h, _ptr(residues), _ptr(offsets), _ptr(pat), len(offsets) - 1,
                                                 C.byref(cnt)))
        return cnt

    def lookup_peptides_read(self, cnt: DbiLookupCounts) -> dict:
        out, bufs = {"counts": cnt}, DbiLookupBuffers()
        for name, (dt, size) in LOOKUP_FIELDS.items():
            out[name] = a = np.empty(int(size(cnt)), dtype=dt)
            setattr(bufs, name, a.ctypes.data)
        self._check(self.lib.dbi_lookup_peptides_read(self._h, C.byref(bufs)))
        return out

    def lookup_peptides(self, seqs, modpat=None) -> dict:
        """dbi_lookup_peptides + dbi_lookup_peptides_read: for every peptide (str / bytes, or a packed
        (residues, offsets) pair) and mod pattern (byte k = position + 1 of the k-th modified residue; None = all
        unmodified) whether the index holds it (status: LOOKUP_ABSENT / _FOUND / _MALFORMED), its mass, index entry,
        first occurrence and protein ids (CSR prot_list_off / prot_ids), as numpy arrays."""
        return self.lookup_peptides_read(self.lookup_peptides_begin(seqs, modpat))

    def entry_keys(self) -> np.ndarray:
        n = C.c_uint64(0)
        self._check(self.lib.dbi_entry_keys(self._h, None, 0, C.byref(n)))
        keys = np.empty(n.value, dtype=np.int32)
        if n.value:
            self._check(self.lib.dbi_entry_keys(self._h, _ptr(keys), n.value, C.byref(n)))
        return keys

    def debug_emitted(self) -> dict:
        n = C.c_uint64(0)
        self._check(self.lib.dbi_debug_emitted(self._h, 0, None, None, None, None, C.byref(n)))
        N = n.value
        out = {"mass": np.empty(N, np.float64), "prot": np.empty(N, np.uint32), "off": np.empty(N, np.uint32),
               "len": np.empty(N, np.uint16)}
        self._check(self.lib.dbi_debug_emitted(self._h, N, _ptr(out["mass"]), _ptr(out["prot"]), _ptr(out["off"]),
                                               _ptr(out["len"]), C.byref(n)))
        return out

    def debug_radix_sort(self, keys: np.ndarray, vals: np.ndarray, begin_bit: int, end_bit: int):
        assert keys.dtype == np.uint64 and vals.dtype == np.uint64 and keys.flags.c_contiguous and vals.flags.c_contiguous
        self._check(self.lib.dbi_debug_radix_sort(self._h, _ptr(keys), _ptr(vals), len(keys), begin_bit, end_bit))

    # ---- host-side helpers -----------------------------------------------------------
    def calculate_mass(self, seq: bytes) -> float:
        m = C.c_double()
        self._check(self.lib.dbi_calculate_mass(self._h, seq, len(seq), C.byref(m)))
        return m.value

    def get_protein(self, pid: int) -> bytes:
        p = C.c_void_p()
        n = C.c_uint64()
        self._check(self.lib.dbi_get_protein(self._h, pid, C.byref(p), C.byref(n)))
        return C.string_at(p, n.value)

    def kernel_launches(self) -> int:
        return int(self.lib.dbi_kernel_launches())
