"""Sharded (multi-GPU) index build and query routing (SURVEY.md 8e): one process per GPU,
torch.distributed for the SMALL collectives only (NCCL on GPUs, gloo on CPU in the tests).

The reference shards its index by mass into `indexFactor` SQLite files
(DBIndexStoreSQLiteMult.java:55-56,215-217) and answers a query from the buckets its range
touches (:333-343).  Here a bucket is a GPU:

  1. every rank is given ITS OWN shard of the FASTA (proteins in rank order, so ids stay global),
     packs it into its place of the global residue buffer (window 0) and pulls the other shards over
     NVLink -- the FASTA crosses PCIe once, not once per GPU;
  2. every rank digests the start positions of its own shard while the other shards arrive (side stream);
  3. exchange 0: key histograms (records, and the groups / variants they will expand to) -> one all-gather -> cuts of
     equal estimated COST (sorting, expansion, expected query hits) -> ONE kernel that partitions the
     records and writes them straight into the owners' arenas (mapped peer memory); rank-ordered arrival
     keeps "first occurrence" global (SURVEY.md Q6);
  4. local sort + merge: every rank owns the unique peptides of its base-mass slice (window 2, mapped by
     the others: a hit whose base peptide lives elsewhere is read through the mapping);
  5. differential mods: every rank lists the variant GROUPS of its own peptides; exchange 1 moves the ones
     whose variant mass crosses a cut (the SAME cuts: most groups stay where their peptide is), with their
     site masks, to the owners of those slices, which sort and expand what they hold;
  6. queries are routed on the host with the splitter masses; a range that straddles a splitter is
     answered by the owners of both slices, exactly like Mult.getSequences walking two buckets.
With differential mods the axis is cut into 2 x world FOLDED slices (slice s on rank s < world ? s :
2 world - 1 - s): the light end is crowded with records, the heavy end with variants, and every rank gets one
slice of each so that the base phase, the variant phase and the search load are all even (dbi_mg_plan).

What crosses torch.distributed: the window-0 descriptors (one all-gather; a second one for the shard sizes
unless the caller passes them); exchange 0 -- ONE all-gather of every rank's three local histograms + window
descriptors (96 KB per rank: every rank derives the global histogram, the cuts and the whole count matrix from
it) and one barrier; exchange 1 -- one all-gather of ~350 bytes per rank (send counts, unique count, window
descriptors) and the barrier (it reuses the cuts of exchange 0); a last barrier before anybody may rebuild.

`ShardEngine` is the device side of one rank.  `GpuShardEngine` drives the C ABI (dbi_mg_*); the tests
plug in a CPU engine so that the orchestration runs under gloo without a GPU.  A host that holds every
handle in ONE process (the Java shim) calls dbi_mg_build_local instead of any of this.
"""
from __future__ import annotations

import os
from typing import Tuple

import numpy as np
import torch
import torch.distributed as dist

MG_BINS = 4096
WIN_PROTEOME, WIN_ARENA, WIN_UNIQUE = 0, 1, 2
DESC_BYTES = 96  # sizeof(dbi_mg_window)


# ---- pure host logic (unit-tested on CPU) -------------------------------------------------------
def pick_splitters(hist: np.ndarray, world: int) -> np.ndarray:
    """Equal-count bin splitters: rank d receives the bins [s[d-1], s[d]).  Bins are never split, so
    equal keys (equal masses) stay on one rank and the merge of equal peptides remains local.
    (Same arithmetic as dbi_mg_plan in capi_mg.inl.)"""
    total = int(hist.sum())
    cum = np.cumsum(hist.astype(np.int64))
    out = np.empty(max(world - 1, 0), dtype=np.uint32)
    for d in range(1, world):
        target = total * d // world
        # first bin boundary at which at least `target` items lie below
        out[d - 1] = int(np.searchsorted(cum, target, side="left")) + 1 if total else 0
    np.minimum(out, len(hist), out=out)
    return np.maximum.accumulate(out) if len(out) else out


def slice_owner(s, n_slices: int, world: int):
    """Rank that holds slice s: slice s itself, or, with 2 * world FOLDED slices, 2 * world - 1 - s for the upper
    half -- every rank holds one light and one heavy slice (mg_slice_owner in kernels.cuh)."""
    s = np.asarray(s)
    return np.where(s < world, s, n_slices - 1 - s)


def plan_exchange(world: int, hist_global: np.ndarray, hist_local: np.ndarray, shift: int, min_mass: float,
                  stage: int = 0, has_mods: bool = False, cost=None, n_slices: int = 0):
    """dbi_mg_plan (host arithmetic of libdbindex_gpu.so, no device needed): (bin splitters [n_slices - 1],
    this rank's send counts, every rank's receive total) from the summed and the own [weighted | plain | groups]
    histograms.  cost = (per item, per estimated group, per unit of weight, per expected hit); None: the
    measured default model of the exchange (dbi_mg_default_cost).  n_slices: world (default) or 2 * world."""
    import ctypes as C
    from .capi import load_library
    lib = load_library()
    lib.dbi_mg_plan.restype = C.c_int
    lib.dbi_mg_plan.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_int] + [C.c_void_p] * 3
    lib.dbi_mg_default_cost.restype = None
    lib.dbi_mg_default_cost.argtypes = [C.c_int, C.c_int, C.c_void_p]
    n_slices = n_slices or world
    c = np.zeros(4, dtype=np.float64)
    if cost is None:
        lib.dbi_mg_default_cost(stage, 1 if has_mods else 0, c.ctypes.data)
    else:
        c[:] = cost
    hg = np.ascontiguousarray(hist_global, dtype=np.uint64)
    hl = np.ascontiguousarray(hist_local, dtype=np.uint64)
    if len(hg) == 2 * MG_BINS:  # no group estimates
        hg = np.concatenate([hg, np.zeros(MG_BINS, np.uint64)])
        hl = np.concatenate([hl, np.zeros(MG_BINS, np.uint64)])
    assert len(hg) == 3 * MG_BINS and len(hl) == 3 * MG_BINS
    split = np.zeros(max(n_slices - 1, 1), dtype=np.uint32)
    send, recv = np.zeros(world, dtype=np.uint64), np.zeros(world, dtype=np.uint64)
    rc = lib.dbi_mg_plan(world, hg.ctypes.data, hl.ctypes.data, int(shift), float(min_mass), c.ctypes.data, int(n_slices),
                         split.ctypes.data, send.ctypes.data, recv.ctypes.data)
    if rc != 0:
        raise RuntimeError((lib.dbi_last_error() or b"").decode(errors="replace"))
    return split[:n_slices - 1].copy(), send, recv


def plan_matrix(world: int, hist_all: np.ndarray, shift: int, min_mass: float, stage: int = 0, has_mods: bool = False,
                cost=None, n_slices: int = 0):
    """dbi_mg_plan_matrix: from EVERY rank's local [weighted | plain | groups] histograms ([world, 3 * MG_BINS]) the
    bin splitters [n_slices - 1] and the whole count matrix [world, world] (row = sender)."""
    import ctypes as C
    from .capi import load_library
    lib = load_library()
    lib.dbi_mg_plan_matrix.restype = C.c_int
    lib.dbi_mg_plan_matrix.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.dbi_mg_default_cost.restype = None
    lib.dbi_mg_default_cost.argtypes = [C.c_int, C.c_int, C.c_void_p]
    n_slices = n_slices or world
    c = np.zeros(4, dtype=np.float64)
    if cost is None:
        lib.dbi_mg_default_cost(stage, 1 if has_mods else 0, c.ctypes.data)
    else:
        c[:] = cost
    ha = np.ascontiguousarray(hist_all, dtype=np.uint64).reshape(world, 3 * MG_BINS)
    split = np.zeros(max(n_slices - 1, 1), dtype=np.uint32)
    matrix = np.zeros((world, world), dtype=np.uint64)
    rc = lib.dbi_mg_plan_matrix(world, ha.ctypes.data, int(shift), float(min_mass), c.ctypes.data, int(n_slices),
                                split.ctypes.data, matrix.ctypes.data)
    if rc != 0:
        raise RuntimeError((lib.dbi_last_error() or b"").decode(errors="replace"))
    return split[:n_slices - 1].copy(), matrix


def splitter_masses(bin_splitters: np.ndarray, shift: int, min_mass: float) -> np.ndarray:
    """The mass at which each splitter sits: radix key = bits(mass) - bits(min_mass)."""
    base = np.float64(min_mass).view(np.uint64)
    keys = (bin_splitters.astype(np.uint64) << np.uint64(shift)) + base
    return keys.view(np.float64)


def route_queries(lo: np.ndarray, hi: np.ndarray, split_mass: np.ndarray, rank: int, world: int) -> np.ndarray:
    """Indices of the queries whose [lo, hi] intersects a slice [split[s-1], split[s]) that `rank` holds.
    len(split_mass) + 1 slices: world of them (slice s on rank s) or 2 * world folded ones (slice_owner)."""
    n_slices = len(split_mass) + 1
    edges = np.concatenate(([-np.inf], np.asarray(split_mass, dtype=np.float64), [np.inf]))
    mine = np.zeros(len(lo), dtype=bool)
    for s in range(n_slices):
        if int(slice_owner(s, n_slices, world)) == rank:
            mine |= (hi >= edges[s]) & (lo < edges[s + 1])
    return np.nonzero(mine)[0]


def owned_mask(masses: np.ndarray, split_mass: np.ndarray, rank: int, world: int) -> np.ndarray:
    """True where an entry of this mass belongs to `rank`: its slice is the number of cuts <= mass."""
    sl = np.searchsorted(np.asarray(split_mass, dtype=np.float64), np.asarray(masses, dtype=np.float64), side="right")
    return slice_owner(sl, len(split_mass) + 1, world) == rank


# ---- tiny collectives ---------------------------------------------------------------------------
def _world() -> int:
    return dist.get_world_size() if dist.is_initialized() else 1


_pinned = [None]  # ONE page-locked staging buffer for every small gather (a pageable D2H of the 768 KB histogram
#                   gather costs ~0.15 ms; allocating pinned memory costs milliseconds, so it happens once)


def _to_host(t: torch.Tensor) -> np.ndarray:
    if t.device.type != "cuda":
        return t.numpy()
    n = t.numel()
    if _pinned[0] is None or _pinned[0].numel() < n:
        _pinned[0] = torch.empty(max(2 * n, 4 << 20), dtype=torch.uint8).pin_memory()
    buf = _pinned[0][:n]
    buf.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return buf.numpy()


def _all_gather_bytes(row, device) -> np.ndarray:
    """Every rank's fixed-size byte row (numpy, or a uint8 tensor already on `device`) on every rank:
    [world, len(row)] (one small all-gather + D2H); the result is only valid until the next call."""
    world = _world()
    t = row if isinstance(row, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(row, dtype=np.uint8)).to(device)
    if world == 1:
        return t.cpu().numpy()[None, :].copy()
    out = torch.empty(world * t.numel(), dtype=torch.uint8, device=device)
    dist.all_gather_into_tensor(out, t.contiguous())
    return _to_host(out).reshape(world, -1)


def _barrier(device):
    """Stream-ordered barrier: work enqueued afterwards runs after every rank has reached this point."""
    if _world() > 1:
        dist.all_reduce(torch.zeros(1, dtype=torch.int32, device=device))


class ShardEngine:
    """Device side of one rank (GpuShardEngine: libdbindex_gpu.so; tests: a CPU model)."""

    device = torch.device("cpu")
    has_mods = False
    min_mass = 0.0

    def begin(self, rank: int, world: int): ...
    def shard_info(self) -> Tuple[int, int]: ...                 # (proteins, residues) of the own shard
    def set_shards(self, shard_proteins, shard_residues) -> np.ndarray: ...   # lays window 0 out; its descriptor
    def window(self, window: int, nbytes: int) -> np.ndarray: ...            # ensure + describe (uint8[96])
    def import_window(self, window: int, rank: int, desc: np.ndarray): ...
    def layout_bytes(self, window: int, stage: int, n_items: int) -> int: ...
    def pull_proteome(self): ...
    def digest(self) -> int: ...
    def hist(self, stage: int) -> Tuple[torch.Tensor, int]: ...   # (int64[3 * MG_BINS] on device, shift)
    def count(self, stage: int, splitters: np.ndarray, n_slices: int) -> np.ndarray: ...   # items per destination under the cuts
    def scatter(self, stage: int, splitters: np.ndarray, n_slices: int, matrix: np.ndarray): ...
    def index_base(self): ...
    def n_unique(self) -> int: ...
    def set_unique(self, rank_unique: np.ndarray): ...
    def groups(self) -> Tuple[int, int]: ...                      # (items that travel, variants)
    def index_variants(self): ...
    def finish(self): ...


def build_sharded(engine: ShardEngine, shard_sizes=None) -> dict:
    """Run the sharded build on this rank.  shard_sizes: (proteins, residues) of EVERY rank's shard, [world, 2], when
    the caller knows them (it cut the FASTA): saves the first all-gather.  Returns routing info: {"split_mass": masses at which the entry
    slices are cut, "unique_off": global id of every rank's first unique peptide, "a2a_bytes": ...}."""
    import time
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist.is_initialized() else (0, 1)
    dev = engine.device
    cuda = dev.type == "cuda"
    info = {"rank": rank, "world": world, "a2a_bytes": 0, "a2a_ms": 0.0, "t": {}}
    t_last = [time.perf_counter()]

    def lap(name):  # host wall-clock per stage (every engine call ends synchronised)
        now = time.perf_counter()
        info["t"][name] = info["t"].get(name, 0.0) + 1e3 * (now - t_last[0])
        t_last[0] = now

    def connect(window: int, descs: np.ndarray):
        for r in range(world):
            if r != rank:
                engine.import_window(window, r, descs[r])

    engine.begin(rank, world)
    # ---- the proteome: own shard over PCIe (already added), the other shards over NVLink
    np_, nr_ = engine.shard_info()
    if shard_sizes is None:
        sizes = _all_gather_bytes(np.array([np_, nr_], dtype=np.uint64).view(np.uint8), dev).copy().view(np.uint64).reshape(world, 2)
    else:
        sizes = np.ascontiguousarray(shard_sizes, dtype=np.uint64).reshape(world, 2)
        assert (int(sizes[rank, 0]), int(sizes[rank, 1])) == (np_, nr_), "shard_sizes disagree with the shard this rank added"
    d0 = engine.set_shards(sizes[:, 0].copy(), sizes[:, 1].copy())
    connect(WIN_PROTEOME, _all_gather_bytes(d0, dev).copy())  # also the barrier: every shard is packed
    engine.pull_proteome()
    lap("proteome")
    engine.digest()
    lap("digest")

    state = {"split": None, "shift": 0}
    # folded slices (one light + one heavy per rank) when differential mods make the phases of a build pull
    # the cuts apart; DBI_MG_FOLD=0 keeps one contiguous slice per rank
    n_slices = 2 * world if (engine.has_mods and world > 1 and os.environ.get("DBI_MG_FOLD", "1") != "0") else world
    info["n_slices"] = n_slices
    # DBI_MG_UNIFIED=0: the variant exchange plans its own cuts (equal cost of the variant work alone; almost
    # every group then leaves its rank).  Default: one set of cuts for the whole index.
    unified = os.environ.get("DBI_MG_UNIFIED", "1") != "0"

    def exchange(stage: int, item_bytes: int):
        """Exchange 0 plans the cuts of the index (local histograms -> one all-gather -> dbi_mg_plan_matrix on every
        rank); exchange 1 reuses them -- a variant lies at most a few shifts above its peptide, so most groups stay
        on the GPU that owns the peptide -- and only needs the counts of the groups that cross a cut."""
        nu = np.array([engine.n_unique()], dtype=np.uint64).view(np.uint8)
        if stage == 0 or not unified:
            # ONE all-gather carries every rank's local histograms and the windows it has: every rank then sums
            # the global histogram, places the same cuts, and knows the whole count matrix and whether anybody's
            # window has to grow (rare after the first build) -- no second collective in the steady state
            hist, shift = engine.hist(stage)
            lap(f"hist{stage}.kernel")
            d1 = engine.window(WIN_ARENA, 0)
            d2 = engine.window(WIN_UNIQUE, 0)
            tail = torch.from_numpy(np.concatenate([nu, d1, d2])).to(dev)
            rows = _all_gather_bytes(torch.cat([hist.view(torch.uint8), tail]), dev)
            hb = 3 * MG_BINS * 8
            hists = rows[:, :hb].copy().view(np.uint64).reshape(world, 3 * MG_BINS)
            lap(f"hist{stage}.gather")
            split, matrix = plan_matrix(world, hists, shift, engine.min_mass, stage, engine.has_mods and unified,
                                        n_slices=n_slices)
            state["split"], state["shift"] = split, shift
            send, recv = matrix[rank], matrix.sum(axis=0, dtype=np.uint64)
            ru = rows[:, hb:hb + 8].copy().view(np.uint64).reshape(world)
            descs = rows[:, hb + 8:].copy()
            lap(f"hist{stage}.plan")
            need_a = [engine.layout_bytes(WIN_ARENA, stage, int(recv[d])) for d in range(world)]
            need_u = [engine.layout_bytes(WIN_UNIQUE, 0, int(recv[d])) if stage == 0 else 0 for d in range(world)]
            cap = lambda d, w: int(descs[d, w * DESC_BYTES + 72:w * DESC_BYTES + 80].copy().view(np.uint64)[0])  # noqa: E731  dbi_mg_window.bytes
            if any(need_a[d] > cap(d, 0) or need_u[d] > cap(d, 1) for d in range(world)):
                d1 = engine.window(WIN_ARENA, need_a[rank])
                d2 = engine.window(WIN_UNIQUE, need_u[rank])
                descs = _all_gather_bytes(np.concatenate([d1, d2]), dev).copy()
                lap(f"plan{stage}.grow")
            arena_desc, uniq_desc = descs[:, :DESC_BYTES], descs[:, DESC_BYTES:2 * DESC_BYTES]
        else:
            split = state["split"]
            send = engine.count(stage, split, n_slices)
            lap(f"count{stage}")
            d1 = engine.window(WIN_ARENA, 0)
            d2 = engine.window(WIN_UNIQUE, 0)
            rows = _all_gather_bytes(np.concatenate([send.view(np.uint8), nu, d1, d2]), dev)  # every rank is past its previous use of the arenas
            lap(f"plan{stage}.gather")
            matrix = rows[:, :8 * world].copy().view(np.uint64).reshape(world, world)
            ru = rows[:, 8 * world:8 * world + 8].copy().view(np.uint64).reshape(world)
            o = 8 * world + 8
            arena_desc, uniq_desc = rows[:, o:o + DESC_BYTES].copy(), rows[:, o + DESC_BYTES:o + 2 * DESC_BYTES].copy()
            # the arenas were sized before the receive totals were known: every rank sees the same matrix and
            # the same capacities, so all agree on whether somebody has to grow (rare after the first build)
            need = [engine.layout_bytes(WIN_ARENA, stage, int(matrix[:, d].sum())) for d in range(world)]
            caps = [int(arena_desc[d, 72:80].copy().view(np.uint64)[0]) for d in range(world)]  # dbi_mg_window.bytes
            if any(n > c for n, c in zip(need, caps)):
                d1 = engine.window(WIN_ARENA, need[rank])
                arena_desc = _all_gather_bytes(d1, dev).copy()
                lap(f"plan{stage}.grow")
        info[f"recv{stage}"] = int(matrix[:, rank].sum())  # items this rank holds after the exchange
        connect(WIN_ARENA, arena_desc)
        connect(WIN_UNIQUE, uniq_desc)
        if stage == 1:
            engine.set_unique(ru)
        lap(f"plan{stage}")
        if cuda:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        engine.scatter(stage, split, n_slices, matrix)
        if cuda:
            e1.record()
            e1.synchronize()
            info["a2a_ms"] += e0.elapsed_time(e1)
        lap(f"scatter{stage}.kernel")
        _barrier(dev)  # every rank's stores into this rank's arena are complete
        info["a2a_bytes"] += int(send.sum() - send[rank]) * item_bytes
        lap(f"scatter{stage}")
        return split, state["shift"]

    base_split, shift = exchange(0, 18)
    engine.index_base()
    lap("index_base")
    if not engine.has_mods:
        ru = _all_gather_bytes(np.array([engine.n_unique()], dtype=np.uint64).view(np.uint8), dev).copy().view(np.uint64).reshape(world)
        engine.set_unique(ru)
        engine.finish()
        _barrier(dev)
        info["unique_off"] = np.concatenate(([0], np.cumsum(ru))).astype(np.int64)
        info["n_unique"] = int(ru.sum())
        info["split_mass"] = splitter_masses(base_split, shift, engine.min_mass)
        lap("finish")
        return info
    # every rank lists the groups of its own peptides: that work is small and nearly even; the
    # expensive part (sort + expansion) is balanced by the variant-weighted splitters
    engine.groups()
    lap("groups")
    var_split, shift = exchange(1, engine.group_bytes())
    engine.index_variants()
    engine.finish()
    _barrier(dev)  # nobody frees or rebuilds its windows while another rank may still read them
    lap("index_variants")
    ru = engine.rank_unique
    info["unique_off"] = np.concatenate(([0], np.cumsum(ru))).astype(np.int64)
    info["n_unique"] = int(ru.sum())
    info["split_mass"] = splitter_masses(var_split, shift, engine.min_mass)
    return info


# ---- the GPU engine ---------------------------------------------------------------------------
class GpuShardEngine(ShardEngine):
    """Drives libdbindex_gpu.so's dbi_mg_* entry points for one rank.  `index` is a
    dbindex_b200.GpuIndex that was given THIS RANK'S shard of the proteins."""

    def __init__(self, index, device: torch.device):
        import ctypes as C
        self.C = C
        self.g = index
        self.lib = index.lib
        self.device = device
        p = index.params
        self.has_mods = p.n_mods > 0 and p.max_mods_per_peptide > 0
        self.min_mass = float(p.min_mass)
        self.rank_unique = None
        vp, u64p = C.c_void_p, C.POINTER(C.c_uint64)
        sig = {
            "dbi_mg_begin": (C.c_int, [vp, C.c_int, C.c_int]),
            "dbi_mg_set_shards": (C.c_int, [vp, vp, vp, u64p]),
            "dbi_mg_window_ensure": (C.c_int, [vp, C.c_int, C.c_uint64, vp]),
            "dbi_mg_window_import": (C.c_int, [vp, C.c_int, C.c_int, vp]),
            "dbi_mg_layout_bytes": (C.c_uint64, [C.c_int, C.c_int, C.c_uint64, C.c_int]),
            "dbi_mg_side_classes": (C.c_int, [vp]),
            "dbi_mg_pull_proteome": (C.c_int, [vp]),
            "dbi_mg_digest": (C.c_int, [vp, u64p]),
            "dbi_mg_hist": (C.c_int, [vp, C.c_int, vp, C.POINTER(C.c_int)]),
            "dbi_mg_count": (C.c_int, [vp, C.c_int, vp, C.c_int, vp]),
            "dbi_mg_scatter": (C.c_int, [vp, C.c_int, vp, C.c_int, vp]),
            "dbi_mg_index_base": (C.c_int, [vp]),
            "dbi_mg_unique_count": (C.c_int, [vp, u64p]),
            "dbi_mg_set_unique": (C.c_int, [vp, vp]),
            "dbi_mg_groups": (C.c_int, [vp, u64p, u64p]),
            "dbi_mg_index_variants": (C.c_int, [vp]),
            "dbi_mg_finish": (C.c_int, [vp]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(self.lib, name)
            fn.restype = res
            fn.argtypes = args
        self.side_classes = self.lib.dbi_mg_side_classes(self.g._h)

    def _ck(self, rc):
        self.g._check(rc)

    def begin(self, rank, world):
        self.rank, self.world = rank, world
        self._ck(self.lib.dbi_mg_begin(self.g._h, rank, world))

    def shard_info(self):
        st = self.g.stats()
        return st["n_proteins"], st["n_residues"]

    def window(self, window, nbytes):
        d = np.zeros(DESC_BYTES, dtype=np.uint8)
        self._ck(self.lib.dbi_mg_window_ensure(self.g._h, window, int(nbytes), d.ctypes.data))
        return d

    def import_window(self, window, rank, desc):
        d = np.ascontiguousarray(desc, dtype=np.uint8)
        self._ck(self.lib.dbi_mg_window_import(self.g._h, window, rank, d.ctypes.data))

    def layout_bytes(self, window, stage, n_items):
        return int(self.lib.dbi_mg_layout_bytes(window, stage, int(n_items), self.side_classes))

    def group_bytes(self):
        return 20 + 8 * self.side_classes if self.side_classes else 16

    def set_shards(self, shard_proteins, shard_residues):
        sp = np.ascontiguousarray(shard_proteins, dtype=np.uint64)
        sr = np.ascontiguousarray(shard_residues, dtype=np.uint64)
        need = self.C.c_uint64()
        self._ck(self.lib.dbi_mg_set_shards(self.g._h, sp.ctypes.data, sr.ctypes.data, self.C.byref(need)))
        d = self.window(WIN_PROTEOME, need.value)
        self._ck(self.lib.dbi_mg_set_shards(self.g._h, sp.ctypes.data, sr.ctypes.data, None))
        return d

    def pull_proteome(self):
        self._ck(self.lib.dbi_mg_pull_proteome(self.g._h))

    def digest(self):
        n = self.C.c_uint64()
        self._ck(self.lib.dbi_mg_digest(self.g._h, self.C.byref(n)))
        return n.value

    def hist(self, stage):
        hist = torch.zeros(3 * MG_BINS, dtype=torch.int64, device=self.device)
        shift = self.C.c_int()
        torch.cuda.current_stream().synchronize()
        self._ck(self.lib.dbi_mg_hist(self.g._h, stage, hist.data_ptr(), self.C.byref(shift)))
        return hist, shift.value

    def count(self, stage, splitters, n_slices):
        sp = np.ascontiguousarray(splitters, dtype=np.uint32)
        out = np.zeros(self.world, dtype=np.uint64)
        self._ck(self.lib.dbi_mg_count(self.g._h, stage, sp.ctypes.data if len(sp) else None, int(n_slices), out.ctypes.data))
        return out

    def scatter(self, stage, splitters, n_slices, matrix):
        sp = np.ascontiguousarray(splitters, dtype=np.uint32)
        m = np.ascontiguousarray(matrix, dtype=np.uint64)
        self._ck(self.lib.dbi_mg_scatter(self.g._h, stage, sp.ctypes.data if len(sp) else None, int(n_slices), m.ctypes.data))

    def index_base(self):
        torch.cuda.current_stream().synchronize()
        self._ck(self.lib.dbi_mg_index_base(self.g._h))

    def n_unique(self):
        u = self.C.c_uint64()
        self._ck(self.lib.dbi_mg_unique_count(self.g._h, self.C.byref(u)))
        return u.value

    def set_unique(self, rank_unique):
        ru = np.ascontiguousarray(rank_unique, dtype=np.uint64)
        self.rank_unique = ru
        self._ck(self.lib.dbi_mg_set_unique(self.g._h, ru.ctypes.data))

    def groups(self):
        n, v = self.C.c_uint64(), self.C.c_uint64()
        self._ck(self.lib.dbi_mg_groups(self.g._h, self.C.byref(n), self.C.byref(v)))
        return n.value, v.value

    def index_variants(self):
        torch.cuda.current_stream().synchronize()
        self._ck(self.lib.dbi_mg_index_variants(self.g._h))

    def finish(self):
        self._ck(self.lib.dbi_mg_finish(self.g._h))


def shard_proteins(residues: np.ndarray, offsets: np.ndarray, rank: int, world: int):
    """Rank's contiguous share of a proteome, balanced by residues: (residues, offsets, first protein id)."""
    n = len(offsets) - 1
    total = int(offsets[-1])
    cuts = [int(np.searchsorted(offsets, total * r // world, side="left")) for r in range(world)] + [n]
    cuts[0] = 0
    cuts = np.minimum(np.maximum.accumulate(cuts), n)
    p0, p1 = int(cuts[rank]), int(cuts[rank + 1])
    off = offsets[p0:p1 + 1] - offsets[p0]
    return residues[int(offsets[p0]):int(offsets[p1])], off.astype(np.uint64), p0


def shard_sizes(offsets: np.ndarray, world: int) -> np.ndarray:
    """(proteins, residues) of every rank's shard under shard_proteins: [world, 2] for build_sharded(shard_sizes=)."""
    n = len(offsets) - 1
    total = int(offsets[-1])
    cuts = [int(np.searchsorted(offsets, total * r // world, side="left")) for r in range(world)] + [n]
    cuts[0] = 0
    cuts = np.minimum(np.maximum.accumulate(cuts), n)
    out = np.zeros((world, 2), dtype=np.uint64)
    for r in range(world):
        out[r] = (cuts[r + 1] - cuts[r], int(offsets[cuts[r + 1]]) - int(offsets[cuts[r]]))
    return out


def build_local(indexes) -> None:
    """dbi_mg_build_local: the whole sharded build when this process holds every handle (`indexes[r]` was
    given shard r).  Same kernels as build_sharded; the small collectives are plain host code."""
    import ctypes as C
    lib = indexes[0].lib
    lib.dbi_mg_build_local.restype = C.c_int
    lib.dbi_mg_build_local.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    arr = (C.c_void_p * len(indexes))(*[g._h for g in indexes])
    indexes[0]._check(lib.dbi_mg_build_local(arr, len(indexes)))


def split_masses(index, world: int) -> np.ndarray:
    """Masses at which the slices of a built sharded index are cut (dbi_mg_slices - 1 values)."""
    import ctypes as C
    lib = index.lib
    lib.dbi_mg_split_masses.restype = C.c_int
    lib.dbi_mg_split_masses.argtypes = [C.c_void_p, C.c_void_p]
    lib.dbi_mg_slices.restype = C.c_int
    lib.dbi_mg_slices.argtypes = [C.c_void_p]
    n = int(lib.dbi_mg_slices(index._h))
    out = np.zeros(max(n - 1, 0), dtype=np.float64)
    index._check(lib.dbi_mg_split_masses(index._h, out.ctypes.data if n > 1 else None))
    return out


def lookup_local(handles, seqs, modpat=None) -> dict:
    """dbi_lookup_peptides on a sharded index whose handles all live in this process: every rank gets the whole
    batch (the mass that decides ownership is computed on the device) and the answers are merged.  A row is found
    on at most one rank, the owner of the slice holding its mass; anything else raises.  Returns the arrays of
    GpuIndex.lookup_peptides, `entry` being an entry of rank `rank` (-1 where nothing was found)."""
    from .capi import LOOKUP_FOUND, pack_peptides
    packed = pack_peptides(seqs)
    world = len(handles)
    split = split_masses(handles[0], world)
    parts = [g.lookup_peptides(packed, modpat) for g in handles]
    n = len(packed[1]) - 1
    rank = np.full(n, -1, dtype=np.int32)
    for r, p in enumerate(parts):
        found = p["status"] == LOOKUP_FOUND
        if np.any(found & (rank >= 0)):
            raise RuntimeError(f"rows {np.nonzero(found & (rank >= 0))[0][:8].tolist()} found on two ranks")
        if not np.all(owned_mask(p["mass"][found], split, r, world)):
            raise RuntimeError(f"rank {r} found rows whose mass lies outside its slices")
        rank[found] = r
    first = parts[0]
    for p in parts[1:]:
        if not (np.array_equal(p["status"] == 2, first["status"] == 2) and np.array_equal(p["mass"], first["mass"])):
            raise RuntimeError("the ranks disagree on the masses or the malformed rows of the batch")
    out = {k: first[k].copy() for k in ("status", "mass", "entry", "first_prot", "first_off")}
    sizes = np.zeros(n, dtype=np.int64)
    ids = [np.zeros(0, np.uint32)] * n
    for r, p in enumerate(parts):
        sel = np.nonzero(rank == r)[0]
        plo = p["prot_list_off"].astype(np.int64)
        for k in ("status", "entry", "first_prot", "first_off"):
            out[k][sel] = p[k][sel]
        sizes[sel] = plo[sel + 1] - plo[sel]
        for i in sel:
            ids[i] = p["prot_ids"][plo[i]:plo[i + 1]]
    out["rank"] = rank
    out["prot_list_off"] = np.concatenate(([0], np.cumsum(sizes))).astype(np.uint64)
    out["prot_ids"] = np.concatenate(ids) if n else np.zeros(0, np.uint32)
    return out


def search_unindexed_local(handles, lo, hi, max_candidates: int = 0) -> dict:
    """dbi_mg_search_unindexed_local: dbi_search_unindexed over a proteome sharded over `handles` of this process
    (`handles[r]` was given shard r, as for build_local).  Returns one query_hits-style answer (one record per hit)
    for the ranges [lo[i], hi[i]], the ranks' hits of every query concatenated, and under "n_candidates" the
    candidate records every rank indexed.  DBI_ERANGE (a rank over max_candidates, 0 = no cap) raises DbiError with
    n_candidates = the largest per-rank count and the per-rank counts in its `rank_candidates`."""
    import ctypes as C
    from .capi import DbiError, DbiHitCounts
    from .indexer import _merge_hits
    lib = handles[0].lib
    lib.dbi_mg_search_unindexed_local.restype = C.c_int
    lib.dbi_mg_search_unindexed_local.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_void_p, C.c_uint64,
                                                  C.c_uint64, C.POINTER(DbiHitCounts), C.c_void_p]
    lo = np.ascontiguousarray(lo, dtype=np.float64)
    hi = np.ascontiguousarray(hi, dtype=np.float64)
    if len(lo) != len(hi):
        raise ValueError(f"{len(lo)} lower and {len(hi)} upper bounds")
    n = len(handles)
    arr = (C.c_void_p * n)(*[g._h for g in handles])
    counts = (DbiHitCounts * n)()
    n_cand = np.zeros(n, dtype=np.uint64)
    rc = lib.dbi_mg_search_unindexed_local(arr, n, lo.ctypes.data, hi.ctypes.data, len(lo), int(max_candidates),
                                           counts, n_cand.ctypes.data)
    if rc != 0:
        err = DbiError(rc, (lib.dbi_last_error() or b"").decode(errors="replace"), int(n_cand.max()))
        err.rank_candidates = n_cand
        raise err
    q = np.arange(len(lo), dtype=np.int64)
    out = _merge_hits([(q, g._read_hits(counts[r], None, None, True)) for r, g in enumerate(handles)], len(lo))
    out["n_candidates"] = n_cand
    return out


def _handles_arg(handles):
    import ctypes as C
    return (C.c_void_p * max(len(handles), 1))(*[g._h for g in handles])


def query_spectra_local(handles, mass, tol, range_off=None, tol_mode: int = 0, index_factor: int = 0) -> dict:
    """dbi_mg_query_spectra_local: GpuIndex.query_spectra on a built sharded index whose handles all live in this
    process (`handles[r]` is rank r, as build_local left them).  Returns one query_hits-style answer (one record per
    hit, one query per spectrum), the ranks' hits of every spectrum concatenated."""
    import ctypes as C
    from .capi import DbiError, DbiHitCounts, _ptr, spectra_arrays
    from .indexer import _merge_hits
    lib = handles[0].lib
    lib.dbi_mg_query_spectra_local.restype = C.c_int
    lib.dbi_mg_query_spectra_local.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64,
                                               C.c_int, C.c_int, C.POINTER(DbiHitCounts)]
    mass, tol, range_off, ns = spectra_arrays(mass, tol, range_off, tol_mode)
    n = len(handles)
    counts = (DbiHitCounts * n)()
    rc = lib.dbi_mg_query_spectra_local(_handles_arg(handles), n, _ptr(mass), _ptr(tol), _ptr(range_off), ns,
                                        int(tol_mode), int(index_factor), counts)
    if rc != 0:
        raise DbiError(rc, (lib.dbi_last_error() or b"").decode(errors="replace"))
    q = np.arange(ns, dtype=np.int64)
    return _merge_hits([(q, g._read_hits(counts[r], None, None, True)) for r, g in enumerate(handles)], ns)


def search_unindexed_spectra_local(handles, mass, tol, range_off=None, tol_mode: int = 0, index_factor: int = 0,
                                   max_candidates: int = 0) -> dict:
    """dbi_mg_search_unindexed_spectra_local: GpuIndex.search_unindexed_spectra over a proteome sharded over
    `handles` of this process (as for search_unindexed_local).  Returns one query_hits-style answer (one query per
    spectrum) and under "n_candidates" the candidate records of every rank.  DBI_ERANGE (a rank over max_candidates,
    0 = no cap) raises DbiError with n_candidates = the largest per-rank count and the per-rank counts in its
    `rank_candidates`."""
    import ctypes as C
    from .capi import DbiError, DbiHitCounts, _ptr, spectra_arrays
    from .indexer import _merge_hits
    lib = handles[0].lib
    lib.dbi_mg_search_unindexed_spectra_local.restype = C.c_int
    lib.dbi_mg_search_unindexed_spectra_local.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                          C.c_uint64, C.c_int, C.c_int, C.c_uint64,
                                                          C.POINTER(DbiHitCounts), C.c_void_p]
    mass, tol, range_off, ns = spectra_arrays(mass, tol, range_off, tol_mode)
    n = len(handles)
    counts = (DbiHitCounts * n)()
    n_cand = np.zeros(n, dtype=np.uint64)
    rc = lib.dbi_mg_search_unindexed_spectra_local(_handles_arg(handles), n, _ptr(mass), _ptr(tol), _ptr(range_off),
                                                   ns, int(tol_mode), int(index_factor), int(max_candidates), counts,
                                                   n_cand.ctypes.data)
    if rc != 0:
        err = DbiError(rc, (lib.dbi_last_error() or b"").decode(errors="replace"), int(n_cand.max()))
        err.rank_candidates = n_cand
        raise err
    q = np.arange(ns, dtype=np.int64)
    out = _merge_hits([(q, g._read_hits(counts[r], None, None, True)) for r, g in enumerate(handles)], ns)
    out["n_candidates"] = n_cand
    return out


class ShardedSearcher:
    """The handles of a sharded proteome in this process as one unindexed searcher.  search_unindexed and
    search_unindexed_spectra have the signatures of GpuIndex's, so indexer.search_unindexed_chunked and
    search_unindexed_spectra_chunked split sharded batches unchanged: their ceil(N_c / cap) + 1 rule acts on the
    largest per-rank count, and every call plans its cuts again."""

    def __init__(self, handles):
        self.handles = list(handles)

    def search_unindexed(self, lo, hi, max_candidates: int = 0) -> dict:
        return search_unindexed_local(self.handles, lo, hi, max_candidates)

    def search_unindexed_spectra(self, mass, tol, range_off=None, tol_mode: int = 0, index_factor: int = 0,
                                 max_candidates: int = 0) -> dict:
        return search_unindexed_spectra_local(self.handles, mass, tol, range_off, tol_mode, index_factor,
                                              max_candidates)
