"""Host-side mirror of the reference's indexer / search API over the C ABI.

Same names, argument meaning and error behaviour as the Java classes, so that a
user of ``DBIndexImpl`` / ``DBIndexer`` finds the calls they know:

* ``DBIndexer``   -- DBIndexer.java (init / run / getSequencesUsing*Tolerance /
  getSequences(ranges) / getProteins)
* ``DBIndexImpl`` -- DBIndexImpl.java, the ``DBIndexInterface`` facade
  (getSequences(mass, tol), getSequences(ranges), getProteins, getIndexedProteinById,
  getProteinSequenceById)

Only string assembly happens here (peptide substrings, flanking residues); all
digestion, sorting, merging and searching runs in libdbindex_gpu.so.  The Java shim
under ``java/`` is the same logic in the reference's own language (INTEGRATION.md).
"""
from __future__ import annotations

import os
import threading
from dataclasses import dataclass
from typing import List, Optional, Sequence, Set, Tuple

import numpy as np

from .capi import (DBI_ERANGE, DBI_TOL_DA, DBI_TOL_PPM, DbiError, DbiHitCounts, DbiParams, GpuIndex, _expand_csr,
                   parse_fasta)

MAX_INDEX_RESIDUE_LEN = 3      # Constants.java:44
MAX_PRECURSOR_MASS = 8000      # Constants.java:20
PRECISION = 1e-6               # Constants.java:50
ONE_MILLION = 1000000.0


class DBIndexStoreException(Exception):
    """edu.scripps.yates.utilities.fasta.dbindex.DBIndexStoreException"""


class DBIndexerException(Exception):
    """DBIndexerException.java:9-18"""


@dataclass
class MassRange:
    precMass: float
    tolerance: float


@dataclass(frozen=True)
class IndexedProtein:
    accession: str
    id: int


@dataclass
class IndexedSequence:
    """What parseAddPeptideInfo builds per hit (DBIndexStoreSQLiteByteIndexMerge.java:452-462):
    IndexedSequence(0, mass, sequence, "", "") + setProteinIds + setResidues.  ``sequenceOffset``
    and ``modPositions`` are the superset north_star asks for (SURVEY.md Q10)."""

    mass: float
    sequence: str
    proteinIds: List[int]
    resLeft: str = ""
    resRight: str = ""
    sequenceOffset: int = -1
    sequenceLen: int = 0
    modPositions: Tuple[int, ...] = ()
    id: int = 0

    def key(self):
        return (np.float64(self.mass).view(np.uint64).item(), self.sequence, self.modPositions)


def get_residues(seq_offset: int, seq_len: int, protein_sequence: str) -> Tuple[str, str]:
    """Util.getResidues (Util.java:130-162), right flank off-by-one kept (SURVEY.md Q8)."""
    prot_len = len(protein_sequence)
    left_i = seq_offset - MAX_INDEX_RESIDUE_LEN if seq_offset >= MAX_INDEX_RESIDUE_LEN else 0
    left_len = min(MAX_INDEX_RESIDUE_LEN, seq_offset)
    left = protein_sequence[left_i:left_i + left_len]
    end = seq_offset + seq_len
    right_len = min(MAX_INDEX_RESIDUE_LEN, prot_len - end - 1)
    right = protein_sequence[end:end + right_len] if (end < prot_len and right_len > 0) else ""
    return left.rjust(MAX_INDEX_RESIDUE_LEN, "-"), right.ljust(MAX_INDEX_RESIDUE_LEN, "-")


def tolerance_in_dalton(actual_mass: float, ppm: float) -> float:
    """IndexUtil.getToleranceInDalton (util/IndexUtil.java:238-240)."""
    return actual_mass * (1 - 1 / (ppm / ONE_MILLION + 1))


def merge_intervals(ranges: Sequence[MassRange]) -> List[Tuple[float, float]]:
    """Interval.massRangeToInterval (Interval.java:27-38) + MergeIntervals.mergeIntervals
    (MergeIntervals.java:16-46)."""
    iv = []
    for r in ranges:
        lo = r.precMass - r.tolerance
        if lo < 0.0:
            lo = 0.0
        iv.append((lo, r.precMass + r.tolerance))
    if len(iv) < 2:
        return iv
    iv.sort(key=lambda t: t[0])  # stable, by start
    out = []
    start, end = iv[0]
    for s, e in iv[1:]:
        if end >= s:
            end = max(end, e)
        else:
            out.append((start, end))
            start, end = s, e
    out.append((start, end))
    return out


def read_fasta(path: str) -> Tuple[List[str], np.ndarray, np.ndarray]:
    """FASTA -> (deflines, residues, offsets) through the native multi-threaded parser
    (capi.parse_fasta; the reference uses the external FastaReader, DBIndexer.java:560-571)."""
    return parse_fasta(path)


# resources/dbindex.properties:3-26, restated (the file itself is configuration of the reference)
DBINDEX_PROPERTIES = {
    "default_index_type": "INDEX_NORMAL", "default_in_memory_index": True, "default_index_factor": 8,
    "default_max_internal_cleavages": 6, "default_max_precursor_mass": 6000.0, "default_min_precursor_mass": 500.0,
    "default_use_index": True, "default_enzyme_nocut_residues": "", "default_enzyme_residues": "KR",
    "default_enzyme_offset": 0, "default_mass_type_parent": "1", "mass_group_factor": 10000,
    "add_h2o_plus_proton": True, "mandatory_internal_AAs": "K", "default_semicleavage": False,
}


@dataclass
class DBIndexSearchParams:
    """io/DBIndexSearchParamsImpl.java:46-75 -- the programmatic parameter object: the kernel-facing
    part is `params` (dbi_params), the rest is what the facade needs."""
    params: DbiParams
    dataBaseName: str
    indexFactor: int = 8
    inMemoryIndex: bool = True
    useIndex: bool = True
    indexType: str = "INDEX_NORMAL"
    enzymeOffset: int = 0          # never reaches the Enzyme (SearchParams.java:303); only named the index file
    useMonoParent: bool = False
    mandatoryInternalAAs: Optional[str] = None
    discardDecoyRegexp: Optional[str] = None
    staticParams: str = ""         # SearchParams.getStaticParams(): text of the static mods, part of the index name

    def key(self) -> str:
        """What getByParam keys its registry on (DBIndexImpl.java:44-49: the full index file name, i.e.
        the database plus every parameter that shapes the index, IndexUtil.java:276-323)."""
        p = self.params
        enz = "".join(chr(i) for i in range(256) if p.is_enzyme[i])
        nocut = "".join(chr(i) for i in range(256) if p.is_nocut[i])
        mods = ",".join(f"{chr(p.mods[i].residue)}{p.mods[i].delta!r}" for i in range(p.n_mods))
        statics = ",".join(f"{i}:{p.residue_mass[i]!r}" for i in range(256) if p.residue_mass[i])
        return "|".join(str(x) for x in (
            self.dataBaseName, self.indexFactor, p.max_missed, p.min_mass, p.max_mass, enz, nocut, self.enzymeOffset,
            self.useMonoParent, p.add_h2o_proton, p.mass_group_factor, p.semi, p.min_len, self.mandatoryInternalAAs,
            self.discardDecoyRegexp, p.max_mods_per_peptide, mods, statics))


def getDefaultDBIndexParams(fastaFilePath, inMemoryIndex: Optional[bool] = None, use_mono: Optional[bool] = None,
                            **overrides) -> DBIndexSearchParams:
    """DBIndexImpl.getDefaultDBIndexParams(File | String [, boolean inMemoryIndex]) (DBIndexImpl.java:243-332):
    the defaults of dbindex.properties -- KR, no no-cut residues, 6 missed cleavages, 500-6000 Da, full
    specificity, H2O + proton added, factor 10000, index factor 8.

    Mass type: the reference reads `default_mass_type_parent=1` with `Boolean.valueOf("1")`, which is
    false, so this factory builds an AVERAGE-mass index (DBIndexImpl.java:281-282; only the proteoform
    factory compares with "1", :407-409).  use_mono=None reproduces that; pass True for monoisotopic."""
    from .capi import default_params
    pr = DBINDEX_PROPERTIES
    mono = bool(use_mono) if use_mono is not None else False
    kw = dict(enzyme=pr["default_enzyme_residues"], nocut=pr["default_enzyme_nocut_residues"],
              max_missed=pr["default_max_internal_cleavages"], min_mass=pr["default_min_precursor_mass"],
              max_mass=pr["default_max_precursor_mass"], mass_group_factor=pr["mass_group_factor"],
              add_h2o_proton=1 if pr["add_h2o_plus_proton"] else 0, semi=1 if pr["default_semicleavage"] else 0)
    kw.update(overrides)
    return DBIndexSearchParams(
        params=default_params(mono=mono, **kw), dataBaseName=os.fspath(fastaFilePath),
        indexFactor=pr["default_index_factor"],
        inMemoryIndex=pr["default_in_memory_index"] if inMemoryIndex is None else bool(inMemoryIndex),
        useIndex=pr["default_use_index"], indexType=pr["default_index_type"],
        enzymeOffset=pr["default_enzyme_offset"], useMonoParent=mono)


def getDefaultDBIndexParamsForCrosslinkerAnalysis(fastaFilePath, inMemoryIndex: Optional[bool] = None,
                                                  use_mono: Optional[bool] = None, **overrides) -> DBIndexSearchParams:
    """DBIndexImpl.getDefaultDBIndexParamsForCrosslinkerAnalysis (DBIndexImpl.java:342-372,443-491): the
    dbindex.properties defaults, but H2O + proton is NOT added to the peptide masses (:473) and every indexed
    peptide needs one of `mandatory_internal_AAs` (= "K") as an internal residue (:477-478; semantics
    DBIndexer.java:334-344 and DBIndexStoreSQLiteMult.java:245-263, applied by the digestion kernels)."""
    kw = dict(add_h2o_proton=0, mandatory_internal=DBINDEX_PROPERTIES["mandatory_internal_AAs"])
    kw.update(overrides)
    sp = getDefaultDBIndexParams(fastaFilePath, inMemoryIndex, use_mono, **kw)
    sp.mandatoryInternalAAs = kw["mandatory_internal"]
    return sp


def getDefaultDBIndexParamsForProteoformAnalysis(*args, **kwargs):
    """DBIndexImpl.java:392-432: needs UniProt annotations and proteoform FASTA expansion -- out of scope."""
    raise DBIndexerException("proteoform analysis needs the UniProt annotation service; out of scope of the GPU index")


def createFullIndexFileName(sparam: "DBIndexSearchParams") -> str:
    """IndexUtil.createFullIndexFileName (util/IndexUtil.java:242-324): <database>_<md5 of the parameters that
    shape the index>, the same fields in the same order and spelling.  Two things cannot be reproduced
    byte for byte and are documented deviations: the reference appends `char[].toString()` of
    mandatoryInternalAAs (a JVM identity hash, different on every run) -- the characters themselves are used
    here -- and it knows no differential mods: they are appended only when present, so indexes without them
    keep the reference's key."""
    import hashlib
    p = sparam.params

    def jbool(b):
        return "true" if b else "false"

    def jdouble(x):  # Double.toString for the magnitudes that occur here
        return repr(float(x))

    enz = "".join(chr(i) for i in range(256) if p.is_enzyme[i])
    nocut = "".join(chr(i) for i in range(256) if p.is_nocut[i])
    u = "enzymeOffset:%d" % sparam.enzymeOffset
    u += ", enzymeResidues:" + enz
    u += ", enzymeNoCutResidues:" + nocut
    u += ", maxCleavages:%d" % p.max_missed
    u += ", minPrecursorMass:" + jdouble(p.min_mass)
    u += ", maxPrecursorMass:" + jdouble(p.max_mass)
    u += ", static:" + sparam.staticParams
    u += ", semiCleave:" + jbool(p.semi)
    if p.filter_aa > 0:
        u += ", pepFilter:%s%d" % (chr(p.filter_aa), p.filter_max)  # PeptideFilterByMaxOccurrencies.toString
    u += ", isH2OPlusProtonAdded:" + jbool(p.add_h2o_proton)
    u += ", massGroupFactor:%d" % p.mass_group_factor
    u += ", massType:" + jbool(sparam.useMonoParent)
    if p.has_mandatory:
        u += ", mandatoryInternalAAs:" + "".join(chr(i) for i in range(256) if p.is_mandatory[i])
    u += ", proteoForms:false, maxVariationsPerPeptide:null, useUniprot:false, uniprotVersion:null"
    u += ", usePhosphoSite:false, phosphoSiteSpecies:null, sufix:null"
    u += ", discardDecoys:" + ("null" if sparam.discardDecoyRegexp is None else sparam.discardDecoyRegexp)
    if p.n_mods > 0 and p.max_mods_per_peptide > 0:
        u += ", diffMods:" + ",".join("%s%r" % (chr(p.mods[i].residue), p.mods[i].delta) for i in range(p.n_mods))
        u += ", maxDiffMods:%d" % p.max_mods_per_peptide
    return sparam.dataBaseName + "_" + hashlib.md5(u.encode("utf-8")).hexdigest()


INDEX_FILE_SUFFIX = ".gpuidx"  # the reference's directory is <name>.idx (DBIndexer.java:63,429-431)

# Unindexed search (useIndex = false): candidate records one dbi_search_unindexed may index.  A candidate of a
# 3-mod parameter set expands to ~26 entries of ~40 bytes while it is indexed, so 2^25 candidates stay well inside
# one GPU's memory and below 2^32 entries.
UNINDEXED_MAX_CANDIDATES = 1 << 25


def _merge_hits(parts, nq: int) -> dict:
    """The per-hit answers of several batches of queries (part = (query ids, query_hits-style dict)) as one answer
    for queries 0 .. nq-1 in that order; a query's hits keep their order."""
    qid = np.concatenate([np.repeat(ids, np.diff(h["hit_off"].astype(np.int64))) for ids, h in parts] +
                         [np.zeros(0, np.int64)]).astype(np.int64)
    perm = np.argsort(qid, kind="stable")

    def cat(k, dt):
        return np.concatenate([h[k] for _, h in parts] + [np.zeros(0, dt)])

    def cat_csr(off_key, data_key, dt):
        offs, base = [], 0
        for _, h in parts:
            offs.append(h[off_key][:-1].astype(np.int64) + base)
            base += int(h[off_key][-1])
        return np.append(np.concatenate(offs + [np.zeros(0, np.int64)]), base), cat(data_key, dt)

    out = {k: cat(k, dt)[perm] for k, dt in (("modpat", np.uint32), ("mass", np.float64), ("first_prot", np.uint32),
                                             ("first_off", np.uint32), ("len", np.uint16))}
    run_base = np.cumsum([0] + [int(h["counts"].n_peps) for _, h in parts])
    out["hit_pep"] = np.concatenate([h["hit_pep"] + run_base[i] for i, (_, h) in enumerate(parts)] +
                                    [np.zeros(0, np.int64)])[perm]
    out["flanks"] = np.ascontiguousarray(cat("flanks", np.uint8).reshape(-1, 6)[perm]).reshape(-1)
    out["seq_off"], out["seq"] = _expand_csr(*cat_csr("seq_off", "seq", np.uint8), perm)
    out["prot_list_off"], out["prot_ids"] = _expand_csr(*cat_csr("prot_list_off", "prot_ids", np.uint32), perm)
    out["hit_off"] = np.concatenate(([0], np.cumsum(np.bincount(qid, minlength=nq)))).astype(np.uint64)
    out["counts"] = DbiHitCounts(nq, len(perm), int(run_base[-1]), len(out["seq"]), len(out["prot_ids"]))
    return out


def search_unindexed_chunked(index: GpuIndex, lo, hi, max_candidates: int) -> dict:
    """query_hits-style answer (one record per hit) of the ranges [lo[i], hi[i]] on an unbuilt handle (or on the
    handles of a sharded proteome: multigpu.ShardedSearcher, whose N_c is the largest per-rank count), through
    dbi_search_unindexed calls of at most max_candidates candidate records each (0 = one call, no cap).  The
    ranges go to the device sorted by mass; a batch whose N_c candidates exceed the cap is split into
    ceil(N_c / cap) + 1 contiguous chunks of the sorted order (again if a chunk still exceeds it), and the answer
    comes back in the caller's order."""
    lo = np.ascontiguousarray(lo, dtype=np.float64)
    hi = np.ascontiguousarray(hi, dtype=np.float64)
    parts = []

    def run(ids):
        try:
            parts.append((ids, index.search_unindexed(lo[ids], hi[ids], max_candidates)))
        except DbiError as e:
            n_c = e.n_candidates or 0
            if e.code != DBI_ERANGE or not max_candidates or n_c <= max_candidates or len(ids) < 2:
                raise
            for chunk in np.array_split(ids, min(len(ids), -(-n_c // max_candidates) + 1)):
                run(chunk)

    run(np.argsort(lo, kind="stable"))
    return _merge_hits(parts, len(lo))


def search_unindexed_spectra_chunked(index: GpuIndex, mass, tol, range_off, tol_mode: int, index_factor: int,
                                     max_candidates: int) -> dict:
    """query_hits-style answer (one query per spectrum) of a dbi_search_unindexed_spectra batch on an unbuilt handle,
    through calls of at most max_candidates candidate records each (0 = one call, no cap).  As in
    search_unindexed_chunked, the spectra go to the device sorted by mass (a Dalton list by its first range) and a
    batch over the cap is split into ceil(N_c / cap) + 1 contiguous chunks of that order, again if needed; a
    spectrum is never split, and the answer comes back in the caller's order."""
    mass = np.ascontiguousarray(mass, dtype=np.float64)
    tol = np.ascontiguousarray(tol, dtype=np.float64)
    if tol_mode == DBI_TOL_PPM:
        n, key = len(mass), mass
        lens = np.ones(n, dtype=np.int64)
        first = np.arange(n, dtype=np.int64)
    else:
        ro = np.asarray(range_off, dtype=np.int64)
        n = len(ro) - 1
        lens, first = np.diff(ro), ro[:-1]
        key = np.zeros(n)
        key[lens > 0] = mass[first[lens > 0]]
    parts = []

    def run(ids):
        if tol_mode == DBI_TOL_PPM:
            args = (mass[ids], tol[ids], None)
        else:
            off = np.concatenate(([0], np.cumsum(lens[ids])))
            rows = np.repeat(first[ids] - off[:-1], lens[ids]) + np.arange(off[-1], dtype=np.int64)
            args = (mass[rows], tol[rows], off.astype(np.uint64))
        try:
            parts.append((ids, index.search_unindexed_spectra(*args, tol_mode=tol_mode, index_factor=index_factor,
                                                              max_candidates=max_candidates)))
        except DbiError as e:
            n_c = e.n_candidates or 0
            if e.code != DBI_ERANGE or not max_candidates or n_c <= max_candidates or len(ids) < 2:
                raise
            for chunk in np.array_split(ids, min(len(ids), -(-n_c // max_candidates) + 1)):
                run(chunk)

    run(np.argsort(key, kind="stable"))
    return _merge_hits(parts, n)


class DBIndexer:
    """DBIndexer.java: the indexer / orchestrator, GPU store behind it."""

    def __init__(self, params: DbiParams, index_factor: int = 8, index_path: Optional[str] = None,
                 use_index: bool = True, devices: Optional[Sequence[int]] = None):
        """index_path: where the finished index lives on disk (None = in-memory index only).  run() skips
        indexing when the file exists ("Found existing index, skipping indexing", DBIndexer.java:522-531)
        and writes it after a fresh build.

        use_index = False is the reference's SEARCH_UNINDEXED mode (DBIndexer.java:58-61, MassRangeFilteringIndex):
        run() only adds the proteins, and every getSequences* digests them again for its batch of ranges on the
        GPU (dbi_search_unindexed), max_candidates candidate records per device call.  No index file is read or
        written.  getNumberSequences, getParentMasses and export_reference_index need an index and raise
        DBIndexStoreException in this mode.

        devices (unindexed mode only; what -Ddbindex.gpu.devices is to the Java shim): one handle per entry, on that
        CUDA device (a device may repeat).  The proteome is cut into residue-balanced shards in file order, proteins
        added later go to the last shard, and every search runs over all of them (dbi_mg_search_unindexed_local)."""
        if devices is not None and use_index:
            raise DBIndexerException("a sharded index is not available here: devices needs use_index = False")
        self.sparam = params
        self.index_factor = index_factor  # dbindex.properties:6; only shapes the ">= MAX_MASS" query rule
        self.index_path = index_path
        self.use_index = use_index
        self.devices = None if devices is None else list(devices)
        self.shards: List[GpuIndex] = []  # the handles of a sharded proteome, rank order
        self._shard_first = [0]           # global id of every shard's first protein, then the total
        self.max_candidates = UNINDEXED_MAX_CANDIDATES
        self.loaded_from_disk = False
        self.inited = False
        self.index: Optional[GpuIndex] = None
        self.deflines: List[str] = []   # ProteinCache.defs
        self._seq_cache: dict = {}
        # Search-engine threads query a built index through one view each (dbi_view_open), so their calls run in
        # parallel; the unindexed and sharded searches go through the owner handles, one thread at a time.
        self._tls = threading.local()
        self._views: List[GpuIndex] = []
        self._views_lock = threading.Lock()
        self._owner_lock = threading.Lock()

    # -- lifecycle: init() (DBIndexer.java:412) -> run() (:508) --------------------------
    def init(self):
        if self.inited:
            raise DBIndexerException("Already inited")  # DBIndexer.java:413-415
        if self.devices is None:
            self.index = GpuIndex(self.sparam)
            self._searcher = self.index
        else:
            from .multigpu import ShardedSearcher
            for d in self.devices:
                p = self.sparam.copy()
                p.device = int(d)
                self.shards.append(GpuIndex(p))
            self.index = self.shards[0]  # the masses (calculate_mass) are every shard's
            self._searcher = ShardedSearcher(self.shards)
        self.inited = True

    def export_reference_index(self, database_id: str) -> dict:
        """Write the built index as the reference's own on-disk index -- directory `<database_id>.idx/` with one
        SQLite file per mass bucket, merged rows (dbindex_b200/sqlite_export.py; DBIndexStoreSQLiteMult.java:101-142,
        DBIndexStoreSQLiteByteIndexMerge.java:696-716) -- so that an unmodified reference finds an existing index
        there (SURVEY.md 8 f3).  Differential-mod variants have no counterpart in that format and are left out."""
        from .sqlite_export import export_sqlite
        self._require_index()
        n = self.index.stats()["n_entries"]
        return export_sqlite(lambda b, c: self.index.fetch(b, c), n, database_id, index_factor=self.index_factor,
                             mass_group_factor=self.sparam.mass_group_factor)

    def _require(self):
        if not self.inited or self.index is None:
            raise DBIndexStoreException("Indexer is not initialized")  # DBIndexStoreSQLiteMult.java:153

    def _require_index(self):
        self._require()
        if not self.use_index:
            raise DBIndexStoreException("not available in unindexed search mode (useIndex = false): there is no index")

    def add_proteins(self, deflines: Sequence[str], residues: np.ndarray, offsets: np.ndarray):
        """protCache.addProtein for a packed batch (DBIndexer.java:605)."""
        self._require()
        self.deflines.extend(d.replace("\t", " ") for d in deflines)  # ProteinCache.java:87-89
        if not self.shards:
            self.index.add_proteins(residues, offsets)
            return
        from .multigpu import shard_proteins
        offsets = np.asarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        if self._shard_first[-1] == 0:  # the first proteins are cut the way the Java shim cuts them
            first = []
            for r, g in enumerate(self.shards):
                res, off, p0 = shard_proteins(residues, offsets, r, len(self.shards))
                g.add_proteins(res, off)
                first.append(p0)
            self._shard_first = first + [n]
        else:  # later ones go to the last shard, so that ids stay in insertion order
            self.shards[-1].add_proteins(residues, offsets)
            self._shard_first[-1] += n

    def run(self, fasta: Optional[str] = None, proteins: Optional[Tuple[Sequence[str], Sequence[str]]] = None):
        """DBIndexer.run(): stream the FASTA, cut every protein, close the store."""
        self._require()
        if self.use_index and self.index_path is not None and os.path.exists(self.index_path):
            # indexStore.indexExists() -> "Found existing index, skipping indexing" (DBIndexer.java:522-531)
            try:
                self.index.load(self.index_path)
            except DbiError as e:
                raise DBIndexerException(str(e)) from e
            self.loaded_from_disk = True
            # the deflines (ProteinCache.defs) are not part of the index file: re-read them when a FASTA is at hand
            if fasta is not None:
                self.deflines = [d.replace("\t", " ") for d in read_fasta(fasta)[0]]
            elif proteins is not None:
                self.deflines = [d.replace("\t", " ") for d in proteins[0]]
            return
        if fasta is not None:
            deflines, residues, offsets = read_fasta(fasta)
            self.add_proteins(deflines, residues, offsets)
        elif proteins is not None:
            deflines, seqs = proteins
            residues = np.frombuffer("".join(seqs).encode("latin-1"), dtype=np.uint8)
            offsets = np.zeros(len(seqs) + 1, dtype=np.uint64)
            np.cumsum([len(s) for s in seqs], out=offsets[1:])
            self.add_proteins(deflines, residues, offsets)
        if not self.use_index:  # SEARCH_UNINDEXED: the proteins are all the store keeps
            return
        try:
            self.index.build()  # cutSeq per protein + stopAddSeq (DBIndexer.java:616,666)
            if self.index_path is not None:
                self.index.save(self.index_path)
        except DbiError as e:
            raise DBIndexerException(str(e)) from e

    def close(self):
        with self._views_lock:
            for v in self._views:
                v.close()
            self._views = []
        for g in self.shards or ([self.index] if self.index is not None else []):
            g.close()
        self.index = None
        self.shards = []
        self.inited = False

    # -- helpers ---------------------------------------------------------------------------
    def getProteinSequence(self, pid: int) -> str:
        s = self._seq_cache.get(pid)
        if s is None:
            if self.shards:
                r = min(int(np.searchsorted(self._shard_first, pid, side="right")) - 1, len(self.shards) - 1)
                s = self.shards[r].get_protein(pid - self._shard_first[r]).decode("latin-1")
            else:
                s = self.index.get_protein(pid).decode("latin-1")
            if len(self._seq_cache) < 100000:
                self._seq_cache[pid] = s
        return s

    def _out_of_buckets(self, lo: float, hi: float) -> bool:
        """DBIndexStoreSQLiteMult.getBucketsForMassRange / the 'unsupported precursor mass'
        early return (Mult:55-56,215-217,333-338): empty answer when a bound reaches MAX_MASS."""
        bucket_range = MAX_PRECURSOR_MASS // self.index_factor
        nb = self.index_factor
        return int(lo) // bucket_range > nb - 1 or int(hi) // bucket_range > nb - 1

    def _view(self) -> GpuIndex:
        """The calling thread's view of the built index, opened on its first query."""
        t = self._tls
        if getattr(t, "owner", None) is not self.index:
            v = self.index.view()
            with self._views_lock:
                self._views.append(v)
            t.owner, t.view = self.index, v
        return t.view

    def _hits(self, lo: np.ndarray, hi: np.ndarray) -> dict:
        """The hit source of every getSequences*: one record per hit of every [lo[i], hi[i]] (query_hits), from
        the index, or in unindexed mode from the proteins (chunked dbi_search_unindexed)."""
        try:
            if self.use_index:
                return self._view().query_hits(lo, hi)
            with self._owner_lock:
                return search_unindexed_chunked(self._searcher, lo, hi, self.max_candidates)
        except DbiError as e:
            raise DBIndexStoreException(str(e)) from e

    def _spectra_hits(self, mass, tol, range_off, tol_mode: int) -> dict:
        """The hit source of the spectrum batches: one query per spectrum (dbi_query_spectra, or in unindexed mode
        the chunked dbi_search_unindexed_spectra), the bucket rule of this index_factor applied on the device."""
        try:
            if self.use_index:
                return self._view().query_spectra(mass, tol, range_off, tol_mode, self.index_factor)
            with self._owner_lock:
                return search_unindexed_spectra_chunked(self._searcher, mass, tol, range_off, tol_mode,
                                                        self.index_factor, self.max_candidates)
        except DbiError as e:
            raise DBIndexStoreException(str(e)) from e

    def _materialise(self, lo: np.ndarray, hi: np.ndarray, keep: Optional[np.ndarray] = None) -> List[List[IndexedSequence]]:
        """getSequences for a batch of ranges in ONE device pass (dbi_query_hits, or dbi_search_unindexed)."""
        return self._sequences(self._hits(lo, hi), len(lo), keep)

    def _sequences(self, h: dict, nq: int, keep: Optional[np.ndarray] = None) -> List[List[IndexedSequence]]:
        """The objects parseAddPeptideInfo builds (DBIndexStoreSQLiteByteIndexMerge.java:452-462) for every query of
        a query_hits-style answer -- sequence, flanks, mass and protein ids all come back from the GPU; only the
        Python objects are made here."""
        ho, so, po = (h[k].astype(np.int64) for k in ("hit_off", "seq_off", "prot_list_off"))
        seq, flanks = h["seq"].tobytes().decode("latin-1"), h["flanks"].tobytes().decode("latin-1")
        out = []
        for q in range(nq):
            if keep is not None and not keep[q]:
                out.append([])
                continue
            lst = []
            for i in range(ho[q], ho[q + 1]):
                pat = int(h["modpat"][i])
                pos = tuple(((pat >> (8 * k)) & 0xFF) - 1 for k in range(4) if (pat >> (8 * k)) & 0xFF)
                lst.append(IndexedSequence(float(h["mass"][i]), seq[so[i]:so[i + 1]], h["prot_ids"][po[i]:po[i + 1]].tolist(),
                                           flanks[6 * i:6 * i + 3], flanks[6 * i + 3:6 * i + 6], int(h["first_off"][i]),
                                           int(h["len"][i]), pos))
            out.append(lst)
        return out

    # -- queries --------------------------------------------------------------------------
    def getSequencesBatch(self, masses: Sequence[float], tolerances: Sequence[float]) -> List[List[IndexedSequence]]:
        """Many getSequences(precMass, tol) in one device call."""
        self._require()
        m = np.asarray(masses, dtype=np.float64)
        t = np.asarray(tolerances, dtype=np.float64)
        lo = np.maximum(m - t, 0.0)  # Mult:324-329
        hi = m + t
        keep = np.array([not self._out_of_buckets(lo[i], hi[i]) for i in range(len(m))], dtype=bool)
        return self._materialise(lo, hi, keep)

    def getSequencesUsingDaltonTolerance(self, precursorMass: float, massToleranceInDa: float) -> List[IndexedSequence]:
        """DBIndexer.java:762-772 -> DBIndexStoreSQLiteMult.getSequences (Mult:315-350)."""
        return self.getSequencesBatch([precursorMass], [massToleranceInDa])[0]

    def getSequencesUsingPPMTolerance(self, precursorMass: float, massToleranceInPPM: float) -> List[IndexedSequence]:
        """DBIndexer.java:787-844: one Dalton query, then exact-mass probes above the upper
        bound until one comes back empty (a batch of one spectrum)."""
        return self.getSequencesUsingPPMToleranceBatch([precursorMass], massToleranceInPPM)[0]

    def getSequencesUsingPPMToleranceBatch(self, masses: Sequence[float], massToleranceInPPM) -> List[List[IndexedSequence]]:
        """getSequencesUsingPPMTolerance for every mass in one device call (dbi_query_spectra, DBI_TOL_PPM; in
        unindexed mode dbi_search_unindexed_spectra): the window and the probe walk of every spectrum run on the GPU.
        massToleranceInPPM: one value, or one per mass.  A sharded proteome runs the walk over its ranks
        (dbi_mg_search_unindexed_spectra_local)."""
        self._require()
        m = np.ascontiguousarray(masses, dtype=np.float64)
        ppm = np.ascontiguousarray(np.broadcast_to(np.asarray(massToleranceInPPM, dtype=np.float64), m.shape))
        return self._sequences(self._spectra_hits(m, ppm, None, DBI_TOL_PPM), len(m))

    def _ppm_probe_loop(self, precursorMass: float, massToleranceInPPM: float) -> List[IndexedSequence]:
        """The reference's probe loop on the host, one device call per probe (kept as the reference of the batch)."""
        tol = tolerance_in_dalton(precursorMass, massToleranceInPPM)
        sequences = self.getSequencesUsingDaltonTolerance(precursorMass, tol)
        have = {s.key() for s in sequences}
        upper = precursorMass + tol
        while True:
            tol2 = tolerance_in_dalton(upper, massToleranceInPPM)
            if upper - tol2 < precursorMass:
                seq2 = self.getSequencesUsingDaltonTolerance(upper, 0.0)
                if not seq2:
                    break
                for s in seq2:
                    if s.key() not in have:
                        have.add(s.key())
                        sequences.append(s)
            else:
                break
            new_upper = upper + PRECISION
            if new_upper == upper:
                break
            upper = new_upper
        return sequences

    def getSequences(self, ranges: Sequence[MassRange]) -> List[IndexedSequence]:
        """DBIndexer.java:855-871 -> Mult.getSequences(List<MassRange>) (Mult:353-430): a batch of one spectrum."""
        self._require()
        return self.getSequencesForSpectra([ranges])[0]

    def getSequencesForSpectra(self, spectra: Sequence[Sequence[MassRange]]) -> List[List[IndexedSequence]]:
        """getSequences(List<MassRange>) for every spectrum of a list in one device call (dbi_query_spectra,
        DBI_TOL_DA; in unindexed mode dbi_search_unindexed_spectra): the intervals of every spectrum are clamped,
        sorted, merged and checked against the bucket rule on the GPU (on every rank of a sharded proteome)."""
        self._require()
        lists = [list(sp) for sp in spectra]
        mass = np.array([r.precMass for sp in lists for r in sp], dtype=np.float64)
        tol = np.array([r.tolerance for sp in lists for r in sp], dtype=np.float64)
        range_off = np.zeros(len(lists) + 1, dtype=np.uint64)
        np.cumsum([len(sp) for sp in lists], out=range_off[1:])
        return self._sequences(self._spectra_hits(mass, tol, range_off, DBI_TOL_DA), len(lists))

    def _protein(self, pid: int) -> IndexedProtein:
        return IndexedProtein(self.deflines[pid] if pid < len(self.deflines) else "", pid)

    def getProteins(self, seq) -> Set[IndexedProtein] | List[IndexedProtein]:
        """getProteins(String) (DBIndexer.java:925-947) / getProteins(IndexedSequence) (:882)."""
        self._require()
        if isinstance(seq, IndexedSequence):
            return [self._protein(i) for i in seq.proteinIds]
        return self.getProteinsBatch([seq])[0]

    def getProteinsBatch(self, seqs: Sequence[str]) -> List[Set[IndexedProtein]]:
        """getProteins(String) for a whole list in one device call (dbi_lookup_peptides): the unmodified entry
        whose peptide equals the string, found by its mass computed the way the index computes it
        (IndexUtil.calculateMass) -- the zero-tolerance getSequences + `s.sequence.equals(seq)` filter of the
        reference.  A mass whose bucket lies beyond MAX_MASS gives the empty set, as that query does.

        Unindexed mode takes the reference's own route (DBIndexer.java:925-947): masses by IndexUtil.calculateMass
        (dbi_calculate_mass), one search with zero-width windows, and the unmodified hit whose sequence equals
        the string."""
        self._require()
        if not self.use_index:
            return self._proteins_unindexed(seqs)
        try:
            r = self._view().lookup_peptides(list(seqs))
        except DbiError as e:
            raise DBIndexStoreException(str(e)) from e
        plo = r["prot_list_off"].astype(np.int64)
        out: List[Set[IndexedProtein]] = []
        for i in range(len(seqs)):
            m = float(r["mass"][i])
            if r["status"][i] != 1 or self._out_of_buckets(m, m):
                out.append(set())
            else:
                out.append({self._protein(p) for p in r["prot_ids"][plo[i]:plo[i + 1]].tolist()})
        return out

    def _proteins_unindexed(self, seqs: Sequence[str]) -> List[Set[IndexedProtein]]:
        bs = [s.encode("latin-1") for s in seqs]
        m = np.array([self.index.calculate_mass(b) for b in bs], dtype=np.float64)
        h = self._hits(m, m)
        ho, so, po = (h[k].astype(np.int64) for k in ("hit_off", "seq_off", "prot_list_off"))
        seq = h["seq"].tobytes()
        out: List[Set[IndexedProtein]] = []
        for i, b in enumerate(bs):
            prots: Set[IndexedProtein] = set()
            if not self._out_of_buckets(m[i], m[i]):
                for j in range(ho[i], ho[i + 1]):
                    if h["modpat"][j] == 0 and seq[so[j]:so[j + 1]] == b:
                        prots = {self._protein(p) for p in h["prot_ids"][po[j]:po[j + 1]].tolist()}
                        break
            out.append(prots)
        return out

    def getNumberSequences(self) -> int:
        self._require_index()
        return int(self.index.stats()["n_entries"])

    def getParentMasses(self) -> List[float]:
        """DBIndexer.java:984-992: entry keys divided back by massGroupFactor."""
        self._require_index()
        f = float(self.sparam.mass_group_factor)
        return [k / f for k in self.index.entry_keys().tolist()]


class DBIndexImpl:
    """DBIndexImpl.java: the DBIndexInterface facade a search engine holds."""

    _by_param_key: dict = {}  # DBIndexImpl.java:35 dbIndexByParamKey

    def __init__(self, params, fasta: Optional[str] = None,
                 proteins: Optional[Tuple[Sequence[str], Sequence[str]]] = None, index_factor: int = 8,
                 devices: Optional[Sequence[int]] = None):
        """params: dbi_params, or a DBIndexSearchParams (then the FASTA is its dataBaseName, as in
        DBIndexImpl(DBIndexSearchParams), DBIndexImpl.java:117-145).  devices: DBIndexer's (unindexed mode)."""
        self.sparam = params if isinstance(params, DBIndexSearchParams) else None
        if self.sparam is not None:
            if fasta is None and proteins is None:
                fasta = self.sparam.dataBaseName
            index_factor = self.sparam.indexFactor
            params = self.sparam.params
        index_path = None
        use_index = self.sparam.useIndex if self.sparam is not None else True
        if self.sparam is not None and use_index and not self.sparam.inMemoryIndex:
            # an on-disk index, named like the reference's (DBIndexer.java:429 createFullIndexFileName)
            index_path = createFullIndexFileName(self.sparam) + INDEX_FILE_SUFFIX
        self.indexer = DBIndexer(params, index_factor, index_path=index_path, use_index=use_index, devices=devices)
        self.indexer.init()
        self.indexer.run(fasta=fasta, proteins=proteins)
        self._proteins_by_seq: dict = {}  # DBIndexImpl.java:33
        if self.sparam is not None:
            DBIndexImpl._by_param_key[self.sparam.key()] = self  # DBIndexImpl.java:137-139

    @staticmethod
    def getByParam(sParam: "DBIndexSearchParams") -> "DBIndexImpl":
        """DBIndexImpl.getByParam (DBIndexImpl.java:44-49): one index per parameter key."""
        hit = DBIndexImpl._by_param_key.get(sParam.key())
        return hit if hit is not None else DBIndexImpl(sParam)

    def getSequences(self, *args) -> List[IndexedSequence]:
        """getSequences(double precursorMass, double massTolerance) (DBIndexImpl.java:180) or
        getSequences(List<MassRange>) (:194)."""
        if len(args) == 2:
            return self.indexer.getSequencesUsingDaltonTolerance(float(args[0]), float(args[1]))
        return self.indexer.getSequences(list(args[0]))

    def getSequencesForSpectra(self, spectra) -> List[List[IndexedSequence]]:
        """getSequences(List<MassRange>) for a list of spectra, one device call (DBIndexer.getSequencesForSpectra)."""
        return self.indexer.getSequencesForSpectra(spectra)

    def getProteins(self, seq):
        """getProteins(String) (DBIndexImpl.java:222-237, memoised), getProteins(IndexedSequence) (:208), or for a
        list of strings the list of their protein sets: the strings not memoised yet go to the device in one call."""
        if isinstance(seq, str):
            return self.getProteins([seq])[0]
        if isinstance(seq, IndexedSequence):
            return self.indexer.getProteins(seq)
        seqs = list(seq)
        todo = list(dict.fromkeys(s for s in seqs if s not in self._proteins_by_seq))
        if todo:
            self._proteins_by_seq.update(zip(todo, self.indexer.getProteinsBatch(todo)))
        return [self._proteins_by_seq[s] for s in seqs]

    def getIndexedProteinById(self, pid: int) -> IndexedProtein:
        return IndexedProtein(self.indexer.deflines[pid], pid)  # DBIndexImpl.java:501-504

    def getProteinSequenceById(self, pid: int) -> str:
        return self.indexer.getProteinSequence(pid)  # DBIndexImpl.java:511-513

    def close(self):
        if self.sparam is not None:
            DBIndexImpl._by_param_key.pop(self.sparam.key(), None)
        self.indexer.close()
