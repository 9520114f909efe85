/*
 * dbindex_gpu.h -- C ABI of the B200-native dbIndex hot path.
 *
 * One handle = one peptide index living in the HBM of ONE GPU:
 *   FASTA residues -> in-silico digestion -> (diff-mod expansion) ->
 *   mass-sorted, de-duplicated peptide index -> batched precursor-mass
 *   range lookup.
 *
 * Plain C: pointers and sizes only, no C++/torch types.  Bindable from JNI,
 * Panama FFM, ctypes or cgo.  There is NO CPU fallback behind these entry
 * points: without a CUDA device every call that needs one returns DBI_ECUDA.
 *
 * Each entry point names the reference interface it replaces.  Paths are
 * relative to src/main/java/edu/scripps/yates/dbindex/ of
 * proteomicsyates/dbIndex.  See INTEGRATION.md for the Java-side binding.
 */
#ifndef DBINDEX_GPU_H
#define DBINDEX_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DBI_ABI_VERSION 3

/* ---- status codes (0 = OK, negative = error) -----------------------------
 * The shim maps them onto the reference's two exception types:
 * DBIndexStoreException ("Indexer is not initialized", DBIndexStoreSQLiteMult.java:153,273,316;
 * "Already intialized", :97-99) and DBIndexerException (DBIndexerException.java:9-18). */
#define DBI_OK 0
#define DBI_ENOTINIT (-1) /* query/fetch before dbi_build()            */
#define DBI_EALREADY (-2) /* add_proteins/build after dbi_build()      */
#define DBI_EINVAL (-3)   /* bad argument / unsupported parameter      */
#define DBI_ENOMEM (-4)   /* host or device allocation failed          */
#define DBI_ECUDA (-5)    /* no device, or a CUDA call failed          */
#define DBI_ENCCL (-6)    /* reserved (the exchanges need no NCCL)     */
#define DBI_ERANGE (-7)   /* a hard limit was exceeded (see below)     */

/* ---- hard limits ---------------------------------------------------------- */
#define DBI_MAX_MODS 16         /* distinct (residue, delta) entries          */
#define DBI_MAX_MODS_PER_PEP 4  /* mod pattern = 4 x 8-bit positions          */
#define DBI_MAX_PEP_LEN 65535   /* len is stored as uint16 (ref: MAX_SEQ_LENGTH 10000, DBIndexer.java:75) */
#define DBI_MAX_MOD_POS 254     /* modified residue position inside a peptide */
#define DBI_MIN_PEP_LENGTH 6    /* Constants.java:10                          */
#define DBI_MASS_GROUP_FACTOR 10000 /* dbindex.properties:20, SearchParamReader.java:705 */

/* One differential (variable) modification: residue -> mass shift.
 * Mirrors model/ModResidue.java:12-44 and the 256-entry table of
 * model/DiffModification.java:11-54 (one shift per residue, last one wins). */
typedef struct dbi_mod {
  uint8_t residue;
  uint8_t _pad[7];
  double delta;
} dbi_mod;

/* Search parameters that reach the hot path (SURVEY.md 5.1).  POD, passed by
 * pointer, copied by dbi_create().  Replaces the SearchParams singleton
 * (SearchParams.java:127-132), DBIndexSearchParamsImpl's 19-arg constructor
 * (io/DBIndexSearchParamsImpl.java:46-75) and the global AssignMass table
 * (external utilities jar; call sites DBIndexer.java:268-271,306). */
typedef struct dbi_params {
  uint32_t abi_version;   /* must be DBI_ABI_VERSION */
  int32_t device;         /* CUDA device ordinal */

  /* AssignMass.getMass(char): residue mass table with static mods already
   * added (AssignMassToStaticParam.java:7-15).  Unknown residues = 0. */
  double residue_mass[256];
  double h2o_proton;      /* AssignMass.H2O_PROTON */
  double nterm;           /* AssignMass.getnTerm() */
  double cterm;           /* AssignMass.getcTerm() */
  int32_t add_h2o_proton; /* sparam.isH2OPlusProtonAdded(), DBIndexer.java:268 */

  /* Enzyme (external utilities jar; DBIndexer.java:314-319).  C-terminal cutter. */
  uint8_t is_enzyme[256]; /* Enzyme.isEnzyme(c)            */
  uint8_t is_nocut[256];  /* sparam.getEnzymeNocutResidues */
  int32_t max_missed;     /* sparam.getMaxMissedCleavages(), DBIndexer.java:246,322 */
  int32_t semi;           /* semi-specific cleavage, Enzyme ctor 3rd arg */
  int32_t min_len;        /* Constants.MIN_PEP_LENGTH = 6, DBIndexer.java:331 */
  double min_mass;        /* sparam.getMinPrecursorMass(), DBIndexer.java:331 */
  double max_mass;        /* sparam.getMaxPrecursorMass(), DBIndexer.java:284,327 */
  int32_t mass_group_factor; /* key = (int)(mass*factor), DBIndexStoreSQLiteByte.java:187 */

  /* Differential mods (io/SearchParamReader.java:631-667,322). */
  int32_t n_mods;
  int32_t max_mods_per_peptide; /* max_num_differential_AA_per_mod */
  dbi_mod mods[DBI_MAX_MODS];

  /* Peptide filters applied while a start position is walked (SURVEY.md 8 f4).
   * mandatoryInternalAAs (DBIndexer.java:248,334-344 + DBIndexStoreSQLiteMult.java:245-263): a
   * qualifying window with none of these residues ENDS the start; one that has them only as its
   * last residue is skipped.  has_mandatory = "the array is not null" (an empty array is legal in
   * the reference and then nothing qualifies).
   * PeptideFilterByMaxOccurrencies (util/PeptideFilterByMaxOccurrencies.java:22-34, break at
   * DBIndexer.java:310-313): the start ends once residue filter_aa occurs more than filter_max times. */
  uint8_t is_mandatory[256];
  int32_t has_mandatory;
  int32_t filter_aa;      /* residue code, 0 = no filter */
  int32_t filter_max;
  int32_t _pad_filters;

  /* Test/diagnostic switches (no reference counterpart). */
  int32_t keep_emitted;   /* keep the raw emitted records for dbi_debug_emitted() */
  int32_t profile;        /* record a CUDA-event pair around every build stage  */
  int32_t reserved[6];
} dbi_params;

/* Counters and per-stage device times (replaces the log4j progress lines,
 * DBIndexStoreSQLiteMult.java:277-280, and getNumberSequences, DBIndexStore.java). */
#define DBI_N_STAGES 12
typedef struct dbi_stats {
  uint64_t n_proteins;
  uint64_t n_residues;
  uint64_t n_emitted;      /* records cutSeq would hand to addSequence           */
  uint64_t n_unique;       /* distinct (mass, sequence) after the merge           */
  uint64_t n_entries;      /* searchable entries = unique peptides x mod variants */
  uint64_t n_hash_retries; /* dedup re-runs caused by a (mass,hash) collision     */
  uint64_t device_bytes;   /* bytes of HBM held by the finished index             */
  uint64_t algo_bytes[DBI_N_STAGES]; /* algorithmic bytes moved per stage (DESIGN.md) */
  float stage_ms[DBI_N_STAGES];      /* device time per stage, only if params.profile */
  uint32_t stage_launches[DBI_N_STAGES]; /* kernels launched per stage            */
  uint32_t sort_bits_base;  /* radix key bits sorted for the base records  */
  uint32_t sort_bits_var;   /* radix key bits sorted for the mod variants  */
  /* The dominant kernel of a build = the onesweep scatter passes of its largest
   * sort (mod variants if any, else the base records); only if params.profile. */
  float dom_ms;                  /* summed device time of those launches      */
  uint32_t dom_launches;         /* how many                                  */
  uint64_t dom_bytes_per_launch; /* algorithmic bytes one launch moves        */
  uint32_t dom_kernel;           /* 0 = <u64 key,u32 val> base, 1 = <u64,u64> variants */
  /* The mod-expansion kernel (grp_expand_kernel: sorted groups -> entries), bracketed the
   * same way; bench.py reports whichever of the two takes more of the build. */
  uint32_t exp_launches;
  float exp_ms;
  uint32_t n_groups;       /* variant groups a compact index holds; 0 = entries expanded (DESIGN.md 2) */
  uint64_t exp_bytes_per_launch;
} dbi_stats;

/* stage ids for dbi_stats arrays */
#define DBI_STAGE_PACK 0
#define DBI_STAGE_DIGEST_COUNT 1
#define DBI_STAGE_DIGEST_EMIT 2
#define DBI_STAGE_SORT_BASE 3
#define DBI_STAGE_DEDUP 4
#define DBI_STAGE_MOD_COUNT 5
#define DBI_STAGE_MOD_EMIT 6
#define DBI_STAGE_SORT_VAR 7
#define DBI_STAGE_GATHER_VAR 8
#define DBI_STAGE_QUERY 9
#define DBI_STAGE_FETCH 10
#define DBI_STAGE_OTHER 11

typedef struct dbi_handle dbi_handle;

/* Fill *p with the published defaults: standard monoisotopic (mono != 0) or
 * average residue masses, H2O+proton added, trypsin (KR), no no-cut residues,
 * 2 missed cleavages, full specificity, 600..6000 Da, factor 10000, no mods.
 * This is the written-down contract for the un-vendored AssignMass / Enzyme
 * (SURVEY.md 8c); a Java host overwrites the tables from the live classes.
 * Mirrors DBIndexImpl.getDefaultDBIndexParams (DBIndexImpl.java:243-303). */
void dbi_default_params(dbi_params* p, int mono);

/* AssignMass.addMass(ch, delta) for a static modification; ignored when
 * delta <= 0 exactly like AssignMassToStaticParam.java:9-10. */
void dbi_params_add_static_mod(dbi_params* p, uint8_t residue, double delta);

/* Enzyme.addCleavePosition(ch) per character (SearchParams.java:301-307). */
void dbi_params_set_enzyme(dbi_params* p, const char* residues, const char* nocut);

/* diff_search_options entry: every residue of `residues` gets shift `delta`
 * (io/SearchParamReader.java:640-660).  Returns DBI_ERANGE past DBI_MAX_MODS. */
int dbi_params_add_diff_mod(dbi_params* p, const char* residues, double delta);

/* new DBIndexer(params, INDEX) + init()  (DBIndexer.java:167,412). */
int dbi_create(const dbi_params* params, dbi_handle** out);

/* Use a caller-owned CUDA stream (cudaStream_t cast to void*) for every kernel
 * and copy of this handle; NULL = the handle's own stream. */
int dbi_set_stream(dbi_handle* h, void* cuda_stream);

/* ---- threads and query views ----------------------------------------------
 * Calls on one handle are serialised by the handle's mutex; calls on different
 * handles or views may run at the same time from different threads.  A pending
 * result (dbi_query_hits, dbi_lookup_peptides) belongs to the handle or view
 * that made it, so a begin / read pair on a handle shared between threads needs
 * a lock of the caller's around both calls.
 *
 * A VIEW of a built handle is a dbi_handle that shares the handle's index (no
 * copy) but has its own CUDA stream (non-blocking), scratch arena, mutex,
 * pending hit result, pending lookup result, error flag and query stats.  The
 * search-engine threads of the reference (DBIndexer.java:468-469) each open one
 * and then query in parallel.  Closed with dbi_destroy(view).
 *
 * - Views accept dbi_query, dbi_query_device, dbi_fetch, dbi_query_hits,
 *   dbi_query_hits_device, dbi_query_hits_read, dbi_query_spectra,
 *   dbi_lookup_peptides, dbi_lookup_peptides_read, dbi_entry_keys,
 *   dbi_stats_get, dbi_set_stream, dbi_calculate_mass, dbi_get_protein,
 *   dbi_mg_slices and dbi_mg_split_masses.  Every answer is byte-identical to
 *   the owner's answer to the same call: on a single-GPU index, a compact
 *   index and one rank of a sharded index (the view reads the other ranks'
 *   window 2 as the owner does).  dbi_get_protein is answered by the owner
 *   under the owner's mutex.
 * - Views refuse (DBI_EINVAL) every call that changes the proteins or the
 *   index or runs across several handles: dbi_add_proteins, dbi_upload,
 *   dbi_reset_index, dbi_build, dbi_build_from_records, dbi_save, dbi_load,
 *   dbi_search_unindexed, dbi_search_unindexed_spectra, every dbi_mg_* staging
 *   and rank-level call, the dbi_mg_*_local calls and dbi_debug_*.  A view of a
 *   view is DBI_EINVAL; a view of an unbuilt handle is DBI_ENOTINIT.
 * - The owner keeps answering queries while views are open, but is pinned:
 *   the calls of that list that change its residues, candidate index or index
 *   tables return DBI_EINVAL ("n views open") until the last view is closed.
 * - dbi_destroy(owner) does not wait for its views: the index memory lives
 *   until the last view is destroyed, and the views keep answering until then.
 * - dbi_stats_get on a view reports the owner's index counters (n_*,
 *   device_bytes, n_groups, sort bits) with the view's own launches,
 *   algorithmic bytes and (params.profile) times; calls on a view leave the
 *   owner's stats alone. */
int dbi_view_open(dbi_handle* h, dbi_handle** view);

/* The per-protein body of DBIndexer.run() (DBIndexer.java:600-616):
 * ProteinCache.addProtein (ProteinCache.java:84-95) for n proteins whose
 * residues are concatenated in `residues`, protein i occupying
 * [offsets[i], offsets[i+1]).  Host memory, copied.  May be called repeatedly;
 * ids are assigned in call order (= FASTA order), 0-based like protNum
 * (DBIndexer.java:70,151,251).  Residue byte 0 is rejected (DBI_EINVAL). */
int dbi_add_proteins(dbi_handle* h, const uint8_t* residues, const uint64_t* offsets, uint32_t n);

/* Copy the proteins added so far into HBM now (idempotent; dbi_build() does it
 * implicitly).  Lets a caller separate the host->device copy of the FASTA
 * residues from the build proper. */
int dbi_upload(dbi_handle* h);

/* Drop the built index but keep the proteins (host and device copies), so that
 * dbi_build() can run again: the analogue of deleting the <fasta>_<md5>.idx
 * directory and re-running DBIndexer.run() (DBIndexer.java:522-531). */
int dbi_reset_index(dbi_handle* h);

/* cutSeq for every protein + indexStore.stopAddSeq() (DBIndexer.java:616,666;
 * DBIndexStoreSQLiteByteIndexMerge.java:64-127,620-719): digest, sort by mass,
 * merge equal peptides, expand differential mods, sort the variants. */
int dbi_build(dbi_handle* h);

/* Index persistence / resume (SURVEY.md 8 f3).  The reference keeps its index on disk under
 * <fasta>_<md5(params)> (util/IndexUtil.java:270-324) and skips indexing when it finds one
 * (DBIndexer.java:522-531).  dbi_save writes the proteins and the finished index of a single-GPU
 * handle to `path` (atomically: temp file + rename); dbi_load restores both into a FRESH handle created
 * with the same search parameters (anything else is DBI_EINVAL) -- afterwards the handle answers queries
 * exactly like the one that was saved.  The file name is the host's business. */
int dbi_save(dbi_handle* h, const char* path);
int dbi_load(dbi_handle* h, const char* path);

/* getNumberSequences() and friends. */
int dbi_stats_get(dbi_handle* h, dbi_stats* out);

/* Batched DBIndexStore.getSequences(precMass, tol) (DBIndexStoreSQLiteMult.java:315-350,
 * DBIndexStoreSQLiteByteIndexMerge.java:146-217).  The caller passes the
 * inclusive exact-double bounds lo = max(0, m - tol), hi = m + tol
 * (Mult:324-329); the answer for query i is the contiguous run of index
 * entries [hit_begin[i], hit_begin[i] + hit_count[i]) with lo <= mass <= hi
 * (the exact filter of Merge:415-419).  Host pointers. */
int dbi_query(dbi_handle* h, const double* lo, const double* hi, uint64_t nq, uint64_t* hit_begin,
              uint64_t* hit_count);

/* Same, with every pointer in DEVICE memory of the handle's GPU (used when the
 * queries are already resident; also the building block of dbi_query). */
int dbi_query_device(dbi_handle* h, const double* d_lo, const double* d_hi, uint64_t nq,
                     uint64_t* d_hit_begin, uint64_t* d_hit_count);

/* Materialise entries [begin, begin+count): what parseAddPeptideInfo builds per
 * hit (DBIndexStoreSQLiteByteIndexMerge.java:386-481).  Any output pointer may
 * be NULL.  prot_list_off has count+1 entries (CSR over prot_ids);
 * *n_prot_ids receives the total id count, so call once with prot_ids == NULL
 * to size it.  first_prot/first_off/len are the first occurrence's protein,
 * offset and length (Merge:678-687); modpat holds up to 4 modified residue
 * positions, byte k = position+1 of the k-th modified residue, 0 = none. */
int dbi_fetch(dbi_handle* h, uint64_t begin, uint64_t count, double* mass, uint32_t* first_prot,
              uint32_t* first_off, uint16_t* len, uint32_t* modpat, uint64_t* prot_list_off,
              uint32_t* prot_ids, uint64_t prot_ids_capacity, uint64_t* n_prot_ids);

/* What DBIndexStore.getSequences RETURNS, for a whole batch of ranges in one pass: every hit of
 * every [lo[i], hi[i]] materialised the way parseAddPeptideInfo does per row
 * (DBIndexStoreSQLiteByteIndexMerge.java:386-481): exact mass, first occurrence (protein, offset,
 * length; Merge:438-447), the peptide residues cut from the protein
 * (ProteinCache.getPeptideSequence, ProteinCache.java:112-127), the +-3 flanking residues of
 * Util.getResidues ('-' padded, right side with the reference's off-by-one; Util.java:130-162,
 * Merge:456-458), the mod pattern and the protein-id list (Merge:449-475).
 *
 * The answer is grouped the way the index is.  A RUN is a maximal sequence of consecutive hits of one
 * query that are variants of ONE peptide with ONE mass (a variant group of the index; without
 * differential mods every hit is a run of its own).  Everything the reference derives from the peptide
 * is delivered once per run, a hit carries only its mod pattern: the hits of run p are
 * [pep_hit_off[p], pep_hit_off[p + 1]) and all of them have mass[p], first_prot[p], ... ; the runs of
 * query i are [pep_off[i], pep_off[i + 1]), its hits [hit_off[i], hit_off[i + 1]).  Nothing is lost
 * against one record per hit (expand with the two CSRs); a 10 ppm window of a 3-mod index holds ~10
 * hits per run, so the batch crosses PCIe in a quarter of the bytes.
 *
 *   dbi_query_hits(h, lo, hi, nq, &n)      device: bounds search, run marking, size scans, gathers (results stay in HBM)
 *   caller allocates from n (dbi_host_alloc gives pinned memory for full-speed DMA)
 *   dbi_query_hits_read(h, &out)           D2H into the caller's buffers; any pointer may be NULL
 *
 * seq_off / prot_list_off [n_peps + 1] are CSRs over seq[] and prot_ids[]; flanks holds 6 bytes per run
 * (3 left, 3 right).  The pending result of a handle is dropped by the next dbi_query_hits,
 * dbi_search_unindexed, a successful read, dbi_reset_index or dbi_destroy. */
typedef struct dbi_hit_counts {
  uint64_t nq, n_hits, n_peps, n_seq_bytes, n_prot_ids;
} dbi_hit_counts;
typedef struct dbi_hit_buffers {
  uint64_t* hit_off;       /* nq + 1      hits of every query                     */
  uint64_t* pep_off;       /* nq + 1      runs of every query                     */
  uint32_t* modpat;        /* n_hits      byte k = position + 1 of the k-th mod   */
  uint64_t* pep_hit_off;   /* n_peps + 1  hits of every run                       */
  double* mass;            /* n_peps      */
  uint32_t* first_prot;    /* n_peps      */
  uint32_t* first_off;     /* n_peps      */
  uint16_t* len;           /* n_peps      */
  uint8_t* flanks;         /* 6 * n_peps  */
  uint64_t* seq_off;       /* n_peps + 1  */
  uint8_t* seq;            /* n_seq_bytes */
  uint64_t* prot_list_off; /* n_peps + 1  */
  uint32_t* prot_ids;      /* n_prot_ids  */
} dbi_hit_buffers;
int dbi_query_hits(dbi_handle* h, const double* lo, const double* hi, uint64_t nq, dbi_hit_counts* counts);
/* same with the bounds already in device memory of the handle's GPU */
int dbi_query_hits_device(dbi_handle* h, const double* d_lo, const double* d_hi, uint64_t nq, dbi_hit_counts* counts);
int dbi_query_hits_read(dbi_handle* h, const dbi_hit_buffers* out);

/* DBIndexer in SEARCH_UNINDEXED mode (DBIndexer.java:58-61; MassRangeFilteringIndex.java:90-108): the hits of a
 * batch of ranges, straight from the proteins added so far, with no index built or kept -- the way to search a
 * proteome whose index does not fit one GPU.  lo / hi are host pointers with the inclusive semantics of
 * dbi_query_hits.  The proteins are digested once per call, keeping only the records that can land in a window
 * (K2u / K4u: base mass + some sum of <= min(max_mods, mod sites) shifts meets the union of the windows); those
 * CANDIDATES are indexed as dbi_build indexes a proteome, the hits materialised, and the candidate index freed.
 * For every query the hits equal what dbi_build followed by dbi_query_hits would return on this handle (the
 * multiset of mass bits, first occurrence, length, residues, flanks, mod pattern and protein list, grouped in
 * maximal runs; ties inside a query have no contractual order).
 *
 * The result is the handle's pending hit result: read it with dbi_query_hits_read (same buffers, same runs).
 * The call drops any earlier pending result.  It needs a handle that is not built (built: DBI_EALREADY) and
 * not part of a sharded build (after dbi_mg_begin: DBI_EINVAL).  The handle stays unbuilt: dbi_add_proteins
 * still works and later searches see the added proteins, dbi_build still builds the normal index, and
 * dbi_query_hits / dbi_lookup_peptides still return DBI_ENOTINIT.  The packed residues (K1) are kept between
 * calls and packed again only when proteins were added since.
 *
 * max_candidates (0 = no cap) bounds the candidate records, N_c, which the count pass knows before anything is
 * allocated.  N_c > max_candidates or N_c >= 2^32: DBI_ERANGE and no pending result, so that the host can split
 * the batch.  *n_candidates (may be NULL) receives N_c in both cases.  The < 2^32 hits rule of dbi_query_hits
 * applies unchanged.  dbi_stats_get afterwards reports this search's candidate pipeline: n_emitted = N_c,
 * n_unique and n_entries of the candidate index, and with params.profile the stage times (K12 windows under
 * DBI_STAGE_OTHER). */
int dbi_search_unindexed(dbi_handle* h, const double* lo, const double* hi, uint64_t nq, uint64_t max_candidates,
                         dbi_hit_counts* counts, uint64_t* n_candidates);

/* A batch of spectra, each answered as the reference answers one spectrum's precursor query, in one call.
 *   DBI_TOL_DA:  spectrum s is the ranges [range_off[s], range_off[s+1]) of (mass, tol in Da), answered as
 *                DBIndexer.getSequences(List<MassRange>) (DBIndexer.java:855-871, Mult:353-430): lo = max(0, m - t),
 *                hi = m + t, stable sort by lo, merge while end >= next start (end = max), and an empty answer when
 *                a merged interval fails the bucket rule; otherwise the hits of every merged interval in order.
 *                No ranges: empty.  One range: the same rules (= getSequences(mass, tol)).
 *   DBI_TOL_PPM: spectrum s is mass[s] at tol[s] ppm (range_off must be NULL), answered as
 *                DBIndexer.getSequencesUsingPPMTolerance (DBIndexer.java:787-844): the window of
 *                tol = m (1 - 1 / (ppm / 1e6 + 1)), then the hits of the exact-mass probes u_0 = m + tol,
 *                u_{k+1} = u_k + 1e-6 while u_k - tol(u_k) < m and u_{k+1} != u_k, up to the first empty probe,
 *                except those the window already holds.
 * The bucket rule (DBIndexStoreSQLiteMult, Mult:55-56,333-338) empties a query whose bound b has
 * (int)b / (8000 / index_factor) > index_factor - 1; index_factor 0 turns it off (1..8000 otherwise).
 * Every double is computed as the host computes it.  Non-finite mass or tol, a decreasing range_off,
 * range_off != NULL with DBI_TOL_PPM, or another tol_mode: DBI_EINVAL, the message naming the spectrum.
 *
 * The result is the handle's pending hit result with one query per spectrum: counts->nq = n_spectra, hit_off and
 * pep_off per spectrum (no run straddles two spectra), read with dbi_query_hits_read; the < 2^32 hits rule applies.
 * dbi_query_spectra needs a built handle (DBI_ENOTINIT).  dbi_search_unindexed_spectra is dbi_search_unindexed
 * for spectra: same handle rules, candidate cap, *n_candidates, DBI_ERANGE without a pending result and stats; its
 * candidate windows are the merged intervals, or per PPM spectrum its window up to a bound of every probe the walk
 * can make, so every answer equals dbi_query_spectra on the built index.  On one rank of a sharded index,
 * dbi_query_spectra answers Dalton lists with that rank's share, but its PPM walk only sees the rank's own
 * entries: ask a sharded index through dbi_mg_query_spectra_local (or dbi_mg_spectra_stops +
 * dbi_mg_query_spectra), and a sharded unindexed search through dbi_mg_search_unindexed_spectra_local. */
#define DBI_TOL_DA 0
#define DBI_TOL_PPM 1
int dbi_query_spectra(dbi_handle* h, const double* mass, const double* tol, const uint64_t* range_off,
                      uint64_t n_spectra, int tol_mode, int index_factor, dbi_hit_counts* counts);
int dbi_search_unindexed_spectra(dbi_handle* h, const double* mass, const double* tol, const uint64_t* range_off,
                                 uint64_t n_spectra, int tol_mode, int index_factor, uint64_t max_candidates,
                                 dbi_hit_counts* counts, uint64_t* n_candidates);

/* Batched DBIndexer.getProteins(String) (DBIndexer.java:925-947, DBIndexImpl.java:222-237): which index entry,
 * and so which proteins, every peptide of a list is.  Peptide i is residues[offsets[i], offsets[i+1]) (the packed
 * layout of dbi_add_proteins; offsets non-decreasing) with mod pattern modpat[i] in the index's own encoding
 * (byte k = position + 1 of the k-th modified residue, ascending, zero bytes only after the last mod; modpat =
 * NULL: every row unmodified).  A row is FOUND iff the index holds an entry whose peptide is byte-equal to the
 * row and whose mod pattern equals modpat[i] -- the reference's `s.sequence.equals(seq)` filter at zero
 * tolerance.  Its mass is computed on the device the way the index computes it (h2o_proton if added, cterm,
 * nterm, the residues left to right, then the shift of every pattern position left to right) and matched bit
 * for bit; a row matches at most one entry.
 *
 * A row is MALFORMED (status 2; the rest of the batch is answered) when its length is 0 or above
 * DBI_MAX_PEP_LEN, its pattern is not strictly ascending or has a nonzero byte after a zero byte, names a position
 * >= its length or above DBI_MAX_MOD_POS, a residue without a differential shift, or more mods than
 * max_mods_per_peptide (any mod at all on an index without differential mods).  A well-formed row the index does
 * not hold (e.g. a variant whose shifted mass is outside [min_mass, max_mass]) is status 0.
 *
 *   dbi_lookup_peptides(h, ..., &n)        device: mass, search, protein lists (results stay in HBM)
 *   dbi_lookup_peptides_read(h, &out)      D2H into the caller's buffers; any pointer may be NULL
 *
 * A sharded handle answers for its own mass slice (the owner of the slice holding a row's mass finds it) and
 * compares residues through the other ranks' mapped window 2; a handle on which a rank's window 2 is not mapped
 * refuses the call (DBI_EINVAL).  The pending lookup result of a handle is separate from that of
 * dbi_query_hits and is dropped by the next dbi_lookup_peptides, a successful read, dbi_reset_index or
 * dbi_destroy. */
typedef struct dbi_lookup_counts {
  uint64_t n, n_found, n_prot_ids;
} dbi_lookup_counts;
typedef struct dbi_lookup_buffers {
  uint8_t* status;         /* n           0 = not in the index, 1 = found, 2 = malformed row                */
  double* mass;            /* n           calculateMass (+ shifts) as the index computes it; 0 if malformed  */
  uint64_t* entry;         /* n           index entry of this handle (for dbi_fetch); UINT64_MAX unless found */
  uint32_t* first_prot;    /* n           first occurrence (Merge:678-687); 0xffffffff unless found          */
  uint32_t* first_off;     /* n                                                                              */
  uint64_t* prot_list_off; /* n + 1       CSR over prot_ids; empty list unless found                         */
  uint32_t* prot_ids;      /* n_prot_ids  every occurrence, insertion order, duplicates kept (Q6)            */
} dbi_lookup_buffers;
int dbi_lookup_peptides(dbi_handle* h, const uint8_t* residues, const uint64_t* offsets, const uint32_t* modpat,
                        uint64_t n, dbi_lookup_counts* counts);
int dbi_lookup_peptides_read(dbi_handle* h, const dbi_lookup_buffers* out);

/* Page-locked host memory for the buffers above (cudaHostAlloc / cudaFreeHost); a JVM cannot pin
 * its own allocations.  Pageable memory works too, at staging-copy speed. */
int dbi_host_alloc(uint64_t bytes, void** out);
int dbi_host_free(void* p);

/* ProteinCache.getProteinSequence(id) (ProteinCache.java; DBIndexImpl.java:511).
 * Returns a pointer into the handle's host copy, valid until the next dbi_add_proteins on this handle or
 * dbi_destroy. */
int dbi_get_protein(dbi_handle* h, uint32_t id, const uint8_t** residues, uint64_t* len);

/* IndexUtil.calculateMass(seq) (util/IndexUtil.java:197-208): same summation
 * order as the digestion, so a zero-tolerance lookup finds the peptide.  Pure host
 * arithmetic on the handle's parameter table (dbi_lookup_peptides computes the
 * same mass on the device for a whole list). */
int dbi_calculate_mass(dbi_handle* h, const uint8_t* seq, uint64_t len, double* mass);

/* DBIndexStore.getEntryKeys(): distinct (int)(mass*factor) row keys in ascending
 * order (DBIndexer.java:984-992 divides them back).  Two-call sizing. */
int dbi_entry_keys(dbi_handle* h, int32_t* keys, uint64_t capacity, uint64_t* n_keys);

/* Test hook: the records cutSeq would pass to addSequence, in call order
 * (protein, start, end ascending).  Needs params.keep_emitted. */
int dbi_debug_emitted(dbi_handle* h, uint64_t capacity, double* mass, uint32_t* prot, uint32_t* off,
                      uint16_t* len, uint64_t* n);

/* Test hook for the store-level known-answer test (the literals of
 * DBIndexStoreSQLiteMult.main, DBIndexStoreSQLiteMult.java:497-524): index
 * caller-supplied (mass, prot, off, len) records instead of digesting.
 * Proteins must have been added so that sequences can be compared. */
int dbi_build_from_records(dbi_handle* h, const double* mass, const uint32_t* prot,
                           const uint32_t* off, const uint16_t* len, uint64_t n);

/* ---- FASTA ingest (host only): the step before the path ------------------------------------
 * Replaces the external FastaReader passes of DBIndexer.run (DBIndexer.java:560-571,600-605): the
 * file is mapped and parsed by n_threads host threads (<= 0: all) into the packed layout
 * dbi_add_proteins takes.  A line starting with '>' opens a record (defline = rest of the line);
 * the sequence is the following non-empty lines, stripped of white space at both ends,
 * concatenated and upper-cased; anything before the first '>' is ignored.
 *   dbi_fasta_open -> dbi_fasta_counts -> (caller allocates) -> dbi_fasta_read -> dbi_fasta_close
 * residues[n_residues], offsets[n_proteins + 1]; deflines[defline_bytes] (not NUL-terminated) and
 * defline_off[n_proteins + 1] may be NULL. */
typedef struct dbi_fasta dbi_fasta;
int dbi_fasta_open(const char* path, int n_threads, dbi_fasta** out);
int dbi_fasta_counts(const dbi_fasta* f, uint32_t* n_proteins, uint64_t* n_residues, uint64_t* defline_bytes);
int dbi_fasta_read(const dbi_fasta* f, uint8_t* residues, uint64_t* offsets, char* deflines, uint64_t* defline_off);
void dbi_fasta_close(dbi_fasta* f);

/* ---- sharded (multi-GPU) build (SURVEY.md 8e) ------------------------------------------------
 * The reference shards its index by mass into `indexFactor` SQLite files
 * (DBIndexStoreSQLiteMult.java:55-56,215-217) and answers a query from the buckets its range touches
 * (:333-343).  Here a bucket is a GPU holding one slice of the mass axis (with differential mods: two
 * FOLDED slices, a light and a heavy one, see dbi_mg_plan).  One handle per GPU
 * = one rank; rank r is given ITS shard of the FASTA (dbi_add_proteins; the shards follow each other in
 * rank order, so protein ids stay global and in file order).  The bulk data moves inside two kernels
 * that write straight into the other GPUs' memory over NVLink (mapped peer memory); the caller only
 * carries small host arrays between the ranks (three 32 KB histograms, a world x world count matrix,
 * 96-byte window descriptors) with whatever transport it has -- torch.distributed / NCCL between
 * processes (dbindex_b200/multigpu.py), nothing at all when one process holds every handle:
 *
 *   dbi_mg_build_local(handles, n)        the whole sharded build, one process (what a Java host calls)
 *
 * or, one process per GPU, stage by stage:
 *
 *   dbi_mg_begin
 *   dbi_mg_set_shards(sizing) -> dbi_mg_window_ensure(0) -> dbi_mg_set_shards -> [exchange window 0] ->
 *   dbi_mg_pull_proteome                  the other shards arrive on a side stream (joined by dbi_mg_index_base)
 *   dbi_mg_digest                         the start positions of the OWN shard (reads nothing else)
 *   dbi_mg_hist(0) .. [all-gather local histograms + window descriptors] .. dbi_mg_plan_matrix (or all-reduce
 *   .. dbi_mg_plan .. all-gather counts) .. dbi_mg_window_ensure(1, 2) [re-gather the descriptors only if a
 *   window grew] .. dbi_mg_window_import .. dbi_mg_scatter(0) .. [barrier]
 *   dbi_mg_index_base                     sort + merge of this rank's mass slice
 *   [all-gather n_unique] dbi_mg_set_unique
 *   no mods:  dbi_mg_finish
 *   mods:     dbi_mg_groups -> dbi_mg_count(1) [the SAME cuts: a variant lives at most 4 shifts above its
 *             peptide, so most groups stay where their peptide is] .. [all-gather counts] ..
 *             dbi_mg_window_ensure(1) .. dbi_mg_scatter(1) .. [barrier] -> dbi_mg_index_variants -> dbi_mg_finish
 *
 * Afterwards dbi_query / dbi_query_hits / dbi_fetch answer for the rank's slice; base peptides owned by
 * another rank are read through its mapped window 2.  Ranks are <= DBI_MG_MAX_RANKS (one NVSwitch box). */
#define DBI_MG_BINS 4096
#define DBI_MG_MAX_RANKS 16
#define DBI_MG_WIN_PROTEOME 0 /* packed residues of all shards + protein starts        */
#define DBI_MG_WIN_ARENA 1    /* what the exchanges deliver to this rank               */
#define DBI_MG_WIN_UNIQUE 2   /* first occurrence + protein lists of the own peptides  */
#define DBI_REMOTE_BASE 0xffffffffu /* first_prot of a hit whose owner's window 2 is not mapped */

/* How another rank maps a window: a CUDA IPC handle between processes, the pointer itself inside one. */
typedef struct dbi_mg_window {
  uint8_t ipc[64];
  uint64_t ptr;
  uint64_t bytes;
  int32_t device;
  int32_t pid;
  uint64_t reserved;
} dbi_mg_window;

int dbi_mg_begin(dbi_handle* h, int rank, int world);
/* shard_proteins / shard_residues [world]: what every rank added.  window0_bytes != NULL: sizing call;
 * NULL: lay the global buffer out in window 0 and pack the own shard into its place. */
int dbi_mg_set_shards(dbi_handle* h, const uint64_t* shard_proteins, const uint64_t* shard_residues,
                      uint64_t* window0_bytes);
/* make the window hold >= bytes (it only grows; bytes = 0 just describes it) and describe it */
int dbi_mg_window_ensure(dbi_handle* h, int window, uint64_t bytes, dbi_mg_window* desc);
int dbi_mg_window_import(dbi_handle* h, int window, int rank, const dbi_mg_window* desc);
/* bytes of window 1 for n_items of exchange `stage`, or of window 2 for n_items records of exchange 0 */
uint64_t dbi_mg_layout_bytes(int window, int stage, uint64_t n_items, int n_classes);
int dbi_mg_side_classes(dbi_handle* h); /* n_classes argument of dbi_mg_layout_bytes for this handle */
int dbi_mg_pull_proteome(dbi_handle* h);
int dbi_mg_digest(dbi_handle* h, uint64_t* n_records);
/* d_hist: u64[3 * DBI_MG_BINS] in device memory, zeroed by the caller: += weighted | plain | groups histogram
 * of the local items of exchange `stage` (0 = digested records: weight = index entries a record will expand
 * to, groups = variant groups it will list, both estimated from its mod sites; 1 = variant groups: weight =
 * their entries, no third part) over key >> *shift */
int dbi_mg_hist(dbi_handle* h, int stage, void* d_hist, int* shift);
/* host arithmetic on the summed (global) and the own (local) histograms: the cuts of the mass axis
 * [n_slices - 1], this rank's send counts [world], every rank's receive total [world].  n_slices = world: slice s
 * lives on rank s; n_slices = 2 * world: FOLDED slices, slice s lives on rank s < world ? s : 2 * world - 1 - s
 * (one light and one heavy slice per rank: what balances every phase of a build with differential mods).
 * cost[4] = {per item, per estimated group, per unit of weight (index entry), per expected query hit}; NULL =
 * equal weight.  The cuts minimise the sum over the phases of a build (base: items; variants: groups + weight;
 * search: hits) of the slowest rank's cost.  shift / min_mass as used by dbi_mg_hist (they give a bin its
 * mass).  dbi_mg_default_cost fills the measured model of an exchange (cost[4]). */
int dbi_mg_plan(int world, const uint64_t* hist_global, const uint64_t* hist_local, int shift, double min_mass,
                const double* cost, int n_slices, uint32_t* bin_splitters, uint64_t* send_counts,
                uint64_t* recv_totals);
/* the same for a rank that holds every rank's local histograms, hist_all[world][3 * DBI_MG_BINS] (one all-gather
 * instead of an all-reduce plus an exchange of the send counts): cuts + the whole count matrix,
 * matrix[src * world + dst] = items rank src sends to rank dst */
int dbi_mg_plan_matrix(int world, const uint64_t* hist_all, int shift, double min_mass, const double* cost,
                       int n_slices, uint32_t* bin_splitters, uint64_t* matrix);
void dbi_mg_default_cost(int stage, int has_mods, double* cost);
/* items of exchange `stage` this rank would send to every rank under the given cuts [world] */
int dbi_mg_count(dbi_handle* h, int stage, const uint32_t* bin_splitters, int n_slices, uint64_t* send_counts);
/* matrix[s * world + d] = items rank s sends to rank d.  Stable multisplit of the local items straight
 * into the mapped arenas of their destinations; every rank's arena must have been ensured for its
 * receive total and imported here.  A barrier across the ranks must follow before anybody consumes. */
int dbi_mg_scatter(dbi_handle* h, int stage, const uint32_t* bin_splitters, int n_slices, const uint64_t* matrix);
int dbi_mg_index_base(dbi_handle* h);
int dbi_mg_unique_count(dbi_handle* h, uint64_t* n_unique);
int dbi_mg_set_unique(dbi_handle* h, const uint64_t* rank_unique);
int dbi_mg_groups(dbi_handle* h, uint64_t* n_items, uint64_t* n_variants);
int dbi_mg_index_variants(dbi_handle* h);
int dbi_mg_finish(dbi_handle* h);
/* masses at which the entry slices are cut: a query [lo, hi] belongs to the owner of every slice s with
 * split[s-1] <= hi and lo < split[s] (DBIndexStoreSQLiteMult.java:333-343 walks buckets the same way);
 * owner(s) = s < world ? s : slices - 1 - s */
int dbi_mg_slices(dbi_handle* h); /* slices of the built sharded index (world or 2 * world) */
int dbi_mg_split_masses(dbi_handle* h, double* split_mass); /* [dbi_mg_slices - 1] */
int dbi_mg_build_local(dbi_handle** handles, int n);

/* dbi_search_unindexed over a proteome spread over n handles of this process, prepared as for dbi_mg_build_local
 * (handles[r] is rank r and was given shard r with dbi_add_proteins, shards in rank order).  Every rank digests
 * only the start positions of its own shard, keeping the records that can land in a window (K2u / K4u); exchange 0
 * moves them to the owners of their mass slices, with cuts planned from the candidates' histograms; every rank
 * indexes its slices (with mods: exchange 1 and the variant index) and materialises its hits through the other
 * ranks' window 2.  Afterwards every rank's candidate index is dropped, once all ranks are idle.
 *
 * Every rank ends with a pending hit result for all nq windows in the caller's order (counts[r].nq == nq), read with
 * dbi_query_hits_read on handles[r]: rank r's hits of a window are those inside the mass slices it owns in this
 * call.  For every query the union over the ranks equals what dbi_search_unindexed returns on one handle holding the
 * whole proteome (first occurrences and protein lists are global; order inside a query is not a contract).  lo / hi
 * are host pointers with the semantics of dbi_query_hits; the < 2^32 hits rule applies per rank.
 *
 * The handles stay unbuilt (a built one: DBI_EALREADY): dbi_query_hits still returns DBI_ENOTINIT and
 * dbi_mg_build_local still builds the normal sharded index.  The packed proteome (window 0) is kept between calls
 * and packed and pulled again only when a handle received proteins, or the handles are not the ones of the last
 * call.  n_candidates[r] (may be NULL) = candidate records rank r would index after the exchange, known before any
 * arena grows: one above max_candidates (0 = no cap) or at >= 2^32, or an own shard digesting to >= 2^32 records,
 * gives DBI_ERANGE with the counts filled in.  No handle has a pending result after any failure.  dbi_stats_get on
 * handles[r] reports rank r's candidate pipeline: n_emitted = candidates digested from its shard, n_unique /
 * n_entries of its slices, the stage times with params.profile; n_emitted and n_entries summed over the ranks equal
 * the single-GPU call's.  Null or repeated handles, handles created with other parameters (the device aside) and n
 * outside 1..DBI_MG_MAX_RANKS are DBI_EINVAL.  n = 1 is dbi_search_unindexed on handles[0]. */
int dbi_mg_search_unindexed_local(dbi_handle** handles, int n, const double* lo, const double* hi, uint64_t nq,
                                  uint64_t max_candidates, dbi_hit_counts* counts, uint64_t* n_candidates);

/* Batches of spectra (dbi_query_spectra) on a sharded index.  Every rank ends with a pending hit result with one
 * query per spectrum (counts.nq = n_spectra), read with dbi_query_hits_read on that handle; for every spectrum the
 * union over the ranks equals dbi_query_spectra on one handle holding the whole index (same bucket rule, same
 * check_spectra errors; order inside a spectrum is not a contract).  Dalton lists need no exchange: every rank
 * merges the same intervals and answers them over its own entries.  The PPM walk does: its probes u_k have one
 * owner each (the owner of the slice holding u_k, a cut at u_k belonging to the upper slice), and only the owner
 * knows whether a probe is empty.  Rank r computes K_r, the probe at which its share of the walk ends (the walk's
 * own end conditions, or a probe it owns without an entry of that mass); the walk ends at K = min over r of K_r,
 * and every rank then answers the window and the probes before K over its own entries.
 *
 * Rank level (one call per rank, with any transport between the ranks):
 *   dbi_mg_spectra_stops    K_r of every PPM spectrum (mass, ppm) on the built handle h, as rank `rank` of
 *                           `world` under the cuts split_mass[n_slices - 1] (dbi_mg_split_masses gives them for a
 *                           sharded index; n_slices = world or 2 * world, owner(s) = s < world ? s : n_slices-1-s).
 *                           stop[s] = UINT64_MAX when the walk cannot end on this rank.
 *   dbi_mg_query_spectra    dbi_query_spectra on one rank; stop = the minimum over the ranks of their stops
 *                           (DBI_TOL_PPM; NULL is DBI_EINVAL), NULL with DBI_TOL_DA.
 * One process holds every rank:
 *   dbi_mg_query_spectra_local             handles[r] must be rank r of one built sharded index of world n
 *                                          (DBI_EINVAL otherwise, DBI_ENOTINIT for an unbuilt handle); n = 1 is
 *                                          dbi_query_spectra.  counts[n].
 *   dbi_mg_search_unindexed_spectra_local  dbi_mg_search_unindexed_local fed with the candidate windows of
 *                                          dbi_search_unindexed_spectra, computed on every rank's GPU; the walk uses
 *                                          that call's cuts.  Same handle rules, per-rank cap, DBI_ERANGE with
 *                                          n_candidates[r], no pending result on any handle after a failure; every
 *                                          candidate index is dropped once all ranks are idle.  n = 1 is
 *                                          dbi_search_unindexed_spectra.
 * Both _local calls drop every handle's earlier pending result; after a failure none holds one. */
int dbi_mg_spectra_stops(dbi_handle* h, const double* mass, const double* ppm, uint64_t n_spectra, int index_factor,
                         const double* split_mass, int n_slices, int rank, int world, uint64_t* stop);
int dbi_mg_query_spectra(dbi_handle* h, const double* mass, const double* tol, const uint64_t* range_off,
                         uint64_t n_spectra, int tol_mode, int index_factor, const uint64_t* stop,
                         dbi_hit_counts* counts);
int dbi_mg_query_spectra_local(dbi_handle** handles, int n, const double* mass, const double* tol,
                               const uint64_t* range_off, uint64_t n_spectra, int tol_mode, int index_factor,
                               dbi_hit_counts* counts);
int dbi_mg_search_unindexed_spectra_local(dbi_handle** handles, int n, const double* mass, const double* tol,
                                          const uint64_t* range_off, uint64_t n_spectra, int tol_mode,
                                          int index_factor, uint64_t max_candidates, dbi_hit_counts* counts,
                                          uint64_t* n_candidates);

/* Test hook for K7: stable radix sort of n host (key, value) pairs on key bits
 * [begin_bit, end_bit), in place, on the handle's GPU. */
int dbi_debug_radix_sort(dbi_handle* h, uint64_t* keys, uint64_t* vals, uint64_t n, int begin_bit, int end_bit);

void dbi_destroy(dbi_handle* h);

/* sizeof(dbi_params) and sizeof(dbi_stats) as compiled: lets a binding check
 * its struct layout before the first call. */
void dbi_abi_sizes(uint64_t* sizeof_params, uint64_t* sizeof_stats);

/* Device buffers are recycled through a process-wide per-device cache (blocks come
 * from cudaMalloc once and are reused by size, like a long-lived SQLite page cache,
 * DBIndexStoreSQLiteAbstract.java:114-121).  This returns the cached, currently
 * unused blocks of `device` to the driver. */
int dbi_release_cached_memory(int device);

/* Thread-local text of the last error on this thread. */
const char* dbi_last_error(void);

/* Number of CUDA kernels this library has launched in this process (all
 * handles); bench.py reports the delta over the timed region as gpu_launches. */
uint64_t dbi_kernel_launches(void);

#ifdef __cplusplus
}
#endif
#endif /* DBINDEX_GPU_H */
