// kernels.cuh -- host-callable launchers of the hand-written sm_100a kernels.
#pragma once
#include "common.cuh"

namespace dbi {

// Device-resident lookup tables, one copy per handle (2 KB + 256 B + 2 KB).
struct DevTables {
  double mass[256];   // AssignMass.getMass(c), static mods included
  double diff[256];   // DiffModification.getDiffModMass(c)
  uint8_t flags[256]; // kFlagEnzyme | kFlagNocut | kFlagDiffMod
  uint8_t cls[256];   // mod class of a residue = index of its shift among the distinct shifts
  double cls_delta[16]; // shift of each class
};

// Scalar digestion parameters, passed by value.
struct DigestCfg {
  double init_mass;  // ((0 + H2O_PROTON) + cTerm) + nTerm, DBIndexer.java:265-271
  double min_mass;
  double max_mass;
  int32_t max_mc;
  int32_t semi;
  int32_t min_len;
  int32_t max_mods;  // 0 = no differential mods
  double mod_hi;     // max(0, largest shift): upper bound of one mod's mass change
  double mod_lo;     // min(0, smallest shift)
  int32_t n_classes; // distinct shift values
  int32_t n_seq;     // class sequences of length <= max_mods: (C^(K+1)-1)/(C-1); 0 if > 32
  int32_t mand_on;   // mandatoryInternalAAs != null (DBIndexer.java:334-344)
  int32_t filt_max;  // PeptideFilterByMaxOccurrencies: break once kFlagFilterAA residues exceed this; < 0 = off
};

constexpr int kDigestTile = 2048;   // start positions per CTA
constexpr int kScanTile = 4096;     // elements per tile of the generic scans
constexpr int kModTile = 256;       // base peptides per CTA of the mod kernels (heavy peptides are clustered)

// K1: residues + offsets -> padded buffer res[] (0 separator before, between and
// after proteins) and pstart[p] = position of protein p's first residue.
// pos_base: buffer position d_res[0] stands for (a rank of a sharded build packs its shard of the FASTA
// into its place of the global buffer; d_res / d_pstart then point at that place).
void launch_pack(const uint8_t* d_raw, const uint64_t* d_off, uint32_t n_prot, uint64_t n_res, uint8_t* d_res,
                 uint32_t* d_pstart, uint32_t pos_base, uint32_t* d_err, cudaStream_t s);

// K2: records cutSeq emits per START position (start_cnt[g - first position of tile0], saturating
// at 255) and per tile.  Tiles [tile0, tile0 + ntiles) of kDigestTile start positions each (a
// multi-GPU rank digests only its own tile range of the replicated buffer).  res_alloc = bytes
// readable at d_res (a multiple of 16: the tiles are staged with 16-byte bulk copies).
// The start positions a digest launch covers: [start_lo, start_hi) of the residue buffer, holding the
// proteins [prot_lo, prot_hi) (a whole buffer: 0, res_end, 0, n_prot; a sharded build: the rank's own
// shard, so that nothing outside it is read for the result -- the other shards may still be in flight).
struct DigestRange {
  uint32_t start_lo, start_hi, prot_lo, prot_hi;
};

// Unindexed search (dbi_search_unindexed): the mass windows of a query batch and the mass shifts a peptide's
// variants can add.  K2u / K4u keep a record of base mass m with n_mod modifiable sites iff for some
// k <= min(max_mods, n_mod) and some shift interval [s_lo, s_hi] of k mods, [m + s_lo, m + s_hi] meets the
// union of the windows.  Windows are sorted by lo; pmax[i] = max(hi[0..i]); a mass interval [a, b] meets the
// union iff the last window with lo <= b has pmax >= a.  Dropped windows (inverted, NaN, outside
// [min_mass, max_mass]) sort last with lo = +inf.  Passed by value: a kernel parameter.
constexpr int kMaxShiftIv = 64;
struct MassWindows {
  const double* lo;
  const double* pmax;
  uint32_t n;
  int32_t kmax;                               // max_mods (0 without differential mods)
  uint8_t k_end[DBI_MAX_MODS_PER_PEP + 1];    // intervals of <= k mods: [0, k_end[k])
  double s_lo[kMaxShiftIv], s_hi[kMaxShiftIv];
};
#ifdef __CUDACC__
__device__ __forceinline__ bool windows_meet(const MassWindows& w, double a, double b) {
  uint32_t lo = 0, hi = w.n;  // upper_bound(lo[], b)
  while (lo < hi) {
    const uint32_t mid = (lo + hi) >> 1;
    if (__ldg(w.lo + mid) <= b) lo = mid + 1; else hi = mid;
  }
  return lo > 0 && __ldg(w.pmax + lo - 1) >= a;
}
// the record filter of K2u / K4u
struct InWindows {
  MassWindows w;
  __device__ __forceinline__ bool operator()(double m, uint32_t n_mod) const {
    const uint32_t k = n_mod < (uint32_t)w.kmax ? n_mod : (uint32_t)w.kmax;
    const int end = w.k_end[k];
    for (int j = 0; j < end; ++j)
      if (windows_meet(w, __dadd_rn(m, w.s_lo[j]), __dadd_rn(m, w.s_hi[j]))) return true;
    return false;
  }
};
#endif
// host: the shift intervals of p's differential mods (distinct sums of k class shifts +- eps for k = 0, 1, ...;
// a k whose sums do not fit any more gets the band [k mod_lo - eps, k mod_hi + eps])
constexpr double kShiftEps = 1e-9;
void shift_intervals(const DevTables& t, const DigestCfg& cfg, MassWindows* w);

// windows: K2 / K4 emit only the records InWindows keeps (nullptr = every record)
void launch_digest_count(const uint8_t* d_res, const DigestRange& rg, uint64_t res_alloc, const DevTables* d_tb,
                         const DigestCfg& cfg, uint32_t tile0, uint32_t ntiles, uint8_t* d_start_cnt,
                         uint32_t* d_tile_counts, uint32_t* d_err, cudaStream_t s,
                         const MassWindows* windows = nullptr);

// K3: exclusive scan of u32 tile counts into u64 offsets; offs[n] = total.
void launch_scan_u32_to_u64(const uint32_t* d_in, uint64_t n, uint64_t* d_offs, cudaStream_t s);

// K4: emit (mass bits, gpos, prot, len) in (protein, start, end) order.
// (one walk per emitting start: the per-start counts of K2 replace the counting walk)
// o_nmod (optional): differential-mod sites of every record, saturating at 255 -- the sharded build
// estimates a record's downstream cost from it
void launch_digest_emit(const uint8_t* d_res, const DigestRange& rg, uint64_t res_alloc, const DevTables* d_tb,
                        const DigestCfg& cfg, uint32_t tile0, uint32_t ntiles, const uint8_t* d_start_cnt,
                        const uint64_t* d_tile_offs, const uint32_t* d_pstart, uint64_t* o_mass,
                        uint32_t* o_gpos, uint32_t* o_prot, uint16_t* o_len, uint8_t* o_nmod, uint32_t* d_err,
                        cudaStream_t s, const MassWindows* windows = nullptr);

// K12 (window.cu): the windows of a batch for InWindows.  K12a: sort records key = bits(clipped lo) - bits(min_mass)
// (dropped windows: drop_key), value = bits(clipped hi); *nbits = key width.  K12b (after the K7 sort): lo and the
// inclusive prefix max of hi in sorted order.
void launch_win_keys(const double* lo, const double* hi, uint64_t n, double min_mass, double max_mass, uint64_t* key,
                     uint64_t* val, cudaStream_t s);
uint64_t win_drop_key(double min_mass, double max_mass);
void launch_win_pmax(const uint64_t* key, const uint64_t* val, uint64_t n, double min_mass, double max_mass,
                     double* w_lo, double* w_pmax, cudaStream_t s);

// ---- sort helpers / K8 dedup -------------------------------------------------
// Hash pre-sort of large builds: hash[i] = seeded hash of the residues of record i (u32, or u64 when
// wide), idx[i] = i; then key[i] = mass_bits[idx[i]] - base_bits
void launch_hash_records(const uint8_t* d_res, const uint32_t* gpos, const uint16_t* len, uint64_t n, uint32_t seed,
                         bool wide, void* hash, uint32_t* idx, cudaStream_t s);
void launch_gather_mass_key(const uint64_t* mass_bits, const uint32_t* idx, uint64_t n, uint64_t base_bits,
                            uint64_t* key, cudaStream_t s);
// key[i] = mass_bits[i] - base_bits, idx[i] = i: the input of the mass-only base sort
void launch_mass_key(const uint64_t* mass_bits, uint64_t n, uint64_t base_bits, uint64_t* key, uint32_t* idx,
                     cudaStream_t s);
// K8r: after the mass sort (skey, sidx), orders every run of equal skey by (hash & mask(hash_bits),
// record index), rewriting its sidx slots, and writes hash[r] (u32, or u64 when hash_bits > 32) of
// every record r of such a run.  alt: n spare u32 slots; list: run_order_list_cap(n) u32; n_list: 1 u32.
uint64_t run_order_list_cap(uint64_t n);
void launch_run_order(const uint8_t* d_res, const uint64_t* skey, uint32_t* sidx, uint32_t* alt,
                      const uint32_t* gpos, const uint16_t* len, uint64_t n, uint32_t seed, int hash_bits, void* hash,
                      uint32_t* list, uint32_t* n_list, cudaStream_t s);
// head flag of every sorted record + per-tile head counts (tile = kScanTile).
// (hash: u32[n] when hash_bits <= 32, else u64[n] of which the low hash_bits order a run; read only
// for records whose sorted neighbour has the same key)
void launch_dedup_flags(const uint8_t* d_res, const uint64_t* skey, const uint32_t* sidx, const void* hash,
                        int hash_bits, const uint32_t* gpos, const uint16_t* len, uint64_t n, uint8_t* flags,
                        uint32_t* tile_counts, uint32_t* d_err, cudaStream_t s);
// unique records + CSR protein lists.
void launch_dedup_emit(const uint64_t* skey, const uint32_t* sidx, const uint8_t* flags, const uint64_t* tile_offs,
                       const uint32_t* gpos, const uint32_t* prot, const uint16_t* len, uint64_t n,
                       uint64_t base_bits, uint64_t n_unique, double* u_mass, uint32_t* u_gpos, uint32_t* u_prot,
                       uint16_t* u_len, uint64_t* u_plo, uint32_t* plist, cudaStream_t s);

// ---- K5/K6 differential-mod expansion ---------------------------------------
// Tiles [tile0, tile0 + ntiles) of kModTile base peptides; counts[] is indexed by the global
// base id, tile_counts[] / tile_offs[] by (tile - tile0).
void launch_mod_count(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg, const double* u_mass,
                      const uint32_t* u_gpos, const uint16_t* u_len, uint64_t n_unique, uint32_t tile0,
                      uint32_t ntiles, uint32_t* counts, uint32_t* tile_counts, uint32_t* d_err, cudaStream_t s);
void launch_mod_emit(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg, const double* u_mass,
                     const uint32_t* u_gpos, const uint16_t* u_len, uint64_t n_unique, uint32_t tile0,
                     uint32_t ntiles, const uint32_t* counts, const uint64_t* tile_offs, uint64_t base_bits,
                     uint64_t id_off, uint64_t* v_key, uint64_t* v_payload, cudaStream_t s);
// entries from sorted (key, payload): mass = bits(key + base), base id, mod pattern
void launch_split_entries(const uint64_t* skey, const uint64_t* spayload, uint64_t n, uint64_t base_bits,
                          double* e_mass, uint32_t* e_base, uint32_t* e_pat, cudaStream_t s);

// Unique-peptide tables of every rank of a sharded index (world = 1: this GPU's own).  A peptide is
// named by its global id; rank r holds ids [uoff[r], uoff[r + 1]).  A rank whose tables are not mapped
// here (nullptr) makes its peptides come back as DBI_REMOTE_BASE.
constexpr int kMaxRanks = 16;
struct UniqView {
  const uint32_t* gpos[kMaxRanks];
  const uint32_t* prot[kMaxRanks];
  const uint16_t* len[kMaxRanks];
  const uint64_t* plo[kMaxRanks];
  const uint32_t* plist[kMaxRanks];
  uint64_t uoff[kMaxRanks + 1];
  int world;
};
#ifdef __CUDACC__
// owner rank and row of a unique peptide named by its global id
__device__ __forceinline__ int uniq_owner(const UniqView& uv, uint64_t gid, uint64_t* row) {
  int r = 0;
  while (r + 1 < uv.world && gid >= uv.uoff[r + 1]) ++r;
  *row = gid - uv.uoff[r];
  return r;
}
#endif
// Group path (class sequences <= 32, mods_grp.cu): one sort record per (peptide, class sequence)
// group; payload = peptide << 32 | sequence << 27 | variant count.
constexpr int kExpTile = 512;  // entries per CTA of the expansion
// cmask[u * C + c] = 64-bit mask of the sites of shift class c in peptide u (all zero for peptides
// longer than 64 residues, which are counted into *n_long).
void launch_site_masks(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg, const uint32_t* u_gpos,
                       const uint16_t* u_len, uint64_t n_unique, uint64_t* cmask, unsigned long long* n_long,
                       cudaStream_t s);
// *n_long += peptides longer than 64 residues in a length table
void launch_count_long(const uint16_t* len, uint64_t n, unsigned long long* n_long, cudaStream_t s);
// K5g: mask[u] (global id) = the class sequences whose group exists (bit 0 always); tile_groups / tile_vars
// per tile; vt_cnt (nullptr = not wanted) [v * ntiles + tile] = groups of class sequence v in the tile.
void launch_grp_count(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg, const double* u_mass,
                      const uint32_t* u_gpos, const uint16_t* u_len, const uint64_t* cmask, uint64_t n_unique,
                      uint32_t tile0, uint32_t ntiles, uint32_t* mask, uint32_t* tile_groups, uint32_t* tile_vars,
                      uint32_t* vt_cnt, uint32_t* d_err, cudaStream_t s);
// K6g: lists = false: peptide-major, goffs[tile] = first group of the tile (scan of tile_groups);
// lists = true: one list per class sequence, goffs[v * ntiles + tile] = v-major scan of vt_cnt.
void launch_grp_emit(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg, const double* u_mass,
                     const uint32_t* u_gpos, const uint16_t* u_len, const uint64_t* cmask, uint64_t n_unique,
                     uint32_t tile0, uint32_t ntiles, const uint32_t* mask, const uint64_t* goffs, bool lists,
                     uint64_t base_bits, uint64_t id_off, uint64_t* g_key, uint64_t* g_pay, uint32_t* d_err,
                     cudaStream_t s);
// K7m (merge.cu): the S sorted group lists of K6g's list layout merged by (key, payload) in one pass.
// Every kGmStride-th record of each list is a sample; the samples whose rank among all samples is a multiple
// of kGmSplit cut the output into tiles of at most (kGmSplit + S) * kGmStride records, each merged in
// shared memory.  The output order is that of a stable key sort of the peptide-major layout.
constexpr int kGrpMaxLists = 32;
constexpr int kGmStride = 32;
constexpr int kGmSplit = 64;
struct GroupLists {
  uint64_t start[kGrpMaxLists + 1];  // list v = records [start[v], start[v + 1])
  uint64_t soff[kGrpMaxLists + 1];   // samples of list v = [soff[v], soff[v + 1]) (group_lists_plan)
  int n_lists;
};
// fills soff from start / n_lists
void group_lists_plan(GroupLists* gl);
size_t group_merge_tmp_bytes(const GroupLists& gl);
// o_cnt[i] = variant count of merged record i (payload & (2^27 - 1)).  A tile over its capacity raises
// kErrMergeCap (cannot happen by construction; checked anyway).
void launch_group_merge(const GroupLists& gl, const uint64_t* key, const uint64_t* pay, uint64_t* o_key,
                        uint64_t* o_pay, uint32_t* o_cnt, void* tmp, uint32_t* d_err, cudaStream_t s);
void launch_grp_extract_cnt(const uint64_t* pay, uint64_t n, uint32_t* cnt, cudaStream_t s);
// first[t] = group holding entry t * kExpTile, t in [0, tiles]; first[tiles] = n_groups - 1
void launch_grp_tile_first(const uint64_t* eoff, uint64_t n_groups, uint64_t n_entries, uint32_t* first,
                           cudaStream_t s);
// entries of the sorted groups; groups of long peptides are listed in long_list and written by a
// second kernel (launched when long_cap > 0).  The payload's peptide field is a ROW of cmask /
// u_gpos / u_len; gid_tab (sharded build: rows are arrival slots of the group exchange) maps a row
// to the peptide's global id, nullptr = the row is the id; uv (with gid_tab) = the tables (of any rank)
// holding (gpos, len) of a peptide, which only the rare peptides longer than 64 residues need.
void launch_grp_expand(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg, const uint32_t* u_gpos,
                       const uint16_t* u_len, const uint64_t* cmask, const uint32_t* gid_tab, const UniqView* uv,
                       const uint64_t* skey, const uint64_t* spay, const uint64_t* eoff, const uint32_t* tile_first,
                       uint64_t n_groups, uint64_t n_entries, uint64_t base_bits, double* e_mass, uint32_t* e_base,
                       uint32_t* e_pat, uint32_t* long_list, uint32_t* long_count, uint32_t long_cap, uint32_t* d_err,
                       cudaStream_t s);

// Compact index (group arrays kept, entries never written): K6q expands entry ranges.  Range q = entries
// [begin[q], begin[q] + c_q) to output positions [out_off[q], out_off[q + 1]); tiles of kExpTile entries,
// tile_q[t] = the range of tile t, tile_off = exclusive scan of the tiles per range.
struct ExpRanges {
  const uint32_t* tile_q;
  const uint64_t* tile_off;
  const uint64_t* begin;
  const uint64_t* out_off;
};
// A compact index's groups for the lookup (K11a over the groups): payloads, entry offsets, site masks.
struct GroupView {
  const uint64_t* pay;
  const uint64_t* eoff;
  const uint64_t* cmask;
  int n_classes;
};
// K6q: (mass, peptide, pattern) of every entry of the ranges, in the order of K6x.  Groups of peptides longer
// than 64 residues are counted into *long_count and listed as (group, tile) pairs while there is room
// (long_cap pairs); the caller runs the kernel again with a larger list when the count exceeds it.
void launch_grp_expand_ranges(const DigestCfg& cfg, const uint64_t* cmask, const double* g_mass, const uint64_t* g_pay,
                              const uint64_t* g_eoff, uint64_t n_groups, const ExpRanges& rg, uint64_t n_tiles,
                              double* o_mass, uint32_t* o_base, uint32_t* o_pat, uint32_t* long_list,
                              uint32_t* long_count, uint32_t long_cap, uint32_t* d_err, cudaStream_t s);
// the windowed K6l over the n_listed pairs K6q listed
void launch_grp_expand_ranges_long(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg,
                                   const uint32_t* u_gpos, const uint16_t* u_len, const double* g_mass,
                                   const uint64_t* g_pay, const uint64_t* g_eoff, const ExpRanges& rg,
                                   const uint32_t* long_list, const uint32_t* long_count, uint32_t n_listed,
                                   double* o_mass, uint32_t* o_base, uint32_t* o_pat, cudaStream_t s);
// key[i] += base_bits: sorted group keys -> group mass bits
void launch_grp_key_mass(uint64_t* key, uint64_t n, uint64_t base_bits, cudaStream_t s);
// group ranges (K9 over the group masses) -> entry ranges through eoff, in place.  cnt32 (optional) = the
// counts as u32, and *over = 1 if one is >= 2^32; ntile32 (optional) = K6q tiles of every range.
void launch_grp_entry_ranges(const uint64_t* eoff, uint64_t nq, uint64_t* begin, uint64_t* count, uint32_t* cnt32,
                             uint32_t* ntile32, uint32_t* over, cudaStream_t s);

// ---- K9/K10 query ----------------------------------------------------------------
// cnt32 (optional): the hit counts again as u32, the input of the hit-offset scan
void launch_query(const double* e_mass, uint64_t n_entries, const double* lo, const double* hi, uint64_t nq,
                  uint64_t* hit_begin, uint64_t* hit_count, uint32_t* cnt32, cudaStream_t s);

// ---- K13/K14 spectra (spectra.cu) --------------------------------------------------
// K13a: the Dalton range lists of n spectra (spectrum s = ranges [range_off[s], range_off[s+1])) clamped, sorted,
// merged and checked against the bucket rule (index_factor 0: off); the merged intervals of s in its slots from
// range_off[s] of o_lo / o_hi, cnt[s] = their number (0: the spectrum is empty).  launch_spec_compact packs them
// at ioff = exclusive scan of cnt.
void launch_spec_intervals(const double* mass, const double* tol, const uint64_t* range_off, uint64_t n,
                           int index_factor, double* o_lo, double* o_hi, uint32_t* cnt, cudaStream_t s);
void launch_spec_compact(const uint64_t* range_off, const uint64_t* ioff, uint64_t n, const double* s_lo,
                         const double* s_hi, double* o_lo, double* o_hi, cudaStream_t s);
// K13b: the window [max(0, m - tol), m + tol] of n PPM spectra; c_lo / c_hi (both NULL or neither): the candidate
// window of an unindexed search, which also holds every probe the walk can make
void launch_spec_ppm_window(const double* mass, const double* ppm, uint64_t n, double* w_lo, double* w_hi,
                            double* c_lo, double* c_hi, cudaStream_t s);
// K14: the exact-mass probe walk of every PPM spectrum over the sorted entry masses; count pass (window + probes per
// spectrum), then the intervals at ioff = exclusive scan of the counts.  stop != NULL (a sharded index): the walk of
// spectrum s ends at probe stop[s] (K14s, minimum over the ranks) instead of at the first probe without an entry.
void launch_spec_probe_count(const double* e_mass, uint64_t n_entries, const double* mass, const double* ppm,
                             const double* w_lo, const double* w_hi, uint64_t n, int index_factor, const uint64_t* stop,
                             uint32_t* cnt, cudaStream_t s);
void launch_spec_probe_emit(const double* e_mass, uint64_t n_entries, const double* mass, const double* ppm,
                            const double* w_lo, const double* w_hi, uint64_t n, int index_factor, const uint64_t* stop,
                            const uint64_t* ioff, double* o_lo, double* o_hi, cudaStream_t s);
// The mass slices of a sharded index as one rank sees them: slice x = [cut[x-1], cut[x]) (cut[-1] = -inf,
// cut[n_slices-1] = +inf); bit x of `mine` is set when the rank owns slice x.  Passed by value (~260 bytes).
struct SliceCuts {
  double cut[2 * kMaxRanks - 1];
  int n_slices;
  uint32_t mine;
};
// K14s: stop[s] = the probe at which this rank's share of spectrum s's walk ends (UINT64_MAX: not on this rank)
void launch_spec_stops(const double* e_mass, uint64_t n_entries, const double* mass, const double* ppm,
                       const double* w_hi, uint64_t n, int index_factor, const SliceCuts& cuts, uint64_t* stop,
                       cudaStream_t s);
// per-interval hit_off / pep_off (K10) -> per-spectrum: hit_off[s] = iv_hit_off[ioff[s]], s = 0..n
void launch_spec_collapse(const uint64_t* ioff, uint64_t n, const uint64_t* iv_hit_off, const uint64_t* iv_pep_off,
                          uint64_t* hit_off, uint64_t* pep_off, cudaStream_t s);

// K10a-c: the hits of a query batch grouped in RUNS (consecutive hits of one query that are variants of
// one peptide with one mass).  hit_off = exclusive scan of the hit counts; pep_off = runs before every
// query; what parseAddPeptideInfo materialises
// (DBIndexStoreSQLiteByteIndexMerge.java:386-481) is written once per run, the mod pattern per hit.
// (a query's hits are cut into segments of 256, one warp each: seg_off = scan of the segment counts,
// seg_q[s] = query of segment s, seg_run_off = scan of the runs that start in every segment)
void launch_hits_seg_count(const uint64_t* hit_count, uint64_t nq, uint32_t* nseg32, cudaStream_t s);
void launch_hits_seg_fill(const uint64_t* seg_off, uint64_t nq, uint32_t* seg_q, cudaStream_t s);
void launch_hits_count_runs(const double* e_mass, const uint32_t* e_base, const uint32_t* seg_q, const uint64_t* seg_off,
                            const uint64_t* hit_begin, const uint64_t* hit_off, uint64_t nseg, uint32_t* nruns32,
                            cudaStream_t s);
void launch_hits_pep_off(const uint64_t* seg_off, const uint64_t* seg_run_off, uint64_t nq, uint64_t* pep_off,
                         cudaStream_t s);
void launch_hits_runs(const double* e_mass, const uint32_t* e_base, uint64_t ent_off, const uint32_t* e_pat,
                      const UniqView& uv, const uint32_t* seg_q, const uint64_t* seg_off, const uint64_t* hit_begin,
                      const uint64_t* hit_off, const uint64_t* seg_run_off, uint64_t nseg, uint32_t* o_pat,
                      uint64_t* pep_hit_off, double* o_mass, uint32_t* pep_entry, uint32_t* len32, uint32_t* np32,
                      cudaStream_t s);
void launch_peps_gather(const uint8_t* d_res, const uint32_t* pstart, const uint32_t* e_base, uint64_t ent_off,
                        const UniqView& uv, const uint32_t* pep_entry, const uint64_t* seq_off, const uint64_t* plo_out,
                        uint64_t n_peps, uint32_t* o_prot, uint32_t* o_off, uint16_t* o_len, uint8_t* o_flanks,
                        uint8_t* o_seq, uint32_t* o_ids, cudaStream_t s);
// per-entry protein-list length for entries [begin, begin+count) + per-tile sums.
// e_base == nullptr means "entry i is unique peptide base_off + i" (no differential mods).
// Base peptides are named by global ids and resolved through uv; a peptide whose owner's tables are
// not mapped has list size 0 and comes back as first_prot = DBI_REMOTE_BASE, first_off = global id.
void launch_fetch_sizes(const uint32_t* e_base, uint64_t base_off, const UniqView& uv, uint64_t begin, uint64_t count,
                        uint32_t* sizes, uint32_t* tile_counts, cudaStream_t s);
// what parseAddPeptideInfo materialises per hit; any output may be nullptr.
void launch_fetch_gather(const double* e_mass, const uint32_t* e_base, uint64_t base_off, const UniqView& uv,
                         const uint32_t* e_pat, const uint32_t* pstart, uint64_t begin, uint64_t count,
                         const uint32_t* sizes, const uint64_t* tile_offs, double* o_mass, uint32_t* o_prot,
                         uint32_t* o_off, uint16_t* o_len, uint32_t* o_pat, uint64_t* o_list_off, uint32_t* o_ids,
                         cudaStream_t s);
// K11 batched peptide lookup (dbi_lookup_peptides).  Row i = q_res[q_off[i] - q_off[0], q_off[i+1] - q_off[0])
// with mod pattern q_pat[i] (nullptr = all unmodified).  K11a: status (0 absent, 1 found, 2 malformed), mass,
// entry (UINT64_MAX unless found), protein-list length o_np, and *n_found += found rows.
void launch_lookup_match(const uint8_t* d_res, const double* e_mass, uint64_t n_entries, const uint32_t* e_base,
                         uint64_t ent_off, const uint32_t* e_pat, const UniqView& uv, const DevTables* d_tb,
                         double init_mass, int max_mods, const uint8_t* q_res, const uint64_t* q_off,
                         const uint32_t* q_pat, uint64_t n, uint8_t* o_status, double* o_mass, uint64_t* o_entry,
                         uint32_t* o_np, unsigned long long* n_found, const GroupView* gv, uint64_t* o_gid,
                         cudaStream_t s);
// K11b: first occurrence + protein ids of the found rows (plo = scan of o_np); 0xffffffff for the others
void launch_lookup_gather(const uint8_t* status, const uint64_t* entry, const uint32_t* e_base, uint64_t ent_off,
                          const UniqView& uv, const uint32_t* pstart, const uint64_t* plo, uint64_t n,
                          uint32_t* o_prot, uint32_t* o_off, uint32_t* o_ids, cudaStream_t s);
// distinct (int)(mass*factor) keys: flags + compaction
void launch_key_flags(const double* e_mass, uint64_t n, double factor, uint8_t* flags, uint32_t* tile_counts,
                      cudaStream_t s);
void launch_key_emit(const double* e_mass, uint64_t n, double factor, const uint8_t* flags,
                     const uint64_t* tile_offs, int32_t* keys, cudaStream_t s);

// ---- multi-GPU exchange helpers (mg.cu) -----------------------------------------------------
constexpr int kMgBins = 4096;  // histogram bins over the top bits of the radix key
// Where the items of one exchange go.  The mass axis is cut into n_thr + 1 SLICES (slice of an item =
// number of thresholds <= key - sub); there are `world` slices, slice s living on rank s, or 2 * world
// FOLDED slices: slice s lives on rank s < world ? s : 2 * world - 1 - s, so that every rank holds one light
// slice (many records, few variants) and one heavy slice (few records, many variants).  This rank's items
// for destination d arrive at rows row0[d] .. of d's arrays (after the items of the lower ranks).
constexpr int kMaxSlices = 2 * kMaxRanks;
struct MgPlan {
  uint64_t thr[kMaxSlices];
  uint64_t row0[kMaxRanks];
  int world;
  int n_thr;
};
__host__ __device__ inline uint32_t mg_slice_owner(uint32_t slice, uint32_t n_slices, uint32_t world) {
  return slice < world ? slice : n_slices - 1u - slice;
}
// hist[0 .. kMgBins) += weight, hist[kMgBins .. 2 kMgBins) += 1, hist[2 kMgBins .. 3 kMgBins) += group estimate
// over min(kMgBins-1, (key[i] - sub) >> shift) (hist is zeroed by the caller); weight of item i =
// wpay ? (wpay[i] & wmask) + wadd  (group records carry their variant count)  :  wtab ? wtab[wcode[i]]
// (records: variants of a peptide with wcode[i] mod sites)  :  1;  group estimate = gtab ? gtab[wcode[i]] : 0.
void launch_mg_hist(const uint64_t* key, uint64_t n, uint64_t sub, int shift, const uint64_t* wpay, uint64_t wmask,
                    uint32_t wadd, const uint8_t* wcode, const uint32_t* wtab, const uint32_t* gtab,
                    unsigned long long* hist, cudaStream_t s);
// counts[d] += items whose destination is d (dest = number of thresholds <= key - sub); counts zeroed by the caller
void launch_mg_count(const uint64_t* key, uint64_t n, uint64_t sub, const MgPlan& pl, unsigned long long* counts,
                     cudaStream_t s);
// destination arrays (mapped peer pointers; the own rank's are local)
struct MgRecDst {
  uint64_t* mass[kMaxRanks];
  uint32_t* gpos[kMaxRanks];
  uint32_t* prot[kMaxRanks];
  uint16_t* len[kMaxRanks];
};
struct MgGrpDst {
  uint64_t* key[kMaxRanks];
  uint64_t* pay[kMaxRanks];
  uint32_t* gid[kMaxRanks];   // global id of the group's peptide, by arrival row
  uint64_t* mask[kMaxRanks];  // its C site masks, [row * C + c]
};
size_t mg_scatter_tmp_bytes(uint64_t n);
// fused multisplit + peer-memory all-to-all (mg.cu); tmp = mg_scatter_tmp_bytes(n) bytes
void launch_mg_scatter_records(const uint64_t* mass, const uint32_t* gpos, const uint32_t* prot, const uint16_t* len,
                               uint64_t n, uint64_t sub, const MgPlan& pl, const MgRecDst& dst, void* tmp,
                               cudaStream_t s);
// The payloads name LOCAL peptide rows (id_off turns them into global ids).  C > 0: group records, the
// payload's peptide field becomes the arrival row and (gid, masks) travel as side tables; C == 0:
// per-variant records, only (key, payload + id_off) travel.
void launch_mg_scatter_groups(const uint64_t* key, const uint64_t* pay, const uint64_t* cmask, int C, uint64_t id_off,
                              uint64_t n, const MgPlan& pl, const MgGrpDst& dst, void* tmp, cudaStream_t s);
// list length of every unique peptide: cnt[u] = plo[u+1] - plo[u]
void launch_plo_to_counts(const uint64_t* plo, uint64_t n, uint32_t* cnt, cudaStream_t s);
// full exclusive scan: offs[i] = sum(in[0..i)), offs[n] = total; tmp = (ntiles + 1) u64 + ntiles u64 (64-bit tile sums)
void launch_full_scan_u32_to_u64(const uint32_t* in, uint64_t n, uint64_t* offs, void* tmp, cudaStream_t s);
size_t full_scan_tmp_bytes(uint64_t n);

}  // namespace dbi
