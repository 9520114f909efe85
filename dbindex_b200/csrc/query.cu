// query.cu -- K9 batched lower/upper bound, K10 hit gather, K11 peptide lookup, entry-key listing.
//
// Replaces DBIndexStoreSQLiteByteIndexMerge.getSequences (Merge:146-217): the
// `SELECT ... WHERE precursor_mass_key BETWEEN minKey AND maxKey` plus the exact
// double filter of parseAddPeptideInfo (Merge:415-419) become one lower_bound and
// one upper_bound on the totally ordered mass array; both ends inclusive (Q5).
#include <cassert>

#include "kernels.cuh"
#include "mods_common.cuh"

namespace dbi {
namespace {

constexpr int Q_THREADS = 256;
constexpr int Q_IPT = kScanTile / Q_THREADS;

// first index with mass >= v
__device__ __forceinline__ uint64_t lower_bound_d(const double* __restrict__ a, uint64_t n, double v) {
  uint64_t lo = 0, len = n;
  while (len > 0) {
    const uint64_t half = len >> 1;
    const double m = __ldg(a + lo + half);
    if (m < v) { lo += half + 1; len -= half + 1; } else { len = half; }
  }
  return lo;
}
// first index with mass > v
__device__ __forceinline__ uint64_t upper_bound_d(const double* __restrict__ a, uint64_t n, double v) {
  uint64_t lo = 0, len = n;
  while (len > 0) {
    const uint64_t half = len >> 1;
    const double m = __ldg(a + lo + half);
    if (m <= v) { lo += half + 1; len -= half + 1; } else { len = half; }
  }
  return lo;
}

__global__ void __launch_bounds__(Q_THREADS)
    query_kernel(const double* __restrict__ e_mass, uint64_t n, const double* __restrict__ lo,
                 const double* __restrict__ hi, uint64_t nq, uint64_t* __restrict__ hit_begin,
                 uint64_t* __restrict__ hit_count, uint32_t* __restrict__ cnt32) {
  const uint64_t q = (uint64_t)blockIdx.x * Q_THREADS + threadIdx.x;
  if (q >= nq) return;
  const double l = lo[q], h = hi[q];
  const uint64_t b = lower_bound_d(e_mass, n, l);  // mass < minMass skipped (Merge:419)
  const uint64_t e = upper_bound_d(e_mass, n, h);  // mass > maxMass stops (Merge:415)
  hit_begin[q] = b;
  hit_count[q] = e > b ? e - b : 0;
  if (cnt32) cnt32[q] = e > b ? (uint32_t)(e - b) : 0u;  // an index holds < 2^32 entries
}

constexpr int HX_WARPS = Q_THREADS / 32;
constexpr uint32_t HX_SEG = 256;  // hits per warp

// The answer to a batch is grouped the way the index is: a RUN = consecutive hits of one query that are
// variants of one peptide with one mass (one variant group of the index, contiguous by construction).
// Everything parseAddPeptideInfo derives from the peptide (first occurrence, residues, flanks, protein
// list) is materialised once per run; a hit carries only its mod pattern.

// first hit of a run?  (hit i of a query that starts at entry b; no differential mods: every entry is a
// peptide of its own)
__device__ __forceinline__ bool run_head(const unsigned long long* __restrict__ mass_bits,
                                         const uint32_t* __restrict__ e_base, uint64_t e, uint32_t i) {
  if (!e_base || i == 0) return true;
  return e_base[e] != e_base[e - 1] || mass_bits[e] != mass_bits[e - 1];
}

// The hits of a query are processed in SEGMENTS of HX_SEG consecutive hits, one warp each, so that a
// +-3 Da window with 10^5 hits and a 10 ppm window with 50 spread over the machine alike.
// seg_off = exclusive scan of ceil(count / HX_SEG) over the queries.
__global__ void __launch_bounds__(Q_THREADS)
    hits_seg_count_kernel(const uint64_t* __restrict__ hit_count, uint64_t nq, uint32_t* __restrict__ nseg32) {
  const uint64_t q = (uint64_t)blockIdx.x * Q_THREADS + threadIdx.x;
  if (q < nq) nseg32[q] = (uint32_t)((hit_count[q] + HX_SEG - 1) / HX_SEG);
}

__global__ void __launch_bounds__(Q_THREADS)
    hits_seg_fill_kernel(const uint64_t* __restrict__ seg_off, uint64_t nq, uint32_t* __restrict__ seg_q) {
  const uint64_t q = (uint64_t)blockIdx.x * HX_WARPS + (threadIdx.x >> 5);
  if (q >= nq) return;
  const uint64_t s0 = seg_off[q], s1 = seg_off[q + 1];
  for (uint64_t s = s0 + lane_id(); s < s1; s += 32) seg_q[s] = (uint32_t)q;
}

struct HitSeg {
  uint64_t b;    // index entry of the segment's first hit
  uint64_t h0;   // its position in the batch's hit list
  uint32_t i0;   // its rank inside its query
  uint32_t n;    // hits in the segment
};
__device__ __forceinline__ HitSeg hit_segment(uint64_t s, const uint32_t* __restrict__ seg_q,
                                              const uint64_t* __restrict__ seg_off,
                                              const uint64_t* __restrict__ hit_begin,
                                              const uint64_t* __restrict__ hit_off) {
  const uint32_t q = seg_q[s];
  const uint64_t k = s - seg_off[q];
  const uint64_t hq = hit_off[q], nq_hits = hit_off[q + 1] - hq;
  HitSeg g;
  g.i0 = (uint32_t)(k * HX_SEG);
  g.n = (uint32_t)min((uint64_t)HX_SEG, nq_hits - g.i0);
  g.b = hit_begin[q] + g.i0;
  g.h0 = hq + g.i0;
  return g;
}

// K10a: one warp per segment, lanes stride its hits (consecutive entries -> coalesced): runs that START
// in the segment.
__global__ void __launch_bounds__(Q_THREADS)
    hits_count_runs_kernel(const double* __restrict__ e_mass, const uint32_t* __restrict__ e_base,
                           const uint32_t* __restrict__ seg_q, const uint64_t* __restrict__ seg_off,
                           const uint64_t* __restrict__ hit_begin, const uint64_t* __restrict__ hit_off, uint64_t nseg,
                           uint32_t* __restrict__ nruns32) {
  const uint64_t sg = (uint64_t)blockIdx.x * HX_WARPS + (threadIdx.x >> 5);
  if (sg >= nseg) return;
  const HitSeg g = hit_segment(sg, seg_q, seg_off, hit_begin, hit_off);
  const unsigned long long* mb = reinterpret_cast<const unsigned long long*>(e_mass);
  uint32_t cnt = 0;
  for (uint32_t i = lane_id(); i < g.n; i += 32) cnt += run_head(mb, e_base, g.b + i, g.i0 + i) ? 1u : 0u;
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if (lane_id() == 0) nruns32[sg] = cnt;
}

// runs of every query: pep_off[q] = runs that start before the first segment of q (nq + 1 values)
__global__ void __launch_bounds__(Q_THREADS)
    hits_pep_off_kernel(const uint64_t* __restrict__ seg_off, const uint64_t* __restrict__ seg_run_off, uint64_t nq,
                        uint64_t* __restrict__ pep_off) {
  const uint64_t q = (uint64_t)blockIdx.x * Q_THREADS + threadIdx.x;
  if (q <= nq) pep_off[q] = seg_run_off[seg_off[q]];
}

// K10b: same mapping.  seg_run_off = exclusive scan of the run counts; a warp numbers the runs of its
// segment on the fly (ballot prefix), writes the mod pattern of every hit, and the first hit of every run
// fills the run's row: where its hits start, the exact mass, the index entry (for K10c), residue count
// and protein-list length (scanned into the two CSRs afterwards).
__global__ void __launch_bounds__(Q_THREADS)
    hits_runs_kernel(const double* __restrict__ e_mass, const uint32_t* __restrict__ e_base, uint64_t ent_off,
                     const uint32_t* __restrict__ e_pat, const __grid_constant__ UniqView uv,
                     const uint32_t* __restrict__ seg_q, const uint64_t* __restrict__ seg_off,
                     const uint64_t* __restrict__ hit_begin, const uint64_t* __restrict__ hit_off,
                     const uint64_t* __restrict__ seg_run_off, uint64_t nseg, uint32_t* __restrict__ o_pat,
                     uint64_t* __restrict__ pep_hit_off, double* __restrict__ o_mass, uint32_t* __restrict__ pep_entry,
                     uint32_t* __restrict__ len32, uint32_t* __restrict__ np32) {
  const uint64_t sg = (uint64_t)blockIdx.x * HX_WARPS + (threadIdx.x >> 5);
  if (sg >= nseg) return;
  const HitSeg g = hit_segment(sg, seg_q, seg_off, hit_begin, hit_off);
  const unsigned long long* mb = reinterpret_cast<const unsigned long long*>(e_mass);
  uint64_t done = seg_run_off[sg];  // runs that start before the current 32 hits
  for (uint32_t j = 0; j < g.n; j += 32) {  // warp-uniform trip count
    const uint32_t i = j + lane_id();
    const bool valid = i < g.n;
    const uint64_t e = g.b + i;
    const bool head = valid && run_head(mb, e_base, e, g.i0 + i);
    const unsigned heads = __ballot_sync(0xffffffffu, head);
    if (valid && o_pat) o_pat[g.h0 + i] = e_pat ? e_pat[e] : 0u;
    if (head) {
      const uint64_t p = done + (uint32_t)__popc(heads & lanemask_lt());
      const uint64_t gid = e_base ? (uint64_t)e_base[e] : ent_off + e;
      uint64_t row;
      const int r = uniq_owner(uv, gid, &row);
      uint32_t len = 0, np = 0;
      if (uv.len[r]) {
        len = uv.len[r][row];
        np = (uint32_t)(uv.plo[r][row + 1] - uv.plo[r][row]);
      }
      pep_hit_off[p] = g.h0 + i;
      o_mass[p] = e_mass[e];
      pep_entry[p] = (uint32_t)e;
      len32[p] = len;
      np32[p] = np;
    }
    done += (uint32_t)__popc(heads);
  }
}

// K10c: a CTA materialises HG_TILE consecutive runs.  Per-run scalars are gathered by one thread per run
// (random reads of the owner tables, coalesced writes); the peptide residues and the flanks, whose
// output regions are contiguous for consecutive runs, are written by the whole CTA in 16-byte chunks:
// a thread finds the run its chunk starts in (binary search over the tile's offsets in shared memory),
// then copies the residues of that run and its successors word by word (aligned 32-bit loads of the
// residue buffer, funnel-shifted into place).
constexpr int HG_TILE = Q_THREADS;

// 4 residue bytes starting at buffer position pos (any alignment)
__device__ __forceinline__ uint32_t ld_res4(const uint8_t* __restrict__ res, uint32_t pos) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(res) + (pos >> 2);
  const uint32_t sh = (pos & 3u) * 8u;
  const uint32_t a = __ldg(w);
  if (sh == 0) return a;
  return __funnelshift_r(a, __ldg(w + 1), sh);
}

// What parseAddPeptideInfo takes from the peptide itself (K10c per run, K11b per found lookup row): the first
// occurrence's protein and offset inside it (Merge:678-687), and every occurrence's protein id in insertion
// order (Merge:449-475) into ids[0 ..).  Row `row` of rank r, whose tables are mapped; any output may be nullptr.
__device__ __forceinline__ void peptide_occurrences(const UniqView& uv, int r, uint64_t row,
                                                    const uint32_t* __restrict__ pstart, uint32_t* o_prot,
                                                    uint32_t* o_off, uint32_t* ids) {
  const uint32_t gp = uv.gpos[r][row], pr = uv.prot[r][row];
  if (o_prot) *o_prot = pr;
  if (o_off) *o_off = gp - pstart[pr];  // sequenceOffset inside the first protein
  if (ids) {
    const uint64_t src = uv.plo[r][row], n = uv.plo[r][row + 1] - src;
    for (uint64_t k = 0; k < n; ++k) ids[k] = uv.plist[r][src + k];
  }
}

__global__ void __launch_bounds__(Q_THREADS)
    peps_gather_kernel(const uint8_t* __restrict__ res, const uint32_t* __restrict__ pstart,
                       const uint32_t* __restrict__ e_base, uint64_t ent_off, const __grid_constant__ UniqView uv,
                       const uint32_t* __restrict__ pep_entry, const uint64_t* __restrict__ seq_off,
                       const uint64_t* __restrict__ plo_out, uint64_t n_peps, uint32_t* __restrict__ o_prot,
                       uint32_t* __restrict__ o_off, uint16_t* __restrict__ o_len, uint8_t* __restrict__ o_flanks,
                       uint8_t* __restrict__ o_seq, uint32_t* __restrict__ o_ids) {
  __shared__ uint32_t s_gpos[HG_TILE];
  __shared__ uint32_t s_soff[HG_TILE + 1];  // seq offsets relative to the tile's first byte
  __shared__ __align__(16) uint8_t s_fl[HG_TILE * 6 + 16];
  const int t = threadIdx.x;
  const uint64_t h0 = (uint64_t)blockIdx.x * HG_TILE;
  const uint32_t tile_n = (uint32_t)min((uint64_t)HG_TILE, n_peps - h0);
  const uint64_t h = h0 + t;
  const uint64_t seq0 = seq_off[h0];
  if (t == 0) s_soff[tile_n] = (uint32_t)(seq_off[h0 + tile_n] - seq0);
  if ((uint32_t)t < tile_n) {
    const uint64_t e = pep_entry[h];
    const uint64_t gid = e_base ? (uint64_t)e_base[e] : ent_off + e;
    uint64_t row;
    const int r = uniq_owner(uv, gid, &row);
    s_soff[t] = (uint32_t)(seq_off[h] - seq0);
    uint8_t* f = s_fl + 6 * t;
    if (!uv.len[r]) {  // the owner's tables are not mapped: the caller resolves the peptide through its owner
      if (o_prot) o_prot[h] = DBI_REMOTE_BASE;
      if (o_off) o_off[h] = (uint32_t)gid;
      if (o_len) o_len[h] = 0;
      s_gpos[t] = 0;
      for (int k = 0; k < 6; ++k) f[k] = '-';
    } else {
      const uint32_t gp = uv.gpos[r][row], len = uv.len[r][row];
      s_gpos[t] = gp;
      if (o_len) o_len[h] = (uint16_t)len;
      // Util.getResidues (Util.java:130-162): up to 3 residues on the left, '-' padded on the left; on
      // the right min(3, protLen - end - 1) residues -- the reference's off-by-one drops the last
      // residue of the protein from the right flank (SURVEY.md Q8) -- '-' padded on the right.
      const uint8_t l2 = ld_res(res, gp - 1);
      const uint8_t l1 = l2 ? ld_res(res, gp - 2) : (uint8_t)0;
      const uint8_t l0 = l1 ? ld_res(res, gp - 3) : (uint8_t)0;
      f[0] = l0 ? l0 : (uint8_t)'-';
      f[1] = l1 ? l1 : (uint8_t)'-';
      f[2] = l2 ? l2 : (uint8_t)'-';
      const uint32_t endp = gp + len;  // first position after the peptide
      uint8_t rr[4];
      uint32_t remaining = 0;          // residues after the peptide, up to 4
      while (remaining < 4 && (rr[remaining] = ld_res(res, endp + remaining)) != 0) ++remaining;
      const uint32_t rl = remaining > 0 ? min(3u, remaining - 1u) : 0u;
      for (uint32_t k = 0; k < 3; ++k) f[3 + k] = k < rl ? rr[k] : (uint8_t)'-';
      peptide_occurrences(uv, r, row, pstart, o_prot ? o_prot + h : nullptr, o_off ? o_off + h : nullptr,
                          o_ids ? o_ids + plo_out[h] : nullptr);
    }
  }
  __syncthreads();
  if (o_flanks) {  // 6 bytes per run, contiguous over the tile
    uint8_t* dst = o_flanks + 6 * h0;
    const uint32_t nb = 6 * tile_n;
    for (uint32_t i = t; i < nb; i += Q_THREADS) dst[i] = s_fl[i];
  }
  if (!o_seq) return;
  // ProteinCache.getPeptideSequence for the whole tile: bytes [seq0, seq0 + total) of o_seq
  const uint32_t total = s_soff[tile_n];
  uint8_t* out = o_seq + seq0;
  const uint32_t head = min(total, (uint32_t)((16 - ((uintptr_t)out & 15)) & 15));  // bytes before the first aligned chunk
  auto run_at = [&](uint32_t p) {  // last run with s_soff <= p
    uint32_t lo = 0, hi = tile_n;
    while (hi - lo > 1) {
      const uint32_t mid = (lo + hi) >> 1;
      if (s_soff[mid] <= p) lo = mid; else hi = mid;
    }
    return lo;
  };
  if ((uint32_t)t < head) {
    const uint32_t i = run_at((uint32_t)t);
    out[t] = ld_res(res, s_gpos[i] + ((uint32_t)t - s_soff[i]));
  }
  const uint32_t n_chunks = (total - head + 15) / 16;
  for (uint32_t c = t; c < n_chunks; c += Q_THREADS) {
    const uint32_t p0 = head + c * 16;
    uint32_t i = run_at(p0);
    uint32_t w[4] = {0, 0, 0, 0};
    const uint32_t nbytes = min(16u, total - p0);
    uint32_t b = 0;
    while (b < nbytes) {
      uint32_t nxt = s_soff[i + 1];
      while (p0 + b >= nxt) nxt = s_soff[++i + 1];  // empty sequences are skipped
      const uint32_t take = min(nbytes - b, nxt - (p0 + b));  // bytes of run i that land in this chunk
      uint32_t src = s_gpos[i] + (p0 + b - s_soff[i]);
      // up to 4 bytes at a time into byte position b of the 16-byte chunk (may straddle two words)
      for (uint32_t k = 0; k < take; k += 4) {
        const uint32_t nb4 = min(4u, take - k);
        uint32_t v = ld_res4(res, src + k);
        if (nb4 < 4) v &= (1u << (8 * nb4)) - 1u;
        const uint32_t at = b + k, wi = at >> 2, sh = (at & 3u) * 8u;
        w[wi] |= v << sh;
        if (sh && wi < 3) w[wi + 1] |= v >> (32 - sh);
      }
      b += take;
    }
    if (nbytes == 16) {
      *reinterpret_cast<uint4*>(out + p0) = make_uint4(w[0], w[1], w[2], w[3]);
    } else {
      for (uint32_t k = 0; k < nbytes; ++k) out[p0 + k] = (uint8_t)(w[k >> 2] >> (8 * (k & 3)));
    }
  }
}

// Entries name their base peptide by GLOBAL id; uv says which rank holds it (world = 1: this GPU).
__global__ void __launch_bounds__(Q_THREADS)
    fetch_sizes_kernel(const uint32_t* __restrict__ e_base, uint64_t base_off, const __grid_constant__ UniqView uv,
                       uint64_t begin, uint64_t count, uint32_t* __restrict__ sizes,
                       uint32_t* __restrict__ tile_counts) {
  __shared__ uint32_t scratch[Q_THREADS / 32 + 1];
  const uint64_t tile_base = (uint64_t)blockIdx.x * kScanTile;
  uint32_t sum = 0;
  for (int k = 0; k < Q_IPT; ++k) {
    const uint64_t i = tile_base + (uint64_t)k * Q_THREADS + threadIdx.x;
    if (i >= count) break;
    const uint64_t gid = e_base ? (uint64_t)e_base[begin + i] : base_off + begin + i;
    uint64_t row;
    const int r = uniq_owner(uv, gid, &row);
    const uint32_t sz = uv.plo[r] ? (uint32_t)(uv.plo[r][row + 1] - uv.plo[r][row]) : 0u;
    sizes[i] = sz;
    sum += sz;
  }
  uint32_t total;
  block_exclusive_sum<uint32_t, Q_THREADS>(sum, scratch, &total);
  if (threadIdx.x == 0) tile_counts[blockIdx.x] = total;
}

__global__ void __launch_bounds__(Q_THREADS)
    fetch_gather_kernel(const double* __restrict__ e_mass, const uint32_t* __restrict__ e_base, uint64_t base_off,
                        const __grid_constant__ UniqView uv, const uint32_t* __restrict__ e_pat,
                        const uint32_t* __restrict__ pstart, uint64_t begin, uint64_t count,
                        const uint32_t* __restrict__ sizes, const uint64_t* __restrict__ tile_offs,
                        double* __restrict__ o_mass, uint32_t* __restrict__ o_prot, uint32_t* __restrict__ o_off,
                        uint16_t* __restrict__ o_len, uint32_t* __restrict__ o_pat, uint64_t* __restrict__ o_list_off,
                        uint32_t* __restrict__ o_ids) {
  __shared__ uint32_t scratch[Q_THREADS / 32 + 1];
  const uint64_t tile_base = (uint64_t)blockIdx.x * kScanTile;
  const uint64_t ntiles = (count + kScanTile - 1) / kScanTile;
  uint64_t running = tile_offs[blockIdx.x];
  if (blockIdx.x == 0 && threadIdx.x == 0 && o_list_off) o_list_off[count] = tile_offs[ntiles];
  for (int k = 0; k < Q_IPT; ++k) {
    const uint64_t i = tile_base + (uint64_t)k * Q_THREADS + threadIdx.x;
    const bool valid = i < count;
    const uint32_t sz = valid ? sizes[i] : 0u;
    uint32_t total;
    const uint32_t ex = block_exclusive_sum<uint32_t, Q_THREADS>(sz, scratch, &total);
    if (valid) {
      const uint64_t e = begin + i;
      const uint64_t gid = e_base ? (uint64_t)e_base[e] : base_off + e;
      uint64_t row;
      const int r = uniq_owner(uv, gid, &row);
      const bool own = uv.len[r] != nullptr;  // else the owner's tables are not mapped here
      const uint32_t pr = own ? uv.prot[r][row] : 0xffffffffu;
      if (o_mass) o_mass[i] = e_mass[e];
      if (o_prot) o_prot[i] = pr;  // DBI_REMOTE_BASE
      if (o_off) o_off[i] = own ? uv.gpos[r][row] - pstart[pr] : (uint32_t)gid;  // sequenceOffset inside the first protein
      if (o_len) o_len[i] = own ? uv.len[r][row] : (uint16_t)0;
      if (o_pat) o_pat[i] = e_pat ? e_pat[e] : 0u;
      const uint64_t lo = running + ex;
      if (o_list_off) o_list_off[i] = lo;
      if (o_ids && own) {
        const uint64_t src = uv.plo[r][row];
        for (uint32_t j = 0; j < sz; ++j) o_ids[lo + j] = uv.plist[r][src + j];
      }
    }
    running += total;
  }
}

// ---- K11 batched peptide lookup: getProteins(String) (DBIndexer.java:925-947) for a whole list ----------------
constexpr uint8_t kLookupAbsent = 0, kLookupFound = 1, kLookupMalformed = 2;
constexpr unsigned kFull = 0xffffffffu;

// lookup_match_kernel<true>: the rank of the variant (sites pos[], of classes cls[]) in its group of
// peptide gid, whose residues are q[0 .. len): K6x's block order over the site masks for peptides of up to 64
// residues, K6l's lexicographic order of the site tuples for longer ones.
__device__ __noinline__ uint64_t group_rank(const GroupView& gv, const DevTables* __restrict__ tb,
                                            const uint8_t* __restrict__ q, uint32_t len, uint64_t gid, int k,
                                            const int* pos, const int* cls) {
  if (len <= 64) {
    const uint64_t* cm = gv.cmask + gid * (uint64_t)gv.n_classes;
    return group_entry_rank(k, pos, k > 0 ? cm[cls[0]] : 0ull, k > 1 ? cm[cls[1]] : 0ull, k > 2 ? cm[cls[2]] : 0ull,
                            k > 3 ? cm[cls[3]] : 0ull);
  }
  // right to left over the sites; S[j] = chains of levels j .. k-1 on the sites seen so far.  A site x of
  // level j's class between the row's sites of levels j-1 and j starts S[j + 1] tuples that precede the row's.
  uint64_t S[DBI_MAX_MODS_PER_PEP + 1] = {};
  S[k] = 1;
  uint64_t rank = 0;
  for (int x = (int)len - 1; x >= 0; --x) {
    const uint8_t c = q[x];
    if (!(__ldg(&tb->flags[c]) & kFlagDiffMod)) continue;
    const int cl = __ldg(&tb->cls[c]);
    for (int j = 0; j < k; ++j) {
      if (cls[j] != cl) continue;
      if (x < pos[j] && (j == 0 || x > pos[j - 1])) rank += S[j + 1];
      S[j] += S[j + 1];
    }
  }
  return rank;
}

// K11a: one warp per row.
//  1. The row's mass in the index's own summation order: init_mass, the residues left to right (digest.cu), then
//     the shift of every pattern position left to right (mods.cu, mods_grp.cu), so that it equals the indexed
//     mass bit for bit.  It is ONE sequential FP64 chain; the lanes load the residue masses side by side and
//     every lane runs the same chain over the shuffled values, so the whole warp holds the mass and the
//     validation verdict without a broadcast.
//  2. A 32-ary search for the first entry with mass >= the row's: each round the lanes probe 32 evenly spaced
//     pivots of the interval (independent loads) and a ballot narrows it 33-fold, ~log33(V) dependent rounds.
//  3. A walk over the run of equal mass bits, 32 entries per step.  A candidate has the row's mod pattern and
//     length; the warp compares its residues with the row's (lane j: positions j, j + 32, ...).  Unique
//     peptides are distinct strings and a (peptide, pattern) pair is indexed once, so the first full match is
//     the answer (a build with -DDBI_DEBUG walks the rest of the run and asserts that no second one exists).
// kGroups (compact index): steps 2 and 3 run over the groups; a candidate group has the class sequence of the
// row's pattern, and the entry is the group's first entry + the rank of the pattern in the group's order.
template <bool kGroups>
__global__ void __launch_bounds__(Q_THREADS)
    lookup_match_kernel(const uint8_t* __restrict__ res, const double* __restrict__ e_mass, uint64_t n_entries,
                        const uint32_t* __restrict__ e_base, uint64_t ent_off, const uint32_t* __restrict__ e_pat,
                        const __grid_constant__ UniqView uv, const DevTables* __restrict__ tb, double init_mass,
                        int max_mods, const uint8_t* __restrict__ q_res, const uint64_t* __restrict__ q_off,
                        const uint32_t* __restrict__ q_pat, uint64_t n, uint8_t* __restrict__ o_status,
                        double* __restrict__ o_mass, uint64_t* __restrict__ o_entry, uint32_t* __restrict__ o_np,
                        unsigned long long* __restrict__ n_found, const GroupView gv, uint64_t* __restrict__ o_gid) {
  const uint64_t i = (uint64_t)blockIdx.x * HX_WARPS + (threadIdx.x >> 5);
  if (i >= n) return;  // warp-uniform
  const unsigned lane = lane_id();
  const uint8_t* q = q_res + (q_off[i] - q_off[0]);
  const uint64_t len = q_off[i + 1] - q_off[i];
  const uint32_t pat = q_pat ? q_pat[i] : 0u;
  bool ok = len >= 1 && len <= DBI_MAX_PEP_LEN;
  uint32_t row_seq = 0;  // kGroups: the class sequence of the pattern, its sites and their classes
  int row_k = 0, row_pos[DBI_MAX_MODS_PER_PEP] = {}, row_cls[DBI_MAX_MODS_PER_PEP] = {};
  double m = init_mass;
  if (ok) {
    for (uint32_t c = 0; c < len; c += 32) {
      const uint32_t p = c + lane;
      const double rm = p < len ? __ldg(&tb->mass[q[p]]) : 0.0;
      const uint32_t k_end = min(32u, (uint32_t)len - c);
      for (uint32_t k = 0; k < k_end; ++k) m = __dadd_rn(m, __shfl_sync(kFull, rm, k));
    }
    // mod pattern: byte k = position + 1 of the k-th modified residue, strictly ascending, zeros only at the end
    uint32_t prev = 0, n_mods = 0;
    if constexpr (kGroups) row_seq = 0;
    bool ended = false;
    for (int k = 0; k < DBI_MAX_MODS_PER_PEP && ok; ++k) {
      const uint32_t b = (pat >> (8 * k)) & 0xFFu;
      if (b == 0) {
        ended = true;
        continue;
      }
      const uint32_t pos = b - 1;
      ok = !ended && b > prev && pos < len && pos <= DBI_MAX_MOD_POS && (int)++n_mods <= max_mods;
      if (!ok) break;
      const uint8_t c = q[pos];
      ok = (__ldg(&tb->flags[c]) & kFlagDiffMod) != 0;
      m = __dadd_rn(m, __ldg(&tb->diff[c]));
      prev = b;
      if constexpr (kGroups) {  // heap numbering of class sequences: children of v are v * C + c + 1
        row_cls[n_mods - 1] = __ldg(&tb->cls[c]);
        row_pos[n_mods - 1] = (int)pos;
        row_seq = row_seq * (uint32_t)gv.n_classes + row_cls[n_mods - 1] + 1u;
      }
    }
    if constexpr (kGroups) row_k = (int)n_mods;
  }
  if (!ok) {
    if (lane == 0) {
      o_status[i] = kLookupMalformed;
      o_mass[i] = 0.0;
      o_entry[i] = UINT64_MAX;
      o_np[i] = 0;
      if constexpr (kGroups) o_gid[i] = 0;
    }
    return;
  }

  // first entry with mass >= m lies in [lo, hi]
  uint64_t lo = 0, hi = n_entries;
  while (hi - lo > 32) {
    const uint64_t w = hi - lo;
    const unsigned below = __ballot_sync(kFull, __ldg(e_mass + lo + (lane + 1) * w / 33) < m);
    const uint64_t k = (uint64_t)__popc(below);  // pivots 0 .. k-1 lie below m
    hi = k < 32 ? lo + (k + 1) * w / 33 : hi;
    lo = k > 0 ? lo + k * w / 33 + 1 : lo;
  }
  const unsigned below = __ballot_sync(kFull, lo + lane < hi && __ldg(e_mass + lo + lane) < m);
  const uint64_t first = lo + (uint64_t)__popc(below);

  const unsigned long long mb = (unsigned long long)__double_as_longlong(m);
  const unsigned long long* e_bits = reinterpret_cast<const unsigned long long*>(e_mass);
  uint64_t hit = UINT64_MAX, hit_gid = 0;
  uint32_t hit_np = 0;
  for (uint64_t e0 = first; e0 < n_entries; e0 += 32) {
    const uint64_t e = e0 + lane;
    const bool eq = e < n_entries && __ldg(e_bits + e) == mb;
    bool cand;
    uint64_t gid = 0;
    if constexpr (kGroups) {
      const uint64_t pay = eq ? __ldg(gv.pay + e) : 0ull;
      cand = eq && (((uint32_t)pay >> 27) & 31u) == row_seq;
      gid = pay >> 32;
    } else {
      cand = eq && (e_pat ? __ldg(e_pat + e) : 0u) == pat;
      if (cand) gid = e_base ? (uint64_t)__ldg(e_base + e) : ent_off + e;
    }
    int r = 0;
    uint64_t row = 0;
    if (cand) {
      r = uniq_owner(uv, gid, &row);
      cand = uv.len[r][row] == len;
    }
    for (unsigned cm = __ballot_sync(kFull, cand); cm; cm &= cm - 1) {
      const int src = __ffs(cm) - 1;
      const int cr = __shfl_sync(kFull, r, src);
      const uint64_t crow = __shfl_sync(kFull, row, src);
      const uint32_t gp = uv.gpos[cr][crow];
      bool same = true;
      for (uint32_t p = lane; p < len; p += 32) same &= q[p] == ld_res(res, gp + p);
      if (__all_sync(kFull, same)) {
#ifdef DBI_DEBUG
        assert(hit == UINT64_MAX);
#endif
        hit = e0 + src;
        hit_gid = __shfl_sync(kFull, gid, src);
        hit_np = (uint32_t)(uv.plo[cr][crow + 1] - uv.plo[cr][crow]);
#ifndef DBI_DEBUG
        break;
#endif
      }
    }
#ifndef DBI_DEBUG
    if (hit != UINT64_MAX) break;
#endif
    if (__ballot_sync(kFull, eq) != kFull) break;  // the run of equal mass bits ends in this step
  }
  if constexpr (kGroups)
    if (hit != UINT64_MAX) hit = __ldg(gv.eoff + hit) + group_rank(gv, tb, q, (uint32_t)len, hit_gid, row_k, row_pos,
                                                                   row_cls);
  if (lane == 0) {
    if constexpr (kGroups) o_gid[i] = hit_gid;
    o_status[i] = hit != UINT64_MAX ? kLookupFound : kLookupAbsent;
    o_mass[i] = m;
    o_entry[i] = hit;
    o_np[i] = hit_np;
    if (hit != UINT64_MAX) atomicAdd(n_found, 1ull);
  }
}

// K11b: one thread per row; found rows get their first occurrence and protein ids (prot_list_off = scan of the
// list lengths K11a wrote), the others first_prot = first_off = 0xffffffff.
__global__ void __launch_bounds__(Q_THREADS)
    lookup_gather_kernel(const uint8_t* __restrict__ status, const uint64_t* __restrict__ entry,
                         const uint32_t* __restrict__ e_base, uint64_t ent_off, const __grid_constant__ UniqView uv,
                         const uint32_t* __restrict__ pstart, const uint64_t* __restrict__ plo, uint64_t n,
                         uint32_t* __restrict__ o_prot, uint32_t* __restrict__ o_off, uint32_t* __restrict__ o_ids) {
  const uint64_t i = (uint64_t)blockIdx.x * Q_THREADS + threadIdx.x;
  if (i >= n) return;
  if (status[i] != kLookupFound) {
    o_prot[i] = 0xffffffffu;
    o_off[i] = 0xffffffffu;
    return;
  }
  const uint64_t e = entry[i];
  uint64_t row;
  const int r = uniq_owner(uv, e_base ? (uint64_t)e_base[e] : ent_off + e, &row);
  peptide_occurrences(uv, r, row, pstart, o_prot + i, o_off + i, o_ids + plo[i]);
}

__device__ __forceinline__ int32_t row_key(double m, double factor) { return (int32_t)(m * factor); }

__global__ void __launch_bounds__(Q_THREADS)
    key_flags_kernel(const double* __restrict__ e_mass, uint64_t n, double factor, uint8_t* __restrict__ flags,
                     uint32_t* __restrict__ tile_counts) {
  __shared__ uint32_t scratch[Q_THREADS / 32 + 1];
  const uint64_t tile_base = (uint64_t)blockIdx.x * kScanTile;
  uint32_t sum = 0;
  for (int k = 0; k < Q_IPT; ++k) {
    const uint64_t i = tile_base + (uint64_t)k * Q_THREADS + threadIdx.x;
    if (i >= n) break;
    const uint8_t f = (i == 0) || row_key(e_mass[i], factor) != row_key(e_mass[i - 1], factor);
    flags[i] = f;
    sum += f;
  }
  uint32_t total;
  block_exclusive_sum<uint32_t, Q_THREADS>(sum, scratch, &total);
  if (threadIdx.x == 0) tile_counts[blockIdx.x] = total;
}

__global__ void __launch_bounds__(Q_THREADS)
    key_emit_kernel(const double* __restrict__ e_mass, uint64_t n, double factor, const uint8_t* __restrict__ flags,
                    const uint64_t* __restrict__ tile_offs, int32_t* __restrict__ keys) {
  __shared__ uint32_t scratch[Q_THREADS / 32 + 1];
  const uint64_t tile_base = (uint64_t)blockIdx.x * kScanTile;
  uint64_t running = tile_offs[blockIdx.x];
  for (int k = 0; k < Q_IPT; ++k) {
    const uint64_t i = tile_base + (uint64_t)k * Q_THREADS + threadIdx.x;
    const bool valid = i < n;
    const uint32_t f = valid ? flags[i] : 0u;
    uint32_t total;
    const uint32_t ex = block_exclusive_sum<uint32_t, Q_THREADS>(f, scratch, &total);
    if (valid && f) keys[running + ex] = row_key(e_mass[i], factor);
    running += total;
  }
}

}  // namespace

void launch_query(const double* e_mass, uint64_t n_entries, const double* lo, const double* hi, uint64_t nq,
                  uint64_t* hit_begin, uint64_t* hit_count, uint32_t* cnt32, cudaStream_t s) {
  if (nq == 0) return;
  const unsigned grid = (unsigned)((nq + Q_THREADS - 1) / Q_THREADS);
  DBI_LAUNCH(query_kernel, grid, Q_THREADS, 0, s, e_mass, n_entries, lo, hi, nq, hit_begin, hit_count, cnt32);
}

void launch_hits_seg_count(const uint64_t* hit_count, uint64_t nq, uint32_t* nseg32, cudaStream_t s) {
  if (nq == 0) return;
  DBI_LAUNCH(hits_seg_count_kernel, (unsigned)((nq + Q_THREADS - 1) / Q_THREADS), Q_THREADS, 0, s, hit_count, nq, nseg32);
}

void launch_hits_seg_fill(const uint64_t* seg_off, uint64_t nq, uint32_t* seg_q, cudaStream_t s) {
  if (nq == 0) return;
  DBI_LAUNCH(hits_seg_fill_kernel, (unsigned)((nq + HX_WARPS - 1) / HX_WARPS), Q_THREADS, 0, s, seg_off, nq, seg_q);
}

void launch_hits_count_runs(const double* e_mass, const uint32_t* e_base, const uint32_t* seg_q, const uint64_t* seg_off,
                            const uint64_t* hit_begin, const uint64_t* hit_off, uint64_t nseg, uint32_t* nruns32,
                            cudaStream_t s) {
  if (nseg == 0) return;
  const unsigned grid = (unsigned)((nseg + HX_WARPS - 1) / HX_WARPS);
  DBI_LAUNCH(hits_count_runs_kernel, grid, Q_THREADS, 0, s, e_mass, e_base, seg_q, seg_off, hit_begin, hit_off, nseg,
             nruns32);
}

void launch_hits_pep_off(const uint64_t* seg_off, const uint64_t* seg_run_off, uint64_t nq, uint64_t* pep_off,
                         cudaStream_t s) {
  DBI_LAUNCH(hits_pep_off_kernel, (unsigned)((nq + 1 + Q_THREADS - 1) / Q_THREADS), Q_THREADS, 0, s, seg_off, seg_run_off,
             nq, pep_off);
}

void launch_hits_runs(const double* e_mass, const uint32_t* e_base, uint64_t ent_off, const uint32_t* e_pat,
                      const UniqView& uv, const uint32_t* seg_q, const uint64_t* seg_off, const uint64_t* hit_begin,
                      const uint64_t* hit_off, const uint64_t* seg_run_off, uint64_t nseg, uint32_t* o_pat,
                      uint64_t* pep_hit_off, double* o_mass, uint32_t* pep_entry, uint32_t* len32, uint32_t* np32,
                      cudaStream_t s) {
  if (nseg == 0) return;
  const unsigned grid = (unsigned)((nseg + HX_WARPS - 1) / HX_WARPS);
  DBI_LAUNCH(hits_runs_kernel, grid, Q_THREADS, 0, s, e_mass, e_base, ent_off, e_pat, uv, seg_q, seg_off, hit_begin,
             hit_off, seg_run_off, nseg, o_pat, pep_hit_off, o_mass, pep_entry, len32, np32);
}

void launch_peps_gather(const uint8_t* d_res, const uint32_t* pstart, const uint32_t* e_base, uint64_t ent_off,
                        const UniqView& uv, const uint32_t* pep_entry, const uint64_t* seq_off, const uint64_t* plo_out,
                        uint64_t n_peps, uint32_t* o_prot, uint32_t* o_off, uint16_t* o_len, uint8_t* o_flanks,
                        uint8_t* o_seq, uint32_t* o_ids, cudaStream_t s) {
  if (n_peps == 0) return;
  const unsigned grid = (unsigned)((n_peps + Q_THREADS - 1) / Q_THREADS);
  DBI_LAUNCH(peps_gather_kernel, grid, Q_THREADS, 0, s, d_res, pstart, e_base, ent_off, uv, pep_entry, seq_off, plo_out,
             n_peps, o_prot, o_off, o_len, o_flanks, o_seq, o_ids);
}

void launch_fetch_sizes(const uint32_t* e_base, uint64_t base_off, const UniqView& uv, uint64_t begin, uint64_t count,
                        uint32_t* sizes, uint32_t* tile_counts, cudaStream_t s) {
  if (count == 0) return;
  const unsigned tiles = (unsigned)((count + kScanTile - 1) / kScanTile);
  DBI_LAUNCH(fetch_sizes_kernel, tiles, Q_THREADS, 0, s, e_base, base_off, uv, begin, count, sizes, tile_counts);
}

void launch_fetch_gather(const double* e_mass, const uint32_t* e_base, uint64_t base_off, const UniqView& uv,
                         const uint32_t* e_pat, const uint32_t* pstart, uint64_t begin, uint64_t count,
                         const uint32_t* sizes, const uint64_t* tile_offs, double* o_mass, uint32_t* o_prot,
                         uint32_t* o_off, uint16_t* o_len, uint32_t* o_pat, uint64_t* o_list_off, uint32_t* o_ids,
                         cudaStream_t s) {
  if (count == 0) return;
  const unsigned tiles = (unsigned)((count + kScanTile - 1) / kScanTile);
  DBI_LAUNCH(fetch_gather_kernel, tiles, Q_THREADS, 0, s, e_mass, e_base, base_off, uv, e_pat, pstart, begin, count,
             sizes, tile_offs, o_mass, o_prot, o_off, o_len, o_pat, o_list_off, o_ids);
}

void launch_lookup_match(const uint8_t* d_res, const double* e_mass, uint64_t n_entries, const uint32_t* e_base,
                         uint64_t ent_off, const uint32_t* e_pat, const UniqView& uv, const DevTables* d_tb,
                         double init_mass, int max_mods, const uint8_t* q_res, const uint64_t* q_off,
                         const uint32_t* q_pat, uint64_t n, uint8_t* o_status, double* o_mass, uint64_t* o_entry,
                         uint32_t* o_np, unsigned long long* n_found, const GroupView* gv, uint64_t* o_gid,
                         cudaStream_t s) {
  if (n == 0) return;
  const unsigned grid = (unsigned)((n + HX_WARPS - 1) / HX_WARPS);
  if (gv)
    DBI_LAUNCH(lookup_match_kernel<true>, grid, Q_THREADS, 0, s, d_res, e_mass, n_entries, e_base, ent_off, e_pat, uv,
               d_tb, init_mass, max_mods, q_res, q_off, q_pat, n, o_status, o_mass, o_entry, o_np, n_found, *gv, o_gid);
  else
    DBI_LAUNCH(lookup_match_kernel<false>, grid, Q_THREADS, 0, s, d_res, e_mass, n_entries, e_base, ent_off, e_pat, uv,
               d_tb, init_mass, max_mods, q_res, q_off, q_pat, n, o_status, o_mass, o_entry, o_np, n_found,
               GroupView{}, nullptr);
}

void launch_lookup_gather(const uint8_t* status, const uint64_t* entry, const uint32_t* e_base, uint64_t ent_off,
                          const UniqView& uv, const uint32_t* pstart, const uint64_t* plo, uint64_t n,
                          uint32_t* o_prot, uint32_t* o_off, uint32_t* o_ids, cudaStream_t s) {
  if (n == 0) return;
  const unsigned grid = (unsigned)((n + Q_THREADS - 1) / Q_THREADS);
  DBI_LAUNCH(lookup_gather_kernel, grid, Q_THREADS, 0, s, status, entry, e_base, ent_off, uv, pstart, plo, n, o_prot,
             o_off, o_ids);
}

void launch_key_flags(const double* e_mass, uint64_t n, double factor, uint8_t* flags, uint32_t* tile_counts,
                      cudaStream_t s) {
  if (n == 0) return;
  const unsigned tiles = (unsigned)((n + kScanTile - 1) / kScanTile);
  DBI_LAUNCH(key_flags_kernel, tiles, Q_THREADS, 0, s, e_mass, n, factor, flags, tile_counts);
}

void launch_key_emit(const double* e_mass, uint64_t n, double factor, const uint8_t* flags,
                     const uint64_t* tile_offs, int32_t* keys, cudaStream_t s) {
  if (n == 0) return;
  const unsigned tiles = (unsigned)((n + kScanTile - 1) / kScanTile);
  DBI_LAUNCH(key_emit_kernel, tiles, Q_THREADS, 0, s, e_mass, n, factor, flags, tile_offs, keys);
}

}  // namespace dbi
