// mods_grp.cu -- differential-mod expansion, group path (class sequences <= 32).
//
// SPEC as in mods.cu (DESIGN.md "Mod expansion SPEC"; the reference only parses the mods,
// io/SearchParamReader.java:631-687, model/DiffModification.java:11-54).
//
// All variants of one peptide whose chosen sites carry the same SEQUENCE of shift classes share
// one mass f_s(base) = ((base + d_s0) + d_s1) + ... -- they are one contiguous run of the final
// index.  So only one record per (peptide, class sequence) group goes through the radix sort and
// the entries are written after the sort, already in place:
//   K5m site_masks : per peptide and shift class, the 64-bit mask of its sites        (thread/peptide)
//   K5g grp_count  : groups and variants per peptide: subsequence-count DP over sites (thread/peptide)
//   K6g grp_emit   : {key = mass bits - base, payload = peptide << 32 | sequence << 27 | count}
//   (single GPU: K6g writes one sorted list per class sequence and K7m (merge.cu) merges them; sharded
//   build: K7 sorts the records after the exchange.  K3 scans the counts into entry offsets)
//   K6t grp_tile_first : first group of every tile of kExpTile consecutive ENTRIES
//   K6x grp_expand_tab : one thread per ENTRY: un-rank the entry inside its group in constant
//                    time (product-set blocks, per-group block tables in shared memory) and write
//                    (mass, peptide, pattern) -- coalesced stores, no divergent per-group enumeration
//   K6l grp_expand_long : groups of peptides longer than 64 residues (no masks): one warp each
//   K6q grp_expand_ranges : compact index (the sorted groups kept, no entry arrays): K6x's tile body over
//                    tiles cut from arbitrary entry ranges, at query time; the windowed K6l for long groups
//
// HBM-bound byte/integer work; no tensor cores.  Algorithmic bytes: K5m 14 + len per peptide read,
// 8 C written; K5g/K6g 25 + 8 C per peptide, 16 per group written; K6x 24 per group + 8 C per
// group (random 32-B sectors) read, 16 per entry written.
#include <cstring>

#include "mods_common.cuh"

namespace dbi {
namespace {

constexpr uint32_t kGrpCntBits = 27;
constexpr uint32_t kGrpCntMask = (1u << kGrpCntBits) - 1;
constexpr int kMaskLen = 64;  // peptides up to this length have site masks

// Subsequence-count DP state of one thread: cnt[v] for every class sequence v (heap numbering:
// children of v are v*C + c + 1), in shared memory, one column per thread (conflict-free).
struct SeqCounts {
  uint32_t* col;  // &smem[threadIdx.x]; cnt[v] = col[v * MD_THREADS]
  __device__ __forceinline__ uint32_t get(int v) const { return col[v * MD_THREADS]; }
  __device__ __forceinline__ void set(int v, uint32_t x) { col[v * MD_THREADS] = x; }
  __device__ __forceinline__ void reset(int n_seq) {
    col[0] = 1u;
    for (int v = 1; v < n_seq; ++v) col[v * MD_THREADS] = 0u;
  }
  // a site of class c extends every sequence's parent; deeper sequences first so that a parent is
  // read before this site updates it
  __device__ __forceinline__ void site(int c, int C, int n_par) {
    for (int p = n_par - 1; p >= 0; --p) {
      const uint32_t up = col[p * MD_THREADS];
      if (up) col[(p * C + c + 1) * MD_THREADS] += up;
    }
  }
};

// mass of the variants of class sequence v: base, then + shift per chosen site left to right
__device__ __forceinline__ double seq_mass(uint32_t v, int C, double base, const double* cls_delta) {
  uint32_t pk;
  const int k = pack_seq(v, C, &pk);
  double m = base;
  for (int j = 0; j < k; ++j) m = __dadd_rn(m, cls_delta[seq_class_at(pk, j)]);
  return m;
}

// Runs the DP of peptide u.  Peptides of up to kMaskLen residues walk their site masks, longer
// ones their residues.  Returns false (and raises kErrModPos) if a site lies beyond position 254.
__device__ __forceinline__ void peptide_dp(SeqCounts& sc, const uint8_t* __restrict__ res,
                                           const uint64_t* __restrict__ cmask, const ModTables& mt,
                                           const DigestCfg& cfg, uint64_t u, uint32_t gpos, uint32_t len, int n_par,
                                           uint32_t* err) {
  const int C = cfg.n_classes;
  sc.reset(cfg.n_seq);
  if (len <= kMaskLen) {
    const uint64_t* cm = cmask + u * (uint64_t)C;
    if (C == 1) {
      for (uint64_t m = cm[0]; m; m &= m - 1) sc.site(0, C, n_par);
    } else if (C == 2) {
      const uint64_t m0 = cm[0], m1 = cm[1];
      for (uint64_t m = m0 | m1; m; m &= m - 1) sc.site((int)(((m1 & (0 - m)) & m) != 0), C, n_par);
    } else {
      uint64_t all = 0;
      for (int c = 0; c < C; ++c) all |= cm[c];
      for (; all; all &= all - 1) {
        const uint64_t bit = all & (0 - all);
        int c = 0;
        while (!(cm[c] & bit)) ++c;
        sc.site(c, C, n_par);
      }
    }
  } else {
    for (uint32_t i = 0; i < len; ++i) {
      const uint8_t r = ld_res(res, gpos + i);
      if (mt.flags[r] & kFlagDiffMod) {
        if (i > DBI_MAX_MOD_POS) {
          atomicOr(err, kErrModPos);
          break;
        }
        sc.site(mt.cls[r], C, n_par);
      }
    }
  }
}

// Can a variant of this peptide reach a mass gate at all?
__device__ __forceinline__ bool gate_reachable(double bm, const DigestCfg& cfg) {
  const int K = cfg.max_mods;
  return !(bm + K * cfg.mod_hi <= cfg.max_mass - 1e-6 && bm + K * cfg.mod_lo >= cfg.min_mass + 1e-6);
}

// ---- K5m ------------------------------------------------------------------------------
__global__ void __launch_bounds__(MD_THREADS)
    site_masks_kernel(const uint8_t* __restrict__ res, const DevTables* __restrict__ tb, int C,
                      const uint32_t* __restrict__ u_gpos, const uint16_t* __restrict__ u_len, uint64_t n_unique,
                      uint64_t* __restrict__ cmask, unsigned long long* __restrict__ n_long) {
  __shared__ uint8_t s_cls[256];  // class + 1 of a modifiable residue, 0 otherwise
  for (int i = threadIdx.x; i < 256; i += MD_THREADS)
    s_cls[i] = (tb->flags[i] & kFlagDiffMod) ? (uint8_t)(tb->cls[i] + 1) : (uint8_t)0;
  __syncthreads();
  const uint64_t u = (uint64_t)blockIdx.x * MD_THREADS + threadIdx.x;
  if (u >= n_unique) return;
  const uint32_t len = u_len[u];
  uint64_t* out = cmask + u * (uint64_t)C;
  if (len > kMaskLen) {  // no masks: all-zero marks the peptide as long (a group with sites has a non-zero mask)
    for (int c = 0; c < C; ++c) out[c] = 0;
    atomicAdd(n_long, 1ull);
    return;
  }
  const uint32_t gp = u_gpos[u];
  if (C <= 4) {
    uint64_t m0 = 0, m1 = 0, m2 = 0, m3 = 0;
    for (uint32_t i = 0; i < len; ++i) {
      const uint32_t c1 = s_cls[ld_res(res, gp + i)];
      const uint64_t bit = 1ull << i;
      if (c1 == 1) m0 |= bit;
      if (c1 == 2) m1 |= bit;
      if (c1 == 3) m2 |= bit;
      if (c1 == 4) m3 |= bit;
    }
    out[0] = m0;
    if (C > 1) out[1] = m1;
    if (C > 2) out[2] = m2;
    if (C > 3) out[3] = m3;
  } else {
    for (int c = 0; c < C; ++c) {
      uint64_t m = 0;
      for (uint32_t i = 0; i < len; ++i)
        if (s_cls[ld_res(res, gp + i)] == (uint32_t)c + 1) m |= 1ull << i;
      out[c] = m;
    }
  }
}

// peptides longer than kMaskLen in a (global) length table
__global__ void __launch_bounds__(MD_THREADS)
    count_long_kernel(const uint16_t* __restrict__ len, uint64_t n, unsigned long long* __restrict__ n_long) {
  const uint64_t i = (uint64_t)blockIdx.x * MD_THREADS + threadIdx.x;
  const bool is = i < n && len[i] > kMaskLen;
  const unsigned m = __ballot_sync(0xffffffffu, is);
  if (m && lane_id() == 0) atomicAdd(n_long, (unsigned long long)__popc(m));
}

// ---- K5g ------------------------------------------------------------------------------
// mask_out[u]: bit v set iff group (u, v) exists (v = 0 always).  vt_cnt (optional, list layout of K6g):
// vt_cnt[v * vt_stride + tile] = groups of class sequence v in the tile.
__global__ void __launch_bounds__(MD_THREADS)
    grp_count_kernel(const uint8_t* __restrict__ res, const DevTables* __restrict__ tb, DigestCfg cfg,
                     const double* __restrict__ u_mass, const uint32_t* __restrict__ u_gpos,
                     const uint16_t* __restrict__ u_len, const uint64_t* __restrict__ cmask, uint64_t n_unique,
                     uint32_t tile0, uint32_t* __restrict__ mask_out, uint32_t* __restrict__ tile_groups,
                     uint32_t* __restrict__ tile_vars, uint32_t* __restrict__ vt_cnt, uint32_t vt_stride,
                     uint32_t* err) {
  extern __shared__ uint32_t s_cnt[];  // [n_seq][MD_THREADS]
  __shared__ ModTables mt;
  __shared__ uint32_t scratch[MD_WARPS + 1];
  __shared__ uint32_t s_vc[32];  // groups of every class sequence in the tile
  if (threadIdx.x < 32) s_vc[threadIdx.x] = 0;
  load_mod_tables(mt, tb);
  __syncthreads();
  const int C = cfg.n_classes;
  const int n_par = (cfg.n_seq - 1) / C;
  const uint64_t u = (uint64_t)(tile0 + blockIdx.x) * kModTile + threadIdx.x;
  uint32_t mask = 0, nv = 0;
  if (u < n_unique) {
    SeqCounts sc{s_cnt + threadIdx.x};
    const double bm = u_mass[u];
    peptide_dp(sc, res, cmask, mt, cfg, u, u_gpos[u], u_len[u], n_par, err);
    const bool gated = gate_reachable(bm, cfg);
    mask = 1;
    nv = 1;  // the unmodified peptide is always present
    for (int v = 1; v < cfg.n_seq; ++v) {
      const uint32_t c = sc.get(v);
      if (c == 0) continue;
      if (gated) {
        const double m = seq_mass((uint32_t)v, C, bm, mt.cls_delta);
        if (!(m >= cfg.min_mass && m <= cfg.max_mass)) continue;
      }
      if (c > kGrpCntMask) atomicOr(err, kErrModPos);  // > 2^27 variants in one group
      mask |= 1u << v;
      nv += c;
    }
    mask_out[u] = mask;
  }
  if (vt_cnt)
    for (int v = 0; v < cfg.n_seq; ++v) {
      const unsigned b = __ballot_sync(0xffffffffu, (mask >> v) & 1u);
      if (lane_id() == 0 && b) atomicAdd(&s_vc[v], (uint32_t)__popc(b));
    }
  uint32_t tot_g;
  block_exclusive_sum<uint32_t, MD_THREADS>((uint32_t)__popc(mask), scratch, &tot_g);  // syncs: s_vc is complete
  if (vt_cnt && (int)threadIdx.x < cfg.n_seq) vt_cnt[(uint64_t)threadIdx.x * vt_stride + blockIdx.x] = s_vc[threadIdx.x];
  // the variant total of a tile is informational (the entry count comes from the 64-bit scan of the sorted
  // groups); summed in 64 bits and saturated so that a wrap can never look like a small number
  __shared__ unsigned long long scratch64[MD_WARPS + 1];
  unsigned long long tot_v;
  block_exclusive_sum<unsigned long long, MD_THREADS>((unsigned long long)nv, scratch64, &tot_v);
  if (threadIdx.x == 0) {
    tile_groups[blockIdx.x] = tot_g;
    tile_vars[blockIdx.x] = tot_v > 0xffffffffull ? 0xffffffffu : (uint32_t)tot_v;
  }
}

// ---- K6g ------------------------------------------------------------------------------
// Peptide-major layout (kLists = false, the sharded build): the groups of a tile from tile_goffs[tile] on,
// peptide by peptide, v ascending.  List layout (kLists = true): the groups of class sequence v form list v,
// in peptide order; group (u, v) goes to goffs[v * vt_stride + tile] + (earlier peptides of the tile with v).
// Either way every list v is strictly increasing in (key, payload): u_mass grows with u, and the rounded
// additions of f_v(base) are monotone in the base.
template <bool kLists>
__global__ void __launch_bounds__(MD_THREADS)
    grp_emit_kernel(const uint8_t* __restrict__ res, const DevTables* __restrict__ tb, DigestCfg cfg,
                    const double* __restrict__ u_mass, const uint32_t* __restrict__ u_gpos,
                    const uint16_t* __restrict__ u_len, const uint64_t* __restrict__ cmask, uint64_t n_unique,
                    uint32_t tile0, const uint32_t* __restrict__ mask_in, const uint64_t* __restrict__ goffs,
                    uint32_t vt_stride, uint64_t base_bits, uint64_t id_off, uint64_t* __restrict__ g_key,
                    uint64_t* __restrict__ g_pay, uint32_t* err) {
  extern __shared__ uint32_t s_cnt[];  // [n_seq][MD_THREADS]
  __shared__ ModTables mt;
  __shared__ uint32_t scratch[MD_WARPS + 1];
  load_mod_tables(mt, tb);
  __syncthreads();
  const int C = cfg.n_classes;
  const int n_par = (cfg.n_seq - 1) / C;
  const uint64_t u = (uint64_t)(tile0 + blockIdx.x) * kModTile + threadIdx.x;
  const bool valid = u < n_unique;
  const uint32_t mask = valid ? mask_in[u] : 0u;
  const int w = threadIdx.x >> 5;
  // list layout: ballot of every class sequence per warp, and where each warp's groups of it start
  __shared__ uint32_t s_bal[kLists ? 32 * MD_WARPS : 1];
  __shared__ uint64_t s_wbase[kLists ? 32 * MD_WARPS : 1];
  uint64_t o = 0;
  if constexpr (kLists) {
    for (int v = 0; v < cfg.n_seq; ++v) {
      const unsigned b = __ballot_sync(0xffffffffu, (mask >> v) & 1u);
      if (lane_id() == 0) s_bal[v * MD_WARPS + w] = b;
    }
    __syncthreads();
    if ((int)threadIdx.x < cfg.n_seq) {
      uint64_t run = goffs[(uint64_t)threadIdx.x * vt_stride + blockIdx.x];
      for (int x = 0; x < MD_WARPS; ++x) {
        s_wbase[threadIdx.x * MD_WARPS + x] = run;
        run += (uint32_t)__popc(s_bal[threadIdx.x * MD_WARPS + x]);
      }
    }
    __syncthreads();
    if (!valid) return;
  } else {
    uint32_t tot;
    const uint32_t ex = block_exclusive_sum<uint32_t, MD_THREADS>((uint32_t)__popc(mask), scratch, &tot);
    if (!valid) return;
    o = goffs[blockIdx.x] + ex;
  }
  auto slot = [&](int v) -> uint64_t {
    if constexpr (kLists)
      return s_wbase[v * MD_WARPS + w] + (uint32_t)__popc(s_bal[v * MD_WARPS + w] & lanemask_lt());
    else
      return o++;
  };
  const double bm = u_mass[u];
  const uint64_t gid = (id_off + u) << 32;  // global id of the peptide (id_off = 0 on a single GPU)
  {
    const uint64_t x = slot(0);
    g_key[x] = (uint64_t)__double_as_longlong(bm) - base_bits;
    g_pay[x] = gid | 1u;
  }
  if (mask == 1u) return;  // no sites, or every modified mass is gated out
  SeqCounts sc{s_cnt + threadIdx.x};
  peptide_dp(sc, res, cmask, mt, cfg, u, u_gpos[u], u_len[u], n_par, err);
  for (int v = 1; v < cfg.n_seq; ++v) {
    if (!((mask >> v) & 1u)) continue;  // no variant, or gated out (K5g)
    const uint32_t c = sc.get(v);
    const double m = seq_mass((uint32_t)v, C, bm, mt.cls_delta);
    const uint64_t x = slot(v);
    g_key[x] = (uint64_t)__double_as_longlong(m) - base_bits;
    g_pay[x] = gid | ((uint64_t)v << kGrpCntBits) | (uint64_t)(c & kGrpCntMask);
  }
}

__global__ void __launch_bounds__(MD_THREADS)
    grp_extract_cnt_kernel(const uint64_t* __restrict__ pay, uint64_t n, uint32_t* __restrict__ cnt) {
  const uint64_t i = (uint64_t)blockIdx.x * MD_THREADS + threadIdx.x;
  if (i < n) cnt[i] = (uint32_t)pay[i] & kGrpCntMask;
}

// ---- K6t ------------------------------------------------------------------------------
// first[t] = the group that holds entry t * kExpTile: last g with eoff[g] <= t * kExpTile.
__global__ void __launch_bounds__(MD_THREADS)
    grp_tile_first_kernel(const uint64_t* __restrict__ eoff, uint64_t n_groups, uint64_t n_tiles,
                          uint32_t* __restrict__ first) {
  const uint64_t t = (uint64_t)blockIdx.x * MD_THREADS + threadIdx.x;
  if (t > n_tiles) return;
  if (t == n_tiles) {  // sentinel: the last group
    first[t] = (uint32_t)(n_groups - 1);
    return;
  }
  const uint64_t e = t * (uint64_t)kExpTile;
  uint64_t lo = 0, hi = n_groups;  // invariant: eoff[lo] <= e < eoff[hi]   (eoff[n_groups] = #entries > e)
  while (hi - lo > 1) {
    const uint64_t mid = (lo + hi) >> 1;
    if (__ldg(eoff + mid) <= e) lo = mid; else hi = mid;
  }
  first[t] = (uint32_t)lo;
}

// ---- K6x ------------------------------------------------------------------------------
// position of the (r+1)-th set bit of m (r < popc(m)): binary search on popcounts, constant cost
__device__ __forceinline__ int select_bit(uint64_t m, uint32_t r) {
  int pos = 0;
  uint32_t c = (uint32_t)__popc((uint32_t)m);
  uint32_t x = (uint32_t)m;
  if (r >= c) { r -= c; pos = 32; x = (uint32_t)(m >> 32); }
  c = (uint32_t)__popc(x & 0xffffu);
  if (r >= c) { r -= c; pos += 16; x >>= 16; }
  c = (uint32_t)__popc(x & 0xffu);
  if (r >= c) { r -= c; pos += 8; x >>= 8; }
  c = (uint32_t)__popc(x & 0xfu);
  if (r >= c) { r -= c; pos += 4; x >>= 4; }
  c = (uint32_t)__popc(x & 0x3u);
  if (r >= c) { r -= c; pos += 2; x >>= 2; }
  if (r >= (x & 1u)) pos += 1;
  return pos;
}

constexpr int EX_GMAX = kExpTile + 1;  // groups that can overlap one tile (every group has >= 1 entry)
constexpr uint8_t kLongGroup = 0xff;   // peptide longer than 64 residues: K6l writes the group
constexpr uint8_t kSlowGroup = 0xfe;   // k = 4, or the tile's list pool is full: every entry un-ranks from the masks

// One thread per ENTRY with constant, convergent work.  The entries of a group are ordered by BLOCKS
// that are product sets:
//   k = 1: one block, the sites of the class, ascending;
//   k = 2: block = first site p;   entries = sites of the second class above p;
//   k = 3: block = MIDDLE site p;  entries = (sites of the first class below p) x (sites of the
//          third class above p), the third site running fastest;
//   k = 4: block = second site p;  entries = (first-class sites below p) x (pairs i2 < i3 above p).
// (The order of the entries INSIDE a group is free: they all have the same mass and peptide.)
// Phase 1 (thread per group) turns the site masks of a group into byte LISTS of site positions in a
// shared pool and appends one record per block that overlaps the tile; phase 2 max-scans the block
// heads so that every entry knows its block; phase 3 (thread per entry) is then
//   rank in block -> (a, b) by one multiplication -> two byte loads -> pattern -> three coalesced stores.
constexpr int ET_THREADS = 128;
constexpr int ET_PER = kExpTile / ET_THREADS;
constexpr int EP_POOL = 3072;  // bytes of site lists shared by the groups of a tile; pool[0] = 0 = "no site"

struct ExpBlk {    // 16 bytes, read with one LDS.128
  int32_t start;   // tile-local entry of the block's first entry (may be negative)
  uint16_t grp;    // tile-local group
  uint16_t a0;     // pool index of the first-level list (0 = none)
  uint16_t b0;     // pool index of the first last-level site of this block
  uint8_t nb;      // last-level sites of this block
  uint8_t p;       // block site
  uint32_t k;      // class-sequence length, or kLongGroup / kSlowGroup
};

struct ExpSmem {
  double mass[EX_GMAX];
  uint32_t base[EX_GMAX];
  uint32_t idx[EX_GMAX];      // row of the group's peptide in the mask table
  uint32_t head[kExpTile];    // (entry << 16 | block slot) at block starts, max-scanned
  ExpBlk blk[kExpTile];       // every listed block owns >= 1 entry of the tile
  uint8_t pool[EP_POOL];
  uint8_t seq[EX_GMAX];
  uint32_t recip[65];         // ceil(2^20 / n): exact quotient for ranks < 4096
  uint32_t nblk, pool_used;
  uint32_t scratch[ET_THREADS / 32 + 1];
};

// appends (position + 1) of every set bit of c, ascending, to the byte pool; the two 32-bit halves are walked
// separately (most peptides have fewer than 33 residues: half the instructions of a 64-bit walk)
__device__ __forceinline__ uint32_t fill_sites(uint64_t c, uint8_t* pool, uint32_t x) {
  uint32_t lo = (uint32_t)c, hi = (uint32_t)(c >> 32);
  for (; lo; lo &= lo - 1) pool[x++] = (uint8_t)__ffs((int)lo);
  for (; hi; hi &= hi - 1) pool[x++] = (uint8_t)(32 + __ffs((int)hi));
  return x;
}

// pattern of entry q of the block at site p, from the masks (slow path)
__device__ __forceinline__ uint32_t block_entry(int k, int p, uint32_t q, uint64_t c0, uint64_t c1, uint64_t c2,
                                                uint64_t c3) {
  if (k == 2) return (uint32_t)(p + 1) | ((uint32_t)(select_bit(c1 & above(p), q) + 1) << 8);
  const uint64_t L = c0 & below(p);
  if (k == 3) {
    const uint64_t R = c2 & above(p);
    const uint32_t nr = (uint32_t)__popcll(R);
    const uint32_t a = q / nr, b = q - a * nr;
    return (uint32_t)(select_bit(L, a) + 1) | ((uint32_t)(p + 1) << 8) | ((uint32_t)(select_bit(R, b) + 1) << 16);
  }
  const uint32_t w2 = pairs_above(p, c2, c3);
  const uint32_t a = q / w2;
  uint32_t b = q - a * w2;
  int i2 = 0;
  uint64_t r3 = 0;
  for (uint64_t m = c2 & above(p); m; m &= m - 1) {
    i2 = __ffsll((long long)m) - 1;
    r3 = c3 & above(i2);
    const uint32_t w = (uint32_t)__popcll(r3);
    if (b < w) break;
    b -= w;
  }
  return (uint32_t)(select_bit(L, a) + 1) | ((uint32_t)(p + 1) << 8) | ((uint32_t)(i2 + 1) << 16) |
         ((uint32_t)(select_bit(r3, b) + 1) << 24);
}

// entry q of a whole group, from the masks (slow path: k = 4, or no room for the lists)
__device__ __forceinline__ uint32_t group_entry_slow(int k, uint32_t q, uint64_t c0, uint64_t c1, uint64_t c2,
                                                     uint64_t c3) {
  if (k == 1) return (uint32_t)select_bit(c0, q) + 1u;
  int p = 0;
  for (uint64_t m = block_sites(k, c0, c1); m; m &= m - 1) {
    p = __ffsll((long long)m) - 1;
    const uint32_t w = block_size(k, p, c0, c1, c2, c3);
    if (q < w) break;
    q -= w;
  }
  return block_entry(k, p, q, c0, c1, c2, c3);
}

// One tile of K6x / K6q: the entries [e0, e0 + tile_n) of the sorted groups, which are the groups g0 ..
// g0 + ngrp - 1, written to positions o0 + 0 .. o0 + tile_n - 1 of the outputs.
// cmask[row * C + c]: the site masks; row = the payload's peptide field.  gid_tab (sharded build: the
// rows are arrival slots of the group exchange) maps a row to the peptide's global id, else row = id.
// Groups of long peptides go to long_list: K6x lists a group once, in the tile where it starts (K6l writes it
// whole); K6q (kWindow) lists every (group, tile) pair, and the windowed K6l writes the tile's share.
template <bool kWindow>
__device__ __forceinline__ void expand_tile(ExpSmem& s, const DigestCfg& cfg, const uint64_t* __restrict__ cmask,
                                            const uint32_t* __restrict__ gid_tab, const uint64_t* __restrict__ skey,
                                            const uint64_t* __restrict__ spay, const uint64_t* __restrict__ eoff,
                                            uint64_t base_bits, uint64_t tile, uint64_t e0, uint32_t tile_n,
                                            uint32_t g0, uint32_t ngrp, uint64_t o0, double* __restrict__ e_mass,
                                            uint32_t* __restrict__ e_base, uint32_t* __restrict__ e_pat,
                                            uint32_t* __restrict__ long_list, uint32_t* __restrict__ long_count,
                                            uint32_t long_cap, uint32_t* err) {
  const int C = cfg.n_classes;
  const int t = threadIdx.x;
  for (int i = t; i < kExpTile; i += ET_THREADS) s.head[i] = 0;
  if (t <= 64) s.recip[t] = t ? ((1u << 20) + (uint32_t)t - 1u) / (uint32_t)t : 0u;
  if (t == 0) {
    s.nblk = 0;
    s.pool_used = 1;
    s.pool[0] = 0;
  }
  __syncthreads();
  // (1) one thread per group: site lists + block records
  for (uint32_t j = t; j < ngrp; j += ET_THREADS) {
    const uint64_t g = (uint64_t)g0 + j;
    const int64_t rel64 = (int64_t)eoff[g] - (int64_t)e0;
    const int32_t rel = (int32_t)max(rel64, (int64_t)INT32_MIN / 2);
    const uint64_t pay = spay[g];
    const uint32_t row = (uint32_t)(pay >> 32);
    const uint32_t seq = ((uint32_t)pay >> kGrpCntBits) & 31u;
    uint32_t pk;
    int k = pack_seq(seq, C, &pk);
    s.mass[j] = __longlong_as_double((long long)(skey[g] + base_bits));
    s.base[j] = gid_tab ? gid_tab[row] : row;
    s.idx[j] = row;
    s.seq[j] = (uint8_t)seq;
    if (rel >= (int32_t)tile_n) continue;  // the group of the NEXT tile's first entry starts right after this tile
    ExpBlk b;
    b.start = rel; b.grp = (uint16_t)j; b.a0 = 0; b.b0 = 0; b.nb = 1; b.p = 0; b.k = (uint32_t)k;
    auto append = [&](const ExpBlk& x) {
      const uint32_t slot = atomicAdd(&s.nblk, 1u);  // < kExpTile: every listed block owns an entry of the tile
      s.blk[slot] = x;
      s.head[x.start > 0 ? x.start : 0] = ((uint32_t)(x.start > 0 ? x.start : 0) << 16) | slot;
    };
    if (k == 0) {
      append(b);
      continue;
    }
    const uint64_t* cm = cmask + (uint64_t)row * (uint64_t)C;
    const int q0 = seq_class_at(pk, 0), q1 = k > 1 ? seq_class_at(pk, 1) : q0, q2 = k > 2 ? seq_class_at(pk, 2) : q0;
    const uint64_t c0 = cm[q0];
    const uint64_t c1 = k > 1 ? cm[q1] : 0ull;
    const uint64_t c2 = k > 2 ? cm[q2] : 0ull;
    if (c0 == 0) {  // a peptide longer than 64 residues: K6l writes this group
      b.k = kLongGroup;
      append(b);
      if constexpr (kWindow) {  // the caller grows the list and runs the tile again when it overflows
        const uint32_t slot = atomicAdd(long_count, 1u);
        if (slot < long_cap) {
          long_list[2 * slot] = (uint32_t)g;
          long_list[2 * slot + 1] = (uint32_t)tile;
        }
      } else if (rel >= 0 && rel < (int32_t)kExpTile) {
        const uint32_t slot = atomicAdd(long_count, 1u);
        if (slot < long_cap) long_list[slot] = (uint32_t)g; else atomicOr(err, kErrModPos);
      }
      continue;
    }
    // lists of the distinct classes of the sequence (a class used at two levels shares its list)
    const uint32_t n0 = (uint32_t)__popcll(c0);
    const uint32_t n1 = (k > 1 && q1 != q0) ? (uint32_t)__popcll(c1) : 0u;
    const uint32_t n2 = (k > 2 && q2 != q0 && q2 != q1) ? (uint32_t)__popcll(c2) : 0u;
    const uint32_t need = n0 + n1 + n2;
    const uint32_t at = k == 4 ? (uint32_t)EP_POOL : atomicAdd(&s.pool_used, need);
    if (at + need > (uint32_t)EP_POOL) {
      b.k = kSlowGroup;
      append(b);
      continue;
    }
    uint32_t x = fill_sites(c0, s.pool, at);
    const uint32_t l0 = at;
    uint32_t l1 = l0, l2 = l0;
    if (n1) {
      l1 = x;
      x = fill_sites(c1, s.pool, x);
    }
    if (k > 2) {
      l2 = q2 == q0 ? l0 : (q2 == q1 ? l1 : x);
      if (n2) x = fill_sites(c2, s.pool, x);
    }
    if (k == 1) {
      b.b0 = (uint16_t)l0;
      b.nb = (uint8_t)n0;
      append(b);
      continue;
    }
    // k = 2: blocks over the first site;  k = 3: blocks over the middle site
    const uint64_t sites = k == 2 ? c0 : c1;
    const uint64_t cb = k == 2 ? c1 : c2;  // last-level class
    const uint32_t lb = k == 2 ? l1 : l2;
    const uint32_t nb_all = (uint32_t)__popcll(cb);
    int32_t run = rel;
    for (uint64_t m = sites; m && run < (int32_t)tile_n; m &= m - 1) {
      const int p = __ffsll((long long)m) - 1;
      const uint32_t nB = (uint32_t)__popcll(cb & above(p));
      const uint32_t nA = k == 3 ? (uint32_t)__popcll(c0 & below(p)) : 1u;
      const uint32_t sz = nA * nB;
      if (sz == 0) continue;
      if (run + (int32_t)sz > 0) {
        b.start = run;
        b.a0 = k == 3 ? (uint16_t)l0 : (uint16_t)0;
        b.b0 = (uint16_t)(lb + nb_all - nB);  // the last nB sites of the list lie above p
        b.nb = (uint8_t)nB;
        b.p = (uint8_t)p;
        append(b);
      }
      run += (int32_t)sz;
    }
  }
  __syncthreads();
  // (2) inclusive max-scan of the heads: entry -> block slot
  {
    uint32_t loc[ET_PER];
    uint32_t run = 0;
#pragma unroll
    for (int i = 0; i < ET_PER; ++i) {
      run = max(run, s.head[t * ET_PER + i]);
      loc[i] = run;
    }
    uint32_t inc = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t n = __shfl_up_sync(0xffffffffu, inc, o);
      if ((int)lane_id() >= o) inc = max(inc, n);
    }
    if (lane_id() == 31) s.scratch[t >> 5] = inc;
    __syncthreads();
    uint32_t carry = 0;
    for (int w = 0; w < (t >> 5); ++w) carry = max(carry, s.scratch[w]);
    const uint32_t prev = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane_id() > 0) carry = max(carry, prev);
#pragma unroll
    for (int i = 0; i < ET_PER; ++i) s.head[t * ET_PER + i] = max(loc[i], carry);
  }
  __syncthreads();
  // (3) one thread per entry, consecutive threads = consecutive entries
  for (uint32_t i = t; i < tile_n; i += ET_THREADS) {
    const uint4 br = reinterpret_cast<const uint4*>(s.blk)[s.head[i] & 0xffffu];
    const uint32_t j = br.y & 0xffffu;
    const uint32_t k = br.w;
    const uint32_t q = (uint32_t)((int32_t)i - (int32_t)br.x);
    uint32_t pat;
    if (k <= 3u) {
      const uint32_t nb = (br.z >> 16) & 0xffu, p1 = (br.z >> 24) + 1u;
      const uint32_t a = (q * s.recip[nb]) >> 20;  // q / nb (q < 4096)
      const uint32_t pa = s.pool[(br.y >> 16) + a];
      const uint32_t pb = s.pool[(br.z & 0xffffu) + (q - a * nb)];
      pat = k == 3u ? (pa | (p1 << 8) | (pb << 16)) : (k == 2u ? (p1 | (pb << 8)) : pb);
    } else if (k == kSlowGroup) {
      uint32_t pk;
      const int kk = pack_seq(s.seq[j], C, &pk);
      const uint64_t* cm = cmask + (uint64_t)s.idx[j] * (uint64_t)C;
      pat = group_entry_slow(kk, q, cm[seq_class_at(pk, 0)], kk > 1 ? cm[seq_class_at(pk, 1)] : 0ull,
                             kk > 2 ? cm[seq_class_at(pk, 2)] : 0ull, kk > 3 ? cm[seq_class_at(pk, 3)] : 0ull);
    } else {
      continue;  // long group: K6l
    }
    const uint64_t e = o0 + i;
    e_mass[e] = s.mass[j];
    e_base[e] = s.base[j];
    e_pat[e] = pat;
  }
}

__global__ void __launch_bounds__(ET_THREADS, 4)
    grp_expand_tab_kernel(DigestCfg cfg, const uint64_t* __restrict__ cmask, const uint32_t* __restrict__ gid_tab,
                          const uint64_t* __restrict__ skey, const uint64_t* __restrict__ spay,
                          const uint64_t* __restrict__ eoff, const uint32_t* __restrict__ tile_first,
                          uint64_t n_entries, uint64_t base_bits, double* __restrict__ e_mass,
                          uint32_t* __restrict__ e_base, uint32_t* __restrict__ e_pat,
                          uint32_t* __restrict__ long_list, uint32_t* __restrict__ long_count, uint32_t long_cap,
                          uint32_t* err) {
  __shared__ __align__(16) ExpSmem s;
  const uint64_t tile = blockIdx.x;
  const uint64_t e0 = tile * (uint64_t)kExpTile;
  const uint32_t tile_n = (uint32_t)min((uint64_t)kExpTile, n_entries - e0);
  const uint32_t g0 = tile_first[tile];
  const uint32_t ngrp = tile_first[tile + 1] - g0 + 1;
  expand_tile<false>(s, cfg, cmask, gid_tab, skey, spay, eoff, base_bits, tile, e0, tile_n, g0, ngrp, e0, e_mass,
                     e_base, e_pat, long_list, long_count, long_cap, err);
}

// ---- K6q ------------------------------------------------------------------------------
// Entry ranges of a compact index: range q = entries [begin[q], begin[q] + c_q) goes to output positions
// [out_off[q], out_off[q + 1]).  Every range is cut into tiles of kExpTile entries; tile_q[t] = its range and
// tile_off = the exclusive scan of the tiles per range.
__device__ __forceinline__ void range_tile(const ExpRanges& rg, uint64_t tile, uint64_t* e0, uint32_t* tile_n,
                                           uint64_t* o0) {
  const uint32_t q = rg.tile_q[tile];
  const uint64_t k = (tile - rg.tile_off[q]) * (uint64_t)kExpTile;
  const uint64_t lo = rg.out_off[q];
  *e0 = rg.begin[q] + k;
  *tile_n = (uint32_t)min((uint64_t)kExpTile, rg.out_off[q + 1] - lo - k);
  *o0 = lo + k;
}

// the group that holds entry e: last g with eoff[g] <= e (eoff[0] = 0, eoff[n_groups] > e)
__device__ __forceinline__ uint32_t group_of(const uint64_t* __restrict__ eoff, uint64_t n_groups, uint64_t e) {
  uint64_t lo = 0, hi = n_groups;
  while (hi - lo > 1) {
    const uint64_t mid = (lo + hi) >> 1;
    if (__ldg(eoff + mid) <= e) lo = mid; else hi = mid;
  }
  return (uint32_t)lo;
}

// compact index: the sorted keys become the group masses in place (key = mass bits - base_bits)
__global__ void __launch_bounds__(MD_THREADS)
    grp_key_mass_kernel(uint64_t* __restrict__ key, uint64_t n, uint64_t base_bits) {
  const uint64_t i = (uint64_t)blockIdx.x * MD_THREADS + threadIdx.x;
  if (i < n) key[i] += base_bits;
}

__global__ void __launch_bounds__(MD_THREADS)
    grp_entry_ranges_kernel(const uint64_t* __restrict__ eoff, uint64_t nq, uint64_t* __restrict__ begin,
                            uint64_t* __restrict__ count, uint32_t* __restrict__ cnt32, uint32_t* __restrict__ ntile32,
                            uint32_t* __restrict__ over) {
  const uint64_t q = (uint64_t)blockIdx.x * MD_THREADS + threadIdx.x;
  if (q >= nq) return;
  const uint64_t g = begin[q];
  const uint64_t b = eoff[g], c = eoff[g + count[q]] - b;
  begin[q] = b;
  count[q] = c;
  if (cnt32) {
    cnt32[q] = (uint32_t)c;
    if (c >> 32) *over = 1u;
  }
  if (ntile32) ntile32[q] = (uint32_t)min((c + kExpTile - 1) / kExpTile, (uint64_t)UINT32_MAX);
}

// g_mass (the groups' masses, as bits) stands where K6x reads key + base_bits
__global__ void __launch_bounds__(ET_THREADS, 4)
    grp_expand_ranges_kernel(DigestCfg cfg, const uint64_t* __restrict__ cmask, const uint64_t* __restrict__ g_mass,
                             const uint64_t* __restrict__ g_pay, const uint64_t* __restrict__ g_eoff, uint64_t n_groups,
                             const ExpRanges rg, double* __restrict__ o_mass, uint32_t* __restrict__ o_base,
                             uint32_t* __restrict__ o_pat, uint32_t* __restrict__ long_list,
                             uint32_t* __restrict__ long_count, uint32_t long_cap, uint32_t* err) {
  __shared__ __align__(16) ExpSmem s;
  const uint64_t tile = blockIdx.x;
  uint64_t e0, o0;
  uint32_t tile_n;
  range_tile(rg, tile, &e0, &tile_n, &o0);
  const uint32_t g0 = group_of(g_eoff, n_groups, e0);
  const uint32_t g1 = group_of(g_eoff, n_groups, e0 + tile_n - 1);
  expand_tile<true>(s, cfg, cmask, nullptr, g_mass, g_pay, g_eoff, 0, tile, e0, tile_n, g0, g1 - g0 + 1, o0, o_mass,
                    o_base, o_pat, long_list, long_count, long_cap, err);
}

// ---- K6l ------------------------------------------------------------------------------
// Groups of peptides longer than 64 residues (rare): one warp per listed group enumerates the
// occurrences from the site list in shared memory; the last matched site is searched by all lanes
// in parallel, the prefix sites by a warp-uniform odometer.  The order is lexicographic in the site
// tuple.  kWindow (after K6q): the list holds (group, tile) pairs, and only the group's entries inside
// the tile are written, at the tile's output positions.
template <bool kWindow>
__global__ void __launch_bounds__(MD_THREADS)
    grp_expand_long_kernel(const uint8_t* __restrict__ res, const DevTables* __restrict__ tb, DigestCfg cfg,
                           const uint32_t* __restrict__ u_gpos, const uint16_t* __restrict__ u_len,
                           const uint32_t* __restrict__ gid_tab, int use_uv, const __grid_constant__ UniqView uv,
                           const uint64_t* __restrict__ skey,
                           const uint64_t* __restrict__ spay, const uint64_t* __restrict__ eoff,
                           const uint32_t* __restrict__ long_list,
                           const uint32_t* __restrict__ long_count, uint64_t base_bits, double* __restrict__ e_mass,
                           uint32_t* __restrict__ e_base, uint32_t* __restrict__ e_pat, const ExpRanges rg) {
  __shared__ ModTables mt;
  __shared__ WarpSites wsites[MD_WARPS];
  load_mod_tables(mt, tb);
  __syncthreads();
  const int w = threadIdx.x >> 5;
  const unsigned l = lane_id();
  WarpSites& ws = wsites[w];
  const int C = cfg.n_classes;
  const uint32_t n_list = *long_count;
  for (uint32_t li = blockIdx.x * MD_WARPS + w; li < n_list; li += gridDim.x * MD_WARPS) {
    const uint64_t g = long_list[kWindow ? 2 * li : li];
    uint64_t w0 = 0, o0 = 0, w1 = UINT64_MAX;  // entries [w0, w1) go to o0 ..
    if constexpr (kWindow) {
      uint32_t tile_n;
      range_tile(rg, long_list[2 * li + 1], &w0, &tile_n, &o0);
      w1 = w0 + tile_n;
    }
    const uint64_t pay = spay[g];
    const uint32_t bb = (uint32_t)(pay >> 32);
    const uint32_t bseq = ((uint32_t)pay >> kGrpCntBits) & 31u;
    const double bmass = __longlong_as_double((long long)(skey[g] + base_bits));
    uint64_t bo = eoff[g];
    uint32_t bpk;
    const int bk = pack_seq(bseq, C, &bpk);
    bool bad = false;
    uint32_t pgpos, plen;
    if (use_uv) {  // sharded build: the peptide's (gpos, len) live with its owner (mapped peer table)
      uint64_t prow;
      const int pr = uniq_owner(uv, gid_tab[bb], &prow);
      pgpos = uv.gpos[pr][prow];
      plen = uv.len[pr][prow];
    } else {
      pgpos = u_gpos[bb];
      plen = u_len[bb];
    }
    const int n = warp_collect_sites(res, pgpos, plen, mt, ws, &bad);
    // odometer over the first bk-1 sites, all lanes in lockstep.  State in registers only:
    // idxp byte L = site ordinal chosen at level L (0xff = none yet), pat = pattern of the prefix.
    uint32_t idxp = 0xffffffffu;
    uint32_t pat = 0;
    int level = 0;
    while (level >= 0) {
      const int want = seq_class_at(bpk, level);
      const int prev = level > 0 ? (int)((idxp >> (8 * (level - 1))) & 0xffu) : -1;  // always set when level > 0
      if (level == bk - 1) {
        // last element: the lanes scan the sites after the prefix for class `want`
        const uint32_t prefix = pat & low_bytes_mask(level);
        for (int j0 = prev + 1; j0 < n; j0 += 32) {
          const int j = j0 + (int)l;
          const bool ok = j < n && (int)mt.cls[ws.res[j]] == want;
          const unsigned om = __ballot_sync(0xffffffffu, ok);
          uint64_t slot = bo + __popc(om & lanemask_lt());
          bool put = ok;
          if (kWindow) {
            put = put && slot >= w0 && slot < w1;
            slot = o0 + (slot - w0);
          }
          if (put) {
            e_mass[slot] = bmass;
            e_base[slot] = gid_tab ? gid_tab[bb] : bb;
            e_pat[slot] = prefix | (((uint32_t)ws.pos[j] + 1u) << (8 * level));
          }
          bo += __popc(om);
          if (kWindow && bo >= w1) break;
        }
        if (kWindow && bo >= w1) break;  // the rest of the group lies after the window
        --level;
        continue;
      }
      // advance this prefix level to its next site of class `want`
      const uint32_t cur = (idxp >> (8 * level)) & 0xffu;
      int j = (cur != 0xffu ? (int)cur : prev) + 1;
      while (j < n && (int)mt.cls[ws.res[j]] != want) ++j;
      if (j >= n) {
        idxp |= 0xffu << (8 * level);  // exhausted: reset and go up
        --level;
      } else {
        idxp = (idxp & ~(0xffu << (8 * level))) | ((uint32_t)j << (8 * level));
        pat = (pat & low_bytes_mask(level)) | (((uint32_t)ws.pos[j] + 1u) << (8 * level));
        ++level;
        if (level < DBI_MAX_MODS_PER_PEP) idxp |= 0xffu << (8 * level);  // the next level starts fresh
      }
    }
    __syncwarp();
  }
}

}  // namespace

void launch_site_masks(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg, const uint32_t* u_gpos,
                       const uint16_t* u_len, uint64_t n_unique, uint64_t* cmask, unsigned long long* n_long,
                       cudaStream_t s) {
  if (n_unique == 0) return;
  DBI_LAUNCH(site_masks_kernel, (unsigned)((n_unique + MD_THREADS - 1) / MD_THREADS), MD_THREADS, 0, s, d_res, d_tb,
             cfg.n_classes, u_gpos, u_len, n_unique, cmask, n_long);
}

void launch_count_long(const uint16_t* len, uint64_t n, unsigned long long* n_long, cudaStream_t s) {
  if (n == 0) return;
  DBI_LAUNCH(count_long_kernel, (unsigned)((n + MD_THREADS - 1) / MD_THREADS), MD_THREADS, 0, s, len, n, n_long);
}

void launch_grp_count(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg, const double* u_mass,
                      const uint32_t* u_gpos, const uint16_t* u_len, const uint64_t* cmask, uint64_t n_unique,
                      uint32_t tile0, uint32_t ntiles, uint32_t* mask, uint32_t* tile_groups, uint32_t* tile_vars,
                      uint32_t* vt_cnt, uint32_t* d_err, cudaStream_t s) {
  if (n_unique == 0 || ntiles == 0) return;
  const size_t smem = (size_t)cfg.n_seq * MD_THREADS * 4;
  DBI_LAUNCH(grp_count_kernel, ntiles, MD_THREADS, smem, s, d_res, d_tb, cfg, u_mass, u_gpos, u_len, cmask, n_unique,
             tile0, mask, tile_groups, tile_vars, vt_cnt, ntiles, d_err);
}

void launch_grp_emit(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg, const double* u_mass,
                     const uint32_t* u_gpos, const uint16_t* u_len, const uint64_t* cmask, uint64_t n_unique,
                     uint32_t tile0, uint32_t ntiles, const uint32_t* mask, const uint64_t* goffs, bool lists,
                     uint64_t base_bits, uint64_t id_off, uint64_t* g_key, uint64_t* g_pay, uint32_t* d_err,
                     cudaStream_t s) {
  if (n_unique == 0 || ntiles == 0) return;
  const size_t smem = (size_t)cfg.n_seq * MD_THREADS * 4;
  if (lists)
    DBI_LAUNCH(grp_emit_kernel<true>, ntiles, MD_THREADS, smem, s, d_res, d_tb, cfg, u_mass, u_gpos, u_len, cmask,
               n_unique, tile0, mask, goffs, ntiles, base_bits, id_off, g_key, g_pay, d_err);
  else
    DBI_LAUNCH(grp_emit_kernel<false>, ntiles, MD_THREADS, smem, s, d_res, d_tb, cfg, u_mass, u_gpos, u_len, cmask,
               n_unique, tile0, mask, goffs, ntiles, base_bits, id_off, g_key, g_pay, d_err);
}

void launch_grp_extract_cnt(const uint64_t* pay, uint64_t n, uint32_t* cnt, cudaStream_t s) {
  if (n == 0) return;
  DBI_LAUNCH(grp_extract_cnt_kernel, (unsigned)((n + MD_THREADS - 1) / MD_THREADS), MD_THREADS, 0, s, pay, n, cnt);
}

void launch_grp_tile_first(const uint64_t* eoff, uint64_t n_groups, uint64_t n_entries, uint32_t* first,
                           cudaStream_t s) {
  if (n_groups == 0) return;
  const uint64_t n_tiles = (n_entries + kExpTile - 1) / kExpTile;
  DBI_LAUNCH(grp_tile_first_kernel, (unsigned)((n_tiles + 1 + MD_THREADS - 1) / MD_THREADS), MD_THREADS, 0, s, eoff,
             n_groups, n_tiles, first);
}

// payload rows index cmask (and gid_tab, when the rows are arrival slots of a sharded build)
void launch_grp_expand(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg, const uint32_t* u_gpos,
                       const uint16_t* u_len, const uint64_t* cmask, const uint32_t* gid_tab, const UniqView* uv,
                       const uint64_t* skey, const uint64_t* spay, const uint64_t* eoff, const uint32_t* tile_first,
                       uint64_t n_groups, uint64_t n_entries, uint64_t base_bits, double* e_mass, uint32_t* e_base,
                       uint32_t* e_pat, uint32_t* long_list, uint32_t* long_count, uint32_t long_cap, uint32_t* d_err,
                       cudaStream_t s) {
  if (n_groups == 0 || n_entries == 0) return;
  const uint64_t n_tiles = (n_entries + kExpTile - 1) / kExpTile;
  DBI_LAUNCH(grp_expand_tab_kernel, (unsigned)n_tiles, ET_THREADS, 0, s, cfg, cmask, gid_tab, skey, spay, eoff,
             tile_first, n_entries, base_bits, e_mass, e_base, e_pat, long_list, long_count, long_cap, d_err);
  if (long_cap > 0) {
    unsigned grid = (long_cap + MD_WARPS - 1) / MD_WARPS;
    if (grid > (unsigned)kNumSMsB200 * 4) grid = (unsigned)kNumSMsB200 * 4;
    UniqView none;
    std::memset(&none, 0, sizeof(none));
    DBI_LAUNCH(grp_expand_long_kernel<false>, grid, MD_THREADS, 0, s, d_res, d_tb, cfg, u_gpos, u_len, gid_tab,
               (uv && gid_tab) ? 1 : 0, uv ? *uv : none, skey, spay, eoff, long_list, long_count, base_bits, e_mass,
               e_base, e_pat, ExpRanges{});
  }
}

void launch_grp_key_mass(uint64_t* key, uint64_t n, uint64_t base_bits, cudaStream_t s) {
  if (n == 0) return;
  DBI_LAUNCH(grp_key_mass_kernel, (unsigned)((n + MD_THREADS - 1) / MD_THREADS), MD_THREADS, 0, s, key, n, base_bits);
}

void launch_grp_entry_ranges(const uint64_t* eoff, uint64_t nq, uint64_t* begin, uint64_t* count, uint32_t* cnt32,
                             uint32_t* ntile32, uint32_t* over, cudaStream_t s) {
  if (nq == 0) return;
  DBI_LAUNCH(grp_entry_ranges_kernel, (unsigned)((nq + MD_THREADS - 1) / MD_THREADS), MD_THREADS, 0, s, eoff, nq, begin,
             count, cnt32, ntile32, over);
}

void launch_grp_expand_ranges(const DigestCfg& cfg, const uint64_t* cmask, const double* g_mass, const uint64_t* g_pay,
                              const uint64_t* g_eoff, uint64_t n_groups, const ExpRanges& rg, uint64_t n_tiles,
                              double* o_mass, uint32_t* o_base, uint32_t* o_pat, uint32_t* long_list,
                              uint32_t* long_count, uint32_t long_cap, uint32_t* d_err, cudaStream_t s) {
  if (n_groups == 0 || n_tiles == 0) return;
  DBI_LAUNCH(grp_expand_ranges_kernel, (unsigned)n_tiles, ET_THREADS, 0, s, cfg, cmask, (const uint64_t*)g_mass, g_pay,
             g_eoff, n_groups, rg, o_mass, o_base, o_pat, long_list, long_count, long_cap, d_err);
}

void launch_grp_expand_ranges_long(const uint8_t* d_res, const DevTables* d_tb, const DigestCfg& cfg,
                                   const uint32_t* u_gpos, const uint16_t* u_len, const double* g_mass,
                                   const uint64_t* g_pay, const uint64_t* g_eoff, const ExpRanges& rg,
                                   const uint32_t* long_list, const uint32_t* long_count, uint32_t n_listed,
                                   double* o_mass, uint32_t* o_base, uint32_t* o_pat, cudaStream_t s) {
  if (n_listed == 0) return;
  unsigned grid = (n_listed + MD_WARPS - 1) / MD_WARPS;
  if (grid > (unsigned)kNumSMsB200 * 4) grid = (unsigned)kNumSMsB200 * 4;
  UniqView none;
  std::memset(&none, 0, sizeof(none));
  DBI_LAUNCH(grp_expand_long_kernel<true>, grid, MD_THREADS, 0, s, d_res, d_tb, cfg, u_gpos, u_len, nullptr, 0, none,
             (const uint64_t*)g_mass, g_pay, g_eoff, long_list, long_count, 0, o_mass, o_base, o_pat, rg);
}

}  // namespace dbi
