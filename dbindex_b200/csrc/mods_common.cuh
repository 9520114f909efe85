// mods_common.cuh -- helpers shared by the differential-mod kernels (mods.cu: one sort record per
// variant; mods_grp.cu: one sort record per (peptide, class sequence) group).
#pragma once
#include "kernels.cuh"

namespace dbi {
namespace {

constexpr int MD_THREADS = 256;
constexpr int MD_WARPS = MD_THREADS / 32;
constexpr int MD_PER_WARP = kModTile / MD_WARPS;  // bases per warp per tile
constexpr int MD_MAX_SITES = DBI_MAX_MOD_POS + 1;  // positions 0..254

struct ModTables {
  double diff[256];
  uint8_t flags[256];
  uint8_t cls[256];
  double cls_delta[16];
};

struct WarpSites {
  uint8_t pos[256];
  uint8_t res[256];
};

__device__ __forceinline__ void load_mod_tables(ModTables& mt, const DevTables* __restrict__ tb) {
  for (int i = threadIdx.x; i < 256; i += blockDim.x) {
    mt.diff[i] = tb->diff[i];
    mt.flags[i] = tb->flags[i];
    mt.cls[i] = tb->cls[i];
    if (i < 16) mt.cls_delta[i] = tb->cls_delta[i];
  }
}

// Heaviest peptides first: the bases are mass-sorted and the variant count grows like the
// cube of the site count, so the last tiles carry orders of magnitude more work.
__device__ __forceinline__ uint32_t mod_tile_local() { return gridDim.x - 1 - blockIdx.x; }

// Gated count of one peptide with one lane per class SEQUENCE (n_seq <= 32).  The variant mass
// depends only on the sequence of shift classes along the chosen sites, so
//   #passing = sum over sequences s of [gate(f_s(base))] * #(occurrences of s as a subsequence
//              of the peptide's site-class string),
// and the occurrence counts follow from one pass over the sites: a site of class c extends every
// sequence's parent (heap numbering: children of v are v*C + c + 1).
// C(m, j) for j <= 4, m <= 255
__device__ __forceinline__ uint32_t binom(uint32_t m, int j) {
  switch (j) {
    case 0: return 1u;
    case 1: return m;
    case 2: return m < 2 ? 0u : m * (m - 1) / 2;
    case 3: return m < 3 ? 0u : m * (m - 1) * (m - 2) / 6;
    default: return m < 4 ? 0u : (uint32_t)((uint64_t)m * (m - 1) * (m - 2) * (m - 3) / 24);
  }
}

// number of subsets of size <= K of n sites
__device__ __forceinline__ uint32_t total_variants(uint32_t n, int K) {
  uint32_t t = 0;
  for (int k = 0; k <= K; ++k) t += binom(n, k);
  return t;
}

// Whole warp: eligible sites of the peptide res[g .. g+len) into ws (positions ascending).
// Returns the number of sites (<= 255); *bad is set if one lies beyond DBI_MAX_MOD_POS.
__device__ __forceinline__ int warp_collect_sites(const uint8_t* __restrict__ res, uint32_t g, uint32_t len,
                                                  const ModTables& mt, WarpSites& ws, bool* bad) {
  const unsigned l = lane_id();
  int n = 0;
  for (uint32_t b = 0; b < len; b += 32) {
    const uint32_t i = b + l;
    const uint8_t c = (i < len) ? ld_res(res, g + i) : (uint8_t)0;
    const bool is = (i < len) && (mt.flags[c] & kFlagDiffMod);
    const unsigned m = __ballot_sync(0xffffffffu, is);
    if (is) {
      if (i > DBI_MAX_MOD_POS) {
        *bad = true;
      } else {
        const int slot = n + __popc(m & lanemask_lt());
        ws.pos[slot] = (uint8_t)i;
        ws.res[slot] = c;
      }
    }
    n += __popc(m);
  }
  *bad = __any_sync(0xffffffffu, *bad);  // warp-uniform verdict
  __syncwarp();                          // the site list is read by other lanes next
  return n > MD_MAX_SITES ? MD_MAX_SITES : n;
}


// Class sequence of heap node v (children of v are v*C + c + 1), packed: nibble j = class of the
// j-th chosen site (site order).  Returns the sequence length.  Register-only on purpose.
__device__ __forceinline__ int pack_seq(uint32_t v, int C, uint32_t* packed) {
  uint32_t pk = 0;
  int depth = 0;
  while (v > 0) {  // leaf to root: the last class first, so shifting left ends with class 0 in nibble 0
    pk = (pk << 4) | ((v - 1) % (uint32_t)C);
    v = (v - 1) / (uint32_t)C;
    ++depth;
  }
  *packed = pk;
  return depth;
}
__device__ __forceinline__ int seq_class_at(uint32_t packed, int j) { return (int)((packed >> (4 * j)) & 15u); }
__device__ __forceinline__ uint32_t low_bytes_mask(int n_bytes) {
  return n_bytes >= 4 ? 0xffffffffu : ((1u << (8 * n_bytes)) - 1u);
}
// bits strictly above position i
__device__ __forceinline__ uint64_t above(int i) { return (~1ull) << i; }
__device__ __forceinline__ uint64_t below(int i) { return ~(~0ull << i); }  // bits strictly below position i


// pairs i2 < i3 above position i (third and fourth class)
__device__ __forceinline__ uint32_t pairs_above(int i, uint64_t c2, uint64_t c3) {
  uint32_t w = 0;
  for (uint64_t m = c2 & above(i); m; m &= m - 1) w += (uint32_t)__popcll(c3 & above(__ffsll((long long)m) - 1));
  return w;
}

// mask of the block sites of a group and the size of the block at site p
__device__ __forceinline__ uint64_t block_sites(int k, uint64_t c0, uint64_t c1) { return k == 2 ? c0 : c1; }
__device__ __forceinline__ uint32_t block_size(int k, int p, uint64_t c0, uint64_t c1, uint64_t c2, uint64_t c3) {
  if (k == 2) return (uint32_t)__popcll(c1 & above(p));
  const uint32_t nl = (uint32_t)__popcll(c0 & below(p));
  if (k == 3) return nl * (uint32_t)__popcll(c2 & above(p));
  return nl ? nl * pairs_above(p, c2, c3) : 0u;
}

// Inverse of the block order of K6x (mods_grp.cu group_entry_slow): the rank inside its group of the variant
// whose level-j site is pos[j] (0-based, ascending), for a peptide of up to 64 residues.  c0..c3 = the site
// masks of the classes of the sequence's levels.
__device__ __forceinline__ uint32_t group_entry_rank(int k, const int* pos, uint64_t c0, uint64_t c1, uint64_t c2,
                                                     uint64_t c3) {
  if (k == 0) return 0u;
  if (k == 1) return (uint32_t)__popcll(c0 & below(pos[0]));
  const int pb = k == 2 ? pos[0] : pos[1];  // the block site
  uint32_t r = 0;                           // entries of the blocks before
  for (uint64_t m = block_sites(k, c0, c1) & below(pb); m; m &= m - 1)
    r += block_size(k, __ffsll((long long)m) - 1, c0, c1, c2, c3);
  if (k == 2) return r + (uint32_t)__popcll(c1 & above(pos[0]) & below(pos[1]));
  const uint32_t a = (uint32_t)__popcll(c0 & below(pos[0]));
  if (k == 3) {
    const uint64_t R = c2 & above(pb);
    return r + a * (uint32_t)__popcll(R) + (uint32_t)__popcll(R & below(pos[2]));
  }
  uint32_t b = (uint32_t)__popcll(c3 & above(pos[2]) & below(pos[3]));  // pairs (i2, i3) before (pos[2], pos[3])
  for (uint64_t m = c2 & above(pb) & below(pos[2]); m; m &= m - 1)
    b += (uint32_t)__popcll(c3 & above(__ffsll((long long)m) - 1));
  return r + a * pairs_above(pb, c2, c3) + b;
}


}  // namespace
}  // namespace dbi
