// dedup.cu -- K8: merge equal peptides after the sort.
//
// Restates DBIndexStoreSQLiteByteIndexMerge.getMergedData (Merge:620-719): records
// with the same peptide STRING collapse into one entry that keeps the first
// occurrence's (mass, offset, length) and the protein ids of every occurrence in
// insertion order, duplicates kept (Merge:658-663,678-687, SURVEY.md Q6).
//
// The records arrive sorted by (mass bits, sequence hash, emission ordinal), so the
// occurrences of one string are adjacent and in insertion order; equal mass does
// NOT imply equal string (permutation isomers), hence the residue comparison.
// Two different strings with equal mass bits AND equal hash would interleave; that case is
// detected here and the caller re-sorts with another seed and a wider hash.  The number of
// distinct-string pairs with equal mass grows with the square of the record count, so the hash
// is 32 bits for small builds and up to 64 bits (two independent 32-bit halves) for large ones.
#include "kernels.cuh"

namespace dbi {
namespace {

constexpr int DD_THREADS = 256;
constexpr int DD_IPT = kScanTile / DD_THREADS;
// K8r: records per CTA of the first kernel, the longest run it sorts itself, and the run length the
// second kernel sorts in one shared-memory pass (longer runs: sorted chunks of it, then merges)
constexpr uint32_t kRunTile = 2048;
constexpr int RT_IPT = kRunTile / DD_THREADS;
constexpr uint32_t kRunTileCap = 64;
constexpr uint32_t kRunBlockCap = 2048;

__device__ __forceinline__ uint32_t fmix32(uint32_t h) {
  h ^= h >> 16;
  h *= 0x85ebca6bu;
  h ^= h >> 13;
  h *= 0xc2b2ae35u;
  h ^= h >> 16;
  return h;
}

// Seeded hash of one record's residues: the 32-bit hash, or (WIDE) it in the low half and a second,
// independent one in the high half.
template <bool WIDE>
__device__ __forceinline__ uint64_t record_hash(const uint8_t* __restrict__ res, uint32_t g, uint32_t l, uint32_t seed) {
  uint32_t h = 0x811c9dc5u ^ seed;
  uint32_t h2 = 0x9747b28cu + seed;
  for (uint32_t k = 0; k < l; ++k) {
    const uint32_t c = ld_res(res, g + k);
    h = (h ^ c) * 16777619u;
    if (WIDE) h2 = (h2 + c + 1u) * 0x9e3779b1u ^ (h2 >> 15);
  }
  const uint32_t lo = fmix32(h ^ (l * 0x9e3779b1u));
  return WIDE ? ((uint64_t)fmix32(h2 ^ l) << 32) | lo : (uint64_t)lo;
}

// hash[i] of every record and idx[i] = i: the input of the hash pre-sort of large builds
template <bool WIDE>
__global__ void __launch_bounds__(DD_THREADS)
    hash_records_kernel(const uint8_t* __restrict__ res, const uint32_t* __restrict__ gpos,
                        const uint16_t* __restrict__ len, uint64_t n, uint32_t seed, void* __restrict__ hash,
                        uint32_t* __restrict__ idx) {
  const uint64_t i = (uint64_t)blockIdx.x * DD_THREADS + threadIdx.x;
  if (i >= n) return;
  const uint64_t hv = record_hash<WIDE>(res, gpos[i], len[i], seed);
  if (WIDE) ((uint64_t*)hash)[i] = hv;
  else ((uint32_t*)hash)[i] = (uint32_t)hv;
  idx[i] = (uint32_t)i;
}

__global__ void __launch_bounds__(DD_THREADS)
    gather_mass_key_kernel(const uint64_t* __restrict__ mass_bits, const uint32_t* __restrict__ idx, uint64_t n,
                           uint64_t base_bits, uint64_t* __restrict__ key) {
  const uint64_t i = (uint64_t)blockIdx.x * DD_THREADS + threadIdx.x;
  if (i < n) key[i] = mass_bits[idx[i]] - base_bits;
}

__global__ void __launch_bounds__(DD_THREADS)
    mass_key_kernel(const uint64_t* __restrict__ mass_bits, uint64_t n, uint64_t base_bits, uint64_t* __restrict__ key,
                    uint32_t* __restrict__ idx) {
  const uint64_t i = (uint64_t)blockIdx.x * DD_THREADS + threadIdx.x;
  if (i < n) {
    key[i] = mass_bits[i] - base_bits;
    idx[i] = (uint32_t)i;
  }
}

// Order of two records of one equal-mass run: (masked hash, arrival index).  Indices are unique,
// so this is a total order and any correct sort of a run gives the same result.
__device__ __forceinline__ bool run_less(uint64_t ha, uint32_t a, uint64_t hb, uint32_t b) {
  return ha < hb || (ha == hb && a < b);
}

// K8r, first kernel: one CTA per kRunTile sorted records.  Every member of an equal-mass run of
// length >= 2 gets its hash (hash[idx], read by K8's flags).  A run that lies inside the tile and
// has at most kRunTileCap members is sorted here by a rank count; the head of any other run
// appends the run's first position to `list` for run_order_long_kernel.
template <bool WIDE>
__global__ void __launch_bounds__(DD_THREADS)
    run_order_tile_kernel(const uint8_t* __restrict__ res, const uint64_t* __restrict__ skey,
                          uint32_t* __restrict__ sidx, const uint32_t* __restrict__ gpos,
                          const uint16_t* __restrict__ len, uint64_t n, uint32_t seed, uint64_t mask,
                          void* __restrict__ hash, uint32_t* __restrict__ list, uint32_t* __restrict__ n_list) {
  __shared__ uint64_t sh_k[kRunTile];
  __shared__ uint64_t sh_h[kRunTile];
  __shared__ uint32_t sh_i[kRunTile];
  const uint64_t tb = (uint64_t)blockIdx.x * kRunTile;
  const uint32_t tn = (uint32_t)min((uint64_t)kRunTile, n - tb);
#pragma unroll
  for (int k = 0; k < RT_IPT; ++k) {
    const uint32_t p = k * DD_THREADS + threadIdx.x;
    if (p < tn) sh_k[p] = skey[tb + p];
  }
  // the keys just outside the tile; ~0 (no mass key) beyond the ends of the array
  const uint64_t key_before = tb > 0 ? skey[tb - 1] : ~0ull;
  const uint64_t key_after = tb + tn < n ? skey[tb + tn] : ~0ull;
  __syncthreads();
  uint32_t member = 0;  // bit k: item k is in a run sorted by this CTA
  uint32_t rs[RT_IPT], re[RT_IPT];
#pragma unroll
  for (int k = 0; k < RT_IPT; ++k) {
    const uint32_t p = k * DD_THREADS + threadIdx.x;
    if (p >= tn) break;
    const uint64_t key = sh_k[p];
    const bool prev_eq = (p > 0 ? sh_k[p - 1] : key_before) == key;
    const bool next_eq = (p + 1 < tn ? sh_k[p + 1] : key_after) == key;
    if (!prev_eq && !next_eq) continue;  // a singleton: stays where it is, needs no hash
    const uint64_t i = tb + p;
    const uint32_t id = sidx[i];
    const uint64_t hv = record_hash<WIDE>(res, gpos[id], len[id], seed);
    if (WIDE) ((uint64_t*)hash)[id] = hv;
    else ((uint32_t*)hash)[id] = (uint32_t)hv;
    sh_h[p] = hv & mask;
    sh_i[p] = id;
    // bounds of the run inside the tile, looking at most kRunTileCap records each way
    uint32_t s = p, e = p + 1;
    while (s > 0 && p - s < kRunTileCap && sh_k[s - 1] == key) --s;
    while (e < tn && e - p <= kRunTileCap && sh_k[e] == key) ++e;
    const bool whole = (s > 0 || key_before != key) && (e < tn || key_after != key);
    if (whole && e - s <= kRunTileCap) {
      member |= 1u << k;
      rs[k] = s;
      re[k] = e;
    } else if (!prev_eq) {  // the head of a run sorted by the second kernel
      list[atomicAdd(n_list, 1u)] = (uint32_t)i;
    }
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < RT_IPT; ++k) {
    if (!(member >> k & 1u)) continue;
    const uint32_t p = k * DD_THREADS + threadIdx.x;
    const uint64_t hp = sh_h[p];
    const uint32_t ip = sh_i[p];
    uint32_t rank = 0;
    for (uint32_t q = rs[k]; q < re[k]; ++q) rank += run_less(sh_h[q], sh_i[q], hp, ip);
    sidx[tb + rs[k] + rank] = ip;
  }
}

// Sorts cnt <= kRunBlockCap (hash, index) pairs in shared memory: bitonic network over the next power
// of two, padded with all-ones pairs, which rank after every real pair.
__device__ __forceinline__ void block_sort_run(uint64_t* sh_h, uint32_t* sh_i, uint32_t cnt) {
  uint32_t P = 2;
  while (P < cnt) P <<= 1;
  for (uint32_t q = cnt + threadIdx.x; q < P; q += blockDim.x) {
    sh_h[q] = ~0ull;
    sh_i[q] = ~0u;
  }
  __syncthreads();
  for (uint32_t k = 2; k <= P; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t t = threadIdx.x; t < P / 2; t += blockDim.x) {
        const uint32_t a = ((t & ~(j - 1)) << 1) | (t & (j - 1)), b = a + j;  // j: a power of two
        const bool up = (a & k) == 0;
        if (run_less(sh_h[b], sh_i[b], sh_h[a], sh_i[a]) == up) {
          const uint64_t th = sh_h[a];
          sh_h[a] = sh_h[b];
          sh_h[b] = th;
          const uint32_t ti = sh_i[a];
          sh_i[a] = sh_i[b];
          sh_i[b] = ti;
        }
      }
      __syncthreads();
    }
  }
}

template <bool WIDE>
__device__ __forceinline__ uint64_t masked_hash(const void* __restrict__ hash, uint64_t mask, uint32_t id) {
  return (WIDE ? ((const uint64_t*)hash)[id] : (uint64_t)((const uint32_t*)hash)[id]) & mask;
}

// K8r, second kernel: one CTA per listed run at a time (grid-stride over the list).  A run of up to
// kRunBlockCap records is sorted in shared memory; a longer one in sorted chunks of kRunBlockCap that
// are then merged pairwise through `alt` (n spare slots), each thread producing one contiguous span
// of every merged pair after a merge-path search.
template <bool WIDE>
__global__ void __launch_bounds__(DD_THREADS)
    run_order_long_kernel(const uint64_t* __restrict__ skey, uint32_t* __restrict__ sidx, uint32_t* __restrict__ alt,
                          uint64_t n, const void* __restrict__ hash, uint64_t mask, const uint32_t* __restrict__ list,
                          const uint32_t* __restrict__ n_list) {
  __shared__ uint64_t sh_h[kRunBlockCap];
  __shared__ uint32_t sh_i[kRunBlockCap];
  __shared__ uint64_t sh_end;
  const uint32_t nl = *n_list;
  for (uint32_t r = blockIdx.x; r < nl; r += gridDim.x) {
    const uint64_t s = list[r];
    const uint64_t key = skey[s];
    // end of the run: the first later position with another key
    if (threadIdx.x == 0) sh_end = n;
    __syncthreads();
    for (uint64_t c = s + 1;; c += blockDim.x) {
      const uint64_t i = c + threadIdx.x;
      if (i < n && skey[i] != key) atomicMin((unsigned long long*)&sh_end, (unsigned long long)i);
      if (__syncthreads_or(sh_end != n || c + blockDim.x >= n)) break;
    }
    const uint64_t e = sh_end;
    const uint64_t L = e - s;
    // sorted chunks of kRunBlockCap
    for (uint64_t c0 = s; c0 < e; c0 += kRunBlockCap) {
      const uint32_t cnt = (uint32_t)min((uint64_t)kRunBlockCap, e - c0);
      for (uint32_t q = threadIdx.x; q < cnt; q += blockDim.x) {
        const uint32_t id = sidx[c0 + q];
        sh_h[q] = masked_hash<WIDE>(hash, mask, id);
        sh_i[q] = id;
      }
      block_sort_run(sh_h, sh_i, cnt);
      for (uint32_t q = threadIdx.x; q < cnt; q += blockDim.x) sidx[c0 + q] = sh_i[q];
      __syncthreads();
    }
    // pairwise merges of sorted spans of width w, ping-ponging between sidx and alt (run offsets fit
    // 32 bits: N < 2^32)
    uint32_t* src = sidx + s;
    uint32_t* dst = alt + s;
    const uint32_t Lr = (uint32_t)L;
    for (uint32_t w = kRunBlockCap; w < Lr; w <<= 1) {
      const uint32_t span = (Lr + blockDim.x - 1) / blockDim.x;
      uint32_t o = threadIdx.x * span;
      const uint32_t o_end = min(Lr, o + span);
      while (o < o_end) {
        const uint32_t a0 = o & ~(2 * w - 1);  // the merged pair [a0, a0 + na + nb)
        const uint32_t na = min(w, Lr - a0), nb = min(w, Lr - a0 - na);
        const uint32_t* A = src + a0;
        const uint32_t* B = A + na;
        const uint32_t stop = min(o_end, a0 + na + nb);
        // merge path: lo records of A and k - lo of B precede output o
        const uint32_t k = o - a0;
        uint32_t lo = k > nb ? k - nb : 0, hi = min(k, na);
        while (lo < hi) {
          const uint32_t m = (lo + hi) / 2;
          const uint32_t am = A[m], bm = B[k - 1 - m];
          if (run_less(masked_hash<WIDE>(hash, mask, am), am, masked_hash<WIDE>(hash, mask, bm), bm)) lo = m + 1;
          else hi = m;
        }
        uint32_t ia = lo, ib = k - lo;
        for (; o < stop; ++o) {
          bool take_a = ib >= nb;
          if (!take_a && ia < na) {
            const uint32_t x = A[ia], y = B[ib];
            take_a = run_less(masked_hash<WIDE>(hash, mask, x), x, masked_hash<WIDE>(hash, mask, y), y);
          }
          dst[o] = take_a ? A[ia++] : B[ib++];
        }
      }
      __syncthreads();
      uint32_t* t = src;
      src = dst;
      dst = t;
    }
    if (src != sidx + s) {
      for (uint32_t q = threadIdx.x; q < Lr; q += blockDim.x) sidx[s + q] = src[q];
    }
    __syncthreads();
  }
}

template <typename H>
__global__ void __launch_bounds__(DD_THREADS)
    dedup_flags_kernel(const uint8_t* __restrict__ res, const uint64_t* __restrict__ skey,
                       const uint32_t* __restrict__ sidx, const H* __restrict__ hash, H hash_mask,
                       const uint32_t* __restrict__ gpos, const uint16_t* __restrict__ len, uint64_t n,
                       uint8_t* __restrict__ flags, uint32_t* __restrict__ tile_counts, uint32_t* err) {
  __shared__ uint32_t scratch[DD_THREADS / 32 + 1];
  const uint64_t tile_base = (uint64_t)blockIdx.x * kScanTile;
  uint32_t heads = 0;
#pragma unroll 4
  for (int k = 0; k < DD_IPT; ++k) {
    const uint64_t i = tile_base + (uint64_t)k * DD_THREADS + threadIdx.x;
    if (i >= n) break;
    uint8_t head = 1;
    if (i > 0 && skey[i] == skey[i - 1]) {
      const uint32_t a = sidx[i], b = sidx[i - 1];
      if (((hash[a] ^ hash[b]) & hash_mask) == 0) {  // only the sorted bits of the hash group the run
        const uint32_t la = len[a], lb = len[b];
        bool same = la == lb;
        if (same) {
          const uint32_t ga = gpos[a], gb = gpos[b];
          if (ga != gb)
            for (uint32_t q = 0; q < la; ++q)
              if (ld_res(res, ga + q) != ld_res(res, gb + q)) { same = false; break; }
        }
        if (same) head = 0;
        else atomicOr(err, kErrHashCollision);  // different strings, same (mass, hash)
      }
    }
    flags[i] = head;
    heads += head;
  }
  uint32_t total;
  block_exclusive_sum<uint32_t, DD_THREADS>(heads, scratch, &total);
  if (threadIdx.x == 0) tile_counts[blockIdx.x] = total;
}

__global__ void __launch_bounds__(DD_THREADS)
    dedup_emit_kernel(const uint64_t* __restrict__ skey, const uint32_t* __restrict__ sidx,
                      const uint8_t* __restrict__ flags, const uint64_t* __restrict__ tile_offs,
                      const uint32_t* __restrict__ gpos, const uint32_t* __restrict__ prot,
                      const uint16_t* __restrict__ len, uint64_t n, uint64_t base_bits, uint64_t n_unique,
                      double* __restrict__ u_mass, uint32_t* __restrict__ u_gpos, uint32_t* __restrict__ u_prot,
                      uint16_t* __restrict__ u_len, uint64_t* __restrict__ u_plo, uint32_t* __restrict__ plist) {
  __shared__ uint32_t scratch[DD_THREADS / 32 + 1];
  const uint64_t tile_base = (uint64_t)blockIdx.x * kScanTile;
  uint64_t running = tile_offs[blockIdx.x];
  if (blockIdx.x == 0 && threadIdx.x == 0) u_plo[n_unique] = n;
  for (int k = 0; k < DD_IPT; ++k) {
    const uint64_t i = tile_base + (uint64_t)k * DD_THREADS + threadIdx.x;
    const bool valid = i < n;
    const uint32_t head = valid ? flags[i] : 0u;
    uint32_t total;
    const uint32_t ex = block_exclusive_sum<uint32_t, DD_THREADS>(head, scratch, &total);
    if (valid) {
      const uint32_t r = sidx[i];
      const uint32_t pr = prot[r];
      plist[i] = pr;  // protein ids of all occurrences, insertion order (Merge:678-681)
      if (head) {     // first occurrence supplies mass / offset / length (Merge:684-687)
        const uint64_t u = running + ex;
        u_mass[u] = __longlong_as_double((long long)(skey[i] + base_bits));
        u_gpos[u] = gpos[r];
        u_prot[u] = pr;
        u_len[u] = len[r];
        u_plo[u] = i;
      }
    }
    running += total;
  }
}

}  // namespace

void launch_hash_records(const uint8_t* d_res, const uint32_t* gpos, const uint16_t* len, uint64_t n, uint32_t seed,
                         bool wide, void* hash, uint32_t* idx, cudaStream_t s) {
  if (n == 0) return;
  const unsigned grid = (unsigned)((n + DD_THREADS - 1) / DD_THREADS);
  if (wide) DBI_LAUNCH(hash_records_kernel<true>, grid, DD_THREADS, 0, s, d_res, gpos, len, n, seed, hash, idx);
  else DBI_LAUNCH(hash_records_kernel<false>, grid, DD_THREADS, 0, s, d_res, gpos, len, n, seed, hash, idx);
}

void launch_gather_mass_key(const uint64_t* mass_bits, const uint32_t* idx, uint64_t n, uint64_t base_bits,
                            uint64_t* key, cudaStream_t s) {
  if (n == 0) return;
  const unsigned grid = (unsigned)((n + DD_THREADS - 1) / DD_THREADS);
  DBI_LAUNCH(gather_mass_key_kernel, grid, DD_THREADS, 0, s, mass_bits, idx, n, base_bits, key);
}

uint64_t run_order_list_cap(uint64_t n) {
  // a listed run crosses a tile edge or is longer than kRunTileCap
  return (n + kRunTile - 1) / kRunTile + n / (kRunTileCap + 1) + 1;
}

void launch_mass_key(const uint64_t* mass_bits, uint64_t n, uint64_t base_bits, uint64_t* key, uint32_t* idx,
                     cudaStream_t s) {
  if (n == 0) return;
  const unsigned grid = (unsigned)((n + DD_THREADS - 1) / DD_THREADS);
  DBI_LAUNCH(mass_key_kernel, grid, DD_THREADS, 0, s, mass_bits, n, base_bits, key, idx);
}

void launch_run_order(const uint8_t* d_res, const uint64_t* skey, uint32_t* sidx, uint32_t* alt,
                      const uint32_t* gpos, const uint16_t* len, uint64_t n, uint32_t seed, int hash_bits, void* hash,
                      uint32_t* list, uint32_t* n_list, cudaStream_t s) {
  if (n == 0) return;
  const uint64_t mask = hash_bits >= 64 ? ~0ull : ((1ull << hash_bits) - 1);
  const bool wide = hash_bits > 32;
  const unsigned tiles = (unsigned)((n + kRunTile - 1) / kRunTile);
  // the number of listed runs stays on the device: a fixed grid walks the list
  const unsigned long_grid = (unsigned)std::min<uint64_t>(tiles, 4 * 148);
  DBI_CUDA(cudaMemsetAsync(n_list, 0, 4, s));
  if (wide) {
    DBI_LAUNCH(run_order_tile_kernel<true>, tiles, DD_THREADS, 0, s, d_res, skey, sidx, gpos, len, n, seed, mask, hash,
               list, n_list);
    DBI_LAUNCH(run_order_long_kernel<true>, long_grid, DD_THREADS, 0, s, skey, sidx, alt, n, hash, mask, list, n_list);
  } else {
    DBI_LAUNCH(run_order_tile_kernel<false>, tiles, DD_THREADS, 0, s, d_res, skey, sidx, gpos, len, n, seed, mask,
               hash, list, n_list);
    DBI_LAUNCH(run_order_long_kernel<false>, long_grid, DD_THREADS, 0, s, skey, sidx, alt, n, hash, mask, list, n_list);
  }
}

void launch_dedup_flags(const uint8_t* d_res, const uint64_t* skey, const uint32_t* sidx, const void* hash,
                        int hash_bits, const uint32_t* gpos, const uint16_t* len, uint64_t n, uint8_t* flags,
                        uint32_t* tile_counts, uint32_t* d_err, cudaStream_t s) {
  if (n == 0) return;
  const unsigned tiles = (unsigned)((n + kScanTile - 1) / kScanTile);
  if (hash_bits > 32) {
    const uint64_t mask = hash_bits >= 64 ? ~0ull : ((1ull << hash_bits) - 1);
    DBI_LAUNCH(dedup_flags_kernel<uint64_t>, tiles, DD_THREADS, 0, s, d_res, skey, sidx, (const uint64_t*)hash, mask,
               gpos, len, n, flags, tile_counts, d_err);
  } else {
    DBI_LAUNCH(dedup_flags_kernel<uint32_t>, tiles, DD_THREADS, 0, s, d_res, skey, sidx, (const uint32_t*)hash,
               0xffffffffu, gpos, len, n, flags, tile_counts, d_err);
  }
}

void launch_dedup_emit(const uint64_t* skey, const uint32_t* sidx, const uint8_t* flags, const uint64_t* tile_offs,
                       const uint32_t* gpos, const uint32_t* prot, const uint16_t* len, uint64_t n,
                       uint64_t base_bits, uint64_t n_unique, double* u_mass, uint32_t* u_gpos, uint32_t* u_prot,
                       uint16_t* u_len, uint64_t* u_plo, uint32_t* plist, cudaStream_t s) {
  if (n == 0) return;
  const unsigned tiles = (unsigned)((n + kScanTile - 1) / kScanTile);
  DBI_LAUNCH(dedup_emit_kernel, tiles, DD_THREADS, 0, s, skey, sidx, flags, tile_offs, gpos, prot, len, n, base_bits,
             n_unique, u_mass, u_gpos, u_prot, u_len, u_plo, plist);
}

}  // namespace dbi
