// window.cu -- K12: the mass windows of an unindexed search (dbi_search_unindexed) in the form the range-filtered
// digest (K2u / K4u, InWindows) tests a record against: windows sorted by their lower bound (K7 onesweep sort on
// key = bits(lo) - bits(min_mass), value = bits(hi)) and the inclusive prefix MAXIMUM of the upper bounds in that
// order.  A mass x lies in the union of the windows iff, for the last sorted window with lo <= x, pmax >= x, so
// the union needs no compaction into disjoint intervals.
#include <math_constants.h>

#include <algorithm>
#include <cstring>
#include <vector>

#include "kernels.cuh"

namespace dbi {
namespace {

constexpr int WK_THREADS = 256;
constexpr int WP_THREADS = 1024;

__device__ __forceinline__ uint64_t dbits_d(double d) { return (uint64_t)__double_as_longlong(d); }

// K12a: clip every window to [min_mass, max_mass] (the index holds no mass outside it); an inverted or clipped-away
// window gets drop_key, which sorts after every kept one, and hi = -inf.  NaN bounds select what K9 selects: a NaN
// lower bound acts as -inf (mass < NaN never holds), a NaN upper bound selects nothing (mass <= NaN never holds).
__global__ void __launch_bounds__(WK_THREADS)
    win_keys_kernel(const double* __restrict__ lo, const double* __restrict__ hi, uint64_t n, double min_mass,
                    double max_mass, uint64_t drop_key, uint64_t* __restrict__ key, uint64_t* __restrict__ val) {
  const uint64_t i = (uint64_t)blockIdx.x * WK_THREADS + threadIdx.x;
  if (i >= n) return;
  const double l = lo[i], h = hi[i];
  const double a = l > min_mass ? l : min_mass;  // NaN and -0.0 become min_mass (>= +0.0: bits sort as unsigned)
  const double b = h < max_mass ? h : max_mass;
  const bool keep = h == h && a <= b;
  key[i] = keep ? dbits_d(a) - dbits_d(min_mass) : drop_key;
  val[i] = keep ? dbits_d(b) : dbits_d(-CUDART_INF);
}

// K12b: one CTA walks the sorted windows in tiles of 1024; warp-shuffle max scan, then a block pass.
__global__ void __launch_bounds__(WP_THREADS)
    win_pmax_kernel(const uint64_t* __restrict__ key, const uint64_t* __restrict__ val, uint64_t n, uint64_t base_bits,
                    uint64_t drop_key, double* __restrict__ w_lo, double* __restrict__ w_pmax) {
  __shared__ double warp_max[WP_THREADS / 32];
  const int w = threadIdx.x >> 5;
  double carry = -CUDART_INF;
  for (uint64_t base = 0; base < n; base += WP_THREADS) {
    const uint64_t i = base + threadIdx.x;
    uint64_t k = drop_key;
    double v = -CUDART_INF;
    if (i < n) {
      k = key[i];
      v = __longlong_as_double((long long)val[i]);
    }
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const double u = __shfl_up_sync(0xffffffffu, v, o);
      if ((int)lane_id() >= o) v = fmax(v, u);
    }
    if (lane_id() == 31) warp_max[w] = v;
    __syncthreads();
    double before = carry;  // max over the earlier tiles and the earlier warps of this tile
    for (int j = 0; j < w; ++j) before = fmax(before, warp_max[j]);
    v = fmax(v, before);
    if (i < n) {
      w_lo[i] = k == drop_key ? CUDART_INF : __longlong_as_double((long long)(k + base_bits));
      w_pmax[i] = v;
    }
    for (int j = 0; j < WP_THREADS / 32; ++j) carry = fmax(carry, warp_max[j]);
    __syncthreads();
  }
}

}  // namespace

uint64_t win_drop_key(double min_mass, double max_mass) {
  uint64_t a, b;
  std::memcpy(&a, &min_mass, 8);
  std::memcpy(&b, &max_mass, 8);
  return b - a + 1;
}

void launch_win_keys(const double* lo, const double* hi, uint64_t n, double min_mass, double max_mass, uint64_t* key,
                     uint64_t* val, cudaStream_t s) {
  if (n == 0) return;
  DBI_LAUNCH(win_keys_kernel, (unsigned)((n + WK_THREADS - 1) / WK_THREADS), WK_THREADS, 0, s, lo, hi, n, min_mass,
             max_mass, win_drop_key(min_mass, max_mass), key, val);
}

void launch_win_pmax(const uint64_t* key, const uint64_t* val, uint64_t n, double min_mass, double max_mass,
                     double* w_lo, double* w_pmax, cudaStream_t s) {
  if (n == 0) return;
  uint64_t base_bits;
  std::memcpy(&base_bits, &min_mass, 8);
  DBI_LAUNCH(win_pmax_kernel, 1, WP_THREADS, 0, s, key, val, n, base_bits, win_drop_key(min_mass, max_mass), w_lo,
             w_pmax);
}

// The shift intervals of InWindows: for k = 0, 1, ..., K the distinct sums of multisets of k class shifts
// (summed in ascending class order), each widened by kShiftEps.  A variant's mass ((m + d1) + d2) + ... and
// m + s differ by a few ulps (< 1e-11 Da at 8000 Da), so the intervals keep every variant; the exact decision
// is K9's on the candidate index.  64 slots: a k whose sums no longer fit (leaving a slot for every later k)
// gets the band [k mod_lo - eps, k mod_hi + eps] instead.
void shift_intervals(const DevTables& t, const DigestCfg& cfg, MassWindows* w) {
  const int K = cfg.max_mods, C = cfg.n_classes;
  w->kmax = K;
  int used = 0;
  std::vector<double> prev{0.0};  // the sum of every multiset of k - 1 classes, and its largest class
  std::vector<int> prev_top{0};
  for (int k = 0; k <= K; ++k) {
    std::vector<double> sums;
    std::vector<int> top;
    if (k == 0) {
      sums = {0.0};
      top = {0};
    } else {  // extend every multiset of k - 1 classes by a class >= its largest
      for (size_t i = 0; i < prev.size(); ++i)
        for (int c = prev_top[i]; c < C; ++c) {
          sums.push_back(prev[i] + t.cls_delta[c]);
          top.push_back(c);
        }
    }
    std::vector<double> distinct = sums;
    std::sort(distinct.begin(), distinct.end());
    distinct.erase(std::unique(distinct.begin(), distinct.end()), distinct.end());
    if (used + (int)distinct.size() + (K - k) <= kMaxShiftIv) {
      for (double s : distinct) {
        w->s_lo[used] = s - kShiftEps;
        w->s_hi[used] = s + kShiftEps;
        ++used;
      }
    } else {
      w->s_lo[used] = k * cfg.mod_lo - kShiftEps;
      w->s_hi[used] = k * cfg.mod_hi + kShiftEps;
      ++used;
    }
    w->k_end[k] = (uint8_t)used;
    prev.swap(sums);
    prev_top.swap(top);
  }
}

}  // namespace dbi
