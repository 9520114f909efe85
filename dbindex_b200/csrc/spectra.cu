// spectra.cu -- K13 / K14: the precursor windows of a batch of spectra (dbi_query_spectra,
// dbi_search_unindexed_spectra) as one flat interval array for K9 / K10.
//
// A spectrum is either a list of (mass, tol in Da) ranges, answered as DBIndexer.getSequences(List<MassRange>)
// answers it (Interval.massRangeToInterval + MergeIntervals.mergeIntervals, then the bucket rule of
// DBIndexStoreSQLiteMult, Mult:333-338,383-387), or a (mass, ppm) pair, answered as
// DBIndexer.getSequencesUsingPPMTolerance (DBIndexer.java:787-844): the Dalton window, then exact-mass probes above
// it until one comes back empty.  Every double below is rounded the way the host computes it: the tolerance, bound
// and probe arithmetic is written with explicit _rn intrinsics so that nvcc cannot contract it into an FMA.
#include <math_constants.h>

#include "kernels.cuh"

namespace dbi {
namespace {

constexpr int SP_THREADS = 256;
constexpr int SP_WARPS = SP_THREADS / 32;
constexpr double kPrecision = 1e-6;  // Constants.PRECISION, the step of the probe walk

// DBIndexer._out_of_buckets for one bound: int(x) // (MAX_PRECURSOR_MASS // f) > f - 1 (f = index_factor,
// 1..8000; 0 = off).  int() truncates and // floors, so a bound below 1 lands in bucket <= 0 and never fails.
__device__ __forceinline__ bool out_of_buckets(double x, int f) {
  if (f <= 0 || !(x >= 1.0)) return false;
  if (x >= 9.0e18) return true;  // beyond long long; bucket >= 9e18 / 8000 > f - 1
  return (long long)x / (long long)(8000 / f) > f - 1;
}

// IndexUtil.getToleranceInDalton: m * (1 - 1 / (ppm / 1e6 + 1)), in that order
__device__ __forceinline__ double tol_in_dalton(double m, double ppm) {
  return __dmul_rn(m, __dsub_rn(1.0, __ddiv_rn(1.0, __dadd_rn(__ddiv_rn(ppm, 1e6), 1.0))));
}

struct Iv {
  double lo, hi;
  uint32_t idx;  // input position: the sort is stable
};

__device__ __forceinline__ bool iv_less(double alo, uint32_t aidx, double blo, uint32_t bidx) {
  return alo < blo || (alo == blo && aidx < bidx);
}

// the clamped interval of range r (massRangeToInterval)
__device__ __forceinline__ Iv range_iv(const double* __restrict__ mass, const double* __restrict__ tol, uint64_t r,
                                       uint32_t idx) {
  const double m = mass[r], t = tol[r];
  double lo = __dsub_rn(m, t);
  if (lo < 0.0) lo = 0.0;
  return Iv{lo, __dadd_rn(m, t), idx};
}

// K13a: one warp per Dalton spectrum.  Up to 32 ranges: one per lane, warp bitonic sort by (lo, input index), then
// the serial merge (end >= next.start, end = max) on every lane from shuffles -- a prefix maximum of hi is not the
// same walk once a negative tolerance makes an interval inverted.  More than 32 ranges: lane 0 sorts and merges the
// spectrum's slots in place (insertion sort, stable).  The merged intervals go to the spectrum's slots
// [range_off[s], ...) of o_lo / o_hi; cnt[s] = their number, 0 when one of them fails the bucket rule.
__global__ void __launch_bounds__(SP_THREADS)
    spec_intervals_kernel(const double* __restrict__ mass, const double* __restrict__ tol,
                          const uint64_t* __restrict__ range_off, uint64_t n, int index_factor, double* __restrict__ o_lo,
                          double* __restrict__ o_hi, uint32_t* __restrict__ cnt) {
  const uint64_t s = (uint64_t)blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
  if (s >= n) return;
  const unsigned lane = lane_id();
  const uint64_t r0 = range_off[s];
  const uint64_t k = range_off[s + 1] - r0;
  uint32_t c = 0;
  bool fail = false;
  if (k == 0) {
  } else if (k <= 32) {
    Iv v = lane < k ? range_iv(mass, tol, r0 + lane, lane) : Iv{CUDART_INF, CUDART_INF, 32u + lane};
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        const double olo = __shfl_xor_sync(0xffffffffu, v.lo, stride);
        const double ohi = __shfl_xor_sync(0xffffffffu, v.hi, stride);
        const uint32_t oidx = __shfl_xor_sync(0xffffffffu, v.idx, stride);
        const bool up = (lane & size) == 0, lower = (lane & stride) == 0;
        const bool take = lower == up ? iv_less(olo, oidx, v.lo, v.idx) : iv_less(v.lo, v.idx, olo, oidx);
        if (take) v = Iv{olo, ohi, oidx};
      }
    }
    double start = __shfl_sync(0xffffffffu, v.lo, 0), end = __shfl_sync(0xffffffffu, v.hi, 0);
    for (uint32_t j = 1; j < k; ++j) {
      const double a = __shfl_sync(0xffffffffu, v.lo, j), b = __shfl_sync(0xffffffffu, v.hi, j);
      if (end >= a) {
        if (b > end) end = b;
      } else {
        if (lane == 0) {
          o_lo[r0 + c] = start;
          o_hi[r0 + c] = end;
        }
        fail |= out_of_buckets(start, index_factor) || out_of_buckets(end, index_factor);
        ++c;
        start = a;
        end = b;
      }
    }
    if (lane == 0) {
      o_lo[r0 + c] = start;
      o_hi[r0 + c] = end;
    }
    fail |= out_of_buckets(start, index_factor) || out_of_buckets(end, index_factor);
    ++c;
  } else if (lane == 0) {
    for (uint64_t j = 0; j < k; ++j) {
      const Iv v = range_iv(mass, tol, r0 + j, 0);
      uint64_t i = j;
      for (; i > 0 && v.lo < o_lo[r0 + i - 1]; --i) {
        o_lo[r0 + i] = o_lo[r0 + i - 1];
        o_hi[r0 + i] = o_hi[r0 + i - 1];
      }
      o_lo[r0 + i] = v.lo;
      o_hi[r0 + i] = v.hi;
    }
    double start = o_lo[r0], end = o_hi[r0];
    for (uint64_t j = 1; j < k; ++j) {
      const double a = o_lo[r0 + j], b = o_hi[r0 + j];
      if (end >= a) {
        if (b > end) end = b;
      } else {
        o_lo[r0 + c] = start;  // c < j: the slot was read already
        o_hi[r0 + c] = end;
        fail |= out_of_buckets(start, index_factor) || out_of_buckets(end, index_factor);
        ++c;
        start = a;
        end = b;
      }
    }
    o_lo[r0 + c] = start;
    o_hi[r0 + c] = end;
    fail |= out_of_buckets(start, index_factor) || out_of_buckets(end, index_factor);
    ++c;
  }
  if (lane == 0) cnt[s] = fail ? 0u : c;
}

// the kept intervals of every spectrum, packed at ioff[s] (one warp per spectrum)
__global__ void __launch_bounds__(SP_THREADS)
    spec_compact_kernel(const uint64_t* __restrict__ range_off, const uint64_t* __restrict__ ioff, uint64_t n,
                        const double* __restrict__ s_lo, const double* __restrict__ s_hi, double* __restrict__ o_lo,
                        double* __restrict__ o_hi) {
  const uint64_t s = (uint64_t)blockIdx.x * SP_WARPS + (threadIdx.x >> 5);
  if (s >= n) return;
  const uint64_t r0 = range_off[s], o = ioff[s], c = ioff[s + 1] - o;
  for (uint64_t i = lane_id(); i < c; i += 32) {
    o_lo[o + i] = s_lo[r0 + i];
    o_hi[o + i] = s_hi[r0 + i];
  }
}

// K13b: one thread per PPM spectrum: the Dalton window [max(0, m - tol), m + tol].  With c_lo: the candidate window
// of an unindexed search, which holds the window and every probe the walk's guard (u - tol(u) < m) admits.  The
// guard computes u / (1 + p) with a relative error of a few ulps, so u <= m (1 + p) (1 + 2^-40) for every admitted
// u; without that form (m <= 0 or 1 + p <= 0) the guard is not bounded and the window reaches up to +inf.
__global__ void __launch_bounds__(SP_THREADS)
    spec_ppm_window_kernel(const double* __restrict__ mass, const double* __restrict__ ppm, uint64_t n,
                           double* __restrict__ w_lo, double* __restrict__ w_hi, double* __restrict__ c_lo,
                           double* __restrict__ c_hi) {
  const uint64_t s = (uint64_t)blockIdx.x * SP_THREADS + threadIdx.x;
  if (s >= n) return;
  const double m = mass[s], p = ppm[s];
  const double t = tol_in_dalton(m, p);
  double lo = __dsub_rn(m, t);
  if (lo < 0.0) lo = 0.0;
  const double hi = __dadd_rn(m, t);
  w_lo[s] = lo;
  w_hi[s] = hi;
  if (!c_lo) return;
  const double p1 = __dadd_rn(__ddiv_rn(p, 1e6), 1.0);
  double ext = m > 0.0 && p1 > 0.0 ? __dmul_rn(__dmul_rn(m, p1), 1.0 + 0x1p-40) : CUDART_INF;
  c_lo[s] = fmin(lo, hi);
  c_hi[s] = fmax(ext, hi);
}

// first index with mass >= v
__device__ __forceinline__ uint64_t lower_bound_d(const double* __restrict__ a, uint64_t n, double v) {
  uint64_t lo = 0, len = n;
  while (len > 0) {
    const uint64_t half = len >> 1;
    if (__ldg(a + lo + half) < v) {
      lo += half + 1;
      len -= half + 1;
    } else {
      len = half;
    }
  }
  return lo;
}

// K14: one thread per PPM spectrum walks the probes u_0 = m + tol, u_{k+1} = u_k + 1e-6 over the entry masses while
// u_k - tol(u_k) < m and u_{k+1} != u_k; the probe [u_k, u_k] is empty (and ends the walk) when u_k < 0, when it
// fails the bucket rule or when no entry has mass u_k.  The spectrum's intervals: its window unless that fails the
// bucket rule, then every continuing probe with k >= 1, and u_0 too when the window does not already hold it
// (inverted or dropped; the reference appends only hits it has not seen).  Count pass (o_lo == nullptr): cnt[s];
// emit pass: the intervals at ioff[s].  kGivenStops (a sharded index, whose probes are spread over the ranks): the
// walk ends at probe stop[s] (K14s, reduced over the ranks) in place of the search for an entry of mass u_k.
template <bool kGivenStops>
__global__ void __launch_bounds__(SP_THREADS)
    spec_probe_kernel(const double* __restrict__ e_mass, uint64_t n_entries, const double* __restrict__ mass,
                      const double* __restrict__ ppm, const double* __restrict__ w_lo, const double* __restrict__ w_hi,
                      uint64_t n, int index_factor, uint32_t* __restrict__ cnt, const uint64_t* __restrict__ ioff,
                      double* __restrict__ o_lo, double* __restrict__ o_hi, const uint64_t* __restrict__ stop) {
  const uint64_t s = (uint64_t)blockIdx.x * SP_THREADS + threadIdx.x;
  if (s >= n) return;
  const double m = mass[s], p = ppm[s], lo = w_lo[s], hi = w_hi[s];
  const uint64_t k_end = kGivenStops ? stop[s] : 0;
  const bool window = !out_of_buckets(lo, index_factor) && !out_of_buckets(hi, index_factor);
  const uint64_t o = o_lo ? ioff[s] : 0;
  uint32_t c = 0;
  if (window) {
    if (o_lo) {
      o_lo[o] = lo;
      o_hi[o] = hi;
    }
    ++c;
  }
  const bool probe0 = !(window && lo <= hi);
  double u = hi;
  for (uint64_t k = 0;; ++k) {
    if (!(__dsub_rn(u, tol_in_dalton(u, p)) < m)) break;
    if (u < 0.0 || out_of_buckets(u, index_factor)) break;
    if constexpr (kGivenStops) {
      if (k >= k_end) break;
    } else {
      const uint64_t b = lower_bound_d(e_mass, n_entries, u);
      if (b >= n_entries || e_mass[b] != u) break;
    }
    if (k > 0 || probe0) {
      if (o_lo) {
        o_lo[o + c] = u;
        o_hi[o + c] = u;
      }
      ++c;
    }
    const double nu = __dadd_rn(u, kPrecision);
    if (nu == u) break;
    u = nu;
  }
  if (!o_lo) cnt[s] = c;
}

// K14s: one thread per PPM spectrum: K_r, where this rank's share of the probe walk of K14 ends when the entries
// are spread over the ranks by mass (slice of u = number of cuts <= u, owner(slice) holds every entry of mass u).
// It ends on the walk's own end conditions, which every rank evaluates alike, and at a probe it owns whose mass
// none of its entries has; a probe it does not own it steps over without a search.  The walk's end is the minimum
// of K_r over the ranks.  Once no slice of this rank meets [u_k, bound] (bound = m (1 + p) (1 + 2^-40) >= every
// probe the guard admits, as K13b computes it) the rank cannot end the walk: stop[s] = UINT64_MAX.
__global__ void __launch_bounds__(SP_THREADS)
    spec_stop_kernel(const double* __restrict__ e_mass, uint64_t n_entries, const double* __restrict__ mass,
                     const double* __restrict__ ppm, const double* __restrict__ w_hi, uint64_t n, int index_factor,
                     const SliceCuts cuts, uint64_t* __restrict__ stop) {
  const uint64_t s = (uint64_t)blockIdx.x * SP_THREADS + threadIdx.x;
  if (s >= n) return;
  const double m = mass[s], p = ppm[s];
  const double p1 = __dadd_rn(__ddiv_rn(p, 1e6), 1.0);
  const double bound = m > 0.0 && p1 > 0.0 ? __dmul_rn(__dmul_rn(m, p1), 1.0 + 0x1p-40) : CUDART_INF;
  double u = w_hi[s];
  uint64_t k = 0;
  for (;; ++k) {
    if (!(__dsub_rn(u, tol_in_dalton(u, p)) < m)) break;
    if (u < 0.0 || out_of_buckets(u, index_factor)) break;
    uint32_t sl = 0;
    for (int x = 0; x + 1 < cuts.n_slices; ++x) sl += cuts.cut[x] <= u ? 1u : 0u;
    if ((cuts.mine >> sl) & 1u) {
      const uint64_t b = lower_bound_d(e_mass, n_entries, u);
      if (b >= n_entries || e_mass[b] != u) break;
    } else {
      // the next slice of this rank above u is slice sl + ffs(above); it starts at cut[sl + ffs(above) - 1]
      const uint32_t above = sl + 1 < 32 ? cuts.mine >> (sl + 1) : 0u;
      if (!above || cuts.cut[sl + __ffs(above) - 1] > bound) {
        k = UINT64_MAX;
        break;
      }
    }
    const double nu = __dadd_rn(u, kPrecision);
    if (nu == u) {
      ++k;
      break;
    }
    u = nu;
  }
  stop[s] = k;
}

// per-interval hit / run offsets (n_iv + 1) -> per-spectrum ones (n + 1): the value at the spectrum's first interval
__global__ void __launch_bounds__(SP_THREADS)
    spec_collapse_kernel(const uint64_t* __restrict__ ioff, uint64_t n, const uint64_t* __restrict__ iv_hit_off,
                         const uint64_t* __restrict__ iv_pep_off, uint64_t* __restrict__ hit_off,
                         uint64_t* __restrict__ pep_off) {
  const uint64_t s = (uint64_t)blockIdx.x * SP_THREADS + threadIdx.x;
  if (s > n) return;
  const uint64_t i = ioff[s];
  hit_off[s] = iv_hit_off[i];
  pep_off[s] = iv_pep_off[i];
}

unsigned grid_threads(uint64_t n) { return (unsigned)((n + SP_THREADS - 1) / SP_THREADS); }
unsigned grid_warps(uint64_t n) { return (unsigned)((n + SP_WARPS - 1) / SP_WARPS); }

}  // namespace

void launch_spec_intervals(const double* mass, const double* tol, const uint64_t* range_off, uint64_t n,
                           int index_factor, double* o_lo, double* o_hi, uint32_t* cnt, cudaStream_t s) {
  if (n == 0) return;
  DBI_LAUNCH(spec_intervals_kernel, grid_warps(n), SP_THREADS, 0, s, mass, tol, range_off, n, index_factor, o_lo,
             o_hi, cnt);
}

void launch_spec_compact(const uint64_t* range_off, const uint64_t* ioff, uint64_t n, const double* s_lo,
                         const double* s_hi, double* o_lo, double* o_hi, cudaStream_t s) {
  if (n == 0) return;
  DBI_LAUNCH(spec_compact_kernel, grid_warps(n), SP_THREADS, 0, s, range_off, ioff, n, s_lo, s_hi, o_lo, o_hi);
}

void launch_spec_ppm_window(const double* mass, const double* ppm, uint64_t n, double* w_lo, double* w_hi,
                            double* c_lo, double* c_hi, cudaStream_t s) {
  if (n == 0) return;
  DBI_LAUNCH(spec_ppm_window_kernel, grid_threads(n), SP_THREADS, 0, s, mass, ppm, n, w_lo, w_hi, c_lo, c_hi);
}

void launch_spec_probe_count(const double* e_mass, uint64_t n_entries, const double* mass, const double* ppm,
                             const double* w_lo, const double* w_hi, uint64_t n, int index_factor, const uint64_t* stop,
                             uint32_t* cnt, cudaStream_t s) {
  if (n == 0) return;
  if (stop)
    DBI_LAUNCH(spec_probe_kernel<true>, grid_threads(n), SP_THREADS, 0, s, e_mass, n_entries, mass, ppm, w_lo, w_hi,
               n, index_factor, cnt, (const uint64_t*)nullptr, (double*)nullptr, (double*)nullptr, stop);
  else
    DBI_LAUNCH(spec_probe_kernel<false>, grid_threads(n), SP_THREADS, 0, s, e_mass, n_entries, mass, ppm, w_lo, w_hi,
               n, index_factor, cnt, (const uint64_t*)nullptr, (double*)nullptr, (double*)nullptr,
               (const uint64_t*)nullptr);
}

void launch_spec_probe_emit(const double* e_mass, uint64_t n_entries, const double* mass, const double* ppm,
                            const double* w_lo, const double* w_hi, uint64_t n, int index_factor, const uint64_t* stop,
                            const uint64_t* ioff, double* o_lo, double* o_hi, cudaStream_t s) {
  if (n == 0) return;
  if (stop)
    DBI_LAUNCH(spec_probe_kernel<true>, grid_threads(n), SP_THREADS, 0, s, e_mass, n_entries, mass, ppm, w_lo, w_hi,
               n, index_factor, (uint32_t*)nullptr, ioff, o_lo, o_hi, stop);
  else
    DBI_LAUNCH(spec_probe_kernel<false>, grid_threads(n), SP_THREADS, 0, s, e_mass, n_entries, mass, ppm, w_lo, w_hi,
               n, index_factor, (uint32_t*)nullptr, ioff, o_lo, o_hi, (const uint64_t*)nullptr);
}

void launch_spec_stops(const double* e_mass, uint64_t n_entries, const double* mass, const double* ppm,
                       const double* w_hi, uint64_t n, int index_factor, const SliceCuts& cuts, uint64_t* stop,
                       cudaStream_t s) {
  if (n == 0) return;
  DBI_LAUNCH(spec_stop_kernel, grid_threads(n), SP_THREADS, 0, s, e_mass, n_entries, mass, ppm, w_hi, n, index_factor,
             cuts, stop);
}

void launch_spec_collapse(const uint64_t* ioff, uint64_t n, const uint64_t* iv_hit_off, const uint64_t* iv_pep_off,
                          uint64_t* hit_off, uint64_t* pep_off, cudaStream_t s) {
  DBI_LAUNCH(spec_collapse_kernel, grid_threads(n + 1), SP_THREADS, 0, s, ioff, n, iv_hit_off, iv_pep_off, hit_off,
             pep_off);
}

}  // namespace dbi
