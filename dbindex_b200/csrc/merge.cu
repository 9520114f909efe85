// merge.cu -- K7m: one-pass multiway merge of the group lists (group path, single GPU).
//
// K6g writes the groups of class sequence v as list v, strictly increasing in (key, payload).  The
// sorted group array is the merge of these S <= 32 lists by (key, payload): every pair is distinct, so
// the order is fully defined, and it is the order a stable key sort of the peptide-major layout gives.
//
//   K7m-a gm_samples : every kGmStride-th record of each list                          (thread/sample)
//   K7m-b gm_rank    : rank of a sample among all samples = its index + a lower bound in every other
//                      list's samples; the samples of rank j * kGmSplit are the splitters  (thread/sample)
//   K7m-c gm_bounds  : a_w(j) = records of list w below splitter j, by a binary search inside one sample
//                      interval (the splitter's own list: exact)                       (warp/splitter, lane/list)
//   K7m-d gm_merge   : tile j = records [a_w(j), a_w(j + 1)) of every list; loads the S segments into shared
//                      memory, merges them with a ceil(log2 S)-level merge-path tree and writes key, payload
//                      and the variant count with coalesced stores                     (CTA/tile)
//
// A tile holds at most (kGmSplit + S) * kGmStride records: between two splitters list w holds s_w samples
// (sum s_w = kGmSplit), so at most (s_w + 1) * kGmStride - 1 records.  HBM bytes: 16 read + 20 written per
// group, plus the samples (32 per kGmStride groups, L2-resident).
#include "kernels.cuh"

namespace dbi {
namespace {

constexpr int GM_THREADS = 256;
constexpr int GM_CAP = (kGmSplit + kGrpMaxLists) * kGmStride;  // records per merge tile, worst case
constexpr size_t GM_SMEM = (size_t)GM_CAP * 32;                 // two (key, payload) buffers
constexpr uint32_t kCntMask = (1u << 27) - 1;                   // variant-count field of the payload

__device__ __forceinline__ bool rec_less(uint64_t ka, uint64_t pa, uint64_t kb, uint64_t pb) {
  return ka < kb || (ka == kb && pa < pb);
}

// first index in [lo, hi) of sorted (key, pay) whose record is not below (xk, xp); the payload is read only
// on a key tie
__device__ __forceinline__ uint64_t lower_bound_rec(const uint64_t* __restrict__ key, const uint64_t* __restrict__ pay,
                                                    uint64_t lo, uint64_t hi, uint64_t xk, uint64_t xp) {
  while (lo < hi) {
    const uint64_t mid = (lo + hi) >> 1;
    const uint64_t k = key[mid];
    if (k < xk || (k == xk && pay[mid] < xp)) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// record a below record b (shared memory; the payloads only on a key tie)
__device__ __forceinline__ bool smem_less(const uint64_t* sk, const uint64_t* sp, uint32_t a, uint32_t b) {
  const uint64_t ka = sk[a], kb = sk[b];
  return ka < kb || (ka == kb && sp[a] < sp[b]);
}

// list of sample s: last v with soff[v] <= s
__device__ __forceinline__ int sample_list(const GroupLists& gl, uint64_t s) {
  int v = 0;
  while (v + 1 < gl.n_lists && gl.soff[v + 1] <= s) ++v;
  return v;
}

// ---- K7m-a ----------------------------------------------------------------------------
__global__ void __launch_bounds__(GM_THREADS)
    gm_samples_kernel(const __grid_constant__ GroupLists gl, const uint64_t* __restrict__ key,
                      const uint64_t* __restrict__ pay, uint64_t* __restrict__ s_key, uint64_t* __restrict__ s_pay) {
  const uint64_t s = (uint64_t)blockIdx.x * GM_THREADS + threadIdx.x;
  if (s >= gl.soff[gl.n_lists]) return;
  const int v = sample_list(gl, s);
  const uint64_t src = gl.start[v] + (s - gl.soff[v]) * kGmStride;
  s_key[s] = key[src];
  s_pay[s] = pay[src];
}

// ---- K7m-b ----------------------------------------------------------------------------
__global__ void __launch_bounds__(GM_THREADS)
    gm_rank_kernel(const __grid_constant__ GroupLists gl, const uint64_t* __restrict__ s_key,
                   const uint64_t* __restrict__ s_pay, uint32_t* __restrict__ spl) {
  const uint64_t s = (uint64_t)blockIdx.x * GM_THREADS + threadIdx.x;
  if (s >= gl.soff[gl.n_lists]) return;
  const int v = sample_list(gl, s);
  const uint64_t xk = s_key[s], xp = s_pay[s];
  uint64_t rank = s - gl.soff[v];
  for (int w = 0; w < gl.n_lists; ++w)
    if (w != v) rank += lower_bound_rec(s_key, s_pay, gl.soff[w], gl.soff[w + 1], xk, xp) - gl.soff[w];
  if (rank % kGmSplit == 0) spl[rank / kGmSplit] = (uint32_t)s;
}

// ---- K7m-c ----------------------------------------------------------------------------
// bnd[j * S + w] = records of list w below splitter j; j = n_spl: the list lengths
__global__ void __launch_bounds__(GM_THREADS)
    gm_bounds_kernel(const __grid_constant__ GroupLists gl, const uint64_t* __restrict__ key,
                     const uint64_t* __restrict__ pay, const uint64_t* __restrict__ s_key,
                     const uint64_t* __restrict__ s_pay, const uint32_t* __restrict__ spl, uint32_t n_spl,
                     uint32_t* __restrict__ bnd) {
  const uint64_t j = ((uint64_t)blockIdx.x * GM_THREADS + threadIdx.x) >> 5;
  const int w = (int)lane_id();
  if (j > n_spl || w >= gl.n_lists) return;
  const uint64_t n_w = gl.start[w + 1] - gl.start[w];
  uint64_t a;
  if (j == n_spl) {
    a = n_w;
  } else {
    const uint64_t s = spl[j];
    const int v = sample_list(gl, s);
    if (w == v) {
      a = (s - gl.soff[v]) * kGmStride;
    } else {
      const uint64_t xk = s_key[s], xp = s_pay[s];
      const uint64_t c = lower_bound_rec(s_key, s_pay, gl.soff[w], gl.soff[w + 1], xk, xp) - gl.soff[w];
      if (c == 0) {
        a = 0;
      } else {  // sample c - 1 lies below the splitter, sample c (if any) above it
        const uint64_t lo = (c - 1) * kGmStride + 1, hi = min(c * kGmStride, n_w);
        a = lower_bound_rec(key + gl.start[w], pay + gl.start[w], lo, hi, xk, xp);
      }
    }
  }
  bnd[j * gl.n_lists + w] = (uint32_t)a;
}

// ---- K7m-d ----------------------------------------------------------------------------
__global__ void __launch_bounds__(GM_THREADS)
    gm_merge_kernel(const __grid_constant__ GroupLists gl, const uint64_t* __restrict__ key,
                    const uint64_t* __restrict__ pay, const uint32_t* __restrict__ bnd, uint64_t* __restrict__ o_key,
                    uint64_t* __restrict__ o_pay, uint32_t* __restrict__ o_cnt, uint32_t* err) {
  extern __shared__ __align__(16) uint64_t gm_smem[];
  __shared__ uint32_t s_lo[kGrpMaxLists];       // first record of each segment, list-local
  __shared__ uint32_t s_off[kGrpMaxLists + 1];  // segment w = tile-local [s_off[w], s_off[w + 1])
  __shared__ uint64_t s_out0;                   // first output position of the tile
  const int S = gl.n_lists;
  const uint32_t t = threadIdx.x;
  const uint32_t* b0 = bnd + (uint64_t)blockIdx.x * S;
  if (t == 0) {
    uint32_t run = 0;
    uint64_t out0 = 0;
    for (int w = 0; w < S; ++w) {
      const uint32_t lo = b0[w];
      s_lo[w] = lo;
      s_off[w] = run;
      run += b0[S + w] - lo;
      out0 += lo;
    }
    s_off[S] = run;
    s_out0 = out0;
  }
  __syncthreads();
  const uint32_t n = s_off[S];
  if (n > (uint32_t)GM_CAP) {
    if (t == 0) atomicOr(err, kErrMergeCap);
    return;
  }
  uint64_t* sk = gm_smem;               // source buffer of the current level
  uint64_t* sp = gm_smem + GM_CAP;
  uint64_t* dk = gm_smem + 2 * GM_CAP;  // destination buffer
  uint64_t* dp = gm_smem + 3 * GM_CAP;
  // load the S segments (consecutive threads = consecutive records of a segment)
  for (uint32_t i = t; i < n; i += GM_THREADS) {
    int lo = 0, hi = S;  // segment of i: last w with s_off[w] <= i
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (s_off[mid] <= i) lo = mid; else hi = mid;
    }
    const uint64_t src = gl.start[lo] + s_lo[lo] + (i - s_off[lo]);
    sk[i] = key[src];
    sp[i] = pay[src];
  }
  __syncthreads();
  // merge-path tree: level `width` merges runs [2k w, 2k w + w) and [2k w + w, 2k w + 2w) of segments.
  // Thread t writes outputs [t per, t per + per); per is odd, so that the 8-byte accesses of a warp at
  // stride per fall into distinct banks.
  const uint32_t per = ((n + GM_THREADS - 1) / GM_THREADS) | 1u;
  for (int width = 1; width < S; width <<= 1) {
    uint32_t p = min(t * per, n);
    const uint32_t p_end = min(p + per, n);
    int k = 0;
    while (p < p_end) {
      while (s_off[min((k + 1) * 2 * width, S)] <= p) ++k;  // the pair whose output holds p
      const uint32_t lo = s_off[k * 2 * width], mid = s_off[min(k * 2 * width + width, S)],
                     hi = s_off[min((k + 1) * 2 * width, S)];
      const uint32_t d = p - lo, nb = hi - mid;
      uint32_t l = d > nb ? d - nb : 0u, r = min(d, mid - lo);
      while (l < r) {  // records of the first run among the first d outputs of the pair
        const uint32_t m = (l + r) >> 1;
        if (smem_less(sk, sp, lo + m, mid + d - 1 - m)) l = m + 1; else r = m;
      }
      uint32_t ia = lo + l, ib = mid + (d - l);
      const uint32_t q_end = min(p_end, hi);
      // the heads of both runs live in registers: one key + payload load per output
      uint64_t ak = 0, ap = 0, bk = 0, bp = 0;
      if (ia < mid) { ak = sk[ia]; ap = sp[ia]; }
      if (ib < hi) { bk = sk[ib]; bp = sp[ib]; }
      for (; p < q_end; ++p) {
        if (ib >= hi || (ia < mid && rec_less(ak, ap, bk, bp))) {
          dk[p] = ak; dp[p] = ap;
          if (++ia < mid) { ak = sk[ia]; ap = sp[ia]; }
        } else {
          dk[p] = bk; dp[p] = bp;
          if (++ib < hi) { bk = sk[ib]; bp = sp[ib]; }
        }
      }
    }
    __syncthreads();
    uint64_t* tk = sk; sk = dk; dk = tk;
    uint64_t* tp = sp; sp = dp; dp = tp;
  }
  const uint64_t o = s_out0;
  for (uint32_t i = t; i < n; i += GM_THREADS) {
    const uint64_t pv = sp[i];
    o_key[o + i] = sk[i];
    o_pay[o + i] = pv;
    o_cnt[o + i] = (uint32_t)pv & kCntMask;
  }
}

uint64_t n_splitters(const GroupLists& gl) { return (gl.soff[gl.n_lists] + kGmSplit - 1) / kGmSplit; }

}  // namespace

void group_lists_plan(GroupLists* gl) {
  gl->soff[0] = 0;
  for (int v = 0; v < gl->n_lists; ++v)
    gl->soff[v + 1] = gl->soff[v] + (gl->start[v + 1] - gl->start[v] + kGmStride - 1) / kGmStride;
}

// samples (key, payload), splitters, bounds
size_t group_merge_tmp_bytes(const GroupLists& gl) {
  const uint64_t ns = gl.soff[gl.n_lists], nt = n_splitters(gl);
  auto al = [](uint64_t x) { return (x + 255) & ~255ull; };
  return al(ns * 8) * 2 + al(nt * 4) + al((nt + 1) * (uint64_t)gl.n_lists * 4);
}

void launch_group_merge(const GroupLists& gl, const uint64_t* key, const uint64_t* pay, uint64_t* o_key,
                        uint64_t* o_pay, uint32_t* o_cnt, void* tmp, uint32_t* d_err, cudaStream_t s) {
  const uint64_t ns = gl.soff[gl.n_lists], nt = n_splitters(gl);
  if (ns == 0) return;
  auto al = [](uint64_t x) { return (x + 255) & ~255ull; };
  uint8_t* p = (uint8_t*)tmp;
  uint64_t* s_key = (uint64_t*)p;
  uint64_t* s_pay = (uint64_t*)(p + al(ns * 8));
  uint32_t* spl = (uint32_t*)(p + 2 * al(ns * 8));
  uint32_t* bnd = (uint32_t*)(p + 2 * al(ns * 8) + al(nt * 4));
  // set on every call: the attribute belongs to the current device, and the call is a host-side table write
  DBI_CUDA(cudaFuncSetAttribute(gm_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GM_SMEM));
  const unsigned sgrid = (unsigned)((ns + GM_THREADS - 1) / GM_THREADS);
  DBI_LAUNCH(gm_samples_kernel, sgrid, GM_THREADS, 0, s, gl, key, pay, s_key, s_pay);
  DBI_LAUNCH(gm_rank_kernel, sgrid, GM_THREADS, 0, s, gl, s_key, s_pay, spl);
  const uint64_t bthreads = (nt + 1) * 32;
  DBI_LAUNCH(gm_bounds_kernel, (unsigned)((bthreads + GM_THREADS - 1) / GM_THREADS), GM_THREADS, 0, s, gl, key, pay,
             s_key, s_pay, spl, (uint32_t)nt, bnd);
  DBI_LAUNCH(gm_merge_kernel, (unsigned)nt, GM_THREADS, GM_SMEM, s, gl, key, pay, bnd, o_key, o_pay, o_cnt, d_err);
}

}  // namespace dbi
