// digest.cu -- K1 pack, K2 digest-count, K3 scan, K4 digest-emit.
//
// Restates DBIndexer.cutSeq (DBIndexer.java:237-405) as a two-pass count / scan /
// emit over a device-resident residue buffer.  Work unit = one START residue:
// a lane walks `end` sequentially and adds residue masses in IEEE double in the
// reference's order (DBIndexer.java:265-271,308), so masses are bit-identical to
// the Java loop (SURVEY.md Q1).  Output order is the reference's addSequence()
// call order (protein, start, end ascending) because the scan runs over starts in
// buffer order and a lane emits its ends in walking order.
//
// Layout: res[] = 0, protein0, 0, protein1, 0, ... ; a 0 byte is "outside the
// protein" on both sides, so `start == 0` and `end == length-1` of the reference
// become "previous / next byte is 0".
//
// sm_100a specifics: a CTA stages its tile of residues (2048 starts + a 272-byte halo, and in K4
// the per-start counts of K2) with 1-D bulk asynchronous copies (cp.async.bulk ->
// UBLKCP, completion on an mbarrier), turns the bytes ONCE into per-position (mass, predicate
// bits) in shared memory, and every walk step is then two shared-memory loads and one DADD -- no
// global load, no table lookup on the critical path.  Walks that run past the halo (only possible
// through zero-mass residue codes) continue from global memory with identical arithmetic.
// K2 keeps the count of every start, so K4 walks only the emitting starts, once (r01: three walks).
//
// HBM bytes: K2 reads 1.13 B / residue and writes 1 B / residue; K4 reads 2.13 B / residue and
// writes 18 B / record.
#include "kernels.cuh"

namespace dbi {
namespace {

constexpr int DG_THREADS = 256;
constexpr int DG_SPT = kDigestTile / DG_THREADS;  // starts per thread
constexpr int DG_HALO = 272;                      // staged bytes past the tile (incl. the byte before it)
constexpr int DG_WIN = kDigestTile + DG_HALO;     // staged window: positions [w0, w0 + DG_WIN), w0 = tile * 2048
static_assert(DG_WIN % 16 == 0 && DG_SPT == 8, "bulk copies move 16-byte units; a thread owns 8 starts");

// per-position predicate bits
constexpr uint8_t I_SEP = 1;    // separator (outside any protein)
constexpr uint8_t I_ENZ = 2;    // Enzyme.isEnzyme(c): counts as an internal cleavage site (DBIndexer.java:314-316)
constexpr uint8_t I_COK = 4;    // C side of checkCleavage holds when the window ENDS here
constexpr uint8_t I_NOK = 8;    // N side of checkCleavage holds when the window STARTS here
constexpr uint8_t I_MAND = 16;  // one of mandatoryInternalAAs
constexpr uint8_t I_FILT = 32;  // the residue PeptideFilterByMaxOccurrencies counts
constexpr uint8_t I_MOD = 64;   // a differential-mod site (sharded build: the cost estimate of a record)

// ---- mbarrier + bulk copy (PTX; SASS: SYNCS.*, UBLKCP) --------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}

// raw class bits of one residue byte
__device__ __forceinline__ uint8_t raw_bits(uint8_t c, const DevTables* __restrict__ tb) {
  if (c == 0) return I_SEP;
  const uint8_t f = __ldg(&tb->flags[c]);
  return (uint8_t)(((f & kFlagEnzyme) ? I_ENZ : 0) | ((f & kFlagNocut) ? 0x80 : 0) | ((f & kFlagMandatory) ? I_MAND : 0) |
                   ((f & kFlagFilterAA) ? I_FILT : 0) | ((f & kFlagDiffMod) ? I_MOD : 0));
}
// Enzyme.checkCleavage, one side each (contract of SURVEY.md 8c): the window may start at a
// residue if it is the protein's first or follows an enzyme residue and is not a no-cut residue;
// it may end at a residue if it is the protein's last or an enzyme residue not followed by a
// no-cut residue.  (0x80 = raw no-cut bit, dropped from the stored byte.)
__device__ __forceinline__ uint8_t compose_bits(uint8_t prev, uint8_t cur, uint8_t next) {
  if (cur & I_SEP) return I_SEP;
  uint8_t o = cur & (I_ENZ | I_MAND | I_FILT | I_MOD);
  if ((prev & I_SEP) || ((prev & I_ENZ) && !(cur & 0x80))) o |= I_NOK;
  if ((next & I_SEP) || ((cur & I_ENZ) && !(next & 0x80))) o |= I_COK;
  return o;
}

struct TileSmem {
  alignas(16) uint8_t raw[DG_WIN];        // residues (bulk copy), then raw class bits in place
  alignas(16) uint8_t cnt8[kDigestTile];  // records per start, saturating (K2 out, K4 in)
  alignas(8) double mass[DG_WIN];         // AssignMass.getMass(residue at this position)
  uint8_t info[DG_WIN];                   // composed predicate bits
  uint16_t list[kDigestTile];             // compacted starts (tile-local, buffer order)
  alignas(8) uint64_t bar;
  uint32_t scratch[DG_THREADS / 32 + 1];
};

struct TileCtx {
  const uint8_t* __restrict__ res;
  const DevTables* __restrict__ tb;
  const TileSmem* s;
  uint32_t w0;  // buffer position of window byte 0
};

// (mass, predicate bits) of buffer position pos: staged window first, global memory beyond it
__device__ __forceinline__ void at_pos(const TileCtx& cx, uint32_t pos, uint8_t* inf, double* m) {
  const uint32_t li = pos - cx.w0;
  if (li < (uint32_t)(DG_WIN - 1)) {
    *inf = cx.s->info[li];
    *m = cx.s->mass[li];
    return;
  }
  const uint8_t c = ld_res(cx.res, pos);
  if (c == 0) {
    *inf = I_SEP;
    *m = 0;
    return;
  }
  *inf = compose_bits(raw_bits(ld_res(cx.res, pos - 1), cx.tb), raw_bits(c, cx.tb), raw_bits(ld_res(cx.res, pos + 1), cx.tb));
  *m = __ldg(&cx.tb->mass[c]);
}

// The body of the reference's `for start` iteration (DBIndexer.java:256-395) for the
// start at buffer position g.  F is called as emit(mass, len, n_mod) for every record that keep(mass, n_mod)
// accepts; a rejected record is neither emitted nor counted, and the walk goes on.
// FILTERS = false compiles the two peptide filters (SURVEY 8 f4) out of the loop.
template <bool FILTERS, typename Keep, typename F>
__device__ __forceinline__ uint32_t walk_start(const TileCtx& cx, uint32_t g, const DigestCfg& cfg, uint32_t* err,
                                               const Keep& keep, F&& emit) {
  uint8_t inf;
  double m;
  at_pos(cx, g, &inf, &m);
  if (inf & I_SEP) return 0;  // separator, not a residue
  const bool n_ok = inf & I_NOK;
  // full specificity: cleavageStatus can never become true for this start, so the
  // reference walks it without ever reaching addSequence -- nothing to emit
  if (!cfg.semi && !n_ok) return 0;
  const bool cok_any = cfg.semi && n_ok;  // semi: the N side alone satisfies checkCleavage

  double mass = cfg.init_mass;  // DBIndexer.java:265-271
  int mc = -1;                  // intMisCleavageCount, :280
  int n_mand = 0;               // mandatory residues strictly before the current one
  int n_filt = 0;
  uint32_t n_mod = 0;           // differential-mod sites of the window so far
  uint32_t len = 0, count = 0;
  uint32_t pos = g;
  while (mass <= cfg.max_mass && !(inf & I_SEP)) {  // :284  (end < length  <=>  not a separator)
    ++len;                                          // pepSize++, :285
    mass = __dadd_rn(mass, m);                      // precMass = precMass + aaMass, :308
    n_mod += (inf >> 6) & 1;                        // I_MOD = 64
    if (FILTERS && (inf & I_FILT) && ++n_filt > cfg.filt_max && cfg.filt_max >= 0) break;  // peptideFilter.isValid, :310-313
    mc += (inf >> 1) & 1;                           // isEnzyme(cur) -> intMisCleavageCount++, :314-316 (I_ENZ = 2)
    if (cok_any || (inf & I_COK)) {                 // cleavageStatus, :318-320
      if (mc > cfg.max_mc) break;                   // :322-324
      if (mass > cfg.max_mass) break;               // :327-329
      if ((int)len >= cfg.min_len && mass >= cfg.min_mass) {  // :331
        bool include = true;
        if (FILTERS && cfg.mand_on) {
          if (n_mand == 0 && !(inf & I_MAND)) break;  // none in the whole window: :334-344
          include = n_mand > 0;                       // only as the last residue: SKIP (Mult:245-263)
        }
        if (include) {
          if (len > DBI_MAX_PEP_LEN) {
            atomicOr(err, kErrPepTooLong);
            break;
          }
          if (keep(mass, n_mod)) {
            emit(mass, len, n_mod);
            ++count;
          }
        }
      }
    }
    if (FILTERS && (inf & I_MAND)) ++n_mand;
    ++pos;  // ++end, :394
    at_pos(cx, pos, &inf, &m);
  }
  return count;
}

// Stage the tile: bulk-copy the residue window (and, in K4, the per-start counts), then derive
// per-position mass and predicate bits.  Ends with a __syncthreads().
__device__ __forceinline__ void stage_tile(TileSmem& s, const uint8_t* __restrict__ res, uint64_t res_alloc,
                                           const DevTables* __restrict__ tb, uint32_t w0,
                                           const uint8_t* __restrict__ start_cnt_tile) {
  const int t = threadIdx.x;
  const uint64_t avail = res_alloc - w0;  // w0 < res_end <= res_alloc
  const uint32_t bytes = avail < (uint64_t)DG_WIN ? (uint32_t)avail : (uint32_t)DG_WIN;  // multiples of 16
  if (t == 0) {
    mbar_init(&s.bar, 1);
    mbar_expect_tx(&s.bar, bytes + (start_cnt_tile ? (uint32_t)kDigestTile : 0u));
    bulk_g2s(s.raw, res + w0, bytes, &s.bar);
    if (start_cnt_tile) bulk_g2s(s.cnt8, start_cnt_tile, kDigestTile, &s.bar);
  }
  for (uint32_t i = bytes + t; i < (uint32_t)DG_WIN; i += DG_THREADS) s.raw[i] = 0;  // past the buffer: separators
  __syncthreads();  // the barrier is initialised before anybody polls it
  mbar_wait(&s.bar, 0);
  for (int i = t; i < DG_WIN; i += DG_THREADS) {
    const uint8_t c = s.raw[i];
    s.mass[i] = c ? __ldg(&tb->mass[c]) : 0.0;
    s.raw[i] = raw_bits(c, tb);
  }
  __syncthreads();
  for (int i = t; i < DG_WIN; i += DG_THREADS)
    s.info[i] = (i == 0 || i == DG_WIN - 1) ? (uint8_t)(s.raw[i] & I_SEP) : compose_bits(s.raw[i - 1], s.raw[i], s.raw[i + 1]);
  __syncthreads();
}

// every record of the walk (the index build)
struct AllRecords {
  __device__ __forceinline__ bool operator()(double, uint32_t) const { return true; }
};

// ---- K2 -----------------------------------------------------------------------------
// Warp-cooperative cleavage-site scan: the CTA compacts the live starts of its tile (for trypsin
// ~11 % of the residues can start a peptide), one lane walks each, and the per-start counts go
// back to HBM for K4.  Keep = AllRecords: the index build; InWindows: K2u of an unindexed search.
template <bool FILTERS, typename Keep>
__global__ void __launch_bounds__(DG_THREADS)
    digest_count_kernel(const uint8_t* __restrict__ res, DigestRange rg, uint64_t res_alloc,
                        const DevTables* __restrict__ tb, DigestCfg cfg, uint32_t tile0,
                        uint8_t* __restrict__ start_cnt, uint32_t* __restrict__ tile_counts, uint32_t* err,
                        const Keep keep) {
  __shared__ TileSmem s;
  const int t = threadIdx.x;
  const uint32_t w0 = (tile0 + blockIdx.x) * (uint32_t)kDigestTile;  // start l of the tile sits at w0 + 1 + l
  stage_tile(s, res, res_alloc, tb, w0, nullptr);
  // thread t owns the DG_SPT consecutive starts t*DG_SPT .. : order is preserved by a block scan
  uint32_t live = 0, n_live = 0;
#pragma unroll
  for (int k = 0; k < DG_SPT; ++k) {
    const uint32_t l = t * DG_SPT + k;
    const uint8_t inf = s.info[l + 1];
    const uint32_t g = w0 + 1 + l;
    if (g >= rg.start_lo && g < rg.start_hi && !(inf & I_SEP) && (cfg.semi || (inf & I_NOK))) {
      live |= 1u << k;
      ++n_live;
    }
  }
  reinterpret_cast<uint2*>(s.cnt8)[t] = make_uint2(0u, 0u);
  uint32_t total;
  uint32_t o = block_exclusive_sum<uint32_t, DG_THREADS>(n_live, s.scratch, &total);
#pragma unroll
  for (int k = 0; k < DG_SPT; ++k)
    if (live & (1u << k)) s.list[o++] = (uint16_t)(t * DG_SPT + k);
  __syncthreads();
  const TileCtx cx{res, tb, &s, w0};
  uint32_t cnt = 0;
  for (uint32_t i = t; i < total; i += DG_THREADS) {
    const uint32_t l = s.list[i];
    const uint32_t c = walk_start<FILTERS>(cx, w0 + 1 + l, cfg, err, keep, [](double, uint32_t, uint32_t) {});
    s.cnt8[l] = (uint8_t)(c < 255u ? c : 255u);
    cnt += c;
  }
  uint32_t tile_total;
  block_exclusive_sum<uint32_t, DG_THREADS>(cnt, s.scratch, &tile_total);  // syncs: cnt8 is complete
  if (t == 0) tile_counts[blockIdx.x] = tile_total;
  reinterpret_cast<uint2*>(start_cnt + (size_t)blockIdx.x * kDigestTile)[t] = reinterpret_cast<const uint2*>(s.cnt8)[t];
}

// ---- K4 -----------------------------------------------------------------------------
// (K4u: the same with the Keep of K2u, so that counts and recounts agree)
template <bool FILTERS, typename Keep>
__global__ void __launch_bounds__(DG_THREADS)
    digest_emit_kernel(const uint8_t* __restrict__ res, DigestRange rg, uint64_t res_alloc,
                       const DevTables* __restrict__ tb, DigestCfg cfg, uint32_t tile0,
                       const uint8_t* __restrict__ start_cnt, const uint64_t* __restrict__ tile_offs,
                       const uint32_t* __restrict__ pstart, uint64_t* __restrict__ o_mass,
                       uint32_t* __restrict__ o_gpos, uint32_t* __restrict__ o_prot, uint16_t* __restrict__ o_len,
                       uint8_t* __restrict__ o_nmod, uint32_t* err, const Keep keep) {
  __shared__ TileSmem s;
  __shared__ uint32_t s_off[kDigestTile];   // first record of each emitting start (tile-local)
  __shared__ uint16_t s_zero[kDigestTile];  // separators between the tile's first start and this one
  __shared__ uint32_t s_zbase;
  const int t = threadIdx.x;
  const uint64_t tile_off = tile_offs[blockIdx.x];
  if (tile_offs[blockIdx.x + 1] == tile_off) return;  // nothing to emit here (CTA-uniform)
  const uint32_t w0 = (tile0 + blockIdx.x) * (uint32_t)kDigestTile;
  stage_tile(s, res, res_alloc, tb, w0, start_cnt + (size_t)blockIdx.x * kDigestTile);
  if (t == 0) {
    // separators at positions <= w0.  Those below the range (rg.start_lo: the other shards of a sharded
    // build, whose bytes may not have arrived yet) are known by count: rg.prot_lo, one per earlier protein.
    // Inside the range: proteins p of [prot_lo, prot_hi] with pstart[p] - 1 <= w0 (pstart[prot_hi] names
    // the separator that ends the range): upper_bound(pstart, w0 + 1)
    uint32_t lo = rg.prot_lo, hi = rg.prot_hi + 1;
    if (w0 < rg.start_lo) hi = lo;
    while (lo < hi) {
      const uint32_t mid = (lo + hi) >> 1;
      if (__ldg(pstart + mid) <= w0 + 1) lo = mid + 1; else hi = mid;
    }
    s_zbase = lo;
  }
  const TileCtx cx{res, tb, &s, w0};
  // thread t owns starts t*8 .. t*8+7: their counts (K2), recounted when saturated
  uint32_t c[DG_SPT];
  uint32_t n_emit = 0, sum = 0, zeros = 0;
  uint32_t sepmask = 0;
  {
    const uint2 packed = reinterpret_cast<const uint2*>(s.cnt8)[t];
#pragma unroll
    for (int k = 0; k < DG_SPT; ++k) {
      c[k] = ((k < 4 ? packed.x : packed.y) >> (8 * (k & 3))) & 0xffu;
      if (c[k] == 255u)
        c[k] = walk_start<FILTERS>(cx, w0 + 1 + t * DG_SPT + k, cfg, err, keep, [](double, uint32_t, uint32_t) {});
      n_emit += c[k] ? 1u : 0u;
      sum += c[k];
      if ((s.info[1 + t * DG_SPT + k] & I_SEP) && w0 + 1 + t * DG_SPT + k >= rg.start_lo) {
        sepmask |= 1u << k;
        ++zeros;
      }
    }
  }
  uint32_t tot_emit, tot_sum, tot_zero;
  uint32_t slot = block_exclusive_sum<uint32_t, DG_THREADS>(n_emit, s.scratch, &tot_emit);
  uint32_t off = block_exclusive_sum<uint32_t, DG_THREADS>(sum, s.scratch, &tot_sum);
  const uint32_t zex = block_exclusive_sum<uint32_t, DG_THREADS>(zeros, s.scratch, &tot_zero);
#pragma unroll
  for (int k = 0; k < DG_SPT; ++k)
    if (c[k]) {
      s.list[slot] = (uint16_t)(t * DG_SPT + k);
      s_off[slot] = off;
      s_zero[slot] = (uint16_t)(zex + __popc(sepmask & ((1u << k) - 1u)));
      ++slot;
      off += c[k];
    }
  __syncthreads();
  const uint32_t zbase = s_zbase;
  for (uint32_t i = t; i < tot_emit; i += DG_THREADS) {
    const uint32_t g = w0 + 1 + s.list[i];
    // protein of this start = separators at positions <= g, minus one
    const uint32_t prot = zbase + s_zero[i] - 1u;
    uint64_t o = tile_off + s_off[i];
    walk_start<FILTERS>(cx, g, cfg, err, keep, [&](double m, uint32_t len, uint32_t n_mod) {
      o_mass[o] = (uint64_t)__double_as_longlong(m);
      o_gpos[o] = g;
      o_prot[o] = prot;
      o_len[o] = (uint16_t)len;
      if (o_nmod) o_nmod[o] = (uint8_t)(n_mod < 255u ? n_mod : 255u);
      ++o;
    });
  }
}

// ---- K1 -----------------------------------------------------------------------------
constexpr int PK_THREADS = 256;
constexpr int PK_BYTES = 16;  // raw bytes per thread

__global__ void __launch_bounds__(PK_THREADS)
    pack_kernel(const uint8_t* __restrict__ raw, const uint64_t* __restrict__ off, uint32_t n_prot, uint64_t n_res,
                uint8_t* __restrict__ res, uint32_t* __restrict__ pstart, uint32_t pos_base, uint32_t* err) {
  const uint64_t tid = (uint64_t)blockIdx.x * PK_THREADS + threadIdx.x;
  // protein starts and separators
  if (tid <= n_prot) {
    const uint64_t ps = off[tid] + tid + 1;  // pstart[n_prot] = one past the last separator
    pstart[tid] = (uint32_t)ps + pos_base;
    res[ps - 1] = 0;  // separator before protein tid (tid == n_prot: the final one)
  }
  const uint64_t b0 = tid * PK_BYTES;
  if (b0 >= n_res) return;
  // protein containing raw byte b0: last p with off[p] <= b0 (empty proteins share an offset)
  uint32_t lo = 0, hi = n_prot;
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (off[mid] <= b0) lo = mid; else hi = mid;
  }
  uint32_t p = lo;
  uint64_t next = off[p + 1];
  const uint64_t b1 = min(b0 + PK_BYTES, n_res);
  for (uint64_t b = b0; b < b1; ++b) {
    while (b >= next) { ++p; next = off[p + 1]; }
    const uint8_t c = raw[b];
    if (c == 0) atomicOr(err, kErrZeroResidue);
    res[b + p + 1] = c;
  }
}

// ---- K3 -----------------------------------------------------------------------------
constexpr int SC_THREADS = 1024;

__global__ void __launch_bounds__(SC_THREADS)
    scan_u32_to_u64_kernel(const uint32_t* __restrict__ in, uint64_t n, uint64_t* __restrict__ offs) {
  __shared__ unsigned long long scratch[SC_THREADS / 32 + 1];
  unsigned long long carry = 0;
  for (uint64_t base = 0; base < n; base += SC_THREADS) {
    const uint64_t i = base + threadIdx.x;
    const unsigned long long v = (i < n) ? in[i] : 0ull;
    unsigned long long total;
    const unsigned long long ex = block_exclusive_sum<unsigned long long, SC_THREADS>(v, scratch, &total);
    if (i < n) offs[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) offs[n] = carry;
}

}  // namespace

void launch_pack(const uint8_t* d_raw, const uint64_t* d_off, uint32_t n_prot, uint64_t n_res, uint8_t* d_res,
                 uint32_t* d_pstart, uint32_t pos_base, uint32_t* d_err, cudaStream_t s) {
  uint64_t threads = (n_res + PK_BYTES - 1) / PK_BYTES;
  if (threads < (uint64_t)n_prot + 1) threads = (uint64_t)n_prot + 1;
  const unsigned grid = (unsigned)((threads + PK_THREADS - 1) / PK_THREADS);
  DBI_LAUNCH(pack_kernel, grid, PK_THREADS, 0, s, d_raw, d_off, n_prot, n_res, d_res, d_pstart, pos_base, d_err);
}

namespace {
template <typename Keep>
void digest_count(const uint8_t* d_res, const DigestRange& rg, uint64_t res_alloc, const DevTables* d_tb,
                  const DigestCfg& cfg, uint32_t tile0, uint32_t ntiles, uint8_t* d_start_cnt, uint32_t* d_tile_counts,
                  uint32_t* d_err, cudaStream_t s, const Keep& keep) {
  // FILTERS = true only when a peptide filter is on
  const auto kern = (cfg.mand_on || cfg.filt_max >= 0) ? digest_count_kernel<true, Keep> : digest_count_kernel<false, Keep>;
  DBI_LAUNCH(kern, ntiles, DG_THREADS, 0, s, d_res, rg, res_alloc,
             d_tb, cfg, tile0, d_start_cnt, d_tile_counts, d_err, keep);
}
template <typename Keep>
void digest_emit(const uint8_t* d_res, const DigestRange& rg, uint64_t res_alloc, const DevTables* d_tb,
                 const DigestCfg& cfg, uint32_t tile0, uint32_t ntiles, const uint8_t* d_start_cnt,
                 const uint64_t* d_tile_offs, const uint32_t* d_pstart, uint64_t* o_mass, uint32_t* o_gpos,
                 uint32_t* o_prot, uint16_t* o_len, uint8_t* o_nmod, uint32_t* d_err, cudaStream_t s, const Keep& keep) {
  // FILTERS = true only when a peptide filter is on
  const auto kern = (cfg.mand_on || cfg.filt_max >= 0) ? digest_emit_kernel<true, Keep> : digest_emit_kernel<false, Keep>;
  DBI_LAUNCH(kern, ntiles, DG_THREADS, 0, s, d_res, rg, res_alloc,
             d_tb, cfg, tile0, d_start_cnt, d_tile_offs, d_pstart, o_mass, o_gpos, o_prot, o_len, o_nmod, d_err, keep);
}
}  // namespace

void launch_digest_count(const uint8_t* d_res, const DigestRange& rg, uint64_t res_alloc, const DevTables* d_tb,
                         const DigestCfg& cfg, uint32_t tile0, uint32_t ntiles, uint8_t* d_start_cnt,
                         uint32_t* d_tile_counts, uint32_t* d_err, cudaStream_t s, const MassWindows* windows) {
  if (ntiles == 0) return;
  if (windows)
    digest_count(d_res, rg, res_alloc, d_tb, cfg, tile0, ntiles, d_start_cnt, d_tile_counts, d_err, s, InWindows{*windows});
  else
    digest_count(d_res, rg, res_alloc, d_tb, cfg, tile0, ntiles, d_start_cnt, d_tile_counts, d_err, s, AllRecords{});
}

void launch_scan_u32_to_u64(const uint32_t* d_in, uint64_t n, uint64_t* d_offs, cudaStream_t s) {
  DBI_LAUNCH(scan_u32_to_u64_kernel, 1, SC_THREADS, 0, s, d_in, n, d_offs);
}

void launch_digest_emit(const uint8_t* d_res, const DigestRange& rg, uint64_t res_alloc, const DevTables* d_tb,
                        const DigestCfg& cfg, uint32_t tile0, uint32_t ntiles, const uint8_t* d_start_cnt,
                        const uint64_t* d_tile_offs, const uint32_t* d_pstart, uint64_t* o_mass,
                        uint32_t* o_gpos, uint32_t* o_prot, uint16_t* o_len, uint8_t* o_nmod, uint32_t* d_err,
                        cudaStream_t s, const MassWindows* windows) {
  if (ntiles == 0) return;
  if (windows)
    digest_emit(d_res, rg, res_alloc, d_tb, cfg, tile0, ntiles, d_start_cnt, d_tile_offs, d_pstart, o_mass, o_gpos,
                o_prot, o_len, o_nmod, d_err, s, InWindows{*windows});
  else
    digest_emit(d_res, rg, res_alloc, d_tb, cfg, tile0, ntiles, d_start_cnt, d_tile_offs, d_pstart, o_mass, o_gpos,
                o_prot, o_len, o_nmod, d_err, s, AllRecords{});
}

}  // namespace dbi
