// capi.cu -- the C ABI (include/dbindex_gpu.h): handle, device memory, build
// orchestration and query / fetch entry points.  Every device step is one of the
// hand-written kernels of this directory; there is no CPU fallback.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "kernels.cuh"
#include "radix_sort.cuh"

namespace dbi {

std::atomic<uint64_t> g_kernel_launches{0};
thread_local uint64_t t_kernel_launches = 0;
static thread_local char t_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_err, sizeof(t_err), fmt, ap);
  va_end(ap);
}

namespace {

// ---- device memory -----------------------------------------------------------------
// A process-wide, per-device caching allocator: blocks come from cudaMalloc once and are
// recycled by size.  Repeated builds (and short-lived handles) then never pay for
// cudaMalloc / VMM remapping again -- measured: cudaMallocAsync cost 1-6 ms per build in
// pool re-mapping for the GB-sized variant buffers.  A handle reuses the blocks it freed
// immediately (same stream, so ordering is implied); they return to the shared cache only
// after the handle's stream has been synchronised at the end of the API call.
class DevCache {
 public:
  static DevCache& of(int device) {
    static DevCache caches[64];
    return caches[device & 63];
  }
  void* get(size_t bytes) {
    {
      std::lock_guard<std::mutex> lk(mu_);
      auto it = free_.lower_bound(bytes);
      if (it != free_.end() && it->first <= bytes + bytes / 4 + 4096) {
        void* p = it->second;
        cached_ -= it->first;
        free_.erase(it);
        return p;
      }
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaErrorMemoryAllocation) {  // give the cached blocks back and retry once
      cudaGetLastError();
      trim();
      e = cudaMalloc(&p, bytes);
    }
    if (e != cudaSuccess) throw CudaError{e, "cudaMalloc", __FILE__, __LINE__};
    return p;
  }
  void put(void* p, size_t bytes) {
    std::lock_guard<std::mutex> lk(mu_);
    free_.emplace(bytes, p);
    cached_ += bytes;
  }
  void trim() {
    std::lock_guard<std::mutex> lk(mu_);
    for (auto& kv : free_) cudaFree(kv.second);
    free_.clear();
    cached_ = 0;
  }
  size_t cached_bytes() {
    std::lock_guard<std::mutex> lk(mu_);
    return cached_;
  }

 private:
  std::mutex mu_;
  std::multimap<size_t, void*> free_;
  size_t cached_ = 0;
};

// Per-handle front end of the cache.
struct DevArena {
  int device = 0;
  std::multimap<size_t, void*> local;  // freed by this handle, reusable by it right away
  static size_t round(size_t b) { return b < 512 ? 512 : (b + 511) & ~(size_t)511; }
  void* get(size_t bytes, size_t* cap) {
    bytes = round(bytes);
    auto it = local.lower_bound(bytes);
    if (it != local.end() && it->first <= bytes + bytes / 4 + 4096) {
      void* p = it->second;
      *cap = it->first;
      local.erase(it);
      return p;
    }
    *cap = bytes;  // blocks handed out by the shared cache may be larger; remember the request
    return DevCache::of(device).get(bytes);
  }
  void put(void* p, size_t cap) { local.emplace(cap, p); }
  // after the stream is idle: hand everything back to the shared cache
  void flush() {
    for (auto& kv : local) DevCache::of(device).put(kv.second, kv.first);
    local.clear();
  }
  ~DevArena() { flush(); }
};

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;  // capacity handed out
  DevArena* a = nullptr;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  void alloc(size_t b, DevArena& arena) {
    release();
    a = &arena;
    p = arena.get(b, &bytes);
  }
  // a view into memory owned by somebody else (a multi-GPU window): release() only forgets it
  void borrow(void* ptr, size_t b) {
    release();
    a = nullptr;
    p = ptr;
    bytes = b;
  }
  void release() {
    if (p) {
      if (a) a->put(p, bytes);
      p = nullptr;
      bytes = 0;
    }
  }
  void swap(DevBuf& o) {
    std::swap(p, o.p);
    std::swap(bytes, o.bytes);
    std::swap(a, o.a);
  }
  ~DevBuf() { release(); }
  template <typename T>
  T* as() const { return (T*)p; }
};

// Emitted records as they leave K4 (or arrive from the other GPUs).
struct RecView {
  const uint64_t* mass;  // IEEE bits
  const uint32_t* gpos;
  const uint32_t* prot;
  const uint16_t* len;
};

// The device buffers of a set of emitted records.
struct RecSet {
  DevBuf mass, gpos, prot, len;  // mass as IEEE bits
  void alloc(uint64_t n, DevArena& arena) {
    mass.alloc(n * 8, arena);
    gpos.alloc(n * 4, arena);
    prot.alloc(n * 4, arena);
    len.alloc(n * 2, arena);
  }
  void release() { mass.release(); gpos.release(); prot.release(); len.release(); }
  void swap(RecSet& o) { mass.swap(o.mass); gpos.swap(o.gpos); prot.swap(o.prot); len.swap(o.len); }
  RecView view() const { return {mass.as<uint64_t>(), gpos.as<uint32_t>(), prot.as<uint32_t>(), len.as<uint16_t>()}; }
};

inline uint64_t dbits(double d) {
  uint64_t u;
  std::memcpy(&u, &d, 8);
  return u;
}
inline int bit_length(uint64_t v) { return v ? 64 - __builtin_clzll(v) : 0; }

}  // namespace
}  // namespace dbi

using namespace dbi;

struct dbi_handle {
  dbi_params p;
  int device = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  std::mutex mu;
  DevArena arena;  // declared before every DevBuf of the handle: destroyed after them

  // The residues go straight from the caller's buffer to the device (dbi_add_proteins); the host
  // keeps the offsets, and a copy of the residues (ProteinCache) only once dbi_get_protein asks.
  std::vector<uint8_t> h_raw;
  bool h_raw_valid = false;
  std::vector<uint64_t> h_off{0};
  uint64_t n_res = 0;  // residues added so far = bytes valid in d_raw

  // device-resident input
  DevBuf d_raw, d_off;
  uint64_t up_prot = UINT64_MAX;

  // index
  bool built = false;
  DevBuf d_tables, d_err;
  // The device arrays of a built index (kIndexBufs below lists them for release, borrow and device_bytes).
  struct IndexBufs {
    DevBuf d_res, d_pstart;  // packed residues + protein starts: outlive the tables (free_tables keeps them)
    DevBuf u_mass, u_gpos, u_prot, u_len, u_plo, plist;
    DevBuf e_mass, e_base, e_pat;  // empty when there are no differential mods (entries == unique peptides)
    // group path: site masks of the unique peptides (u_cmask[u * C + c]), valid for cmask_n peptides;
    // d_nlong = how many peptides are longer than 64 residues (they have no masks)
    DevBuf u_cmask, d_nlong;
    // compact layout (single GPU, group path): the sorted groups instead of the entry arrays.  g_mass = group
    // mass, g_pay = peptide << 32 | class sequence << 27 | variant count, g_eoff = entries before each group
    // (n_groups + 1).
    DevBuf g_mass, g_pay, g_eoff;
  } ix;
  struct TableCounts {  // the sizes of the tables; free_tables resets them
    uint64_t n_emitted = 0, n_unique = 0, n_entries = 0;
    uint64_t n_groups = 0;  // 0 when the entries are expanded
    uint64_t n_long = 0;    // peptides longer than 64 residues
    uint64_t cmask_n = UINT64_MAX;
  } cnt;
  struct ResLayout {  // what d_res / d_pstart hold; free_index resets it
    uint64_t packed_prot = UINT64_MAX;  // proteins d_res / d_pstart hold (K1 ran on them)
    uint32_t res_end = 0;
    uint64_t res_alloc = 0;  // bytes readable at d_res (multiple of 16: tiles are staged with bulk copies)
    bool mg_layout = false;  // dbi_mg_set_shards done (d_res / d_pstart are views of window 0)
  } lay;
  RecSet kept;  // kept raw records (params.keep_emitted)

  // ---- sharded build (dbi_mg_*, capi_mg.inl) ----
  // Three WINDOWS per rank are visible to the other ranks (mapped peer memory over NVLink):
  //   0 proteome: the packed residues of ALL ranks + their protein starts (every rank packs its own
  //     shard in place and pulls the others);  1 arena: what the exchanges deliver to this rank;
  //   2 unique tables: first occurrence + protein lists of the peptides this rank owns.
  struct MgWindow {  // the block this rank owns (exportable)
    void* p = nullptr;
    uint64_t cap = 0;
  };
  struct MgPeers {  // mapped base of every rank's window (own rank: MgWindow::p)
    void* peer[kMaxRanks] = {};
    uint64_t peer_cap[kMaxRanks] = {};
  };
  bool mg_begun = false;  // dbi_mg_begin was called
  MgWindow win[3];
  // Where a query finds the other ranks' proteins, peptides and mass slices.  Set by the stages that lay them
  // out; free_sharded_tables resets ent_base_off and uoff.
  struct MgRoute {
    int mg_rank = 0, mg_world = 1;
    MgPeers win[3];
    uint64_t prot_off[kMaxRanks + 1] = {};  // global id of every rank's first protein
    uint64_t pos_off[kMaxRanks + 1] = {};   // buffer position of every rank's first separator
    uint64_t ent_base_off = 0;              // global id of this rank's first unique peptide (0 on a single GPU)
    uint64_t uoff[kMaxRanks + 1] = {};      // global id of every rank's first unique peptide
    uint64_t uniq_cap[kMaxRanks] = {};      // layout capacity of every rank's window 2
    uint64_t mg_thr[2][kMaxSlices] = {};    // key thresholds of the two exchanges
    int mg_nthr[2] = {};                    // how many: slices - 1
  } rt;
  cudaStream_t side_stream = nullptr;  // carries the peer pulls of the proteome next to the digest
  cudaEvent_t pull_done = nullptr;
  bool pull_pending = false;
  // world of the sharded unindexed search whose layout window 0 still holds (0 = none): the next search of the
  // same handles with the same shards reuses it (dbi_mg_search_unindexed_local)
  int mg_search_world = 0;
  struct MgStaged {            // the local items between the stages of a sharded build
    RecSet mg_rec;             // local records between digest and exchange
    DevBuf mg_nmod;            // their mod-site counts
    uint64_t mg_n = 0;
    DevBuf mg_vkey, mg_vpay;   // local groups / variants between listing and exchange
    uint64_t mg_v = 0;
    uint64_t mg_recv[2] = {};  // items delivered to this rank by exchange 0 / 1
    void release() {
      mg_rec.release(); mg_nmod.release(); mg_vkey.release(); mg_vpay.release();
      mg_n = mg_v = 0;
      mg_recv[0] = mg_recv[1] = 0;
    }
  } mgs;
  DevBuf mg_wtab;  // variants of a peptide with n sites

  // pending result of dbi_query_hits (device side), read by dbi_query_hits_read
  struct HitResult {
    bool valid = false;
    dbi_hit_counts n{};
    DevBuf hit_off, pep_off, pat, pep_hit_off, mass, prot, off, len, flanks, seq_off, seq, plo, ids;
    void drop() {
      valid = false;
      hit_off.release(); pep_off.release(); pat.release(); pep_hit_off.release(); mass.release(); prot.release();
      off.release(); len.release(); flanks.release(); seq_off.release(); seq.release(); plo.release(); ids.release();
    }
  } hits;

  // pending result of dbi_lookup_peptides, read by dbi_lookup_peptides_read
  struct LookupResult {
    bool valid = false;
    dbi_lookup_counts n{};
    DevBuf status, mass, entry, prot, off, plo, ids;
    void drop() {
      valid = false;
      status.release(); mass.release(); entry.release(); prot.release(); off.release(); plo.release(); ids.release();
    }
  } lookup;

  DigestCfg cfg{};
  MassWindows shifts{};  // the shift intervals of an unindexed search (no windows yet)
  dbi_stats st{};
  // profiling (params.profile): event pairs recorded on the stream without any extra
  // synchronisation and resolved after the final sync of the call
  struct Span { int kind; cudaEvent_t a, b; };
  std::vector<cudaEvent_t> ev_pool;
  size_t ev_used = 0;
  std::vector<Span> spans;
  cudaEvent_t get_event() {
    if (ev_used == ev_pool.size()) {
      cudaEvent_t e;
      DBI_CUDA(cudaEventCreate(&e));
      ev_pool.push_back(e);
    }
    return ev_pool[ev_used++];
  }

  // query views (dbi_view_open): a view names its owner; an owner counts its open views and, when destroyed while
  // some are open, lives on (orphaned) until the last of them is destroyed
  dbi_handle* owner = nullptr;
  std::atomic<int> n_views{0};
  std::mutex view_mu;  // guards the last-view / orphaned hand-over
  bool orphaned = false;

  const double* entry_mass() const { return ix.e_mass.p ? ix.e_mass.as<double>() : ix.u_mass.as<double>(); }
  const uint32_t* entry_base() const { return ix.e_base.as<uint32_t>(); }
  const uint32_t* entry_pat() const { return ix.e_pat.as<uint32_t>(); }
  // what K9 / K14 / the key listing search: the groups of a compact index, else the entries
  const double* key_mass() const { return cnt.n_groups ? ix.g_mass.as<double>() : entry_mass(); }
  uint64_t n_keys() const { return cnt.n_groups ? cnt.n_groups : cnt.n_entries; }
};

// Every array of an index, once.  kResidues: only free_index releases it (the tables of a rebuild reuse the
// packed residues).  kCompact: device_bytes counts it only in a compact index, which needs the site masks to
// expand its groups.  kUncounted: device_bytes never counts it.
enum BufUse { kResidues, kCounted, kCompact, kUncounted };
using IB = dbi_handle::IndexBufs;
using IndexBuf = DevBuf IB::*;
constexpr struct { IndexBuf buf; BufUse use; } kIndexBufs[] = {
    {&IB::d_res, kResidues}, {&IB::d_pstart, kResidues}, {&IB::u_mass, kCounted},    {&IB::u_gpos, kCounted},
    {&IB::u_prot, kCounted}, {&IB::u_len, kCounted},     {&IB::u_plo, kCounted},     {&IB::plist, kCounted},
    {&IB::e_mass, kCounted}, {&IB::e_base, kCounted},    {&IB::e_pat, kCounted},     {&IB::u_cmask, kCompact},
    {&IB::d_nlong, kUncounted}, {&IB::g_mass, kCompact}, {&IB::g_pay, kCompact},     {&IB::g_eoff, kCompact},
};

namespace {

// DBI_TRACE=1: host wall-clock marks inside dbi_build, printed to stderr (diagnostic only).
struct HostTrace {
  bool on = std::getenv("DBI_TRACE") != nullptr;
  std::vector<std::pair<const char*, double>> marks;
  static double now() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
  }
  void mark(const char* what) {
    if (on) marks.emplace_back(what, now());
  }
  void dump() {
    if (!on || marks.empty()) return;
    fprintf(stderr, "[dbi trace]");
    for (size_t i = 1; i < marks.size(); ++i) fprintf(stderr, " %s=%.3f", marks[i].first, marks[i].second - marks[i - 1].second);
    fprintf(stderr, " total=%.3f ms\n", marks.back().second - marks.front().second);
    marks.clear();
  }
};
thread_local HostTrace g_trace;
#define TR(x) g_trace.mark(x)

int fail_cuda(const CudaError& e) {
  set_error("CUDA error %d (%s) at %s:%d: %s", (int)e.e, cudaGetErrorString(e.e), e.file, e.line, e.what);
  cudaGetLastError();  // clear the sticky-free error state
  return e.e == cudaErrorMemoryAllocation ? DBI_ENOMEM : DBI_ECUDA;
}

// Runs at the end of every API call, after the call's local DevBufs are gone: once the stream
// is idle the blocks they freed may be shared with other handles.
struct ArenaFlush {
  dbi_handle* h;
  explicit ArenaFlush(dbi_handle* h_) : h(h_) {}
  ~ArenaFlush();
};

#define DBI_API_BEGIN(h)                      \
  if (!(h)) {                                 \
    set_error("null handle");                 \
    return DBI_EINVAL;                        \
  }                                           \
  std::lock_guard<std::mutex> _lk((h)->mu);   \
  ArenaFlush _af(h);                          \
  try {                                       \
    DBI_CUDA(cudaSetDevice((h)->device));

// A call that only an owner may make: one that changes the proteins or the index, or joins several handles.
#define DBI_OWNER_ONLY(h)                                                        \
  if ((h)->owner) {                                                              \
    set_error("%s is not available on a query view (dbi_view_open)", __func__); \
    return DBI_EINVAL;                                                           \
  }

// A call that changes the residues, the candidate index or the index tables: refused on a view, and on an owner
// while views of it are open (they read the same memory).  After DBI_API_BEGIN, so under the owner's mutex,
// which dbi_view_open holds too.
#define DBI_MUTATES(h)                                           \
  DBI_OWNER_ONLY(h)                                              \
  if (const int nv_ = (h)->n_views.load()) {                     \
    set_error("%s: %d views open on this handle", __func__, nv_); \
    return DBI_EINVAL;                                           \
  }

#define DBI_API_END                              \
  }                                              \
  catch (const CudaError& e) { return fail_cuda(e); } \
  catch (const std::bad_alloc&) {                \
    set_error("host allocation failed");         \
    return DBI_ENOMEM;                           \
  }

constexpr int kSpanDominant = 100;  // span kind of a dominant-kernel launch
constexpr int kSpanExpand = 101;    // span kind of the expansion kernel

ArenaFlush::~ArenaFlush() {
  if (h->arena.local.empty()) return;
  cudaStreamSynchronize(h->stream);
  h->arena.flush();
}

// CUDA-event stage timer (only when params.profile) + launch accounting.
struct Stage {
  dbi_handle* h;
  int id;
  uint64_t l0;
  cudaEvent_t a = nullptr;
  Stage(dbi_handle* h_, int id_) : h(h_), id(id_) {
    l0 = t_kernel_launches;
    if (h->p.profile) {
      a = h->get_event();
      cudaEventRecord(a, h->stream);
    }
  }
  ~Stage() {  // never throws: a failed event creation only loses this stage's timing
    h->st.stage_launches[id] += (uint32_t)(t_kernel_launches - l0);
    if (h->p.profile && a) {
      try {
        cudaEvent_t b = h->get_event();
        cudaEventRecord(b, h->stream);
        h->spans.push_back({id, a, b});
      } catch (...) {
        cudaGetLastError();
      }
    }
  }
};

// Brackets every scatter pass of one sort with an event pair.
struct DomProbe : PassProbe {
  dbi_handle* h;
  cudaEvent_t a = nullptr;
  explicit DomProbe(dbi_handle* h_) : h(h_) {}
  void before_pass(int) override {
    a = h->get_event();
    cudaEventRecord(a, h->stream);
  }
  void after_pass(int) override {
    cudaEvent_t b = h->get_event();
    cudaEventRecord(b, h->stream);
    h->spans.push_back({kSpanDominant, a, b});
  }
};

// After the stream has been synchronised: turn the recorded spans into stats.
void resolve_spans(dbi_handle* h) {
  for (const auto& sp : h->spans) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, sp.a, sp.b) != cudaSuccess) { cudaGetLastError(); continue; }
    if (sp.kind == kSpanDominant) {
      h->st.dom_ms += ms;
      h->st.dom_launches++;
    } else if (sp.kind == kSpanExpand) {
      h->st.exp_ms += ms;
      h->st.exp_launches++;
    } else {
      h->st.stage_ms[sp.kind] += ms;
    }
  }
  h->spans.clear();
  h->ev_used = 0;
}

uint32_t read_err(dbi_handle* h) {
  uint32_t e = 0;
  DBI_CUDA(cudaMemcpyAsync(&e, h->d_err.p, 4, cudaMemcpyDeviceToHost, h->stream));
  DBI_CUDA(cudaStreamSynchronize(h->stream));
  return e;
}

void clear_err(dbi_handle* h) {
  const uint32_t zero = 0;
  DBI_CUDA(cudaMemcpyAsync(h->d_err.p, &zero, 4, cudaMemcpyHostToDevice, h->stream));
}

uint64_t read_u64(dbi_handle* h, const uint64_t* d) {
  uint64_t v = 0;
  DBI_CUDA(cudaMemcpyAsync(&v, d, 8, cudaMemcpyDeviceToHost, h->stream));
  DBI_CUDA(cudaStreamSynchronize(h->stream));
  return v;
}

// The tables an index build derives from the packed residues: unique peptides, protein lists, entries.
void free_tables(dbi_handle* h) {
  for (const auto& b : kIndexBufs)
    if (b.use != kResidues) (h->ix.*b.buf).release();
  h->cnt = {};
  h->kept.release();
}

// The pending results of dbi_query_hits / dbi_search_unindexed and dbi_lookup_peptides.
void drop_results(dbi_handle* h) {
  h->hits.drop();
  h->lookup.drop();
}

// The index tables and the sharded state between the stages of a build; the packed residues stay.
void free_sharded_tables(dbi_handle* h) {
  h->built = false;
  free_tables(h);
  h->mgs.release();
  h->rt.ent_base_off = 0;
  std::memset(h->rt.uoff, 0, sizeof(h->rt.uoff));
}

void free_index(dbi_handle* h) {
  if (h->pull_pending) {  // peer copies into d_res still in flight
    cudaStreamSynchronize(h->side_stream);
    h->pull_pending = false;
  }
  drop_results(h);
  for (const auto& b : kIndexBufs)
    if (b.use == kResidues) (h->ix.*b.buf).release();
  h->lay = {};
  free_sharded_tables(h);
  h->mg_search_world = 0;
  h->spans.clear();
  h->ev_used = 0;
  const uint64_t np = h->st.n_proteins, nr = h->st.n_residues;
  std::memset(&h->st, 0, sizeof(h->st));
  h->st.n_proteins = np;
  h->st.n_residues = nr;
}

void upload_tables(dbi_handle* h) {
  DevTables t;
  std::memset(&t, 0, sizeof(t));
  const dbi_params& p = h->p;
  for (int i = 0; i < 256; ++i) {
    t.mass[i] = p.residue_mass[i];
    t.flags[i] = (p.is_enzyme[i] ? kFlagEnzyme : 0) | (p.is_nocut[i] ? kFlagNocut : 0) |
                 ((p.has_mandatory && p.is_mandatory[i]) ? kFlagMandatory : 0) |
                 ((p.filter_aa > 0 && p.filter_aa == i) ? kFlagFilterAA : 0);
  }
  const bool mods = p.n_mods > 0 && p.max_mods_per_peptide > 0;
  if (mods)
    for (int i = 0; i < p.n_mods; ++i) {  // DiffModification.setDiffModMass: last one wins
      t.diff[p.mods[i].residue] = p.mods[i].delta;
      t.flags[p.mods[i].residue] |= kFlagDiffMod;
    }
  double init = 0;  // DBIndexer.java:265-271, same order
  if (p.add_h2o_proton) init += p.h2o_proton;
  init += p.cterm;
  init += p.nterm;
  h->cfg.init_mass = init;
  h->cfg.min_mass = p.min_mass;
  h->cfg.max_mass = p.max_mass;
  h->cfg.max_mc = p.max_missed;
  h->cfg.semi = p.semi ? 1 : 0;
  h->cfg.min_len = p.min_len;
  h->cfg.max_mods = mods ? p.max_mods_per_peptide : 0;
  h->cfg.mod_hi = 0;
  h->cfg.mod_lo = 0;
  h->cfg.n_classes = 0;
  h->cfg.n_seq = 0;
  h->cfg.mand_on = p.has_mandatory ? 1 : 0;
  h->cfg.filt_max = p.filter_aa > 0 ? std::max(p.filter_max, 0) : -1;
  if (mods) {
    // mod classes = distinct shift values (two residues with the same shift are interchangeable
    // for the mass); class sequences of length <= K number (C^(K+1)-1)/(C-1)
    int nc = 0;
    for (int i = 0; i < 256; ++i)
      if (t.flags[i] & kFlagDiffMod) {
        h->cfg.mod_hi = std::max(h->cfg.mod_hi, t.diff[i]);
        h->cfg.mod_lo = std::min(h->cfg.mod_lo, t.diff[i]);
        int c = 0;
        while (c < nc && t.cls_delta[c] != t.diff[i]) ++c;
        if (c == nc) t.cls_delta[nc++] = t.diff[i];
        t.cls[i] = (uint8_t)c;
      }
    h->cfg.n_classes = nc;
    uint64_t g = 0, pw = 1;
    for (int k = 0; k <= p.max_mods_per_peptide; ++k) { g += pw; pw *= (uint64_t)nc; }
    h->cfg.n_seq = g <= 32 ? (int)g : 0;
    if (std::getenv("DBI_NO_GROUPS")) h->cfg.n_seq = 0;  // diagnostic: force the per-variant path
  }
  shift_intervals(t, h->cfg, &h->shifts);
  h->d_tables.alloc(sizeof(DevTables), h->arena);
  DBI_CUDA(cudaMemcpyAsync(h->d_tables.p, &t, sizeof(t), cudaMemcpyHostToDevice, h->stream));
  DBI_CUDA(cudaStreamSynchronize(h->stream));  // `t` is on this stack frame
}

// H2D of the protein offsets (idempotent); the residues are already on the device.
void ensure_uploaded(dbi_handle* h) {
  const uint64_t n_prot = h->h_off.size() - 1;
  if (h->up_prot == n_prot) return;
  if (!h->d_raw.p) h->d_raw.alloc(16, h->arena);
  h->d_off.alloc((n_prot + 1) * 8, h->arena);
  DBI_CUDA(cudaMemcpyAsync(h->d_off.p, h->h_off.data(), (n_prot + 1) * 8, cudaMemcpyHostToDevice, h->stream));
  h->up_prot = n_prot;
}

int check_err_bits(uint32_t e) {
  if (e & kErrZeroResidue) {
    set_error("residue byte 0 in the protein buffer");
    return DBI_EINVAL;
  }
  if (e & kErrPepTooLong) {
    set_error("a peptide window exceeds DBI_MAX_PEP_LEN (%d residues)", DBI_MAX_PEP_LEN);
    return DBI_ERANGE;
  }
  if (e & kErrModPos) {
    set_error("a modifiable residue lies beyond position %d of a peptide", DBI_MAX_MOD_POS);
    return DBI_ERANGE;
  }
  return DBI_OK;
}

// K1: padded residue buffer + protein starts.
void pack_residues(dbi_handle* h) {
  Stage sg(h, DBI_STAGE_PACK);
  const uint64_t n_res = h->n_res;
  const uint32_t n_prot = (uint32_t)(h->h_off.size() - 1);
  const uint64_t res_end = n_res + n_prot + 1;
  const uint64_t padded = (res_end + 64 + 15) & ~15ull;
  h->lay.res_end = (uint32_t)res_end;
  h->lay.res_alloc = padded;
  h->ix.d_res.alloc(padded, h->arena);
  h->ix.d_pstart.alloc(((uint64_t)n_prot + 1) * 4, h->arena);
  DBI_CUDA(cudaMemsetAsync((uint8_t*)h->ix.d_res.p + res_end, 0, padded - res_end, h->stream));
  launch_pack(h->d_raw.as<uint8_t>(), h->d_off.as<uint64_t>(), n_prot, n_res, h->ix.d_res.as<uint8_t>(),
              h->ix.d_pstart.as<uint32_t>(), 0u, h->d_err.as<uint32_t>(), h->stream);
  h->lay.packed_prot = n_prot;
  h->st.algo_bytes[DBI_STAGE_PACK] += 2 * n_res + (uint64_t)n_prot * 12;
}

// The start of a single-GPU build: protein offsets on the device, error bits cleared, K1.
void build_begin(dbi_handle* h) {
  ensure_uploaded(h);
  clear_err(h);
  pack_residues(h);
}

// K2 (count) and K4 (emit) over the start positions of rg in tiles [t0, t0 + nt); with windows only the records
// that can land in one of them (K2u / K4u).  Each kernel is charged 2 * span residue bytes.  The caller checks the
// error bits and the record count between count() and emit().
struct Digest {
  dbi_handle* h;
  DigestRange rg;
  uint32_t t0, nt;
  uint64_t span;
  const MassWindows* windows;
  DevBuf tile_counts, tile_offs, start_cnt;  // what K2 leaves for K4
  uint64_t n = 0;

  // K2 and the scan of its tile counts: the number of records K4 emits
  uint64_t count() {
    tile_counts.alloc((uint64_t)nt * 4, h->arena);
    tile_offs.alloc(((uint64_t)nt + 1) * 8, h->arena);
    start_cnt.alloc((uint64_t)nt * kDigestTile, h->arena);
    if (!nt) return n = 0;
    Stage sg(h, DBI_STAGE_DIGEST_COUNT);
    launch_digest_count(h->ix.d_res.as<uint8_t>(), rg, h->lay.res_alloc, h->d_tables.as<DevTables>(), h->cfg, t0, nt,
                        start_cnt.as<uint8_t>(), tile_counts.as<uint32_t>(), h->d_err.as<uint32_t>(), h->stream, windows);
    launch_scan_u32_to_u64(tile_counts.as<uint32_t>(), nt, tile_offs.as<uint64_t>(), h->stream);
    n = read_u64(h, tile_offs.as<uint64_t>() + nt);
    h->st.algo_bytes[DBI_STAGE_DIGEST_COUNT] += 2 * span + (uint64_t)nt * 16;
    return n;
  }
  // K4 into out, allocated for the counted records; nmod (optional): their mod-site counts
  void emit(RecSet& out, DevBuf* nmod) {
    out.alloc(n, h->arena);
    if (nmod) nmod->alloc(std::max<uint64_t>(n, 1), h->arena);
    {
      Stage sg(h, DBI_STAGE_DIGEST_EMIT);
      launch_digest_emit(h->ix.d_res.as<uint8_t>(), rg, h->lay.res_alloc, h->d_tables.as<DevTables>(), h->cfg, t0, nt,
                         start_cnt.as<uint8_t>(), tile_offs.as<uint64_t>(), h->ix.d_pstart.as<uint32_t>(),
                         out.mass.as<uint64_t>(), out.gpos.as<uint32_t>(), out.prot.as<uint32_t>(),
                         out.len.as<uint16_t>(), nmod ? nmod->as<uint8_t>() : nullptr, h->d_err.as<uint32_t>(),
                         h->stream, windows);
      h->st.algo_bytes[DBI_STAGE_DIGEST_EMIT] += 2 * span + n * 18;
    }
    tile_counts.release();
    tile_offs.release();
    start_cnt.release();
  }
};

// The digest of a single-GPU build or unindexed search: every start position, none when there are no windows.
Digest whole_digest(dbi_handle* h, const MassWindows* windows) {
  const uint32_t nt =
      windows && !windows->n ? 0u : (uint32_t)(((uint64_t)h->lay.res_end + kDigestTile - 1) / kDigestTile);
  return {h, DigestRange{0u, h->lay.res_end, 0u, (uint32_t)(h->h_off.size() - 1)}, 0u, nt, h->lay.res_end, windows};
}

// Radix key of a mass: bits(mass) - bits(lo); every mass of a build lies in [lo, hi].
struct KeySpace {
  uint64_t base_bits;
  int nbits;
  KeySpace(double lo, double hi) : base_bits(dbits(lo)), nbits(bit_length(dbits(hi) - dbits(lo))) {}
};

inline uint64_t al256(uint64_t x) { return (x + 255) & ~255ull; }

// Window 2 of a sharded build: the unique tables of one rank, laid out by the CAPACITY of the window
// (= the number of records exchange 0 delivered to that rank), which every rank knows.
struct UniqLayout {
  uint64_t gpos, prot, len, plo, plist, total;
  explicit UniqLayout(uint64_t cap) {
    gpos = 0;
    prot = gpos + al256(4 * cap);
    len = prot + al256(4 * cap);
    plo = len + al256(2 * cap);
    plist = plo + al256(8 * (cap + 1));
    total = plist + al256(4 * cap);
  }
};

// Test hook: DBI_GROUP_RADIX sends the single-GPU group path through the K7 sort of the sharded build
// (peptide-major records) instead of K6g's sorted lists + the K7m merge; the results are identical.
bool group_radix(const dbi_handle*) { return std::getenv("DBI_GROUP_RADIX") != nullptr; }
// Test hook: DBI_COMPACT_VARIANTS keeps a single-GPU group-path index compact even below 2^32 entries, so that
// tests and benchmarks can compare the two layouts on small proteomes
bool compact_variants(const dbi_handle*) { return std::getenv("DBI_COMPACT_VARIANTS") != nullptr; }

// The hash pre-sort of large builds (K7 twice): idx[0] <- the records in (mass, hash & mask(hash_bits),
// arrival order), hash <- every record's hash; returns the buffer index of the sorted mass keys.
int hash_presort(dbi_handle* h, const RecView& r, uint64_t N, const KeySpace& ks, uint32_t seed, int hash_bits,
                 DevBuf& hash, DevBuf* idx, DevBuf* hkey, DevBuf* mkey, DevBuf& tmp) {
  cudaStream_t s = h->stream;
  const bool wide = hash_bits > 32;
  const int nbits = ks.nbits;
  Stage sg(h, DBI_STAGE_SORT_BASE);
  hash.alloc(N * (wide ? 8 : 4), h->arena);
  hkey[0].alloc(N * (wide ? 8 : 4), h->arena);
  hkey[1].alloc(N * (wide ? 8 : 4), h->arena);
  launch_hash_records(h->ix.d_res.as<uint8_t>(), r.gpos, r.len, N, seed, wide, hash.p, idx[0].as<uint32_t>(), s);
  DBI_CUDA(cudaMemcpyAsync(hkey[0].p, hash.p, N * (wide ? 8 : 4), cudaMemcpyDeviceToDevice, s));
  // less significant key first: sequence hash ...
  uint32_t* ix[2] = {idx[0].as<uint32_t>(), idx[1].as<uint32_t>()};
  int r1;
  if (wide) {
    uint64_t* hk[2] = {hkey[0].as<uint64_t>(), hkey[1].as<uint64_t>()};
    r1 = radix_sort_pairs<uint64_t, uint32_t>(hk, ix, N, 0, hash_bits, tmp.p, s, nullptr);
  } else {
    uint32_t* hk[2] = {hkey[0].as<uint32_t>(), hkey[1].as<uint32_t>()};
    r1 = radix_sort_pairs<uint32_t, uint32_t>(hk, ix, N, 0, 32, tmp.p, s, nullptr);
  }
  DomProbe base_probe(h);
  // the largest K7 sort of the build: the base sort, unless the variant groups go through K7 too
  const bool base_is_dominant =
      h->p.profile && (h->cfg.max_mods == 0 || (h->cfg.n_seq > 0 && h->rt.mg_world <= 1 && !group_radix(h)));
  if (base_is_dominant) {  // a retry re-runs the sort: count only the final attempt
    h->spans.erase(std::remove_if(h->spans.begin(), h->spans.end(),
                                  [](const dbi_handle::Span& sp) { return sp.kind == kSpanDominant; }),
                   h->spans.end());
    h->st.dom_kernel = 0;
    h->st.dom_bytes_per_launch = N * 24ull;
  }
  // ... then the exact mass bits (stable), so order = (mass, hash, arrival order)
  launch_gather_mass_key(r.mass, ix[r1], N, ks.base_bits, mkey[0].as<uint64_t>(), s);
  uint64_t* mk[2] = {mkey[0].as<uint64_t>(), mkey[1].as<uint64_t>()};
  uint32_t* ix2[2] = {ix[r1], ix[r1 ^ 1]};
  const int r2 = radix_sort_pairs<uint64_t, uint32_t>(mk, ix2, N, 0, nbits, tmp.p, s,
                                                      base_is_dominant ? &base_probe : nullptr);
  // normalise: sorted idx in idx[0]
  if (ix2[r2] != idx[0].as<uint32_t>()) idx[0].swap(idx[1]);
  const int hpasses = (hash_bits + 7) / 8, mpasses = (nbits + 7) / 8;
  const uint64_t hw = wide ? 8 : 4;
  h->st.algo_bytes[DBI_STAGE_SORT_BASE] += N * (16 /*hash: len + gpos*/ + 3 * hw + 4 + 8 + 8 + 4) +
                                           N * 2 * (hw + 4) * hpasses + N * 24ull * mpasses + N * 20;
  return r2;
}

// Builds of fewer records than this order the base records with the mass-only K7 + K8r; larger ones keep
// the hash pre-sort.  Records with bit-equal masses (isomers and repeats) grow with N: at cfg1 / cfg2
// size (2.7 M records) the longest equal-mass run has 244 records and K8r costs less than the four hash
// passes it replaces, while at 514 M (cfg3) runs are long enough that one CTA per run loses to K7.
constexpr uint64_t kRunOrderMaxRecords = 1ull << 23;

// K7 (+ K8r) + K8: sort N records by (mass, sequence hash, arrival order), merge equal peptides into
// the handle's unique tables (u_*, plist).  Below kRunOrderMaxRecords K7 sorts by mass alone (stable,
// so every run of equal mass sits in arrival order) and K8r then orders each such run by (hash, arrival
// order), hashing only records that share their mass bits with another one.  Above it K7 sorts by the
// hash of every record and then, stably, by mass.  Both give the same order.
int sort_dedup(dbi_handle* h, const RecView& r, uint64_t N, const KeySpace& ks) {
  cudaStream_t s = h->stream;
  if (N >= (1ull << 32)) {
    set_error("more than 2^32 emitted records on one GPU (%llu)", (unsigned long long)N);
    return DBI_ERANGE;
  }
  h->cnt.n_unique = 0;
  h->st.n_unique = 0;
  if (N == 0) {
    if (h->rt.mg_world > 1 && h->win[2].p) h->ix.u_plo.borrow((uint8_t*)h->win[2].p + UniqLayout(h->rt.uniq_cap[h->rt.mg_rank]).plo, 8);
    else h->ix.u_plo.alloc(8, h->arena);
    DBI_CUDA(cudaMemsetAsync(h->ix.u_plo.p, 0, 8, s));
    return DBI_OK;
  }
  const uint64_t base_bits = ks.base_bits;
  const int nbits = ks.nbits;
  h->st.sort_bits_base = (uint32_t)nbits + 32;

  DevBuf hash, idx[2], hkey[2], mkey[2], tmp, flags, tile_counts, tile_offs, rlist;
  const bool run_order = N < kRunOrderMaxRecords;
  const uint64_t tiles = (N + kScanTile - 1) / kScanTile;
  TR("ir_begin");
  // Width of the sequence hash: the number of distinct-string pairs with bit-equal mass grows with
  // N^2, so two more bits per doubling of N beyond 4 M records; a detected collision adds 8.
  int hash_bits = 32;
  for (uint64_t m = N >> 22; m > 1; m >>= 1) hash_bits += 2;
  hash_bits = std::min(hash_bits, 64);
  if (const char* e = std::getenv("DBI_HASH_BITS")) {  // test hook: force the wide-hash path on small inputs
    const int v = std::atoi(e);
    if (v >= 32 && v <= 64) hash_bits = v;
  }
  idx[0].alloc(N * 4, h->arena); idx[1].alloc(N * 4, h->arena);
  mkey[0].alloc(N * 8, h->arena); mkey[1].alloc(N * 8, h->arena);
  tmp.alloc(radix_sort_tmp_bytes(N), h->arena);
  flags.alloc(N, h->arena);
  tile_counts.alloc(tiles * 4, h->arena);
  tile_offs.alloc((tiles + 1) * 8, h->arena);
  if (run_order) rlist.alloc((run_order_list_cap(N) + 1) * 4, h->arena);  // [0]: count, then the listed run heads

  TR("ir_alloc");
  int sorted = 0;
  if (run_order) {
    Stage sg(h, DBI_STAGE_SORT_BASE);
    launch_mass_key(r.mass, N, base_bits, mkey[0].as<uint64_t>(), idx[0].as<uint32_t>(), s);
    DomProbe base_probe(h);
    // the largest K7 sort of the build: the base sort, unless the variant groups go through K7 too
    const bool base_is_dominant =
        h->p.profile && (h->cfg.max_mods == 0 || (h->cfg.n_seq > 0 && h->rt.mg_world <= 1 && !group_radix(h)));
    if (base_is_dominant) {  // count only this sort's passes
      h->spans.erase(std::remove_if(h->spans.begin(), h->spans.end(),
                                    [](const dbi_handle::Span& sp) { return sp.kind == kSpanDominant; }),
                     h->spans.end());
      h->st.dom_kernel = 0;
      h->st.dom_bytes_per_launch = N * 24ull;
    }
    uint64_t* mk[2] = {mkey[0].as<uint64_t>(), mkey[1].as<uint64_t>()};
    uint32_t* ix[2] = {idx[0].as<uint32_t>(), idx[1].as<uint32_t>()};
    sorted = radix_sort_pairs<uint64_t, uint32_t>(mk, ix, N, 0, nbits, tmp.p, s, base_is_dominant ? &base_probe : nullptr);
    // normalise: sorted keys in mkey[sorted], sorted idx in idx[0]
    if (sorted) idx[0].swap(idx[1]);
    const int mpasses = (nbits + 7) / 8;
    h->st.algo_bytes[DBI_STAGE_SORT_BASE] += N * (8 + 8 + 4) /*keys*/ + N * 8 /*histogram*/ + N * 24ull * mpasses;
  }
  uint64_t n_unique = 0;
  for (uint32_t attempt = 0;; ++attempt) {
    const bool wide = hash_bits > 32;
    h->st.sort_bits_base = (uint32_t)(nbits + hash_bits);
    const uint32_t seed = 0x9e3779b9u * attempt;
    if (!run_order) sorted = hash_presort(h, r, N, ks, seed, hash_bits, hash, idx, hkey, mkey, tmp);
    {
      Stage sg(h, DBI_STAGE_DEDUP);
      // K8r: equal-mass runs by (hash, arrival order); independent of the order a previous attempt left
      if (run_order) {
        hash.alloc(N * (wide ? 8 : 4), h->arena);
        launch_run_order(h->ix.d_res.as<uint8_t>(), mkey[sorted].as<uint64_t>(), idx[0].as<uint32_t>(),
                         idx[1].as<uint32_t>(), r.gpos, r.len, N, seed, hash_bits, hash.p, rlist.as<uint32_t>() + 1,
                         rlist.as<uint32_t>(), s);
      }
      launch_dedup_flags(h->ix.d_res.as<uint8_t>(), mkey[sorted].as<uint64_t>(), idx[0].as<uint32_t>(), hash.p,
                         hash_bits, r.gpos, r.len, N, flags.as<uint8_t>(), tile_counts.as<uint32_t>(),
                         h->d_err.as<uint32_t>(), s);
      launch_scan_u32_to_u64(tile_counts.as<uint32_t>(), tiles, tile_offs.as<uint64_t>(), s);
      n_unique = read_u64(h, tile_offs.as<uint64_t>() + tiles);
      // K8r streams the keys and indices (the hashing of run members is not counted); K8 flags
      h->st.algo_bytes[DBI_STAGE_DEDUP] += (run_order ? N * (8 + 4) : 0) + N * (8 + 4 + 1);
    }
    const uint32_t e = read_err(h);
    TR("ir_sort+flags+sync");
    if (e & kErrHashCollision) {
      // two different sequences with equal mass bits and equal hash: re-order the runs with another
      // seed and a wider hash (on the K8r path the mass sort stays valid)
      h->st.n_hash_retries++;
      const uint32_t cleared = e & ~kErrHashCollision;
      DBI_CUDA(cudaMemcpyAsync(h->d_err.p, &cleared, 4, cudaMemcpyHostToDevice, s));
      DBI_CUDA(cudaStreamSynchronize(s));
      if (attempt >= 8) {
        set_error("sequence-hash collisions persist after %u re-seeds (%d hash bits)", attempt, hash_bits);
        return DBI_ERANGE;
      }
      hash_bits = std::min(64, std::max(hash_bits + 8, 40));
      continue;
    }
    break;
  }
  {
    Stage sg(h, DBI_STAGE_DEDUP);
    h->cnt.n_unique = n_unique;
    h->st.n_unique = n_unique;
    h->ix.u_mass.alloc(n_unique * 8, h->arena);
    if (h->rt.mg_world > 1) {  // the other ranks read these through their mapping of window 2
      const UniqLayout L(h->rt.uniq_cap[h->rt.mg_rank]);
      uint8_t* base = (uint8_t*)h->win[2].p;
      if (!base || h->win[2].cap < L.total || h->rt.uniq_cap[h->rt.mg_rank] < N) {
        set_error("window 2 (unique tables) is smaller than the %llu records delivered", (unsigned long long)N);
        return DBI_EINVAL;
      }
      h->ix.u_gpos.borrow(base + L.gpos, n_unique * 4);
      h->ix.u_prot.borrow(base + L.prot, n_unique * 4);
      h->ix.u_len.borrow(base + L.len, n_unique * 2);
      h->ix.u_plo.borrow(base + L.plo, (n_unique + 1) * 8);
      h->ix.plist.borrow(base + L.plist, N * 4);
    } else {
      h->ix.u_gpos.alloc(n_unique * 4, h->arena);
      h->ix.u_prot.alloc(n_unique * 4, h->arena);
      h->ix.u_len.alloc(n_unique * 2, h->arena);
      h->ix.u_plo.alloc((n_unique + 1) * 8, h->arena);
      h->ix.plist.alloc(N * 4, h->arena);
    }
    launch_dedup_emit(mkey[sorted].as<uint64_t>(), idx[0].as<uint32_t>(), flags.as<uint8_t>(),
                      tile_offs.as<uint64_t>(), r.gpos, r.prot, r.len, N, base_bits, n_unique,
                      h->ix.u_mass.as<double>(), h->ix.u_gpos.as<uint32_t>(), h->ix.u_prot.as<uint32_t>(),
                      h->ix.u_len.as<uint16_t>(), h->ix.u_plo.as<uint64_t>(), h->ix.plist.as<uint32_t>(), s);
    h->st.algo_bytes[DBI_STAGE_DEDUP] += N * (1 + 4 + 4 + 4) + n_unique * (8 + 4 + 4 + 2 + 8 + 10);
  }
  TR("ir_dedup_emit");
  return DBI_OK;
}

// K5 + K6 over base tiles [tile0, tile0 + ntiles) of the unique tables: (key, payload) pairs of
// every variant into freshly allocated vkey / vpay; *V = how many.
int emit_variants(dbi_handle* h, uint32_t tile0, uint32_t ntiles, const KeySpace& ks, DevBuf& vkey, DevBuf& vpay,
                  uint64_t* V_out) {
  cudaStream_t s = h->stream;
  const uint64_t n_unique = h->cnt.n_unique;
  *V_out = 0;
  if (ntiles == 0 || n_unique == 0) {
    vkey.alloc(8, h->arena);
    vpay.alloc(8, h->arena);
    return DBI_OK;
  }
  DevBuf counts, ucounts, uoffs;
  counts.alloc(n_unique * 4, h->arena);  // indexed by global base id
  ucounts.alloc((uint64_t)ntiles * 4, h->arena);
  uoffs.alloc(((uint64_t)ntiles + 1) * 8, h->arena);
  const uint64_t n_in_tiles = std::min<uint64_t>((uint64_t)ntiles * kModTile, n_unique - (uint64_t)tile0 * kModTile);
  uint64_t V = 0;
  {
    Stage sg(h, DBI_STAGE_MOD_COUNT);
    launch_mod_count(h->ix.d_res.as<uint8_t>(), h->d_tables.as<DevTables>(), h->cfg, h->ix.u_mass.as<double>(),
                     h->ix.u_gpos.as<uint32_t>(), h->ix.u_len.as<uint16_t>(), n_unique, tile0, ntiles,
                     counts.as<uint32_t>(), ucounts.as<uint32_t>(), h->d_err.as<uint32_t>(), s);
    launch_scan_u32_to_u64(ucounts.as<uint32_t>(), ntiles, uoffs.as<uint64_t>(), s);
    V = read_u64(h, uoffs.as<uint64_t>() + ntiles);
    h->st.algo_bytes[DBI_STAGE_MOD_COUNT] += n_in_tiles * (8 + 4 + 2 + 4 + 20);
  }
  if (int rc = check_err_bits(read_err(h))) return rc;
  TR("ir_modcount+sync");
  vkey.alloc(V * 8, h->arena);
  vpay.alloc(V * 8, h->arena);
  TR("ir_valloc");
  {
    Stage sg(h, DBI_STAGE_MOD_EMIT);
    launch_mod_emit(h->ix.d_res.as<uint8_t>(), h->d_tables.as<DevTables>(), h->cfg, h->ix.u_mass.as<double>(),
                    h->ix.u_gpos.as<uint32_t>(), h->ix.u_len.as<uint16_t>(), n_unique, tile0, ntiles,
                    counts.as<uint32_t>(), uoffs.as<uint64_t>(), ks.base_bits, h->rt.ent_base_off, vkey.as<uint64_t>(),
                    vpay.as<uint64_t>(), s);
    h->st.algo_bytes[DBI_STAGE_MOD_EMIT] += n_in_tiles * (8 + 4 + 2 + 4 + 20) + V * 16;
  }
  TR("ir_modemit");
  *V_out = V;
  return DBI_OK;
}

// K7 on V (key, payload) variant pairs (clobbered) -> the handle's entry arrays.
int sort_variants(dbi_handle* h, uint64_t* key_in, uint64_t* pay_in, uint64_t V, const KeySpace& ks) {
  cudaStream_t s = h->stream;
  if (V >= (1ull << 32)) {
    set_error("more than 2^32 index entries on one GPU (%llu)", (unsigned long long)V);
    return DBI_ERANGE;
  }
  DevBuf key2, pay2, vtmp;
  key2.alloc(V * 8, h->arena);
  pay2.alloc(V * 8, h->arena);
  vtmp.alloc(radix_sort_tmp_bytes(V), h->arena);
  h->ix.e_mass.alloc(V * 8, h->arena);
  h->ix.e_base.alloc(V * 4, h->arena);
  h->ix.e_pat.alloc(V * 4, h->arena);
  TR("ir_ealloc");
  {
    // the last pass of the sort writes the final entry arrays (mass, base id, mod pattern)
    Stage sg(h, DBI_STAGE_SORT_VAR);
    uint64_t* vk[2] = {key_in, key2.as<uint64_t>()};
    uint64_t* vp[2] = {pay_in, pay2.as<uint64_t>()};
    DomProbe var_probe(h);
    if (h->p.profile) {
      h->st.dom_kernel = 1;
      h->st.dom_bytes_per_launch = V * 32ull;
    }
    SplitOut<uint64_t> split{h->ix.e_mass.as<uint64_t>(), ks.base_bits, h->ix.e_base.as<uint32_t>(),
                             h->ix.e_pat.as<uint32_t>()};
    const int passes = (ks.nbits + 7) / 8;
    if (V > 1 && passes > 0) {
      radix_sort_pairs<uint64_t, uint64_t>(vk, vp, V, 0, ks.nbits, vtmp.p, s, h->p.profile ? &var_probe : nullptr, &split);
    } else {  // nothing to sort: plain split
      launch_split_entries(vk[0], vp[0], V, ks.base_bits, h->ix.e_mass.as<double>(), h->ix.e_base.as<uint32_t>(),
                           h->ix.e_pat.as<uint32_t>(), s);
    }
    h->st.sort_bits_var = (uint32_t)ks.nbits;
    h->st.algo_bytes[DBI_STAGE_SORT_VAR] += V * 8 + V * 32ull * passes;
  }
  TR("ir_sortvar");
  h->cnt.n_entries = V;
  h->st.n_entries = V;
  return DBI_OK;
}

// Group path (class sequences <= 32): K5m + K5g + K6g over base tiles [tile0, tile0 + ntiles): one
// {key, payload} record per (peptide, class sequence) group.  *NG = groups, *V = variants.
constexpr uint64_t kGrpCntMask = (1ull << 27) - 1;

// K5m over the whole unique table (once per table: the multi-GPU build replaces the table).
void ensure_site_masks(dbi_handle* h) {
  if (h->cnt.cmask_n == h->cnt.n_unique && h->ix.u_cmask.p) return;
  Stage sg(h, DBI_STAGE_MOD_COUNT);
  h->ix.u_cmask.alloc(std::max<uint64_t>(1, h->cnt.n_unique) * (uint64_t)h->cfg.n_classes * 8, h->arena);
  h->ix.d_nlong.alloc(16, h->arena);
  DBI_CUDA(cudaMemsetAsync(h->ix.d_nlong.p, 0, 16, h->stream));
  launch_site_masks(h->ix.d_res.as<uint8_t>(), h->d_tables.as<DevTables>(), h->cfg, h->ix.u_gpos.as<uint32_t>(),
                    h->ix.u_len.as<uint16_t>(), h->cnt.n_unique, h->ix.u_cmask.as<uint64_t>(),
                    (unsigned long long*)h->ix.d_nlong.p, h->stream);
  h->cnt.cmask_n = h->cnt.n_unique;
  h->st.algo_bytes[DBI_STAGE_MOD_COUNT] += h->cnt.n_unique * (4 + 2 + 12 + 8ull * h->cfg.n_classes);
}

// lists != nullptr (single GPU): K6g writes one sorted list per class sequence, described in *lists (the
// input of K7m); nullptr (sharded build): peptide-major records, sorted after the exchange by K7.
int emit_groups(dbi_handle* h, uint32_t tile0, uint32_t ntiles, const KeySpace& ks, DevBuf& gkey, DevBuf& gpay,
                uint64_t* NG_out, uint64_t* V_out, GroupLists* lists = nullptr) {
  cudaStream_t s = h->stream;
  const uint64_t n_unique = h->cnt.n_unique;
  const int S = h->cfg.n_seq;
  *NG_out = 0;
  *V_out = 0;
  if (lists) {
    std::memset(lists, 0, sizeof(*lists));
    lists->n_lists = S;
  }
  if (ntiles == 0 || n_unique == 0) {
    gkey.alloc(8, h->arena);
    gpay.alloc(8, h->arena);
    return DBI_OK;
  }
  ensure_site_masks(h);
  DevBuf mask, tg, tv, goffs, voffs, vt, vtmp;
  mask.alloc(n_unique * 4, h->arena);  // indexed by global peptide id
  tg.alloc((uint64_t)ntiles * 4, h->arena);
  tv.alloc((uint64_t)ntiles * 4, h->arena);
  voffs.alloc(((uint64_t)ntiles + 1) * 8, h->arena);
  const uint64_t n_vt = (uint64_t)S * ntiles;  // list layout: (class sequence, tile) counts, v-major
  if (lists) {
    vt.alloc(n_vt * 4, h->arena);
    goffs.alloc((n_vt + 1) * 8, h->arena);
    vtmp.alloc(full_scan_tmp_bytes(n_vt), h->arena);
  } else {
    goffs.alloc(((uint64_t)ntiles + 1) * 8, h->arena);
  }
  const uint64_t n_in_tiles = std::min<uint64_t>((uint64_t)ntiles * kModTile, n_unique - (uint64_t)tile0 * kModTile);
  const uint64_t per_pep = 8 + 4 + 2 + 4 + 8ull * h->cfg.n_classes;
  uint64_t NG = 0, V = 0;
  {
    Stage sg(h, DBI_STAGE_MOD_COUNT);
    launch_grp_count(h->ix.d_res.as<uint8_t>(), h->d_tables.as<DevTables>(), h->cfg, h->ix.u_mass.as<double>(),
                     h->ix.u_gpos.as<uint32_t>(), h->ix.u_len.as<uint16_t>(), h->ix.u_cmask.as<uint64_t>(), n_unique,
                     tile0, ntiles, mask.as<uint32_t>(), tg.as<uint32_t>(), tv.as<uint32_t>(),
                     lists ? vt.as<uint32_t>() : nullptr, h->d_err.as<uint32_t>(), s);
    if (lists) launch_full_scan_u32_to_u64(vt.as<uint32_t>(), n_vt, goffs.as<uint64_t>(), vtmp.p, s);
    else launch_scan_u32_to_u64(tg.as<uint32_t>(), ntiles, goffs.as<uint64_t>(), s);
    launch_scan_u32_to_u64(tv.as<uint32_t>(), ntiles, voffs.as<uint64_t>(), s);
    uint32_t e = 0;
    if (lists)  // list v starts at goffs[v * ntiles]; goffs[S * ntiles] = NG
      DBI_CUDA(cudaMemcpy2DAsync(lists->start, 8, goffs.p, (size_t)ntiles * 8, 8, (size_t)S + 1,
                                 cudaMemcpyDeviceToHost, s));
    else
      DBI_CUDA(cudaMemcpyAsync(&NG, goffs.as<uint64_t>() + ntiles, 8, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaMemcpyAsync(&V, voffs.as<uint64_t>() + ntiles, 8, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaMemcpyAsync(&e, h->d_err.p, 4, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaStreamSynchronize(s));
    if (lists) {
      NG = lists->start[S];
      group_lists_plan(lists);
    }
    h->st.algo_bytes[DBI_STAGE_MOD_COUNT] += n_in_tiles * per_pep + (lists ? n_vt * (4 + 8) : 0);
    if (int rc = check_err_bits(e)) return rc;
  }
  TR("ir_modcount+sync");
  gkey.alloc(NG * 8, h->arena);
  gpay.alloc(NG * 8, h->arena);
  TR("ir_valloc");
  {
    Stage sg(h, DBI_STAGE_MOD_EMIT);
    launch_grp_emit(h->ix.d_res.as<uint8_t>(), h->d_tables.as<DevTables>(), h->cfg, h->ix.u_mass.as<double>(),
                    h->ix.u_gpos.as<uint32_t>(), h->ix.u_len.as<uint16_t>(), h->ix.u_cmask.as<uint64_t>(), n_unique,
                    tile0, ntiles, mask.as<uint32_t>(), goffs.as<uint64_t>(), lists != nullptr, ks.base_bits,
                    h->rt.ent_base_off, gkey.as<uint64_t>(), gpay.as<uint64_t>(), h->d_err.as<uint32_t>(), s);
    h->st.algo_bytes[DBI_STAGE_MOD_EMIT] += n_in_tiles * per_pep + NG * 16;
  }
  TR("ir_modemit");
  *NG_out = NG;
  *V_out = V;
  return DBI_OK;
}

// K7 on NG group records (clobbered), then K6x: expand the sorted groups into the entry arrays.
// side (sharded build): the groups arrived from any rank; their payload names an ARRIVAL ROW, and the
// row's site masks / peptide global id travelled with the group (side tables in the arena).
struct GroupSide {
  const uint64_t* cmask = nullptr;   // [row * C + c]
  const uint32_t* gid = nullptr;     // [row]
  const UniqView* uv = nullptr;      // where the peptides' (gpos, len) live: only peptides longer than 64 residues need it
};
// lists (single GPU, K6g's list layout): K7m merges the lists instead of the sort.
// in_bufs (single GPU): the buffers of key_in / pay_in, which a compact index keeps when they hold the result.
int sort_expand_groups(dbi_handle* h, uint64_t* key_in, uint64_t* pay_in, uint64_t NG, const KeySpace& ks,
                       const GroupSide* side = nullptr, const GroupLists* lists = nullptr,
                       DevBuf* const* in_bufs = nullptr) {
  cudaStream_t s = h->stream;
  if (NG >= (1ull << 32)) {
    set_error("more than 2^32 variant groups on one GPU (%llu)", (unsigned long long)NG);
    return DBI_ERANGE;
  }
  if (NG == 0) {
    h->ix.e_mass.alloc(8, h->arena); h->ix.e_base.alloc(8, h->arena); h->ix.e_pat.alloc(8, h->arena);
    h->cnt.n_entries = 0;
    h->st.n_entries = 0;
    return DBI_OK;
  }
  const bool sharded = side != nullptr;
  if (!sharded) ensure_site_masks(h);
  DevBuf key2, pay2, vtmp, cnt;
  key2.alloc(NG * 8, h->arena);
  pay2.alloc(NG * 8, h->arena);
  cnt.alloc(NG * 4, h->arena);
  uint64_t* vk[2] = {key_in, key2.as<uint64_t>()};
  uint64_t* vp[2] = {pay_in, pay2.as<uint64_t>()};
  int r = 0;
  if (lists) {
    vtmp.alloc(group_merge_tmp_bytes(*lists), h->arena);
    Stage sg(h, DBI_STAGE_SORT_VAR);
    launch_group_merge(*lists, key_in, pay_in, vk[1], vp[1], cnt.as<uint32_t>(), vtmp.p, h->d_err.as<uint32_t>(), s);
    r = 1;
    h->st.sort_bits_var = 0;
    // records read once, written once with their count; samples gathered, ranked and searched in L2
    const uint64_t ns = lists->soff[lists->n_lists];
    h->st.algo_bytes[DBI_STAGE_SORT_VAR] += NG * (16 + 20) + ns * 16 * 2;
  } else {
    vtmp.alloc(radix_sort_tmp_bytes(NG), h->arena);
    Stage sg(h, DBI_STAGE_SORT_VAR);
    DomProbe var_probe(h);
    if (h->p.profile) {
      h->st.dom_kernel = 1;
      h->st.dom_bytes_per_launch = NG * 32ull;
    }
    r = radix_sort_pairs<uint64_t, uint64_t>(vk, vp, NG, 0, ks.nbits, vtmp.p, s, h->p.profile ? &var_probe : nullptr);
    h->st.sort_bits_var = (uint32_t)ks.nbits;
    h->st.algo_bytes[DBI_STAGE_SORT_VAR] += NG * 8 + NG * 32ull * ((ks.nbits + 7) / 8);
  }
  TR("ir_sortvar");
  DevBuf eoff, stmp, tfirst, llist, lcount;
  eoff.alloc((NG + 1) * 8, h->arena);
  stmp.alloc(full_scan_tmp_bytes(NG), h->arena);
  lcount.alloc(16, h->arena);
  uint64_t V = 0, n_long = 0;
  {
    Stage sg(h, DBI_STAGE_GATHER_VAR);
    if (!lists) launch_grp_extract_cnt(vp[r], NG, cnt.as<uint32_t>(), s);  // K7m wrote the counts
    launch_full_scan_u32_to_u64(cnt.as<uint32_t>(), NG, eoff.as<uint64_t>(), stmp.p, s);
    DBI_CUDA(cudaMemsetAsync(lcount.p, 0, 16, s));
    DBI_CUDA(cudaMemcpyAsync(&V, eoff.as<uint64_t>() + NG, 8, cudaMemcpyDeviceToHost, s));
    if (!sharded) DBI_CUDA(cudaMemcpyAsync(&n_long, h->ix.d_nlong.p, 8, cudaMemcpyDeviceToHost, s));
    uint32_t e = 0;
    DBI_CUDA(cudaMemcpyAsync(&e, h->d_err.p, 4, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaStreamSynchronize(s));
    if (e & kErrMergeCap) {
      set_error("a tile of the group merge exceeds its capacity of %d records",
                (kGmSplit + kGrpMaxLists) * kGmStride);
      return DBI_ERANGE;
    }
    if (sharded) n_long = NG;  // unknown here: any received group may belong to a long peptide
    if (!sharded && in_bufs && (V >= (1ull << 32) || compact_variants(h))) {
      // compact layout: keep the sorted groups, their masses and entry offsets; queries expand what they return
      launch_grp_key_mass(vk[r], NG, ks.base_bits, s);
      h->ix.g_mass.swap(r ? key2 : *in_bufs[0]);
      h->ix.g_pay.swap(r ? pay2 : *in_bufs[1]);
      h->ix.g_eoff.swap(eoff);
      h->ix.e_mass.release(); h->ix.e_base.release(); h->ix.e_pat.release();
      h->cnt.n_groups = NG;
      h->cnt.n_long = n_long;
      h->st.n_groups = (uint32_t)NG;
      h->st.algo_bytes[DBI_STAGE_GATHER_VAR] += NG * ((lists ? 0 : 8 + 4) + 16);
      h->cnt.n_entries = V;
      h->st.n_entries = V;
      return DBI_OK;
    }
    if (V >= (1ull << 32)) {
      set_error("more than 2^32 index entries on one GPU (%llu)", (unsigned long long)V);
      return DBI_ERANGE;
    }
    // groups of long peptides that can land here: at most every modified class sequence of each
    const uint64_t long_cap = std::min<uint64_t>(sharded ? std::min<uint64_t>(NG, 1u << 22) : NG,
                                                 n_long * (uint64_t)(h->cfg.n_seq - 1));
    const uint64_t tiles = (V + kExpTile - 1) / kExpTile;
    h->ix.e_mass.alloc(V * 8, h->arena);
    h->ix.e_base.alloc(V * 4, h->arena);
    h->ix.e_pat.alloc(V * 4, h->arena);
    tfirst.alloc((tiles + 1) * 4, h->arena);
    llist.alloc(std::max<uint64_t>(1, long_cap) * 4, h->arena);
    TR("ir_ealloc");
    launch_grp_tile_first(eoff.as<uint64_t>(), NG, V, tfirst.as<uint32_t>(), s);
    cudaEvent_t xa = nullptr;
    if (h->p.profile) {
      xa = h->get_event();
      cudaEventRecord(xa, s);
    }
    launch_grp_expand(h->ix.d_res.as<uint8_t>(), h->d_tables.as<DevTables>(), h->cfg, h->ix.u_gpos.as<uint32_t>(),
                      h->ix.u_len.as<uint16_t>(), sharded ? side->cmask : h->ix.u_cmask.as<uint64_t>(),
                      sharded ? side->gid : nullptr, sharded ? side->uv : nullptr, vk[r], vp[r], eoff.as<uint64_t>(),
                      tfirst.as<uint32_t>(), NG, V, ks.base_bits, h->ix.e_mass.as<double>(),
                      h->ix.e_base.as<uint32_t>(), h->ix.e_pat.as<uint32_t>(), llist.as<uint32_t>(),
                      lcount.as<uint32_t>(), (uint32_t)long_cap, h->d_err.as<uint32_t>(), s);
    if (h->p.profile) {
      cudaEvent_t xb = h->get_event();
      cudaEventRecord(xb, s);
      h->spans.push_back({kSpanExpand, xa, xb});
      // per group: offset + key + payload + tile bookkeeping read, <= max_mods site masks gathered;
      // per entry: mass + peptide + pattern written
      h->st.exp_bytes_per_launch = NG * (8 + 8 + 8 + 8ull * h->cfg.max_mods) + V * 16;
    }
    h->st.algo_bytes[DBI_STAGE_GATHER_VAR] +=
        NG * ((lists ? 0 : 8 + 4) + 8 + 8 + 8 + 8ull * h->cfg.max_mods) + V * 16;
  }
  TR("ir_expand");
  h->cnt.n_entries = V;
  h->st.n_entries = V;
  return DBI_OK;
}

// Single-GPU: sort + merge + (mods) expand + sort on N emitted records already on the device.
// lo_mass / hi_mass bound every record mass (they fix the radix key width).
int index_records(dbi_handle* h, const RecView& r, uint64_t N, double lo_mass, double hi_mass) {
  h->cnt.n_emitted = N;
  h->st.n_emitted = N;
  const KeySpace ks(lo_mass, hi_mass);
  h->st.n_groups = 0;  // set again if the build keeps the compact layout
  if (int rc = sort_dedup(h, r, N, ks)) return rc;
  h->rt.ent_base_off = 0;
  if (h->cfg.max_mods == 0 || h->cnt.n_unique == 0) {
    h->cnt.n_entries = h->cnt.n_unique;
    h->st.n_entries = h->cnt.n_unique;
    h->built = true;
    return DBI_OK;
  }
  const uint32_t utiles = (uint32_t)((h->cnt.n_unique + kModTile - 1) / kModTile);
  DevBuf vkey, vpay;
  uint64_t V = 0, NG = 0;
  if (h->cfg.n_seq > 0) {  // group path: one record per (peptide, class sequence), merged from sorted lists
    GroupLists lists;
    GroupLists* gl = group_radix(h) ? nullptr : &lists;
    if (int rc = emit_groups(h, 0, utiles, ks, vkey, vpay, &NG, &V, gl)) return rc;
    DevBuf* in_bufs[2] = {&vkey, &vpay};
    if (int rc = sort_expand_groups(h, vkey.as<uint64_t>(), vpay.as<uint64_t>(), NG, ks, nullptr, gl, in_bufs)) return rc;
  } else {  // many shift classes: one record per variant
    if (int rc = emit_variants(h, 0, utiles, ks, vkey, vpay, &V)) return rc;
    if (int rc = sort_variants(h, vkey.as<uint64_t>(), vpay.as<uint64_t>(), V, ks)) return rc;
  }
  h->built = true;
  return DBI_OK;
}

void finish_stats(dbi_handle* h) {
  resolve_spans(h);
  h->st.device_bytes = 0;
  for (const auto& b : kIndexBufs)
    if (b.use != kUncounted && (b.use != kCompact || h->cnt.n_groups))
      h->st.device_bytes += (h->ix.*b.buf).bytes;
}

// The end of a single-GPU build: the index of the N records in recs, whose masses lie in [lo_mass, hi_mass].  A
// failure leaves the handle unbuilt with its proteins; params.keep_emitted keeps the records.
int build_end(dbi_handle* h, RecSet& recs, uint64_t N, double lo_mass, double hi_mass) {
  int rc = index_records(h, recs.view(), N, lo_mass, hi_mass);
  TR("index_records");
  if (rc == DBI_OK) rc = check_err_bits(read_err(h));
  if (rc != DBI_OK) {
    free_index(h);
    return rc;
  }
  if (h->p.keep_emitted) h->kept.swap(recs);
  DBI_CUDA(cudaStreamSynchronize(h->stream));
  finish_stats(h);
  TR("final_sync");
  return DBI_OK;
}

// The unique-peptide tables a fetch resolves base peptides through: this GPU's own, and in a
// sharded build the mapped tables of every connected rank.
UniqView uniq_view(dbi_handle* h) {
  UniqView uv;
  std::memset(&uv, 0, sizeof(uv));
  if (h->rt.mg_world <= 1) {
    uv.world = 1;
    uv.gpos[0] = h->ix.u_gpos.as<uint32_t>();
    uv.prot[0] = h->ix.u_prot.as<uint32_t>();
    uv.len[0] = h->ix.u_len.as<uint16_t>();
    uv.plo[0] = h->ix.u_plo.as<uint64_t>();
    uv.plist[0] = h->ix.plist.as<uint32_t>();
    uv.uoff[0] = 0;
    uv.uoff[1] = h->cnt.n_unique;
    return uv;
  }
  uv.world = h->rt.mg_world;
  for (int r = 0; r < h->rt.mg_world; ++r) {
    uv.uoff[r] = h->rt.uoff[r];
    uint8_t* base = (uint8_t*)h->rt.win[2].peer[r];
    if (!base) continue;  // not connected: its peptides come back as DBI_REMOTE_BASE
    const UniqLayout L(h->rt.uniq_cap[r]);
    uv.gpos[r] = (const uint32_t*)(base + L.gpos);
    uv.prot[r] = (const uint32_t*)(base + L.prot);
    uv.len[r] = (const uint16_t*)(base + L.len);
    uv.plo[r] = (const uint64_t*)(base + L.plo);
    uv.plist[r] = (const uint32_t*)(base + L.plist);
  }
  uv.uoff[h->rt.mg_world] = h->rt.uoff[h->rt.mg_world];
  return uv;
}

// K9 over the handle's masses: entry ranges [d_b, d_b + d_c).  On a compact index K9 finds group ranges,
// which become entry ranges through g_eoff; cnt32 / ntile32 / over as in launch_grp_entry_ranges.
void query_ranges(dbi_handle* h, const double* d_lo, const double* d_hi, uint64_t nq, uint64_t* d_b, uint64_t* d_c,
                  uint32_t* cnt32, uint32_t* ntile32 = nullptr, uint32_t* over = nullptr) {
  launch_query(h->key_mass(), h->n_keys(), d_lo, d_hi, nq, d_b, d_c, h->cnt.n_groups ? nullptr : cnt32, h->stream);
  h->st.algo_bytes[DBI_STAGE_QUERY] += nq * (32 + 2ull * 32 * (uint64_t)bit_length(h->n_keys()));
  if (h->cnt.n_groups) {
    launch_grp_entry_ranges(h->ix.g_eoff.as<uint64_t>(), nq, d_b, d_c, cnt32, ntile32, over, h->stream);
    h->st.algo_bytes[DBI_STAGE_QUERY] += nq * (16 + 2 * 32 + 16 + (cnt32 ? 4 : 0) + (ntile32 ? 4 : 0));
  }
}

// K6q and the windowed K6l: the entries of the ranges rg (n_tiles tiles, n_out entries) of a compact index into
// x_mass / x_base / x_pat, in output order.  The groups of long peptides are listed per (group, tile); a
// proteome without peptides over 64 residues reads nothing back.
void expand_ranges(dbi_handle* h, const ExpRanges& rg, uint64_t n_tiles, uint64_t n_out, DevBuf& x_mass,
                   DevBuf& x_base, DevBuf& x_pat) {
  cudaStream_t s = h->stream;
  x_mass.alloc(std::max<uint64_t>(n_out, 1) * 8, h->arena);
  x_base.alloc(std::max<uint64_t>(n_out, 1) * 4, h->arena);
  x_pat.alloc(std::max<uint64_t>(n_out, 1) * 4, h->arena);
  Stage sg(h, DBI_STAGE_FETCH);
  DevBuf lcount, llist;
  lcount.alloc(16, h->arena);
  // one (group, tile) pair per tile is the common case; a tile can hold up to kExpTile + 1 long groups (peptides
  // over 64 residues with few sites), and then the list overflows and the tiles run again with room for all
  uint64_t cap = h->cnt.n_long ? n_tiles + 1024 : 0;
  for (;;) {
    llist.alloc(std::max<uint64_t>(cap, 1) * 8, h->arena);
    DBI_CUDA(cudaMemsetAsync(lcount.p, 0, 4, s));
    launch_grp_expand_ranges(h->cfg, h->ix.u_cmask.as<uint64_t>(), h->ix.g_mass.as<double>(),
                             h->ix.g_pay.as<uint64_t>(), h->ix.g_eoff.as<uint64_t>(), h->cnt.n_groups, rg, n_tiles,
                             x_mass.as<double>(), x_base.as<uint32_t>(), x_pat.as<uint32_t>(), llist.as<uint32_t>(),
                             lcount.as<uint32_t>(), (uint32_t)cap, h->d_err.as<uint32_t>(), s);
    if (!h->cnt.n_long) break;
    uint32_t n_listed = 0;
    DBI_CUDA(cudaMemcpyAsync(&n_listed, lcount.p, 4, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaStreamSynchronize(s));
    if (n_listed <= cap) {
      launch_grp_expand_ranges_long(h->ix.d_res.as<uint8_t>(), h->d_tables.as<DevTables>(), h->cfg,
                                    h->ix.u_gpos.as<uint32_t>(), h->ix.u_len.as<uint16_t>(), h->ix.g_mass.as<double>(),
                                    h->ix.g_pay.as<uint64_t>(), h->ix.g_eoff.as<uint64_t>(), rg, llist.as<uint32_t>(),
                                    lcount.as<uint32_t>(), n_listed, x_mass.as<double>(), x_base.as<uint32_t>(),
                                    x_pat.as<uint32_t>(), s);
      break;
    }
    cap = n_listed;  // the list overflowed: run the tiles again with room for every pair
  }
  // per tile: the range and two searches of g_eoff; per entry 16 written.  The group records a tile reads (offset,
  // mass, payload, site masks; between 1 and kExpTile + 1 of them) are not counted.
  h->st.algo_bytes[DBI_STAGE_FETCH] += n_tiles * (28 + 16ull * (uint64_t)bit_length(h->cnt.n_groups)) + n_out * 16;
}

void mg_release(dbi_handle* h);  // capi_mg.inl

// A view runs the query helpers unchanged: it borrows every index buffer of its owner and copies the scalars that
// describe the index, next to its own stream, arena, d_err, pending results and stats.  The owner is pinned while
// views are open (DBI_MUTATES), so none of this can go stale.  The windows keep only their peer mappings: a view
// reads the other ranks' tables as its owner does, and never hands a window back (mg_release).
void view_share_index(dbi_handle* v, const dbi_handle* o) {
  v->d_tables.borrow(o->d_tables.p, o->d_tables.bytes);
  for (const auto& b : kIndexBufs) (v->ix.*b.buf).borrow((o->ix.*b.buf).p, (o->ix.*b.buf).bytes);
  v->built = o->built;
  v->cnt = o->cnt;
  v->lay = o->lay;
  v->rt = o->rt;
  v->cfg = o->cfg;
  v->shifts = o->shifts;
  // the owner's index counters; the launches, bytes and times are the view's own
  v->st = o->st;
  std::memset(v->st.algo_bytes, 0, sizeof(v->st.algo_bytes));
  std::memset(v->st.stage_ms, 0, sizeof(v->st.stage_ms));
  std::memset(v->st.stage_launches, 0, sizeof(v->st.stage_launches));
  v->st.dom_ms = v->st.exp_ms = 0;
  v->st.dom_launches = v->st.exp_launches = 0;
}

}  // namespace

extern "C" {

int dbi_create(const dbi_params* params, dbi_handle** out) {
  if (!params || !out) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  *out = nullptr;
  if (params->abi_version != DBI_ABI_VERSION) {
    set_error("dbi_params.abi_version %u != %u", params->abi_version, DBI_ABI_VERSION);
    return DBI_EINVAL;
  }
  const dbi_params& p = *params;
  // Constants.MAX_PRECURSOR_MASS = 8000 (Constants.java:20): masses beyond it have no bucket
  // in the reference (DBIndexStoreSQLiteMult.java:282-287)
  if (!(p.min_mass >= 0) || !(p.max_mass >= p.min_mass) || !(p.max_mass <= 8000.0)) {
    set_error("mass range [%g, %g] must satisfy 0 <= min <= max <= 8000", p.min_mass, p.max_mass);
    return DBI_EINVAL;
  }
  if (p.min_len < 1 || p.max_missed < 0 || p.mass_group_factor < 1 || p.n_mods < 0 || p.n_mods > DBI_MAX_MODS ||
      p.max_mods_per_peptide < 0 || p.max_mods_per_peptide > DBI_MAX_MODS_PER_PEP) {
    set_error("parameter out of range (min_len %d, max_missed %d, factor %d, n_mods %d, max_mods_per_peptide %d)",
              p.min_len, p.max_missed, p.mass_group_factor, p.n_mods, p.max_mods_per_peptide);
    return DBI_EINVAL;
  }
  for (int i = 0; i < 256; ++i)
    if (!(p.residue_mass[i] >= 0)) {
      set_error("residue_mass[%d] is negative or NaN", i);
      return DBI_EINVAL;
    }
  dbi_handle* h = nullptr;
  try {
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev <= 0 || p.device < 0 || p.device >= ndev) {
      set_error("no usable CUDA device (count %d, requested %d): %s; this library has no CPU fallback", ndev,
                p.device, cudaGetErrorString(ce));
      cudaGetLastError();
      return DBI_ECUDA;
    }
    h = new dbi_handle();
    h->p = p;
    h->device = p.device;
    DBI_CUDA(cudaSetDevice(h->device));
    DBI_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    h->arena.device = h->device;
    h->d_err.alloc(4, h->arena);
    DBI_CUDA(cudaMemsetAsync(h->d_err.p, 0, 4, h->stream));
    upload_tables(h);
    *out = h;
    return DBI_OK;
  } catch (const CudaError& e) {
    delete h;
    return fail_cuda(e);
  } catch (const std::bad_alloc&) {
    delete h;
    set_error("host allocation failed");
    return DBI_ENOMEM;
  }
}

int dbi_view_open(dbi_handle* h, dbi_handle** view) {
  if (!view) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  *view = nullptr;
  DBI_API_BEGIN(h)
  if (h->owner) {
    set_error("a view of a view: open views on the owner");
    return DBI_EINVAL;
  }
  if (!h->built) {
    set_error("Indexer is not initialized: a view needs a built index");
    return DBI_ENOTINIT;
  }
  dbi_handle* v = new dbi_handle();
  try {
    v->p = h->p;
    v->device = h->device;
    DBI_CUDA(cudaStreamCreateWithFlags(&v->own_stream, cudaStreamNonBlocking));
    v->stream = v->own_stream;
    v->arena.device = v->device;
    v->d_err.alloc(4, v->arena);
    DBI_CUDA(cudaMemsetAsync(v->d_err.p, 0, 4, v->stream));
    DBI_CUDA(cudaStreamSynchronize(v->stream));
  } catch (...) {
    dbi_destroy(v);  // nothing borrowed yet: torn down like a fresh handle
    throw;
  }
  view_share_index(v, h);
  v->owner = h;
  {
    std::lock_guard<std::mutex> lk(h->view_mu);
    h->n_views.fetch_add(1);
  }
  *view = v;
  return DBI_OK;
  DBI_API_END
}

int dbi_set_stream(dbi_handle* h, void* cuda_stream) {
  DBI_API_BEGIN(h)
  DBI_CUDA(cudaStreamSynchronize(h->stream));
  h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
  return DBI_OK;
  DBI_API_END
}

int dbi_add_proteins(dbi_handle* h, const uint8_t* residues, const uint64_t* offsets, uint32_t n) {
  DBI_API_BEGIN(h)
  DBI_MUTATES(h)
  if (h->built) {
    set_error("index already built");  // "Already intialized", DBIndexStoreSQLiteMult.java:97-99
    return DBI_EALREADY;
  }
  if (n == 0) return DBI_OK;
  if (!residues || !offsets) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  for (uint32_t i = 0; i < n; ++i)
    if (offsets[i + 1] < offsets[i]) {
      set_error("offsets must be non-decreasing (protein %u)", i);
      return DBI_EINVAL;
    }
  const uint64_t add = offsets[n] - offsets[0];
  const uint64_t total_res = h->n_res + add;
  const uint64_t total_prot = h->h_off.size() - 1 + n;
  if (total_res + total_prot + 1 + 4096 >= (1ull << 32) || total_prot >= (1ull << 31)) {
    set_error("more than 2^32 residues on one GPU: shard the FASTA across handles");
    return DBI_ERANGE;
  }
  const uint64_t base = h->n_res;
  cudaStream_t s = h->stream;
  if (total_res > h->d_raw.bytes) {  // grow geometrically; the residues added so far move over
    DevBuf bigger;
    bigger.alloc(std::max<uint64_t>(total_res, h->d_raw.bytes + h->d_raw.bytes / 2), h->arena);
    if (base) DBI_CUDA(cudaMemcpyAsync(bigger.p, h->d_raw.p, base, cudaMemcpyDeviceToDevice, s));
    h->d_raw.swap(bigger);
  }
  // DMA straight from the caller's buffer (pinned memory makes it asynchronous) while the host
  // appends the offsets; the buffer is the caller's again when this call returns
  if (add)
    DBI_CUDA(cudaMemcpyAsync((uint8_t*)h->d_raw.p + base, residues + offsets[0], add, cudaMemcpyHostToDevice, s));
  h->h_off.reserve(h->h_off.size() + n);
  for (uint32_t i = 1; i <= n; ++i) h->h_off.push_back(base + (offsets[i] - offsets[0]));
  // the host copy behind dbi_get_protein is rebuilt on demand: pointers handed out before this call end here
  h->h_raw_valid = false;
  h->n_res = total_res;
  DBI_CUDA(cudaStreamSynchronize(s));
  h->st.n_proteins = total_prot;
  h->st.n_residues = total_res;
  return DBI_OK;
  DBI_API_END
}

int dbi_upload(dbi_handle* h) {
  DBI_API_BEGIN(h)
  DBI_MUTATES(h)
  ensure_uploaded(h);
  DBI_CUDA(cudaStreamSynchronize(h->stream));
  return DBI_OK;
  DBI_API_END
}

int dbi_reset_index(dbi_handle* h) {
  DBI_API_BEGIN(h)
  DBI_MUTATES(h)
  free_index(h);
  DBI_CUDA(cudaStreamSynchronize(h->stream));
  return DBI_OK;
  DBI_API_END
}

int dbi_build(dbi_handle* h) {
  DBI_API_BEGIN(h)
  DBI_MUTATES(h)
  if (h->built) {
    set_error("index already built");
    return DBI_EALREADY;
  }
  TR("begin");
  build_begin(h);
  TR("pack");
  Digest dg = whole_digest(h, nullptr);
  const uint64_t N = dg.count();
  if (int rc = check_err_bits(read_err(h))) {
    free_index(h);
    return rc;
  }
  TR("count+sync");
  RecSet recs;
  dg.emit(recs, nullptr);
  TR("emit");
  if (int rc = build_end(h, recs, N, h->p.min_mass, h->p.max_mass)) return rc;
  g_trace.dump();
  return DBI_OK;
  DBI_API_END
}

int dbi_build_from_records(dbi_handle* h, const double* mass, const uint32_t* prot, const uint32_t* off,
                           const uint16_t* len, uint64_t n) {
  DBI_API_BEGIN(h)
  DBI_MUTATES(h)
  if (h->built) {
    set_error("index already built");
    return DBI_EALREADY;
  }
  if (n && (!mass || !prot || !off || !len)) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  cudaStream_t s = h->stream;
  const uint32_t n_prot = (uint32_t)(h->h_off.size() - 1);
  double lo = 0, hi = 0;
  std::vector<uint32_t> gpos(n);
  for (uint64_t i = 0; i < n; ++i) {
    if (prot[i] >= n_prot || (uint64_t)off[i] + len[i] > h->h_off[prot[i] + 1] - h->h_off[prot[i]] || !(mass[i] >= 0)) {
      set_error("record %llu does not lie inside protein %u (or negative mass)", (unsigned long long)i, prot[i]);
      return DBI_EINVAL;
    }
    gpos[i] = (uint32_t)(h->h_off[prot[i]] + prot[i] + 1 + off[i]);
    lo = i ? std::min(lo, mass[i]) : mass[i];
    hi = i ? std::max(hi, mass[i]) : mass[i];
  }
  build_begin(h);
  RecSet recs;
  recs.alloc(n, h->arena);
  if (n) {
    DBI_CUDA(cudaMemcpyAsync(recs.mass.p, mass, n * 8, cudaMemcpyHostToDevice, s));
    DBI_CUDA(cudaMemcpyAsync(recs.gpos.p, gpos.data(), n * 4, cudaMemcpyHostToDevice, s));
    DBI_CUDA(cudaMemcpyAsync(recs.prot.p, prot, n * 4, cudaMemcpyHostToDevice, s));
    DBI_CUDA(cudaMemcpyAsync(recs.len.p, len, n * 2, cudaMemcpyHostToDevice, s));
    DBI_CUDA(cudaStreamSynchronize(s));
  }
  // mod variants may move masses outside [lo, hi]: widen by the gate
  if (h->cfg.max_mods > 0) {
    lo = std::min(lo, h->p.min_mass);
    hi = std::max(hi, h->p.max_mass);
  }
  return build_end(h, recs, n, lo, hi);
  DBI_API_END
}

int dbi_stats_get(dbi_handle* h, dbi_stats* out) {
  if (!h || !out) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  std::lock_guard<std::mutex> lk(h->mu);
  *out = h->st;
  return DBI_OK;
}

int dbi_query_device(dbi_handle* h, const double* d_lo, const double* d_hi, uint64_t nq, uint64_t* d_hit_begin,
                     uint64_t* d_hit_count) {
  DBI_API_BEGIN(h)
  if (!h->built) {
    set_error("Indexer is not initialized");  // DBIndexStoreSQLiteMult.java:316-318
    return DBI_ENOTINIT;
  }
  Stage sg(h, DBI_STAGE_QUERY);
  query_ranges(h, d_lo, d_hi, nq, d_hit_begin, d_hit_count, nullptr);
  return DBI_OK;
  DBI_API_END
}

int dbi_query(dbi_handle* h, const double* lo, const double* hi, uint64_t nq, uint64_t* hit_begin,
              uint64_t* hit_count) {
  DBI_API_BEGIN(h)
  if (!h->built) {
    set_error("Indexer is not initialized");
    return DBI_ENOTINIT;
  }
  if (nq == 0) return DBI_OK;
  if (!lo || !hi || !hit_begin || !hit_count) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  cudaStream_t s = h->stream;
  DevBuf io;  // lo | hi | begin | count
  io.alloc(nq * 32, h->arena);
  double* d_lo = io.as<double>();
  double* d_hi = d_lo + nq;
  uint64_t* d_b = (uint64_t*)(d_hi + nq);
  uint64_t* d_c = d_b + nq;
  DBI_CUDA(cudaMemcpyAsync(d_lo, lo, nq * 8, cudaMemcpyHostToDevice, s));
  DBI_CUDA(cudaMemcpyAsync(d_hi, hi, nq * 8, cudaMemcpyHostToDevice, s));
  {
    Stage sg(h, DBI_STAGE_QUERY);
    query_ranges(h, d_lo, d_hi, nq, d_b, d_c, nullptr);
  }
  DBI_CUDA(cudaMemcpyAsync(hit_begin, d_b, nq * 8, cudaMemcpyDeviceToHost, s));
  DBI_CUDA(cudaMemcpyAsync(hit_count, d_c, nq * 8, cudaMemcpyDeviceToHost, s));
  DBI_CUDA(cudaStreamSynchronize(s));
  resolve_spans(h);
  return DBI_OK;
  DBI_API_END
}

int dbi_fetch(dbi_handle* h, uint64_t begin, uint64_t count, double* mass, uint32_t* first_prot,
              uint32_t* first_off, uint16_t* len, uint32_t* modpat, uint64_t* prot_list_off, uint32_t* prot_ids,
              uint64_t prot_ids_capacity, uint64_t* n_prot_ids) {
  DBI_API_BEGIN(h)
  if (!h->built) {
    set_error("Indexer is not initialized");
    return DBI_ENOTINIT;
  }
  if (begin > h->cnt.n_entries || count > h->cnt.n_entries - begin) {
    set_error("entry range [%llu, +%llu) outside the index (%llu entries)", (unsigned long long)begin,
              (unsigned long long)count, (unsigned long long)h->cnt.n_entries);
    return DBI_EINVAL;
  }
  if (n_prot_ids) *n_prot_ids = 0;
  if (count == 0) {
    if (prot_list_off) prot_list_off[0] = 0;
    return DBI_OK;
  }
  cudaStream_t s = h->stream;
  const uint64_t tiles = (count + kScanTile - 1) / kScanTile;
  const UniqView uv = uniq_view(h);
  const double* em = h->entry_mass();
  const uint32_t* eb = h->entry_base();
  const uint32_t* ep = h->entry_pat();
  uint64_t fb = begin;
  DevBuf x_mass, x_base, x_pat, rng;
  if (h->cnt.n_groups) {  // compact index: K6q expands the range first
    const uint64_t NT = (count + kExpTile - 1) / kExpTile;
    const uint64_t hr[5] = {begin, 0, count, 0, NT};  // begin | out_off | tile_off
    rng.alloc(40 + NT * 4, h->arena);
    uint64_t* d_r = rng.as<uint64_t>();
    DBI_CUDA(cudaMemcpyAsync(d_r, hr, 40, cudaMemcpyHostToDevice, s));
    uint32_t* tile_q = (uint32_t*)(d_r + 5);
    DBI_CUDA(cudaMemsetAsync(tile_q, 0, NT * 4, s));
    expand_ranges(h, ExpRanges{tile_q, d_r + 3, d_r, d_r + 1}, NT, count, x_mass, x_base, x_pat);
    DBI_CUDA(cudaStreamSynchronize(s));  // hr leaves scope
    em = x_mass.as<double>();
    eb = x_base.as<uint32_t>();
    ep = x_pat.as<uint32_t>();
    fb = 0;
  }
  DevBuf sizes, tcnt, toff;
  sizes.alloc(count * 4, h->arena);
  tcnt.alloc(tiles * 4, h->arena);
  toff.alloc((tiles + 1) * 8, h->arena);
  uint64_t total_ids = 0;
  {
    Stage sg(h, DBI_STAGE_FETCH);
    launch_fetch_sizes(eb, h->rt.ent_base_off, uv, fb, count, sizes.as<uint32_t>(), tcnt.as<uint32_t>(), s);
    launch_scan_u32_to_u64(tcnt.as<uint32_t>(), tiles, toff.as<uint64_t>(), s);
    total_ids = read_u64(h, toff.as<uint64_t>() + tiles);
  }
  if (n_prot_ids) *n_prot_ids = total_ids;
  const bool want_ids = prot_ids != nullptr;
  if (want_ids && prot_ids_capacity < total_ids) {
    set_error("prot_ids capacity %llu < %llu", (unsigned long long)prot_ids_capacity, (unsigned long long)total_ids);
    return DBI_ERANGE;
  }
  DevBuf o_mass, o_prot, o_off, o_len, o_pat, o_lo, o_ids;
  if (mass) o_mass.alloc(count * 8, h->arena);
  if (first_prot) o_prot.alloc(count * 4, h->arena);
  if (first_off) o_off.alloc(count * 4, h->arena);
  if (len) o_len.alloc(count * 2, h->arena);
  if (modpat) o_pat.alloc(count * 4, h->arena);
  if (prot_list_off) o_lo.alloc((count + 1) * 8, h->arena);
  if (want_ids) o_ids.alloc(total_ids * 4, h->arena);
  {
    Stage sg(h, DBI_STAGE_FETCH);
    launch_fetch_gather(em, eb, h->rt.ent_base_off, uv, ep, h->ix.d_pstart.as<uint32_t>(), fb, count, sizes.as<uint32_t>(), toff.as<uint64_t>(),
                        o_mass.as<double>(), o_prot.as<uint32_t>(), o_off.as<uint32_t>(), o_len.as<uint16_t>(),
                        o_pat.as<uint32_t>(), o_lo.as<uint64_t>(), o_ids.as<uint32_t>(), s);
    h->st.algo_bytes[DBI_STAGE_FETCH] += count * (20 + 8 + 26) + total_ids * 8;
  }
  if (mass) DBI_CUDA(cudaMemcpyAsync(mass, o_mass.p, count * 8, cudaMemcpyDeviceToHost, s));
  if (first_prot) DBI_CUDA(cudaMemcpyAsync(first_prot, o_prot.p, count * 4, cudaMemcpyDeviceToHost, s));
  if (first_off) DBI_CUDA(cudaMemcpyAsync(first_off, o_off.p, count * 4, cudaMemcpyDeviceToHost, s));
  if (len) DBI_CUDA(cudaMemcpyAsync(len, o_len.p, count * 2, cudaMemcpyDeviceToHost, s));
  if (modpat) DBI_CUDA(cudaMemcpyAsync(modpat, o_pat.p, count * 4, cudaMemcpyDeviceToHost, s));
  if (prot_list_off) DBI_CUDA(cudaMemcpyAsync(prot_list_off, o_lo.p, (count + 1) * 8, cudaMemcpyDeviceToHost, s));
  if (want_ids && total_ids) DBI_CUDA(cudaMemcpyAsync(prot_ids, o_ids.p, total_ids * 4, cudaMemcpyDeviceToHost, s));
  DBI_CUDA(cudaStreamSynchronize(s));
  resolve_spans(h);
  return DBI_OK;
  DBI_API_END
}

}  // extern "C"

namespace {
// dbi_query_hits with the bounds already on the device
int query_hits_impl(dbi_handle* h, const double* d_lo, const double* d_hi, uint64_t nq, dbi_hit_counts* counts) {
  cudaStream_t s = h->stream;
  dbi_handle::HitResult& r = h->hits;
  r.drop();
  std::memset(counts, 0, sizeof(*counts));
  counts->nq = nq;
  r.n = *counts;
  r.hit_off.alloc((nq + 1) * 8, h->arena);
  if (nq == 0) {
    r.pep_off.alloc(8, h->arena); r.pep_hit_off.alloc(8, h->arena); r.seq_off.alloc(8, h->arena); r.plo.alloc(8, h->arena);
    for (DevBuf* z : {&r.hit_off, &r.pep_off, &r.pep_hit_off, &r.seq_off, &r.plo}) DBI_CUDA(cudaMemsetAsync(z->p, 0, 8, s));
    DBI_CUDA(cudaStreamSynchronize(s));
    r.valid = true;
    return DBI_OK;
  }
  DevBuf io, cnt32, stmp, len32, np32, stmp2, nseg32, seg_off, ntile32, tile_off;
  io.alloc(nq * 16 + 8, h->arena);  // begin | count | over
  uint64_t* d_b = io.as<uint64_t>();
  uint64_t* d_c = d_b + nq;
  uint32_t* d_over = (uint32_t*)(d_c + nq);
  cnt32.alloc(nq * 4, h->arena);
  stmp.alloc(full_scan_tmp_bytes(nq), h->arena);
  const bool compact = h->cnt.n_groups > 0;
  uint64_t H = 0, NS = 0, NT = 0;
  uint32_t over = 0;
  {
    Stage sg(h, DBI_STAGE_QUERY);
    if (compact) {  // and the K6q tiles of every query
      ntile32.alloc(nq * 4, h->arena);
      tile_off.alloc((nq + 1) * 8, h->arena);
      DBI_CUDA(cudaMemsetAsync(d_over, 0, 4, s));
    }
    query_ranges(h, d_lo, d_hi, nq, d_b, d_c, cnt32.as<uint32_t>(), ntile32.as<uint32_t>(), d_over);
    launch_full_scan_u32_to_u64(cnt32.as<uint32_t>(), nq, r.hit_off.as<uint64_t>(), stmp.p, s);
    if (compact) {
      launch_full_scan_u32_to_u64(ntile32.as<uint32_t>(), nq, tile_off.as<uint64_t>(), stmp.p, s);
      DBI_CUDA(cudaMemcpyAsync(&NT, tile_off.as<uint64_t>() + nq, 8, cudaMemcpyDeviceToHost, s));
      DBI_CUDA(cudaMemcpyAsync(&over, d_over, 4, cudaMemcpyDeviceToHost, s));
    }
    // the hits of a query are materialised in segments of 256 (one warp each)
    nseg32.alloc(nq * 4, h->arena);
    seg_off.alloc((nq + 1) * 8, h->arena);
    launch_hits_seg_count(d_c, nq, nseg32.as<uint32_t>(), s);
    launch_full_scan_u32_to_u64(nseg32.as<uint32_t>(), nq, seg_off.as<uint64_t>(), stmp.p, s);
    DBI_CUDA(cudaMemcpyAsync(&H, r.hit_off.as<uint64_t>() + nq, 8, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaMemcpyAsync(&NS, seg_off.as<uint64_t>() + nq, 8, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaStreamSynchronize(s));
  }
  if (H >= (1ull << 32) || over) {
    set_error("%s hits in one batch: split the batch (< 2^32 hits per call)",
              over ? "2^32 or more" : std::to_string(H).c_str());
    r.drop();
    return DBI_ERANGE;
  }
  const UniqView uv = uniq_view(h);
  // where K10 reads the hits: the index's entries, or on a compact index the hits expanded by K6q (hit h of
  // the batch at position h: the queries' hits begin at hit_off)
  const double* em = h->entry_mass();
  const uint32_t* eb = h->entry_base();
  const uint32_t* ep = h->entry_pat();
  const uint64_t* hb = d_b;
  uint64_t eo = h->rt.ent_base_off;
  DevBuf x_mass, x_base, x_pat, tile_q;
  if (compact && H) {
    tile_q.alloc(NT * 4, h->arena);
    launch_hits_seg_fill(tile_off.as<uint64_t>(), nq, tile_q.as<uint32_t>(), s);
    const ExpRanges rg{tile_q.as<uint32_t>(), tile_off.as<uint64_t>(), d_b, r.hit_off.as<uint64_t>()};
    expand_ranges(h, rg, NT, H, x_mass, x_base, x_pat);
    em = x_mass.as<double>();
    eb = x_base.as<uint32_t>();
    ep = x_pat.as<uint32_t>();
    hb = r.hit_off.as<uint64_t>();
    eo = 0;
  }
  r.pep_off.alloc((nq + 1) * 8, h->arena);
  uint64_t NP = 0, SB = 0, PI = 0;
  if (H) {
    Stage sg(h, DBI_STAGE_FETCH);
    DevBuf seg_q, nruns32, seg_run_off, pep_entry, stmp3;
    seg_q.alloc(NS * 4, h->arena);
    nruns32.alloc(NS * 4, h->arena);
    seg_run_off.alloc((NS + 1) * 8, h->arena);
    stmp3.alloc(full_scan_tmp_bytes(NS), h->arena);
    r.pat.alloc(H * 4, h->arena);
    launch_hits_seg_fill(seg_off.as<uint64_t>(), nq, seg_q.as<uint32_t>(), s);
    launch_hits_count_runs(em, eb, seg_q.as<uint32_t>(), seg_off.as<uint64_t>(), hb, r.hit_off.as<uint64_t>(), NS,
                           nruns32.as<uint32_t>(), s);
    launch_full_scan_u32_to_u64(nruns32.as<uint32_t>(), NS, seg_run_off.as<uint64_t>(), stmp3.p, s);
    launch_hits_pep_off(seg_off.as<uint64_t>(), seg_run_off.as<uint64_t>(), nq, r.pep_off.as<uint64_t>(), s);
    NP = read_u64(h, seg_run_off.as<uint64_t>() + NS);
    r.pep_hit_off.alloc((NP + 1) * 8, h->arena);
    r.mass.alloc(NP * 8, h->arena);
    r.seq_off.alloc((NP + 1) * 8, h->arena);
    r.plo.alloc((NP + 1) * 8, h->arena);
    pep_entry.alloc(NP * 4, h->arena);
    len32.alloc(NP * 4, h->arena);
    np32.alloc(NP * 4, h->arena);
    stmp2.alloc(full_scan_tmp_bytes(NP), h->arena);
    launch_hits_runs(em, eb, eo, ep, uv, seg_q.as<uint32_t>(), seg_off.as<uint64_t>(), hb, r.hit_off.as<uint64_t>(),
                     seg_run_off.as<uint64_t>(), NS,
                     r.pat.as<uint32_t>(), r.pep_hit_off.as<uint64_t>(), r.mass.as<double>(), pep_entry.as<uint32_t>(),
                     len32.as<uint32_t>(), np32.as<uint32_t>(), s);
    DBI_CUDA(cudaMemcpyAsync(r.pep_hit_off.as<uint64_t>() + NP, r.hit_off.as<uint64_t>() + nq, 8, cudaMemcpyDeviceToDevice, s));
    launch_full_scan_u32_to_u64(len32.as<uint32_t>(), NP, r.seq_off.as<uint64_t>(), stmp2.p, s);
    launch_full_scan_u32_to_u64(np32.as<uint32_t>(), NP, r.plo.as<uint64_t>(), stmp2.p, s);
    DBI_CUDA(cudaMemcpyAsync(&SB, r.seq_off.as<uint64_t>() + NP, 8, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaMemcpyAsync(&PI, r.plo.as<uint64_t>() + NP, 8, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaStreamSynchronize(s));
    r.prot.alloc(NP * 4, h->arena);
    r.off.alloc(NP * 4, h->arena);
    r.len.alloc(NP * 2, h->arena);
    r.flanks.alloc(NP * 6, h->arena);
    r.seq.alloc(std::max<uint64_t>(SB, 1), h->arena);
    r.ids.alloc(std::max<uint64_t>(PI, 1) * 4, h->arena);
    launch_peps_gather(h->ix.d_res.as<uint8_t>(), h->ix.d_pstart.as<uint32_t>(), eb, eo, uv,
                       pep_entry.as<uint32_t>(), r.seq_off.as<uint64_t>(), r.plo.as<uint64_t>(), NP,
                       r.prot.as<uint32_t>(), r.off.as<uint32_t>(), r.len.as<uint16_t>(), r.flanks.as<uint8_t>(),
                       r.seq.as<uint8_t>(), r.ids.as<uint32_t>(), s);
    // per hit: entry read twice (12 + 16), pattern written (4); per run: peptide tables (4 + 4 + 2 + 16)
    // read, 56 written; residues and ids copied
    h->st.algo_bytes[DBI_STAGE_FETCH] += H * (28 + 4) + NP * (26 + 56 + 12) + 2 * SB + 8 * PI;
  } else {
    r.pep_hit_off.alloc(8, h->arena);
    r.seq_off.alloc(8, h->arena);
    r.plo.alloc(8, h->arena);
    DBI_CUDA(cudaMemsetAsync(r.pep_off.p, 0, (nq + 1) * 8, s));
    DBI_CUDA(cudaMemsetAsync(r.pep_hit_off.p, 0, 8, s));
    DBI_CUDA(cudaMemsetAsync(r.seq_off.p, 0, 8, s));
    DBI_CUDA(cudaMemsetAsync(r.plo.p, 0, 8, s));
  }
  DBI_CUDA(cudaStreamSynchronize(s));
  resolve_spans(h);
  counts->n_hits = H;
  counts->n_peps = NP;
  counts->n_seq_bytes = SB;
  counts->n_prot_ids = PI;
  r.n = *counts;
  r.valid = true;
  return DBI_OK;
}

// The start of an unindexed search on one handle: its candidate pipeline replaces the stats of the previous one.
void search_begin(dbi_handle* h) {
  h->spans.clear();
  h->ev_used = 0;
  const uint64_t np = h->st.n_proteins, nr = h->st.n_residues;
  std::memset(&h->st, 0, sizeof(h->st));
  h->st.n_proteins = np;
  h->st.n_residues = nr;
  ensure_uploaded(h);
  clear_err(h);
}

// K12: a batch's windows on the handle's GPU, sorted by lo, with the prefix maximum of hi.  io = lo | hi (the
// caller's order, for the materialisation) | sorted lo | prefix max of hi; *win = the handle's shift intervals
// over those windows.  lo / hi are host pointers, or device pointers with kind = cudaMemcpyDeviceToDevice.
void upload_windows(dbi_handle* h, const double* lo, const double* hi, uint64_t nq, DevBuf& io, MassWindows* win,
                    cudaMemcpyKind kind = cudaMemcpyHostToDevice) {
  cudaStream_t s = h->stream;
  io.alloc(std::max<uint64_t>(nq, 1) * 32, h->arena);
  double* d_lo = io.as<double>();
  double* d_hi = d_lo + nq;
  double* w_lo = d_hi + nq;
  double* w_pmax = w_lo + nq;
  *win = h->shifts;
  win->lo = w_lo;
  win->pmax = w_pmax;
  win->n = (uint32_t)nq;
  if (!nq) return;
  DBI_CUDA(cudaMemcpyAsync(d_lo, lo, nq * 8, kind, s));
  DBI_CUDA(cudaMemcpyAsync(d_hi, hi, nq * 8, kind, s));
  Stage sg(h, DBI_STAGE_OTHER);
  DevBuf wk[2], wv[2], wtmp;
  for (int i = 0; i < 2; ++i) {
    wk[i].alloc(nq * 8, h->arena);
    wv[i].alloc(nq * 8, h->arena);
  }
  wtmp.alloc(radix_sort_tmp_bytes(nq), h->arena);
  launch_win_keys(d_lo, d_hi, nq, h->p.min_mass, h->p.max_mass, wk[0].as<uint64_t>(), wv[0].as<uint64_t>(), s);
  uint64_t* kk[2] = {wk[0].as<uint64_t>(), wk[1].as<uint64_t>()};
  uint64_t* vv[2] = {wv[0].as<uint64_t>(), wv[1].as<uint64_t>()};
  const int nbits = bit_length(win_drop_key(h->p.min_mass, h->p.max_mass));
  const int r = radix_sort_pairs<uint64_t, uint64_t>(kk, vv, nq, 0, nbits, wtmp.p, s, nullptr);
  launch_win_pmax(kk[r], vv[r], nq, h->p.min_mass, h->p.max_mass, w_lo, w_pmax, s);
  h->st.algo_bytes[DBI_STAGE_OTHER] += nq * (16 + 16) + nq * 32ull * ((nbits + 7) / 8) + nq * 32;
}

// An unindexed search needs an unbuilt handle that is not part of a sharded build.
int check_unindexed(dbi_handle* h) {
  if (h->built) {
    set_error("the index is built: query it with dbi_query_hits");
    return DBI_EALREADY;
  }
  if (h->mg_begun) {
    set_error("an unindexed search runs on one GPU; this handle is part of a sharded build");
    return DBI_EINVAL;
  }
  return DBI_OK;
}

// The candidate index of an unindexed search lives for one call only; the pending result does not depend on it.
struct DropCandidates {
  dbi_handle* h;
  bool armed = true;
  ~DropCandidates() {
    if (!armed) return;
    free_tables(h);
    h->built = false;
  }
};

// K12 windows, K2u / K4u candidates, and their index on the handle (h->built until the caller's DropCandidates
// drops it) for the windows [lo[i], hi[i]] (kind: where lo / hi live).  io = upload_windows' buffer, whose first
// 2 nq doubles are lo | hi on the device.  N_c over max_candidates (or at 2^32): DBI_ERANGE with *n_candidates set.
int index_candidates(dbi_handle* h, const double* lo, const double* hi, uint64_t nq, cudaMemcpyKind kind,
                     uint64_t max_candidates, uint64_t* n_candidates, DevBuf& io) {
  if (nq >= (1ull << 32)) {
    set_error("%llu windows in one batch (< 2^32)", (unsigned long long)nq);
    return DBI_ERANGE;
  }
  search_begin(h);
  const uint32_t n_prot = (uint32_t)(h->h_off.size() - 1);
  if (h->lay.packed_prot != n_prot) pack_residues(h);  // K1 only when proteins were added since the last pack

  MassWindows win;
  upload_windows(h, lo, hi, nq, io, &win, kind);
  // K2u: the records that can land in a window, counted before anything is allocated
  Digest dg = whole_digest(h, &win);
  const uint64_t N = dg.count();
  if (int rc = check_err_bits(read_err(h))) return rc;
  if (n_candidates) *n_candidates = N;
  h->st.n_emitted = N;
  if ((max_candidates && N > max_candidates) || N >= (1ull << 32)) {
    set_error("%llu candidate records exceed the cap of %llu (and 2^32): split the batch", (unsigned long long)N,
              (unsigned long long)(max_candidates ? max_candidates : (1ull << 32) - 1));
    resolve_spans(h);
    return DBI_ERANGE;
  }
  RecSet cand;
  if (N) dg.emit(cand, nullptr);  // K4u
  DropCandidates drop_candidates{h};
  if (int rc = index_records(h, cand.view(), N, h->p.min_mass, h->p.max_mass)) return rc;
  if (int rc = check_err_bits(read_err(h))) return rc;
  drop_candidates.armed = false;
  return DBI_OK;
}

// ---- batches of spectra (dbi_query_spectra, dbi_search_unindexed_spectra; K13 / K14 in spectra.cu) ----
int check_spectra(const double* mass, const double* tol, const uint64_t* range_off, uint64_t n, int tol_mode,
                  int index_factor, const dbi_hit_counts* counts) {
  if (tol_mode != DBI_TOL_DA && tol_mode != DBI_TOL_PPM) {
    set_error("tol_mode %d is neither DBI_TOL_DA nor DBI_TOL_PPM", tol_mode);
    return DBI_EINVAL;
  }
  if (tol_mode == DBI_TOL_PPM && range_off) {
    set_error("DBI_TOL_PPM takes one mass per spectrum: range_off must be NULL");
    return DBI_EINVAL;
  }
  if (index_factor < 0 || index_factor > 8000) {
    set_error("index_factor %d outside 0..8000", index_factor);
    return DBI_EINVAL;
  }
  if (!counts || (n && (!mass || !tol || (tol_mode == DBI_TOL_DA && !range_off)))) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  for (uint64_t sp = 0; sp < n; ++sp) {
    const uint64_t r0 = tol_mode == DBI_TOL_DA ? range_off[sp] : sp;
    const uint64_t r1 = tol_mode == DBI_TOL_DA ? range_off[sp + 1] : sp + 1;
    if (r1 < r0) {
      set_error("spectrum %llu: range_off decreases (%llu -> %llu)", (unsigned long long)sp, (unsigned long long)r0,
                (unsigned long long)r1);
      return DBI_EINVAL;
    }
    for (uint64_t r = r0; r < r1; ++r)
      if (!std::isfinite(mass[r]) || !std::isfinite(tol[r])) {
        set_error("spectrum %llu: non-finite mass or tolerance (%g, %g)", (unsigned long long)sp, mass[r], tol[r]);
        return DBI_EINVAL;
      }
  }
  return DBI_OK;
}

// A batch of spectra on the device.  in = mass | tol (| range_off for Dalton lists).  Dalton: K13a merges every
// list, iv = the kept intervals of all spectra, spectrum s owning [ioff[s], ioff[s+1]).  PPM: K13b writes win =
// window lo | hi (| candidate lo | hi), and spectra_probe (K14, on the handle's entries) makes iv and ioff.
struct SpectraBatch {
  uint64_t n = 0, n_ranges = 0, n_iv = 0;
  int mode = DBI_TOL_DA, factor = 0;
  DevBuf in, win, cnt, ioff, stmp, iv;
  const double* mass() const { return in.as<double>(); }
  const double* tol() const { return in.as<double>() + n_ranges; }
  const uint64_t* range_off() const { return (const uint64_t*)(in.as<double>() + 2 * n_ranges); }
  const double* iv_lo() const { return iv.as<double>(); }
  const double* iv_hi() const { return iv.as<double>() + n_iv; }
};

// scan of cnt into ioff, then iv sized for the intervals
void spectra_offsets(dbi_handle* h, SpectraBatch& b) {
  b.ioff.alloc((b.n + 1) * 8, h->arena);
  b.stmp.alloc(full_scan_tmp_bytes(b.n), h->arena);
  launch_full_scan_u32_to_u64(b.cnt.as<uint32_t>(), b.n, b.ioff.as<uint64_t>(), b.stmp.p, h->stream);
  b.n_iv = read_u64(h, b.ioff.as<uint64_t>() + b.n);
  b.iv.alloc(std::max<uint64_t>(b.n_iv, 1) * 16, h->arena);
}

// upload and K13; with `candidates` (PPM) also the candidate windows of an unindexed search
void spectra_prepare(dbi_handle* h, SpectraBatch& b, const double* mass, const double* tol, const uint64_t* range_off,
                     uint64_t n, int mode, int factor, bool candidates) {
  cudaStream_t s = h->stream;
  b.n = n;
  b.mode = mode;
  b.factor = factor;
  b.n_ranges = mode == DBI_TOL_DA ? (n ? range_off[n] : 0) : n;
  const uint64_t R = b.n_ranges;
  b.in.alloc(std::max<uint64_t>(2 * R + (mode == DBI_TOL_DA ? n + 1 : 0), 1) * 8, h->arena);
  if (R) {
    DBI_CUDA(cudaMemcpyAsync(b.in.p, mass, R * 8, cudaMemcpyHostToDevice, s));
    DBI_CUDA(cudaMemcpyAsync(b.in.as<double>() + R, tol, R * 8, cudaMemcpyHostToDevice, s));
  }
  b.cnt.alloc(std::max<uint64_t>(n, 1) * 4, h->arena);
  Stage sg(h, DBI_STAGE_QUERY);
  if (mode == DBI_TOL_DA) {
    if (n) DBI_CUDA(cudaMemcpyAsync((void*)b.range_off(), range_off, (n + 1) * 8, cudaMemcpyHostToDevice, s));
    b.win.alloc(std::max<uint64_t>(R, 1) * 16, h->arena);
    double* s_lo = b.win.as<double>();
    double* s_hi = s_lo + R;
    launch_spec_intervals(b.mass(), b.tol(), b.range_off(), n, factor, s_lo, s_hi, b.cnt.as<uint32_t>(), s);
    spectra_offsets(h, b);
    launch_spec_compact(b.range_off(), b.ioff.as<uint64_t>(), n, s_lo, s_hi, b.iv.as<double>(),
                        b.iv.as<double>() + b.n_iv, s);
    // per range: (mass, tol) read, slot written, interval packed (16 + 16 + 32); per spectrum: offsets and count
    h->st.algo_bytes[DBI_STAGE_QUERY] += R * 64 + n * (16 + 4 + 16);
  } else {
    b.win.alloc(std::max<uint64_t>(n, 1) * (candidates ? 32 : 16), h->arena);
    double* w = b.win.as<double>();
    launch_spec_ppm_window(b.mass(), b.tol(), n, w, w + n, candidates ? w + 2 * n : nullptr,
                           candidates ? w + 3 * n : nullptr, s);
    h->st.algo_bytes[DBI_STAGE_QUERY] += n * (16 + (candidates ? 32 : 16));
  }
}

// K14: the window and the continuing probes of every PPM spectrum, over the handle's (or candidate) index.
// d_stop (device, n u64): the walks of a sharded index end at the given probes (the minimum of K14s over the ranks).
void spectra_probe(dbi_handle* h, SpectraBatch& b, const uint64_t* d_stop = nullptr) {
  cudaStream_t s = h->stream;
  Stage sg(h, DBI_STAGE_QUERY);
  const double* w_lo = b.win.as<double>();
  const double* w_hi = w_lo + b.n;
  launch_spec_probe_count(h->key_mass(), h->n_keys(), b.mass(), b.tol(), w_lo, w_hi, b.n, b.factor, d_stop,
                          b.cnt.as<uint32_t>(), s);
  spectra_offsets(h, b);
  launch_spec_probe_emit(h->key_mass(), h->n_keys(), b.mass(), b.tol(), w_lo, w_hi, b.n, b.factor, d_stop,
                         b.ioff.as<uint64_t>(), b.iv.as<double>(), b.iv.as<double>() + b.n_iv, s);
  // both passes: (mass, ppm, window) read, one lower bound (or one stop) per spectrum; count, offsets, interval
  const uint64_t probe = d_stop ? 8 : 32 + 8ull * (uint64_t)bit_length(h->n_keys());
  h->st.algo_bytes[DBI_STAGE_QUERY] += 2 * b.n * (32 + probe) + b.n * (4 + 8) + b.n_iv * 16;
}

// K14s on the handle's entries for the PPM batch b (K13b done): stop[s] = K_r of this rank, copied to the host
void spectra_stops(dbi_handle* h, SpectraBatch& b, const SliceCuts& cuts, uint64_t* stop) {
  cudaStream_t s = h->stream;
  if (!b.n) return;
  DevBuf d_stop;
  d_stop.alloc(b.n * 8, h->arena);
  {
    Stage sg(h, DBI_STAGE_QUERY);
    launch_spec_stops(h->key_mass(), h->n_keys(), b.mass(), b.tol(), b.win.as<double>() + b.n, b.n, b.factor, cuts,
                      d_stop.as<uint64_t>(), s);
    h->st.algo_bytes[DBI_STAGE_QUERY] += b.n * (24 + 32 + 8ull * (uint64_t)bit_length(h->n_keys()) + 8);
  }
  DBI_CUDA(cudaMemcpyAsync(stop, d_stop.p, b.n * 8, cudaMemcpyDeviceToHost, s));
  DBI_CUDA(cudaStreamSynchronize(s));
}

// spectra_probe with the host stops of every PPM spectrum
void spectra_probe_stops(dbi_handle* h, SpectraBatch& b, const uint64_t* stop) {
  DevBuf d_stop;
  d_stop.alloc(std::max<uint64_t>(b.n, 1) * 8, h->arena);
  if (b.n) DBI_CUDA(cudaMemcpyAsync(d_stop.p, stop, b.n * 8, cudaMemcpyHostToDevice, h->stream));
  spectra_probe(h, b, d_stop.as<uint64_t>());
}

// K9 / K10 over the intervals, then the per-interval offsets of the pending result collapsed to per-spectrum ones
int spectra_answer(dbi_handle* h, SpectraBatch& b, dbi_hit_counts* counts) {
  if (b.n_iv >= (1ull << 32)) {
    set_error("%llu intervals in one batch (< 2^32): split the batch", (unsigned long long)b.n_iv);
    return DBI_ERANGE;
  }
  if (int rc = query_hits_impl(h, b.iv_lo(), b.iv_hi(), b.n_iv, counts)) return rc;
  dbi_handle::HitResult& r = h->hits;
  DevBuf hit_off, pep_off;
  hit_off.alloc((b.n + 1) * 8, h->arena);
  pep_off.alloc((b.n + 1) * 8, h->arena);
  launch_spec_collapse(b.ioff.as<uint64_t>(), b.n, r.hit_off.as<uint64_t>(), r.pep_off.as<uint64_t>(),
                       hit_off.as<uint64_t>(), pep_off.as<uint64_t>(), h->stream);
  DBI_CUDA(cudaStreamSynchronize(h->stream));
  r.hit_off.swap(hit_off);
  r.pep_off.swap(pep_off);
  counts->nq = b.n;
  r.n.nq = b.n;
  return DBI_OK;
}
}  // namespace

extern "C" {

int dbi_query_hits(dbi_handle* h, const double* lo, const double* hi, uint64_t nq, dbi_hit_counts* counts) {
  DBI_API_BEGIN(h)
  if (!h->built) {
    set_error("Indexer is not initialized");
    return DBI_ENOTINIT;
  }
  if (!counts || (nq && (!lo || !hi))) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  DevBuf io;  // lo | hi
  io.alloc(std::max<uint64_t>(nq, 1) * 16, h->arena);
  if (nq) {
    DBI_CUDA(cudaMemcpyAsync(io.p, lo, nq * 8, cudaMemcpyHostToDevice, h->stream));
    DBI_CUDA(cudaMemcpyAsync(io.as<double>() + nq, hi, nq * 8, cudaMemcpyHostToDevice, h->stream));
  }
  return query_hits_impl(h, io.as<double>(), io.as<double>() + nq, nq, counts);
  DBI_API_END
}

int dbi_query_hits_device(dbi_handle* h, const double* d_lo, const double* d_hi, uint64_t nq, dbi_hit_counts* counts) {
  DBI_API_BEGIN(h)
  if (!h->built) {
    set_error("Indexer is not initialized");
    return DBI_ENOTINIT;
  }
  if (!counts || (nq && (!d_lo || !d_hi))) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  return query_hits_impl(h, d_lo, d_hi, nq, counts);
  DBI_API_END
}

int dbi_query_hits_read(dbi_handle* h, const dbi_hit_buffers* out) {
  DBI_API_BEGIN(h)
  dbi_handle::HitResult& r = h->hits;
  if (!r.valid) {
    set_error("no pending dbi_query_hits result on this handle");
    return DBI_ENOTINIT;
  }
  if (!out) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  cudaStream_t s = h->stream;
  const uint64_t H = r.n.n_hits;
  auto d2h = [&](void* dst, const DevBuf& src, uint64_t bytes) {
    if (dst && bytes) DBI_CUDA(cudaMemcpyAsync(dst, src.p, bytes, cudaMemcpyDeviceToHost, s));
  };
  const uint64_t NP = r.n.n_peps;
  d2h(out->hit_off, r.hit_off, (r.n.nq + 1) * 8);
  d2h(out->pep_off, r.pep_off, (r.n.nq + 1) * 8);
  d2h(out->modpat, r.pat, H * 4);
  d2h(out->pep_hit_off, r.pep_hit_off, (NP + 1) * 8);
  d2h(out->mass, r.mass, NP * 8);
  d2h(out->first_prot, r.prot, NP * 4);
  d2h(out->first_off, r.off, NP * 4);
  d2h(out->len, r.len, NP * 2);
  d2h(out->flanks, r.flanks, NP * 6);
  d2h(out->seq_off, r.seq_off, (NP + 1) * 8);
  d2h(out->seq, r.seq, r.n.n_seq_bytes);
  d2h(out->prot_list_off, r.plo, (NP + 1) * 8);
  d2h(out->prot_ids, r.ids, r.n.n_prot_ids * 4);
  DBI_CUDA(cudaStreamSynchronize(s));
  r.drop();
  return DBI_OK;
  DBI_API_END
}

int dbi_search_unindexed(dbi_handle* h, const double* lo, const double* hi, uint64_t nq, uint64_t max_candidates,
                         dbi_hit_counts* counts, uint64_t* n_candidates) {
  DBI_API_BEGIN(h)
  DBI_MUTATES(h)
  if (int rc = check_unindexed(h)) return rc;
  if (!counts || (nq && (!lo || !hi))) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  drop_results(h);
  if (n_candidates) *n_candidates = 0;
  DevBuf io;
  if (int rc = index_candidates(h, lo, hi, nq, cudaMemcpyHostToDevice, max_candidates, n_candidates, io)) return rc;
  DropCandidates drop_candidates{h};
  return query_hits_impl(h, io.as<double>(), io.as<double>() + nq, nq, counts);
  DBI_API_END
}

int dbi_query_spectra(dbi_handle* h, const double* mass, const double* tol, const uint64_t* range_off,
                      uint64_t n_spectra, int tol_mode, int index_factor, dbi_hit_counts* counts) {
  DBI_API_BEGIN(h)
  if (!h->built) {
    set_error("Indexer is not initialized");
    return DBI_ENOTINIT;
  }
  if (int rc = check_spectra(mass, tol, range_off, n_spectra, tol_mode, index_factor, counts)) return rc;
  h->hits.drop();
  SpectraBatch b;
  spectra_prepare(h, b, mass, tol, range_off, n_spectra, tol_mode, index_factor, false);
  if (tol_mode == DBI_TOL_PPM) spectra_probe(h, b);
  return spectra_answer(h, b, counts);
  DBI_API_END
}

int dbi_search_unindexed_spectra(dbi_handle* h, const double* mass, const double* tol, const uint64_t* range_off,
                                 uint64_t n_spectra, int tol_mode, int index_factor, uint64_t max_candidates,
                                 dbi_hit_counts* counts, uint64_t* n_candidates) {
  DBI_API_BEGIN(h)
  DBI_MUTATES(h)
  if (int rc = check_unindexed(h)) return rc;
  if (int rc = check_spectra(mass, tol, range_off, n_spectra, tol_mode, index_factor, counts)) return rc;
  drop_results(h);
  if (n_candidates) *n_candidates = 0;
  SpectraBatch b;
  spectra_prepare(h, b, mass, tol, range_off, n_spectra, tol_mode, index_factor, true);
  // the candidate windows: the merged intervals, or [min(lo, u_0), bound of the probes] of every PPM spectrum
  const bool da = tol_mode == DBI_TOL_DA;
  const uint64_t nw = da ? b.n_iv : n_spectra;
  const double* c_lo = da ? b.iv_lo() : b.win.as<double>() + 2 * n_spectra;
  const double* c_hi = da ? b.iv_hi() : b.win.as<double>() + 3 * n_spectra;
  DevBuf io;
  if (int rc = index_candidates(h, c_lo, c_hi, nw, cudaMemcpyDeviceToDevice, max_candidates, n_candidates, io))
    return rc;
  DropCandidates drop_candidates{h};
  io.release();
  if (!da) spectra_probe(h, b);
  return spectra_answer(h, b, counts);
  DBI_API_END
}

int dbi_lookup_peptides(dbi_handle* h, const uint8_t* residues, const uint64_t* offsets, const uint32_t* modpat,
                        uint64_t n, dbi_lookup_counts* counts) {
  DBI_API_BEGIN(h)
  if (!h->built) {
    set_error("Indexer is not initialized");
    return DBI_ENOTINIT;
  }
  if (!counts || (n && !offsets)) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  for (uint64_t i = 0; i < n; ++i)
    if (offsets[i + 1] < offsets[i]) {
      set_error("offsets must be non-decreasing (row %llu)", (unsigned long long)i);
      return DBI_EINVAL;
    }
  const uint64_t R = n ? offsets[n] - offsets[0] : 0;
  if (R && !residues) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  const UniqView uv = uniq_view(h);
  for (int r = 0; r < uv.world; ++r)
    if (uv.uoff[r + 1] > uv.uoff[r] && !uv.len[r]) {
      set_error("rank %d's unique-peptide window is not mapped on this handle: its peptides cannot be compared", r);
      return DBI_EINVAL;
    }
  cudaStream_t s = h->stream;
  dbi_handle::LookupResult& L = h->lookup;
  L.drop();
  std::memset(counts, 0, sizeof(*counts));
  counts->n = n;
  L.status.alloc(std::max<uint64_t>(n, 1), h->arena);
  L.mass.alloc(std::max<uint64_t>(n, 1) * 8, h->arena);
  L.entry.alloc(std::max<uint64_t>(n, 1) * 8, h->arena);
  L.prot.alloc(std::max<uint64_t>(n, 1) * 4, h->arena);
  L.off.alloc(std::max<uint64_t>(n, 1) * 4, h->arena);
  L.plo.alloc((n + 1) * 8, h->arena);
  if (n == 0) {
    DBI_CUDA(cudaMemsetAsync(L.plo.p, 0, 8, s));
    DBI_CUDA(cudaStreamSynchronize(s));
    L.n = *counts;
    L.valid = true;
    return DBI_OK;
  }
  // input: residues | offsets | patterns | found counter
  const uint64_t res_bytes = (R + 7) & ~7ull, pat_bytes = modpat ? (n * 4 + 7) & ~7ull : 0;
  DevBuf in, np32, stmp, gid;
  in.alloc(res_bytes + (n + 1) * 8 + pat_bytes + 8, h->arena);
  uint8_t* d_q = in.as<uint8_t>();
  uint64_t* d_off = (uint64_t*)(d_q + res_bytes);
  uint32_t* d_pat = modpat ? (uint32_t*)(d_off + n + 1) : nullptr;
  unsigned long long* d_found = (unsigned long long*)((uint8_t*)(d_off + n + 1) + pat_bytes);
  if (R) DBI_CUDA(cudaMemcpyAsync(d_q, residues + offsets[0], R, cudaMemcpyHostToDevice, s));
  DBI_CUDA(cudaMemcpyAsync(d_off, offsets, (n + 1) * 8, cudaMemcpyHostToDevice, s));
  if (modpat) DBI_CUDA(cudaMemcpyAsync(d_pat, modpat, n * 4, cudaMemcpyHostToDevice, s));
  DBI_CUDA(cudaMemsetAsync(d_found, 0, 8, s));
  np32.alloc(n * 4, h->arena);
  stmp.alloc(full_scan_tmp_bytes(n), h->arena);
  uint64_t n_found = 0, PI = 0;
  {
    Stage sg(h, DBI_STAGE_QUERY);
    // compact index: the search runs over the groups, and gid[row] = the peptide found (K11b's input)
    const GroupView gv{h->ix.g_pay.as<uint64_t>(), h->ix.g_eoff.as<uint64_t>(), h->ix.u_cmask.as<uint64_t>(),
                       h->cfg.n_classes};
    if (h->cnt.n_groups) gid.alloc(n * 8, h->arena);
    launch_lookup_match(h->ix.d_res.as<uint8_t>(), h->key_mass(), h->n_keys(), h->entry_base(), h->rt.ent_base_off,
                        h->entry_pat(), uv, h->d_tables.as<DevTables>(), h->cfg.init_mass, h->cfg.max_mods, d_q, d_off,
                        d_pat, n, L.status.as<uint8_t>(), L.mass.as<double>(), L.entry.as<uint64_t>(),
                        np32.as<uint32_t>(), d_found, h->cnt.n_groups ? &gv : nullptr, gid.as<uint64_t>(), s);
    int rounds = 1;  // the last one probes <= 32 consecutive entries
    for (uint64_t w = h->n_keys(); w > 32; w = w / 33 + 1) ++rounds;
    // rows read (residues, offset, pattern), 32 eight-byte probes per search round, the row's residues compared
    // once with its candidate, status + mass + entry + list length written
    h->st.algo_bytes[DBI_STAGE_QUERY] += 2 * R + n * (12 + 256ull * rounds + 21);
  }
  {
    Stage sg(h, DBI_STAGE_FETCH);
    launch_full_scan_u32_to_u64(np32.as<uint32_t>(), n, L.plo.as<uint64_t>(), stmp.p, s);
    DBI_CUDA(cudaMemcpyAsync(&PI, L.plo.as<uint64_t>() + n, 8, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaMemcpyAsync(&n_found, d_found, 8, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaStreamSynchronize(s));
    L.ids.alloc(std::max<uint64_t>(PI, 1) * 4, h->arena);
    if (h->cnt.n_groups)
      launch_lookup_gather(L.status.as<uint8_t>(), gid.as<uint64_t>(), nullptr, 0, uv, h->ix.d_pstart.as<uint32_t>(),
                           L.plo.as<uint64_t>(), n, L.prot.as<uint32_t>(), L.off.as<uint32_t>(), L.ids.as<uint32_t>(), s);
    else
      launch_lookup_gather(L.status.as<uint8_t>(), L.entry.as<uint64_t>(), h->entry_base(), h->rt.ent_base_off, uv,
                           h->ix.d_pstart.as<uint32_t>(), L.plo.as<uint64_t>(), n, L.prot.as<uint32_t>(),
                           L.off.as<uint32_t>(), L.ids.as<uint32_t>(), s);
    // list lengths scanned (4 read, 8 written); per row status + list offset read, first occurrence written;
    // per found row entry, base id, peptide tables (4 + 4 + 16) and protein start read; ids copied
    h->st.algo_bytes[DBI_STAGE_FETCH] += n * (12 + 9 + 8) + n_found * (8 + 4 + 24 + 4) + 8 * PI;
  }
  DBI_CUDA(cudaStreamSynchronize(s));
  resolve_spans(h);
  counts->n_found = n_found;
  counts->n_prot_ids = PI;
  L.n = *counts;
  L.valid = true;
  return DBI_OK;
  DBI_API_END
}

int dbi_lookup_peptides_read(dbi_handle* h, const dbi_lookup_buffers* out) {
  DBI_API_BEGIN(h)
  dbi_handle::LookupResult& L = h->lookup;
  if (!L.valid) {
    set_error("no pending dbi_lookup_peptides result on this handle");
    return DBI_ENOTINIT;
  }
  if (!out) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  cudaStream_t s = h->stream;
  const uint64_t n = L.n.n;
  auto d2h = [&](void* dst, const DevBuf& src, uint64_t bytes) {
    if (dst && bytes) DBI_CUDA(cudaMemcpyAsync(dst, src.p, bytes, cudaMemcpyDeviceToHost, s));
  };
  d2h(out->status, L.status, n);
  d2h(out->mass, L.mass, n * 8);
  d2h(out->entry, L.entry, n * 8);
  d2h(out->first_prot, L.prot, n * 4);
  d2h(out->first_off, L.off, n * 4);
  d2h(out->prot_list_off, L.plo, (n + 1) * 8);
  d2h(out->prot_ids, L.ids, L.n.n_prot_ids * 4);
  DBI_CUDA(cudaStreamSynchronize(s));
  L.drop();
  return DBI_OK;
  DBI_API_END
}

int dbi_host_alloc(uint64_t bytes, void** out) {
  if (!out) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  *out = nullptr;
  const cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault);
  if (e != cudaSuccess) {
    set_error("cudaHostAlloc(%llu): %s", (unsigned long long)bytes, cudaGetErrorString(e));
    cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? DBI_ENOMEM : DBI_ECUDA;
  }
  return DBI_OK;
}

int dbi_host_free(void* p) {
  if (p && cudaFreeHost(p) != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaFreeHost failed");
    return DBI_ECUDA;
  }
  return DBI_OK;
}

int dbi_get_protein(dbi_handle* h, uint32_t id, const uint8_t** residues, uint64_t* len) {
  if (!h || !residues || !len) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  if (h->owner) h = h->owner;  // the host copy is built lazily, once, by the owner under its mutex
  std::lock_guard<std::mutex> lk(h->mu);
  if ((uint64_t)id + 1 >= h->h_off.size()) {
    set_error("protein id %u out of range", id);
    return DBI_EINVAL;
  }
  if (!h->h_raw_valid) {  // first use: bring the residues back once (ProteinCache on demand)
    try {
      DBI_CUDA(cudaSetDevice(h->device));
      h->h_raw.resize(h->n_res);
      if (h->n_res) DBI_CUDA(cudaMemcpyAsync(h->h_raw.data(), h->d_raw.p, h->n_res, cudaMemcpyDeviceToHost, h->stream));
      DBI_CUDA(cudaStreamSynchronize(h->stream));
      h->h_raw_valid = true;
    } catch (const CudaError& e) {
      return fail_cuda(e);
    }
  }
  *residues = h->h_raw.data() + h->h_off[id];
  *len = h->h_off[id + 1] - h->h_off[id];
  return DBI_OK;
}

int dbi_calculate_mass(dbi_handle* h, const uint8_t* seq, uint64_t len, double* mass) {
  if (!h || (!seq && len) || !mass) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  const dbi_params& p = h->p;
  double m = 0;  // util/IndexUtil.java:198-207
  if (p.add_h2o_proton) m += p.h2o_proton;
  m += p.cterm;
  m += p.nterm;
  for (uint64_t i = 0; i < len; ++i) m += p.residue_mass[seq[i]];
  *mass = m;
  return DBI_OK;
}

int dbi_entry_keys(dbi_handle* h, int32_t* keys, uint64_t capacity, uint64_t* n_keys) {
  DBI_API_BEGIN(h)
  if (!h->built) {
    set_error("Indexer is not initialized");
    return DBI_ENOTINIT;
  }
  if (!n_keys) {
    set_error("null argument");
    return DBI_EINVAL;
  }
  *n_keys = 0;
  const uint64_t n = h->n_keys();  // equal masses are adjacent: the groups give the same keys as the entries
  if (n == 0) return DBI_OK;
  cudaStream_t s = h->stream;
  const uint64_t tiles = (n + kScanTile - 1) / kScanTile;
  DevBuf flags, tcnt, toff, out;
  flags.alloc(n, h->arena);
  tcnt.alloc(tiles * 4, h->arena);
  toff.alloc((tiles + 1) * 8, h->arena);
  Stage sg(h, DBI_STAGE_OTHER);
  launch_key_flags(h->key_mass(), n, (double)h->p.mass_group_factor, flags.as<uint8_t>(), tcnt.as<uint32_t>(), s);
  launch_scan_u32_to_u64(tcnt.as<uint32_t>(), tiles, toff.as<uint64_t>(), s);
  const uint64_t nk = read_u64(h, toff.as<uint64_t>() + tiles);
  *n_keys = nk;
  if (!keys) return DBI_OK;
  if (capacity < nk) {
    set_error("keys capacity %llu < %llu", (unsigned long long)capacity, (unsigned long long)nk);
    return DBI_ERANGE;
  }
  out.alloc(nk * 4, h->arena);
  launch_key_emit(h->key_mass(), n, (double)h->p.mass_group_factor, flags.as<uint8_t>(), toff.as<uint64_t>(),
                  out.as<int32_t>(), s);
  DBI_CUDA(cudaMemcpyAsync(keys, out.p, nk * 4, cudaMemcpyDeviceToHost, s));
  DBI_CUDA(cudaStreamSynchronize(s));
  return DBI_OK;
  DBI_API_END
}

int dbi_debug_emitted(dbi_handle* h, uint64_t capacity, double* mass, uint32_t* prot, uint32_t* off, uint16_t* len,
                      uint64_t* n) {
  DBI_API_BEGIN(h)
  DBI_OWNER_ONLY(h)
  if (!h->built || !h->p.keep_emitted) {
    set_error("emitted records were not kept (params.keep_emitted) or the index is not built");
    return DBI_ENOTINIT;
  }
  if (n) *n = h->cnt.n_emitted;
  if (capacity < h->cnt.n_emitted) {
    if (!mass && !prot && !off && !len) return DBI_OK;  // sizing call
    set_error("capacity %llu < %llu", (unsigned long long)capacity, (unsigned long long)h->cnt.n_emitted);
    return DBI_ERANGE;
  }
  const uint64_t N = h->cnt.n_emitted;
  cudaStream_t s = h->stream;
  std::vector<uint32_t> gpos(N), pr(N);
  if (N) {
    DBI_CUDA(cudaMemcpyAsync(gpos.data(), h->kept.gpos.p, N * 4, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaMemcpyAsync(pr.data(), h->kept.prot.p, N * 4, cudaMemcpyDeviceToHost, s));
    if (mass) DBI_CUDA(cudaMemcpyAsync(mass, h->kept.mass.p, N * 8, cudaMemcpyDeviceToHost, s));
    if (len) DBI_CUDA(cudaMemcpyAsync(len, h->kept.len.p, N * 2, cudaMemcpyDeviceToHost, s));
    DBI_CUDA(cudaStreamSynchronize(s));
  }
  for (uint64_t i = 0; i < N; ++i) {
    if (prot) prot[i] = pr[i];
    if (off) off[i] = gpos[i] - (uint32_t)(h->h_off[pr[i]] + pr[i] + 1);
  }
  return DBI_OK;
  DBI_API_END
}

int dbi_debug_radix_sort(dbi_handle* h, uint64_t* keys, uint64_t* vals, uint64_t n, int begin_bit, int end_bit) {
  DBI_API_BEGIN(h)
  DBI_OWNER_ONLY(h)
  if (n == 0) return DBI_OK;
  if (!keys || !vals || begin_bit < 0 || end_bit > 64 || end_bit < begin_bit) {
    set_error("bad argument");
    return DBI_EINVAL;
  }
  cudaStream_t s = h->stream;
  DevBuf k[2], v[2], tmp;
  for (int i = 0; i < 2; ++i) {
    k[i].alloc(n * 8, h->arena);
    v[i].alloc(n * 8, h->arena);
  }
  tmp.alloc(radix_sort_tmp_bytes(n), h->arena);
  DBI_CUDA(cudaMemcpyAsync(k[0].p, keys, n * 8, cudaMemcpyHostToDevice, s));
  DBI_CUDA(cudaMemcpyAsync(v[0].p, vals, n * 8, cudaMemcpyHostToDevice, s));
  uint64_t* kk[2] = {k[0].as<uint64_t>(), k[1].as<uint64_t>()};
  uint64_t* vv[2] = {v[0].as<uint64_t>(), v[1].as<uint64_t>()};
  const int r = radix_sort_pairs<uint64_t, uint64_t>(kk, vv, n, begin_bit, end_bit, tmp.p, s, nullptr);
  DBI_CUDA(cudaMemcpyAsync(keys, kk[r], n * 8, cudaMemcpyDeviceToHost, s));
  DBI_CUDA(cudaMemcpyAsync(vals, vv[r], n * 8, cudaMemcpyDeviceToHost, s));
  DBI_CUDA(cudaStreamSynchronize(s));
  return DBI_OK;
  DBI_API_END
}

void dbi_destroy(dbi_handle* h) {
  if (!h) return;
  dbi_handle* owner = h->owner;
  if (!owner) {  // the index memory lives until the last view is destroyed
    std::lock_guard<std::mutex> lk(h->view_mu);
    if (h->n_views.load()) {
      h->orphaned = true;
      return;
    }
  }
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  free_index(h);  // on a view: forgets the borrowed buffers
  if (!owner) mg_release(h);
  h->d_raw.release();
  h->d_off.release();
  h->mg_wtab.release();
  h->d_tables.release();
  h->d_err.release();
  cudaStreamSynchronize(h->stream);
  h->arena.flush();
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  if (h->side_stream) {
    cudaStreamSynchronize(h->side_stream);
    cudaStreamDestroy(h->side_stream);
    cudaEventDestroy(h->pull_done);
  }
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  if (owner) {
    bool last = false;
    {
      std::lock_guard<std::mutex> lk(owner->view_mu);
      last = owner->n_views.fetch_sub(1) == 1 && owner->orphaned;
    }
    if (last) dbi_destroy(owner);
  }
}

int dbi_release_cached_memory(int device) {
  if (device < 0 || device >= 64) {
    set_error("bad device ordinal %d", device);
    return DBI_EINVAL;
  }
  if (cudaSetDevice(device) != cudaSuccess) {
    cudaGetLastError();
    set_error("no such CUDA device %d", device);
    return DBI_ECUDA;
  }
  DevCache::of(device).trim();
  return DBI_OK;
}

const char* dbi_last_error(void) { return t_err; }

uint64_t dbi_kernel_launches(void) { return g_kernel_launches.load(); }

}  // extern "C"

#include "capi_mg.inl"
#include "capi_persist.inl"
