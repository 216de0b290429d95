// C ABI of libfrg.so (include/frg.h): store life-cycle, ingest, match dispatch, merge.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <new>

#include "frg_internal.cuh"

namespace frg {

static thread_local char g_err[512] = "";
static thread_local int g_launches = 0;
static thread_local const char* g_variant = "none";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  set_error("CUDA error %d (%s) at %s:%d: %s", int(e), cudaGetErrorString(e), file, line, what);
  return e == cudaErrorMemoryAllocation ? FRG_ERR_NOMEM : FRG_ERR_CUDA;
}

void note_launch(const char* variant) {
  ++g_launches;
  if (variant) g_variant = variant;
}
void reset_launches() { g_launches = 0; g_variant = "none"; }

struct ProfileSpan { cudaEvent_t a, b; int launches; int stage; };
static thread_local int g_profile = 0;      // 0 off, 1 every stage, 2 the dominant kernel only, 3 = 2 on every 4th match
static thread_local unsigned g_match_seq = 0;
constexpr unsigned kProfileSampleEvery = 4;
static thread_local std::vector<ProfileSpan> g_spans;
static thread_local cudaEvent_t g_open = nullptr;
static thread_local int g_open_stage = 0;
static thread_local float g_stage_ms[FRG_PROFILE_STAGES] = {0};

void profile_begin(cudaStream_t st, int stage) {
  if (!g_profile || (g_profile >= 2 && stage != kStageDominant)) return;
  if (g_profile == 3 && (g_match_seq % kProfileSampleEvery) != 0) return;
  if (cudaEventCreate(&g_open) != cudaSuccess) { g_open = nullptr; return; }
  g_open_stage = stage;
  cudaEventRecord(g_open, st);
}

void profile_end(cudaStream_t st, int launches) {
  if (!g_profile || !g_open) return;
  ProfileSpan sp{g_open, nullptr, launches, g_open_stage};
  g_open = nullptr;
  if (cudaEventCreate(&sp.b) != cudaSuccess) { cudaEventDestroy(sp.a); return; }
  cudaEventRecord(sp.b, st);
  g_spans.push_back(sp);
}

int device_info(int device, DeviceInfo* out) {
  static std::mutex mu;
  static std::vector<DeviceInfo> cache;
  std::lock_guard<std::mutex> lk(mu);
  if (device < 0) { set_error("negative device"); return FRG_ERR_INVALID; }
  if (int(cache.size()) <= device) cache.resize(device + 1);
  DeviceInfo& d = cache[device];
  if (d.sm_count == 0) {
    cudaDeviceProp p;
    FRG_CUDA(cudaGetDeviceProperties(&p, device));
    d.sm_count = p.multiProcessorCount;
    d.cc_major = p.major;
    d.cc_minor = p.minor;
    d.smem_optin = p.sharedMemPerBlockOptin;
  }
  *out = d;
  return FRG_OK;
}

int store_begin_write(frg_store* s, cudaStream_t stream) {
  for (cudaStream_t r : s->readers) {
    if (r == stream) continue;
    cudaEvent_t ev;
    FRG_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    FRG_CUDA(cudaEventRecord(ev, r));
    FRG_CUDA(cudaStreamWaitEvent(stream, ev, 0));
    FRG_CUDA(cudaEventDestroy(ev));   // destruction is deferred until the event completes
  }
  s->readers.clear();
  if (s->has_write) FRG_CUDA(cudaStreamWaitEvent(stream, s->last_write, 0));
  return FRG_OK;
}

int store_end_write(frg_store* s, cudaStream_t stream) {
  FRG_CUDA(cudaEventRecord(s->last_write, stream));
  s->has_write = true;
  s->version++;
  return FRG_OK;
}

int store_begin_read(frg_store* s, cudaStream_t stream) {
  if (s->has_write) FRG_CUDA(cudaStreamWaitEvent(stream, s->last_write, 0));
  bool seen = false;
  for (cudaStream_t r : s->readers) seen |= (r == stream);
  if (!seen) s->readers.push_back(stream);
  return FRG_OK;
}

// after a stream synchronisation: has a kernel of this store reported a broken pipeline?
static int store_fault(const frg_store* s) {
  const uint32_t f = s->fault_host ? *static_cast<volatile uint32_t*>(s->fault_host) : 0u;
  if (!f) return FRG_OK;
  set_error("a tensor-core pipeline barrier of this store's match kernels timed out (code %u): results since are "
            "void; destroy the store and create it again", f);
  return FRG_ERR_CUDA;
}

static bool has_master(const frg_store* s) { return !(s->flags & FRG_STORE_BF16_ONLY); }
static bool has_plane(const frg_store* s) { return (s->flags & (FRG_STORE_BF16_PLANE | FRG_STORE_BF16_ONLY)) != 0; }
// a unit store with a full master scans an int8 plane (tc_match.cu); raw and bf16-only stores keep a bf16 one
static bool has_plane8(const frg_store* s) {
  return (s->flags & FRG_STORE_BF16_PLANE) && !(s->flags & (FRG_STORE_RAW | FRG_STORE_BF16_ONLY));
}
// bytes of one scan-plane row
static size_t plane_row_bytes(const frg_store* s) {
  if (!has_plane(s)) return 0;
  return has_plane8(s) ? size_t(s->dim) : size_t(s->plane_dim) * sizeof(__nv_bfloat16);
}

static size_t row_bytes(const frg_store* s) {
  return size_t(s->dim) * (has_master(s) ? sizeof(float) : 0) + plane_row_bytes(s) + sizeof(int32_t);
}

// p: the scan plane, bf16 or int8 (has_plane8) - its element type is the caller's to know
static int alloc_arrays(frg_store* s, int64_t cap, float** m, void** p, int32_t** t) {
  *m = nullptr; *p = nullptr; *t = nullptr;
  const int64_t c = cap > 0 ? cap : 1;
  cudaError_t e = cudaSuccess;
  if (has_master(s)) e = cudaMalloc(reinterpret_cast<void**>(m), size_t(c) * s->dim * sizeof(float));
  if (e == cudaSuccess && has_plane(s)) e = cudaMalloc(p, size_t(c) * plane_row_bytes(s));
  if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(t), size_t(c) * sizeof(int32_t));
  if (e != cudaSuccess) {
    cudaFree(*m); cudaFree(*p); cudaFree(*t);
    *m = nullptr; *p = nullptr; *t = nullptr;
    return cuda_fail(e, "cudaMalloc(store arrays)", __FILE__, __LINE__);
  }
  return FRG_OK;
}
static void* plane_ptr(const frg_store* s) { return s->plane8 ? static_cast<void*>(s->plane8) : static_cast<void*>(s->plane); }
static void set_plane(frg_store* s, void* p) {
  if (has_plane8(s)) s->plane8 = static_cast<int8_t*>(p);
  else s->plane = static_cast<__nv_bfloat16*>(p);
}

// grow to at least `cap` rows; s->mu held.  Synchronous (rare, off the hot path).
static int grow_locked(frg_store* s, int64_t cap) {
  if (cap <= s->capacity) return FRG_OK;
  FRG_CUDA(cudaDeviceSynchronize());
  float* m; void* p; int32_t* t;
  FRG_CHECK(alloc_arrays(s, cap, &m, &p, &t));
  if (s->rows > 0) {
    if (m) FRG_CUDA(cudaMemcpy(m, s->master, size_t(s->rows) * s->dim * sizeof(float), cudaMemcpyDeviceToDevice));
    if (p) FRG_CUDA(cudaMemcpy(p, plane_ptr(s), size_t(s->rows) * plane_row_bytes(s), cudaMemcpyDeviceToDevice));
    FRG_CUDA(cudaMemcpy(t, s->tags, size_t(s->rows) * sizeof(int32_t), cudaMemcpyDeviceToDevice));
  }
  cudaFree(s->master); cudaFree(plane_ptr(s)); cudaFree(s->tags);
  s->master = m; set_plane(s, p); s->tags = t;
  s->capacity = cap;
  s->readers.clear();
  s->has_write = false;
  return FRG_OK;
}

static int64_t next_capacity(int64_t have, int64_t need) {
  int64_t c = have > 0 ? have : 1024;
  while (c < need) c += c / 2 + 1024;
  return c;
}

// exact live-row recount (synchronous; s->mu held): mutators only mark the count stale
static int count_live(frg_store* s) {
  FRG_CUDA(cudaDeviceSynchronize());
  std::vector<int32_t> t(static_cast<size_t>(s->rows));
  if (s->rows > 0)
    FRG_CUDA(cudaMemcpy(t.data(), s->tags, size_t(s->rows) * sizeof(int32_t), cudaMemcpyDeviceToHost));
  int64_t live = 0;
  for (int32_t v : t) live += v >= 0;
  s->live = live;
  return FRG_OK;
}

// ---- tenant extents (frg_store::extents); s->mu held
static void extent_add(frg_store* s, int32_t tag, int64_t lo, int64_t hi) {
  if (tag < 0 || hi <= lo) return;
  auto it = s->extents.find(tag);
  if (it == s->extents.end()) { s->extents.emplace(tag, frg_store::Extent{lo, hi}); return; }
  if (lo < it->second.lo) it->second.lo = lo;
  if (hi > it->second.hi) it->second.hi = hi;
}

// interval [lo, hi) of tag -> its span set (merged with what it touches)
static void span_add(frg_store* s, int32_t tag, int64_t lo, int64_t hi) {
  if (tag < 0 || hi <= lo) return;
  frg_store::Spans& sp = s->spans[tag];
  if (sp.scattered) return;
  auto it = sp.iv.upper_bound(lo);
  if (it != sp.iv.begin()) {
    auto pv = std::prev(it);
    if (pv->second >= lo) { lo = pv->first; if (pv->second > hi) hi = pv->second; sp.covered -= pv->second - pv->first; it = sp.iv.erase(pv); }
  }
  while (it != sp.iv.end() && it->first <= hi) {
    if (it->second > hi) hi = it->second;
    sp.covered -= it->second - it->first;
    it = sp.iv.erase(it);
  }
  sp.iv.emplace(lo, hi);
  sp.covered += hi - lo;
  if (sp.iv.size() > frg_store::kMaxSpans) { sp.scattered = true; sp.iv.clear(); }
}

// rows / tags are HOST arrays (or null: append at `base` / tag 0)
static void extents_note_upsert(frg_store* s, const int64_t* hrows, const int32_t* htags, int64_t n, int64_t base) {
  {
    // exact runs of consecutive rows with one tag -> span intervals
    int64_t i = 0;
    while (i < n) {
      const int32_t tag = htags ? htags[i] : 0;
      const int64_t lo = hrows ? hrows[i] : base + i;
      int64_t j = i + 1;
      while (j < n && (htags ? htags[j] : 0) == tag && (hrows ? hrows[j] : base + j) == lo + (j - i)) ++j;
      span_add(s, tag, lo, lo + (j - i));
      i = j;
    }
  }
  if (!htags && !hrows) { extent_add(s, 0, base, base + n); return; }
  // runs of equal tags over consecutive rows (bulk loads) cost one map update each
  int64_t i = 0;
  while (i < n) {
    const int32_t tag = htags ? htags[i] : 0;
    int64_t lo = hrows ? hrows[i] : base + i, hi = lo + 1;
    int64_t j = i + 1;
    while (j < n && (htags ? htags[j] : 0) == tag) {
      const int64_t r = hrows ? hrows[j] : base + j;
      if (r < lo) lo = r;
      if (r + 1 > hi) hi = r + 1;
      ++j;
    }
    extent_add(s, tag, lo, hi);
    i = j;
  }
}

// the whole gallery, or - for a tenant-filtered call whose tag extents are known - only the row window that
// tenant's rows can sit in
static GalleryWindow window_of(const frg_store* s, int32_t tenant, bool for_tc = false) {
  GalleryWindow w;
  w.master = s->master; w.plane = s->plane; w.plane8 = s->plane8; w.tags = s->tags; w.gmax_bits = s->gmax_bits; w.fault = s->fault_dev;
  w.rows = s->rows; w.row0 = 0; w.dim = s->dim; w.plane_dim = s->plane_dim; w.flags = s->flags;
  w.maybe_dead = s->maybe_dead;
  if (tenant >= 0 && s->extents_known) {
    int64_t lo = 0, hi = 0;
    auto it = s->extents.find(tenant);
    if (it != s->extents.end()) { lo = it->second.lo; hi = it->second.hi < s->rows ? it->second.hi : s->rows; }
    if (hi < lo) hi = lo;
    // A window that is mostly other tenants' rows (a company's block + one person re-enrolled at the far end):
    // keep the WHOLE store as the window and let the tensor-core kernels walk only the tiles of the tenant's
    // intervals.  (The exact scan and first_match still take the bounding window.)
    auto sp = s->spans.find(tenant);
    if (for_tc && sp != s->spans.end() && !sp->second.scattered && hi - lo >= 32768 &&
        sp->second.covered * 4 <= hi - lo) {
      w.owner = const_cast<frg_store*>(s);
      w.want_tile_list = true;
      w.list_tenant = tenant;
      return w;                             // row0 = 0, rows = s->rows: tile indices are absolute
    }
    w.row0 = lo; w.rows = hi - lo;
    if (w.master) w.master += lo * s->dim;
    if (w.plane) w.plane += lo * s->plane_dim;
    if (w.plane8) w.plane8 += lo * s->dim;
    w.tags += lo;
  }
  return w;
}

int store_tile_list(frg_store* s, int32_t tenant, int gran, cudaStream_t st, const int32_t** list, int* n) {
  *list = nullptr; *n = 0;
  auto sp = s->spans.find(tenant);
  if (sp == s->spans.end() || sp->second.scattered || !s->extents_known) return FRG_OK;
  frg_store::TileList& tl = s->tile_lists[std::make_pair(tenant, gran)];
  if (tl.version != s->version) {
    // rebuild: tiles touched by the intervals, ascending, clipped to the rows in use
    std::vector<int32_t> tiles;
    int64_t last = -1;
    for (const auto& iv : sp->second.iv) {
      const int64_t hi = iv.second < s->rows ? iv.second : s->rows;
      if (hi <= iv.first) continue;
      int64_t t0 = iv.first / gran;
      const int64_t t1 = (hi - 1) / gran;
      if (t0 <= last) t0 = last + 1;
      for (int64_t t = t0; t <= t1; ++t) tiles.push_back(int32_t(t));
      if (t1 > last) last = t1;
    }
    const int64_t all_tiles = (s->rows + gran - 1) / gran;
    tl.version = s->version;
    tl.n = int(tiles.size());
    tl.use = !tiles.empty() && int64_t(tiles.size()) * 2 <= all_tiles;
    if (tl.use) {
      if (int64_t(tiles.size()) > tl.cap) {
        // a bigger buffer; the old one may still be read by matches in flight: freed with the store
        if (tl.dev) s->retired.push_back(tl.dev);
        tl.cap = int64_t(tiles.size()) * 2 + 64;
        tl.dev = nullptr;
        FRG_CUDA(cudaMalloc(reinterpret_cast<void**>(&tl.dev), size_t(tl.cap) * sizeof(int32_t)));
      }
      if (!tl.ready) FRG_CUDA(cudaEventCreateWithFlags(&tl.ready, cudaEventDisableTiming));
      // Overwriting in place is safe: this match was ordered (store_begin_read) after the mutation that bumped
      // the version, and that mutation after every match that read the previous list.  Pageable source: the
      // call returns once the vector has been staged.
      FRG_CUDA(cudaMemcpyAsync(tl.dev, tiles.data(), tiles.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
      FRG_CUDA(cudaEventRecord(tl.ready, st));
    }
  }
  if (!tl.use) return FRG_OK;
  FRG_CUDA(cudaStreamWaitEvent(st, tl.ready, 0));        // another stream may have uploaded it
  *list = tl.dev; *n = tl.n;
  return FRG_OK;
}

}  // namespace frg

using namespace frg;

extern "C" {

int frg_abi_version(void) { return FRG_ABI_VERSION; }
const char* frg_last_error(void) { return g_err; }
int frg_last_launch_count(void) { return g_launches; }
const char* frg_last_variant(void) { return g_variant; }

int frg_profile_enable(int32_t on) {
  g_profile = on < 0 ? 0 : (on > 3 ? 1 : on);
  g_match_seq = 0;
  return FRG_OK;
}

int frg_profile_collect(float* dominant_ms, int32_t* dominant_launches) {
  float total = 0.f;
  int launches = 0;
  int rc = FRG_OK;
  for (float& v : g_stage_ms) v = 0.f;
  for (auto& sp : g_spans) {
    float ms = 0.f;
    cudaError_t e = cudaEventSynchronize(sp.b);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, sp.a, sp.b);
    if (e != cudaSuccess && rc == FRG_OK) rc = cuda_fail(e, "profile events", __FILE__, __LINE__);
    if (sp.stage >= 0 && sp.stage < FRG_PROFILE_STAGES) g_stage_ms[sp.stage] += ms;
    if (sp.stage == kStageDominant) { total += ms; launches += sp.launches; }
    cudaEventDestroy(sp.a);
    cudaEventDestroy(sp.b);
  }
  g_spans.clear();
  if (dominant_ms) *dominant_ms = total;
  if (dominant_launches) *dominant_launches = launches;
  return rc;
}

int frg_profile_stage_ms(int32_t stage, float* ms) {
  if (stage < 0 || stage >= FRG_PROFILE_STAGES || !ms) { set_error("bad profile stage"); return FRG_ERR_INVALID; }
  *ms = g_stage_ms[stage];
  return FRG_OK;
}

int frg_device_count(int32_t* count) {
  if (!count) { set_error("count is NULL"); return FRG_ERR_INVALID; }
  int n = 0;
  *count = 0;
  FRG_CUDA(cudaGetDeviceCount(&n));
  *count = n;
  return FRG_OK;
}

int frg_store_create(int32_t device, int32_t dim, int64_t capacity, uint32_t flags, frg_store** out) {
  if (!out) { set_error("out is NULL"); return FRG_ERR_INVALID; }
  *out = nullptr;
  if (dim <= 0 || dim % 8 != 0) { set_error("dim %d must be a positive multiple of 8", dim); return FRG_ERR_INVALID; }
  if (capacity < 0) { set_error("negative capacity"); return FRG_ERR_INVALID; }
  if ((flags & FRG_STORE_BF16_ONLY) && (flags & FRG_STORE_RAW)) {
    set_error("a bf16-only store holds unit rows for the cosine filter; it cannot be raw");
    return FRG_ERR_INVALID;
  }
  DeviceInfo di;
  FRG_CHECK(device_info(device, &di));
  DeviceGuard g(device);
  if (!g.ok) { set_error("cannot select device %d", device); return FRG_ERR_CUDA; }
  frg_store* s = new (std::nothrow) frg_store();
  if (!s) { set_error("out of host memory"); return FRG_ERR_NOMEM; }
  s->device = device; s->dim = dim; s->flags = flags;
  // a raw store's scan plane is the Euclidean one (norm terms in kEuclidPad more columns) where the
  // tensor-core tile shapes cover it; other raw stores keep a plain image nobody scans
  const char* why = "";
  s->plane_dim = ((flags & FRG_STORE_RAW) && (flags & FRG_STORE_BF16_PLANE) && tc_supported(dim, FRG_METRIC_EUCLIDEAN, &why))
                     ? dim + kEuclidPad : dim;
  void* plane = nullptr;
  int rc = alloc_arrays(s, capacity, &s->master, &plane, &s->tags);
  set_plane(s, plane);
  if (rc == FRG_OK) {
    cudaError_t eg = cudaMalloc(reinterpret_cast<void**>(&s->gmax_bits), 2 * sizeof(uint32_t));
    if (eg == cudaSuccess) eg = cudaMemset(s->gmax_bits, 0, 2 * sizeof(uint32_t));
    if (eg != cudaSuccess) {
      cudaFree(s->master); cudaFree(plane_ptr(s)); cudaFree(s->tags); cudaFree(s->gmax_bits);
      rc = cuda_fail(eg, "cudaMalloc(gmax)", __FILE__, __LINE__);
    }
  }
  if (rc == FRG_OK) {
    cudaError_t ef = cudaHostAlloc(reinterpret_cast<void**>(&s->fault_host), sizeof(uint32_t), cudaHostAllocMapped);
    if (ef == cudaSuccess) {
      *s->fault_host = 0;
      ef = cudaHostGetDevicePointer(reinterpret_cast<void**>(&s->fault_dev), s->fault_host, 0);
    }
    if (ef != cudaSuccess) {
      cudaFree(s->master); cudaFree(plane_ptr(s)); cudaFree(s->tags); cudaFree(s->gmax_bits);
      if (s->fault_host) cudaFreeHost(s->fault_host);
      rc = cuda_fail(ef, "cudaHostAlloc(fault word)", __FILE__, __LINE__);
    }
  }
  if (rc != FRG_OK) { delete s; return rc; }
  s->capacity = capacity > 0 ? capacity : 1;
  cudaError_t e = cudaEventCreateWithFlags(&s->last_write, cudaEventDisableTiming);
  if (e != cudaSuccess) { frg_store_destroy(s); return cuda_fail(e, "cudaEventCreate", __FILE__, __LINE__); }
  // keep stream-ordered workspaces cached instead of returning them to the OS after every match
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t keep = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  *out = s;
  return FRG_OK;
}

int frg_store_destroy(frg_store* s) {
  if (!s) return FRG_OK;
  {
    DeviceGuard g(s->device);
    cudaDeviceSynchronize();
    cudaFree(s->master); cudaFree(plane_ptr(s)); cudaFree(s->tags); cudaFree(s->gmax_bits);
    if (s->fault_host) cudaFreeHost(s->fault_host);
    for (auto& kv : s->tile_lists) { cudaFree(kv.second.dev); if (kv.second.ready) cudaEventDestroy(kv.second.ready); }
    for (void* p : s->retired) cudaFree(p);
    if (s->last_write) cudaEventDestroy(s->last_write);
  }
  delete s;
  return FRG_OK;
}

int frg_store_reserve(frg_store* s, int64_t capacity) {
  if (!s) { set_error("store is NULL"); return FRG_ERR_INVALID; }
  DeviceGuard g(s->device);
  std::lock_guard<std::mutex> lk(s->mu);
  return grow_locked(s, capacity);
}

int frg_store_stats(frg_store* s, frg_store_stats_t* out) {
  if (!s || !out) { set_error("NULL argument"); return FRG_ERR_INVALID; }
  DeviceGuard g(s->device);
  std::lock_guard<std::mutex> lk(s->mu);
  memset(out, 0, sizeof(*out));
  if (s->live < 0) FRG_CHECK(count_live(s));   // lazily recounted after device-side mutations
  out->rows = s->rows; out->live = s->live; out->capacity = s->capacity; out->version = s->version;
  out->bytes = int64_t(row_bytes(s)) * s->capacity;
  out->dim = s->dim; out->device = s->device; out->flags = s->flags;
  out->faults = s->fault_host ? *s->fault_host : 0u;
  return FRG_OK;
}

// hrows / htags: HOST copies of rows / tags when the caller has them (host_known), for the tenant extents
static int upsert_impl(frg_store* s, const int64_t* rows, const float* vecs, const int32_t* tags,
                       int64_t n, uint32_t flags, void* stream, bool tags_may_be_negative,
                       bool host_known, const int64_t* hrows, const int32_t* htags) {
  if (!s || (n > 0 && !vecs) || n < 0) { set_error("upsert: bad argument"); return FRG_ERR_INVALID; }
  if (n == 0) return FRG_OK;
  DeviceGuard g(s->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::lock_guard<std::mutex> lk(s->mu);
  if (!rows && s->rows + n > s->capacity) FRG_CHECK(grow_locked(s, next_capacity(s->capacity, s->rows + n)));
  FRG_CHECK(store_begin_write(s, st));
  const bool normalise = !(flags & FRG_ROWS_PRENORMALISED) && !(s->flags & FRG_STORE_RAW);
  FRG_CHECK(launch_ingest(vecs, rows, tags, n, s->rows, s->dim, normalise, s->master, s->plane, s->plane8,
                          s->plane_dim, s->gmax_bits, s->tags, st));
  if (host_known) extents_note_upsert(s, hrows, htags, n, s->rows);
  else s->extents_known = false;             // positions / tags live in device memory only
  if (!rows) s->rows += n;
  s->live = -1;
  if (tags && tags_may_be_negative) s->maybe_dead = true;
  return store_end_write(s, st);
}

int frg_store_upsert(frg_store* s, const int64_t* rows, const float* vecs, const int32_t* tags,
                     int64_t n, uint32_t flags, void* stream) {
  // device-resident tags cannot be inspected here: assume they may carry -1 (tombstones)
  return upsert_impl(s, rows, vecs, tags, n, flags, stream, true, !rows && !tags, nullptr, nullptr);
}



// Small host batches (online enrolment: a few templates between query batches, BASELINE config 5) are
// staged through a per-thread ring of pinned bounce buffers: the caller's arrays are copied out at once, the
// H2D copy + ingest are enqueued and the call returns WITHOUT waiting for the device - a match enqueued next
// is ordered after the mutation on the device (store_begin_read).  A slot is reused only after the copy
// that read it has completed (event).  Large batches (bulk loads) keep the direct, synchronous path.
struct PinnedRing {
  static constexpr int kSlots = 4;
  static constexpr size_t kMaxBytes = 4u << 20;
  unsigned char* p[kSlots] = {nullptr, nullptr, nullptr, nullptr};
  size_t cap[kSlots] = {0, 0, 0, 0};
  cudaEvent_t done[kSlots] = {nullptr, nullptr, nullptr, nullptr};
  bool pending[kSlots] = {false, false, false, false};
  int next = 0;
  ~PinnedRing() {
    for (int i = 0; i < kSlots; ++i) {
      if (pending[i]) cudaEventSynchronize(done[i]);
      if (done[i]) cudaEventDestroy(done[i]);
      if (p[i]) cudaFreeHost(p[i]);
    }
  }
  unsigned char* acquire(size_t bytes, int* slot) {
    const int i = next;
    next = (next + 1) % kSlots;
    if (pending[i]) { cudaEventSynchronize(done[i]); pending[i] = false; }
    if (!done[i] && cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming) != cudaSuccess) { done[i] = nullptr; return nullptr; }
    if (bytes > cap[i]) {
      if (p[i]) cudaFreeHost(p[i]);
      p[i] = nullptr; cap[i] = 0;
      const size_t want = (bytes + 65535) & ~size_t(65535);
      if (cudaHostAlloc(reinterpret_cast<void**>(&p[i]), want, cudaHostAllocDefault) != cudaSuccess) { p[i] = nullptr; return nullptr; }
      cap[i] = want;
    }
    *slot = i;
    return p[i];
  }
  void release(int slot, cudaStream_t st) {
    if (cudaEventRecord(done[slot], st) == cudaSuccess) pending[slot] = true;
  }
};
static thread_local PinnedRing g_upload_ring;

int frg_store_upsert_host(frg_store* s, const int64_t* rows, const float* vecs, const int32_t* tags,
                          int64_t n, uint32_t flags) {
  if (!s || (n > 0 && !vecs) || n < 0) { set_error("upsert_host: bad argument"); return FRG_ERR_INVALID; }
  if (n == 0) return FRG_OK;
  DeviceGuard g(s->device);
  {
    std::lock_guard<std::mutex> lk(s->mu);
    if (rows)
      for (int64_t i = 0; i < n; ++i)
        if (rows[i] < 0 || rows[i] >= s->rows) {
          set_error("upsert_host: row %lld out of range [0, %lld)", (long long)rows[i], (long long)s->rows);
          return FRG_ERR_STATE;
        }
  }
  // stream-ordered staging (no cudaMalloc / cudaFree: those synchronise the whole device and would
  // stall every match in flight): one allocation [vecs | rows | tags], ingest
  cudaStream_t st = cudaStreamPerThread;
  const size_t vbytes = size_t(n) * s->dim * sizeof(float);
  const size_t vb = (vbytes + 255) & ~size_t(255);
  const size_t rb = rows ? ((size_t(n) * sizeof(int64_t) + 255) & ~size_t(255)) : 0;
  const size_t tb = tags ? size_t(n) * sizeof(int32_t) : 0;
  bool negative = false;
  if (tags) for (int64_t i = 0; i < n; ++i) negative |= tags[i] < 0;
  unsigned char* d = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&d), vb + rb + tb + 16, st));
  float* dv = reinterpret_cast<float*>(d);
  int64_t* dr = rows ? reinterpret_cast<int64_t*>(d + vb) : nullptr;
  int32_t* dt = tags ? reinterpret_cast<int32_t*>(d + vb + rb) : nullptr;

  int slot = -1;
  unsigned char* h = vb + rb + tb <= PinnedRing::kMaxBytes ? g_upload_ring.acquire(vb + rb + tb, &slot) : nullptr;
  if (h) {
    // asynchronous: the caller's arrays are consumed here, the device is not waited for
    memcpy(h, vecs, vbytes);
    if (rows) memcpy(h + vb, rows, size_t(n) * sizeof(int64_t));
    if (tags) memcpy(h + vb + rb, tags, tb);
    cudaError_t e = cudaMemcpyAsync(d, h, vb + rb + tb, cudaMemcpyHostToDevice, st);
    g_upload_ring.release(slot, st);
    int rc = e == cudaSuccess ? upsert_impl(s, dr, dv, dt, n, flags, st, negative, true, rows, tags)
                              : cuda_fail(e, "upsert_host staging", __FILE__, __LINE__);
    cudaError_t ef = cudaFreeAsync(d, st);
    if (rc == FRG_OK && ef != cudaSuccess) rc = cuda_fail(ef, "cudaFreeAsync", __FILE__, __LINE__);
    return rc;
  }
  (void)cudaGetLastError();
  // bulk load: copy straight from the caller's arrays, one stream synchronize so that they may be reused
  cudaError_t e = cudaMemcpyAsync(dv, vecs, vbytes, cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess && rows) e = cudaMemcpyAsync(dr, rows, size_t(n) * sizeof(int64_t), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess && tags) e = cudaMemcpyAsync(dt, tags, size_t(n) * sizeof(int32_t), cudaMemcpyHostToDevice, st);
  int rc = e == cudaSuccess ? FRG_OK : cuda_fail(e, "upsert_host staging", __FILE__, __LINE__);
  if (rc == FRG_OK) rc = upsert_impl(s, dr, dv, dt, n, flags, st, negative, true, rows, tags);
  cudaError_t ef = cudaFreeAsync(d, st);
  if (rc == FRG_OK) {
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize", __FILE__, __LINE__);
    else if (ef != cudaSuccess) rc = cuda_fail(ef, "cudaFreeAsync", __FILE__, __LINE__);
  }
  return rc;
}

int frg_store_remove(frg_store* s, const int64_t* rows, int64_t n, void* stream) {
  if (!s || (n > 0 && !rows) || n < 0) { set_error("remove: bad argument"); return FRG_ERR_INVALID; }
  if (n == 0) return FRG_OK;
  DeviceGuard g(s->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::lock_guard<std::mutex> lk(s->mu);
  FRG_CHECK(store_begin_write(s, st));
  FRG_CHECK(launch_tombstone(rows, n, s->rows, s->tags, st));
  s->live = -1;
  s->maybe_dead = true;
  return store_end_write(s, st);
}

int frg_store_remove_host(frg_store* s, const int64_t* rows, int64_t n) {
  if (!s || (n > 0 && !rows) || n < 0) { set_error("remove_host: bad argument"); return FRG_ERR_INVALID; }
  if (n == 0) return FRG_OK;
  DeviceGuard g(s->device);
  cudaStream_t st = cudaStreamPerThread;
  const size_t bytes = size_t(n) * sizeof(int64_t);
  int64_t* dr = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&dr), bytes, st));
  int slot = -1;
  unsigned char* h = bytes <= PinnedRing::kMaxBytes ? g_upload_ring.acquire(bytes, &slot) : nullptr;
  if (h) {
    memcpy(h, rows, bytes);                       // asynchronous, as frg_store_upsert_host
    cudaError_t e = cudaMemcpyAsync(dr, h, bytes, cudaMemcpyHostToDevice, st);
    g_upload_ring.release(slot, st);
    int rc = e == cudaSuccess ? frg_store_remove(s, dr, n, st) : cuda_fail(e, "cudaMemcpyAsync", __FILE__, __LINE__);
    cudaFreeAsync(dr, st);
    return rc;
  }
  (void)cudaGetLastError();
  cudaError_t e = cudaMemcpyAsync(dr, rows, bytes, cudaMemcpyHostToDevice, st);
  int rc = e == cudaSuccess ? frg_store_remove(s, dr, n, st) : cuda_fail(e, "cudaMemcpyAsync", __FILE__, __LINE__);
  cudaFreeAsync(dr, st);
  if (rc == FRG_OK) {
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize", __FILE__, __LINE__);
  }
  return rc;
}

int frg_store_compact(frg_store* s, int64_t* old_to_new) {
  if (!s) { set_error("store is NULL"); return FRG_ERR_INVALID; }
  DeviceGuard g(s->device);
  std::lock_guard<std::mutex> lk(s->mu);
  FRG_CUDA(cudaDeviceSynchronize());
  const int64_t n = s->rows;
  std::vector<int32_t> t(static_cast<size_t>(n));
  if (n > 0) FRG_CUDA(cudaMemcpy(t.data(), s->tags, size_t(n) * sizeof(int32_t), cudaMemcpyDeviceToHost));
  std::vector<int64_t> src;
  src.reserve(size_t(n));
  for (int64_t r = 0; r < n; ++r) {
    if (t[size_t(r)] >= 0) {
      if (old_to_new) old_to_new[r] = int64_t(src.size());
      src.push_back(r);
    } else if (old_to_new) {
      old_to_new[r] = -1;
    }
  }
  const int64_t m = int64_t(src.size());
  // the host copy of the tags gives the extents exactly, at the rows' NEW positions - built aside and swapped
  // in only once the rows have really moved: a failed compaction must leave windows that match the data
  std::unordered_map<int32_t, frg_store::Extent> fresh;
  for (int64_t i = 0; i < m; ++i) {
    const int32_t tag = t[size_t(src[size_t(i)])];
    auto it = fresh.find(tag);
    if (it == fresh.end()) fresh.emplace(tag, frg_store::Extent{i, i + 1});
    else it->second.hi = i + 1;
  }
  // Stable compaction IN PLACE, chunk by chunk through a bounce buffer: a row only ever moves to a lower
  // position (src[i] >= i), so once the sources of destination chunk [a, b) sit in the bounce buffer, writing
  // [a, b) cannot touch a source of any later chunk (those are >= b).  No second full-capacity copy: a 100 M-row
  // store compacts with ~200 MB of scratch.  Rows [0, first) stay where they are.
  int64_t first = 0;
  while (first < m && src[size_t(first)] == first) ++first;
  if (first < m) {
    constexpr int64_t chunk_rows = 65536;
    const int64_t chunk = m - first < chunk_rows ? m - first : chunk_rows;
    float* bm; void* bp; int32_t* bt;
    int64_t* dsrc = nullptr;
    FRG_CHECK(alloc_arrays(s, chunk, &bm, &bp, &bt));            // nothing has changed yet if this fails
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&dsrc), size_t(chunk) * sizeof(int64_t));
    if (e != cudaSuccess) { cudaFree(bm); cudaFree(bp); cudaFree(bt); return cuda_fail(e, "compact staging", __FILE__, __LINE__); }
    int rc = FRG_OK;
    for (int64_t a = first; a < m && rc == FRG_OK; a += chunk) {
      const int64_t cnt = m - a < chunk ? m - a : chunk;
      e = cudaMemcpy(dsrc, src.data() + a, size_t(cnt) * sizeof(int64_t), cudaMemcpyHostToDevice);
      if (e != cudaSuccess) { rc = cuda_fail(e, "compact staging", __FILE__, __LINE__); break; }
      rc = launch_gather_rows(dsrc, cnt, s->dim, int(plane_row_bytes(s)), s->master, plane_ptr(s), s->tags, bm, bp, bt,
                              nullptr);
      if (rc != FRG_OK) break;
      if (bm) e = cudaMemcpyAsync(s->master + a * s->dim, bm, size_t(cnt) * s->dim * sizeof(float), cudaMemcpyDeviceToDevice, nullptr);
      if (e == cudaSuccess && bp)
        e = cudaMemcpyAsync(static_cast<unsigned char*>(plane_ptr(s)) + a * plane_row_bytes(s), bp,
                            size_t(cnt) * plane_row_bytes(s), cudaMemcpyDeviceToDevice, nullptr);
      if (e == cudaSuccess) e = cudaMemcpyAsync(s->tags + a, bt, size_t(cnt) * sizeof(int32_t), cudaMemcpyDeviceToDevice, nullptr);
      if (e != cudaSuccess) rc = cuda_fail(e, "compact move", __FILE__, __LINE__);
    }
    if (rc == FRG_OK) {
      e = cudaDeviceSynchronize();
      if (e != cudaSuccess) rc = cuda_fail(e, "cudaDeviceSynchronize", __FILE__, __LINE__);
    }
    cudaFree(dsrc); cudaFree(bm); cudaFree(bp); cudaFree(bt);
    if (rc != FRG_OK) {
      // a device failure in the middle (a sticky CUDA error: the context is gone anyway) - never trust windows
      // computed for a layout that was not reached
      s->extents_known = false;
      return rc;
    }
  }
  s->extents.swap(fresh);
  s->extents_known = true;
  s->spans.clear();
  for (int64_t i = 0; i < m;) {                       // exact runs at the rows' new positions
    const int32_t tag = t[size_t(src[size_t(i)])];
    int64_t j = i + 1;
    while (j < m && t[size_t(src[size_t(j)])] == tag) ++j;
    span_add(s, tag, i, j);
    i = j;
  }
  s->live = m; s->maybe_dead = false;
  if (m != n) { s->rows = m; s->version++; }
  return FRG_OK;
}

int frg_store_read_host(frg_store* s, int64_t row0, int64_t n, float* vecs, int32_t* tags) {
  if (!s || n < 0 || row0 < 0) { set_error("read_host: bad argument"); return FRG_ERR_INVALID; }
  DeviceGuard g(s->device);
  std::lock_guard<std::mutex> lk(s->mu);
  if (row0 + n > s->rows) { set_error("read_host: rows [%lld, %lld) beyond %lld", (long long)row0, (long long)(row0 + n), (long long)s->rows); return FRG_ERR_STATE; }
  FRG_CUDA(cudaDeviceSynchronize());
  if (n == 0) return FRG_OK;
  if (vecs && s->master) {
    FRG_CUDA(cudaMemcpy(vecs, s->master + row0 * s->dim, size_t(n) * s->dim * sizeof(float), cudaMemcpyDeviceToHost));
  } else if (vecs) {
    // bf16-only store: copy the plane and widen on the host (bf16 -> fp32 is exact)
    std::vector<uint16_t> h(size_t(n) * s->dim);
    FRG_CUDA(cudaMemcpy(h.data(), s->plane + row0 * s->dim, h.size() * sizeof(uint16_t), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < h.size(); ++i) {
      const uint32_t b = uint32_t(h[i]) << 16;
      memcpy(vecs + i, &b, sizeof(float));
    }
  }
  if (tags) FRG_CUDA(cudaMemcpy(tags, s->tags + row0, size_t(n) * sizeof(int32_t), cudaMemcpyDeviceToHost));
  return FRG_OK;
}

int frg_store_fill_synthetic(frg_store* s, int64_t n, int64_t global_row0, uint64_t seed, int32_t tag,
                             void* stream) {
  if (!s || n < 0) { set_error("fill_synthetic: bad argument"); return FRG_ERR_INVALID; }
  if (s->dim > 1024) { set_error("fill_synthetic: dim > 1024 not built"); return FRG_ERR_UNSUPPORTED; }
  if (n == 0) return FRG_OK;
  DeviceGuard g(s->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::lock_guard<std::mutex> lk(s->mu);
  if (s->rows + n > s->capacity) FRG_CHECK(grow_locked(s, s->rows + n));
  FRG_CHECK(store_begin_write(s, st));
  FRG_CHECK(launch_synth(n, s->rows, global_row0, seed, tag, s->dim, s->master, s->plane, s->plane8, s->plane_dim,
                         s->gmax_bits, s->tags, st));
  extent_add(s, tag, s->rows, s->rows + n);
  span_add(s, tag, s->rows, s->rows + n);
  s->rows += n;
  if (s->live >= 0 && tag >= 0) s->live += n;
  if (tag < 0) s->maybe_dead = true;
  return store_end_write(s, st);
}

// --------------------------------------------------------------------------------------------- match
static int pick_variant(const frg_store* s, const frg_match_params_t* p, int nq) {
  const char* why = "";
  // Raw stores queried with the cosine metric (cluster means) and caller-normalised queries always
  // take the exact scan.
  // Cosine filter: its error bound assumes unit rows and queries.  Euclidean filter: needs the raw
  // store's augmented plane (norm terms), its bound scales with the norms (queries.cu).
  const bool unit = !(s->flags & FRG_STORE_RAW) && !(p->flags & FRG_QUERY_PRENORMALISED);
  const bool fits = p->metric == FRG_METRIC_EUCLIDEAN ? s->plane_dim == s->dim + kEuclidPad : unit;
  const bool tc_ok = (p->metric == FRG_METRIC_EUCLIDEAN ? s->plane != nullptr : (s->plane || s->plane8)) && fits &&
                     tc_supported(s->dim, p->metric, &why);
  if (p->variant != FRG_VARIANT_AUTO) return p->variant;
  if (!s->master) return FRG_VARIANT_TC_BF16;          // bf16-only store: the coarse scores are the scores
  // dispatch table (DESIGN.md): the tensor-core filter reads 1 B/element (int8 plane) instead of 4 and wins from
  // the smallest batches on; the exact scan remains for galleries without a scan plane, for the
  // Euclidean metric and for dims the tile shapes do not cover.
  (void)nq;
  return tc_ok ? FRG_VARIANT_TC_EXACT : FRG_VARIANT_SCAN_F32;
}

// Row-sharded gallery: where the local result goes next.  active: out_rows / out_scores of the match are the
// caller's LOCAL scratch, the merged result of all ranks goes to fin_*.
struct ExchangeTail {
  bool active = false;
  bool merge = true;       // false: FRG_XCHG_PUSH_ONLY - push this shard's result, the caller merges later
  XPush x;
  int64_t* fin_rows = nullptr;
  float* fin_scores = nullptr;
  uint8_t* fin_accept = nullptr;
};

static int match_scan(const GalleryWindow* s, const float* q, int nq, int k, const frg_match_params_t* p, int sm_count,
                      int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st,
                      const ExchangeTail& tail = ExchangeTail()) {
  if (!s->master && s->rows > 0) {
    set_error("match: a bf16-only store has no fp32 master for the exact scan (use FRG_VARIANT_TC_BF16 / AUTO)");
    return FRG_ERR_UNSUPPORTED;
  }
  ScanArgs a;
  a.master = s->master; a.tags = s->tags; a.rows = s->rows; a.dim = s->dim;
  a.nq = nq; a.k = k; a.metric = p->metric; a.tenant = p->tenant; a.sm_count = sm_count;
  size_t part_bytes = 0;
  FRG_CHECK(scan_f32_workspace_bytes(a, &part_bytes));
  const size_t qn_bytes = (size_t(nq) * s->dim * sizeof(float) + 255) & ~size_t(255);
  unsigned char* ws = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), qn_bytes + part_bytes, st));
  float* qn = reinterpret_cast<float*>(ws);
  a.qn = qn;
  int rc = launch_normalise_queries(q, nq, s->dim, p->metric == FRG_METRIC_COSINE && !(p->flags & FRG_QUERY_PRENORMALISED), qn, nullptr, nullptr, nullptr, nullptr, st);
  if (rc == FRG_OK)
    rc = launch_scan_f32(a, ws + qn_bytes, p->row_offset, p->threshold, out_rows, out_scores, out_accept, st);
  if (rc == FRG_OK && tail.active)       // no select stage here: a push kernel sends every query (and the hello)
    rc = launch_exchange_push(tail.x, out_rows, out_scores, nq, k, sm_count, st);
  if (rc == FRG_OK && tail.active && tail.merge)
    rc = launch_exchange_merge(tail.x, nq, k, p->metric, p->threshold, sm_count, tail.fin_rows, tail.fin_scores,
                               tail.fin_accept, st);
  g_variant = "scan_f32";
  cudaError_t e = cudaFreeAsync(ws, st);
  if (rc == FRG_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync", __FILE__, __LINE__);
  return rc;
}

static int match_tc(const GalleryWindow* s, const float* q, int nq, int k, const frg_match_params_t* p, bool rescore,
                    int sm_count, int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st,
                    const ExchangeTail& tail = ExchangeTail()) {
  const char* why = "";
  const bool euclid = p->metric == FRG_METRIC_EUCLIDEAN;
  if (!s->plane && !s->plane8) { set_error("match: the store was created without FRG_STORE_BF16_PLANE"); return FRG_ERR_UNSUPPORTED; }
  if (!tc_supported(s->dim, p->metric, &why)) { set_error("match: %s", why); return FRG_ERR_UNSUPPORTED; }
  if (euclid) {
    if (!s->plane || s->plane_dim != s->dim + kEuclidPad) {
      set_error("match: the Euclidean tensor-core filter needs a FRG_STORE_RAW store with a scan plane");
      return FRG_ERR_UNSUPPORTED;
    }
    if (!rescore) {
      set_error("match: FRG_VARIANT_TC_BF16 is cosine-only (a distance from the bf16 score would cancel near d = 0)");
      return FRG_ERR_UNSUPPORTED;
    }
  } else if ((s->flags & FRG_STORE_RAW) || (p->flags & FRG_QUERY_PRENORMALISED)) {
    set_error("match: the cosine tensor-core variants need unit-norm rows and queries (raw store / prenormalised query given)");
    return FRG_ERR_UNSUPPORTED;
  }
  if (s->rows > 0x7fffffff) { set_error("match: more than 2^31-1 rows in one shard"); return FRG_ERR_UNSUPPORTED; }
  if (s->rows == 0) return match_scan(s, q, nq, k, p, sm_count, out_rows, out_scores, out_accept, st, tail);
  if (rescore && !s->master) {
    set_error("match: FRG_VARIANT_TC_EXACT needs the fp32 master; this store is bf16-only");
    return FRG_ERR_UNSUPPORTED;
  }
  const char* variant_name = rescore ? "tc_exact" : "tc_bf16";
  // int8 plane (unit store with a master): there are no bf16 scores to return - FRG_VARIANT_TC_BF16 is served
  // with exact scores, which meet its tolerance a fortiori
  const bool i8 = !euclid && s->plane8 != nullptr;
  if (i8) rescore = true;
  const size_t qn_bytes = (size_t(nq) * s->dim * sizeof(float) + 255) & ~size_t(255);
  const size_t qb_bytes = (size_t(nq) * (s->dim + (euclid ? kEuclidQPad : 0)) * (i8 ? 1 : sizeof(__nv_bfloat16)) + 255) & ~size_t(255);
  const size_t eps_bytes = (size_t(nq) * sizeof(float) + 255) & ~size_t(255);     // per-query filter error bound
  const size_t qb2_bytes = euclid ? qb_bytes : 0;                                 // the pre-pass (lower-bound) image
  // Euclidean: the bound coefficients [nq][4]; int8: the per-query step of the integer scores [nq]
  const size_t coef_bytes = euclid ? ((size_t(nq) * 4 * sizeof(float) + 255) & ~size_t(255)) : i8 ? eps_bytes : 0;
  const int32_t* tile_list = nullptr;
  int n_list = 0;
  const int64_t plan_rows = tc_effective_rows(s, nq, st, &tile_list, &n_list);
  if (plan_rows < 0) return FRG_ERR_CUDA;
  const int plan_dim = euclid ? -s->dim : s->dim;          // (negative: Euclidean plane, tc_plan)
  const size_t tc_bytes = tc_workspace_bytes(plan_rows, plan_dim, nq, k, sm_count, false, i8);
  unsigned char* ws = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), qn_bytes + qb_bytes + eps_bytes + qb2_bytes + coef_bytes + tc_bytes, st));
  float* qn = reinterpret_cast<float*>(ws);
  __nv_bfloat16* qb = reinterpret_cast<__nv_bfloat16*>(ws + qn_bytes);
  float* eps = reinterpret_cast<float*>(ws + qn_bytes + qb_bytes);
  __nv_bfloat16* qb2 = euclid ? reinterpret_cast<__nv_bfloat16*>(ws + qn_bytes + qb_bytes + eps_bytes) : nullptr;
  float* coef = (euclid || i8) ? reinterpret_cast<float*>(ws + qn_bytes + qb_bytes + eps_bytes + qb2_bytes) : nullptr;
  unsigned char* tc_ws = ws + qn_bytes + qb_bytes + eps_bytes + qb2_bytes + coef_bytes;
  int* flagged = nullptr; int* n_flagged = nullptr;
  void* keys = nullptr; int* ct0 = nullptr; int* nf0 = nullptr;
  tc_workspace_init_targets(plan_rows, plan_dim, nq, k, sm_count, tc_ws, &keys, &ct0, &nf0, false, i8);
  int8_t* qi8 = i8 ? reinterpret_cast<int8_t*>(qb) : nullptr;
  profile_begin(st, kStagePrep);
  int rc = euclid ? launch_prepare_queries_euclid(q, nq, s->dim, s->gmax_bits, qn, qb, qb2, coef, eps,
                                                  static_cast<uint32_t*>(keys), ct0, nf0, st)
           : i8   ? launch_prepare_queries_i8(q, nq, s->dim, qn, qi8, coef, eps, s->gmax_bits,
                                              static_cast<unsigned long long*>(keys), ct0, nf0, st)
                  : launch_normalise_queries(q, nq, s->dim, !(p->flags & FRG_QUERY_PRENORMALISED), qn, qb,
                                             static_cast<uint32_t*>(keys), ct0, nf0, st, eps, s->gmax_bits);
  profile_end(st, 1);
  if (rc == FRG_OK)
    rc = launch_tc_match(s, p->metric, qn, i8 ? nullptr : qb, eps, nq, k, p->tenant, rescore, p->threshold,
                         p->row_offset, tc_ws, sm_count, tail.active ? tail.x : XPush(), out_rows, out_scores,
                         out_accept, &flagged, &n_flagged, st, plan_rows, tile_list, n_list, qb2,
                         euclid ? coef : nullptr, qi8, i8 ? coef : nullptr);
  if (rc == FRG_OK) {
    // queries whose candidate lists overflowed are redone exactly, inside the same enqueue
    ScanArgs a;
    a.master = s->master; a.plane = s->plane; a.tags = s->tags; a.rows = s->rows; a.dim = s->dim;
    a.qn = qn; a.nq = nq; a.k = k; a.metric = p->metric; a.tenant = p->tenant; a.sm_count = sm_count;
    profile_begin(st, kStageFallback);
    rc = launch_scan_f32_flagged(a, flagged, n_flagged, p->row_offset, p->threshold,
                                 tail.active ? tail.x : XPush(), out_rows, out_scores, out_accept, st);
    profile_end(st, 1);
  }
  if (rc == FRG_OK && tail.active && tail.merge)
    // select has pushed every query it settled, the fallback's last CTA the ones it redid: what is left is
    // to wait for every rank's packets and merge each query's `world` lists as they arrive
    rc = launch_exchange_merge(tail.x, nq, k, p->metric, p->threshold, sm_count, tail.fin_rows, tail.fin_scores,
                               tail.fin_accept, st);
  g_variant = variant_name;
  cudaError_t e = cudaFreeAsync(ws, st);
  if (rc == FRG_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync", __FILE__, __LINE__);
  return rc;
}

// the match itself, s->mu held and the read ordered (store_begin_read)
static int match_locked(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                        int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st,
                        const ExchangeTail& tail, int sm_count) {
  struct SeqBump { ~SeqBump() { ++g_match_seq; } } bump;      // sampled profiling: every 4th match is bracketed
  // a tenant-filtered call scans only the rows that tenant can sit in (the whole gallery otherwise)
  const int variant = pick_variant(s, p, nq);
  const GalleryWindow w = window_of(s, p->tenant, variant == FRG_VARIANT_TC_EXACT || variant == FRG_VARIANT_TC_BF16);
  frg_match_params_t pw = *p;
  pw.row_offset += w.row0;
  switch (variant) {
    case FRG_VARIANT_SCAN_F32:
      return match_scan(&w, q, nq, k, &pw, sm_count, out_rows, out_scores, out_accept, st, tail);
    case FRG_VARIANT_TC_EXACT:
      return match_tc(&w, q, nq, k, &pw, true, sm_count, out_rows, out_scores, out_accept, st, tail);
    case FRG_VARIANT_TC_BF16:
      return match_tc(&w, q, nq, k, &pw, false, sm_count, out_rows, out_scores, out_accept, st, tail);
    default:
      set_error("match: unknown variant %d", p->variant);
      return FRG_ERR_INVALID;
  }
}

static int match_impl(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                      int64_t* out_rows, float* out_scores, uint8_t* out_accept, void* stream,
                      const ExchangeTail& tail) {
  reset_launches();
  if (!s || !p || nq < 0 || (nq > 0 && (!q || !out_rows || !out_scores))) { set_error("match: bad argument"); return FRG_ERR_INVALID; }
  if (k < 1 || k > FRG_MAX_K) { set_error("match: k=%d out of range 1..%d", k, FRG_MAX_K); return FRG_ERR_INVALID; }
  if (p->metric != FRG_METRIC_COSINE && p->metric != FRG_METRIC_EUCLIDEAN) { set_error("match: unknown metric %d", p->metric); return FRG_ERR_INVALID; }
  if (nq == 0) return FRG_OK;
  DeviceGuard g(s->device);
  if (!g.ok) { set_error("cannot select device %d", s->device); return FRG_ERR_CUDA; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceInfo di;
  FRG_CHECK(device_info(s->device, &di));

  std::lock_guard<std::mutex> lk(s->mu);   // enqueue under the lock: the snapshot a match sees is the
                                           // store as of this call (peopleCount.py:816-819 semantics)
  FRG_CHECK(store_begin_read(s, st));
  return match_locked(s, q, nq, k, p, out_rows, out_scores, out_accept, st, tail, di.sm_count);
}

int frg_match(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
              int64_t* out_rows, float* out_scores, uint8_t* out_accept, void* stream) {
  return match_impl(s, q, nq, k, p, out_rows, out_scores, out_accept, stream, ExchangeTail());
}

// ---- per-query tenants (frg_match_tenants)
}  // extern "C"

int frg::stage_upload(void* dev, const void* host, size_t bytes, cudaStream_t st) {
  if (bytes == 0) return FRG_OK;
  int slot = -1;
  unsigned char* h = bytes <= PinnedRing::kMaxBytes ? g_upload_ring.acquire(bytes, &slot) : nullptr;
  if (!h) {
    (void)cudaGetLastError();
    FRG_CUDA(cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, st));   // pageable: staged before it returns
    return FRG_OK;
  }
  memcpy(h, host, bytes);
  cudaError_t e = cudaMemcpyAsync(dev, h, bytes, cudaMemcpyHostToDevice, st);
  g_upload_ring.release(slot, st);
  if (e != cudaSuccess) return cuda_fail(e, "stage_upload", __FILE__, __LINE__);
  return FRG_OK;
}

extern "C" {

// Tiles a tenant's rows can sit in, in kTcTileRows-row tiles: its cached tile list when that is shorter than its
// extent's tile range, else that range (other tenants' rows in it are masked by the filter's tag check), else every
// tile (tenant < 0, or extents not known).  A tag no row carries: no tiles.  s->mu held.
static int tenant_tiles(frg_store* s, int32_t tenant, cudaStream_t st, TcTenantGroup* g) {
  g->tile0 = 0; g->n_tiles = int((s->rows + kTcTileRows - 1) / kTcTileRows); g->list = nullptr;
  if (tenant < 0 || !s->extents_known) return FRG_OK;
  auto it = s->extents.find(tenant);
  const int64_t lo = it != s->extents.end() ? it->second.lo : 0;
  const int64_t hi = it != s->extents.end() ? (it->second.hi < s->rows ? it->second.hi : s->rows) : 0;
  if (hi <= lo) { g->n_tiles = 0; return FRG_OK; }
  g->tile0 = int(lo / kTcTileRows);
  g->n_tiles = int((hi - 1) / kTcTileRows) - g->tile0 + 1;
  const int32_t* list = nullptr;
  int n = 0;
  FRG_CHECK(store_tile_list(s, tenant, kTcTileRows, st, &list, &n));
  if (list && n < g->n_tiles) { g->list = list; g->n_tiles = n; }
  return FRG_OK;
}

static int match_tenants_impl(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                              const int32_t* tenants, int64_t* out_rows, float* out_scores, uint8_t* out_accept,
                              cudaStream_t st) {
  reset_launches();
  if (!s || !p || nq < 0 || (nq > 0 && (!q || !out_rows || !out_scores || !tenants))) {
    set_error("match_tenants: bad argument");
    return FRG_ERR_INVALID;
  }
  if (k < 1 || k > FRG_MAX_K) { set_error("match: k=%d out of range 1..%d", k, FRG_MAX_K); return FRG_ERR_INVALID; }
  if (p->metric != FRG_METRIC_COSINE && p->metric != FRG_METRIC_EUCLIDEAN) { set_error("match: unknown metric %d", p->metric); return FRG_ERR_INVALID; }
  if (nq == 0) return FRG_OK;
  // stable sort by tenant (every negative tag means "all tenants")
  auto norm = [&](int32_t i) { return tenants[i] < 0 ? int32_t(-1) : tenants[i]; };
  std::vector<int32_t> perm(static_cast<size_t>(nq));
  for (int32_t i = 0; i < nq; ++i) perm[size_t(i)] = i;
  std::stable_sort(perm.begin(), perm.end(), [&](int32_t a, int32_t b) { return norm(a) < norm(b); });
  frg_match_params_t pg = *p;
  if (norm(perm.front()) == norm(perm.back())) {            // one tenant: exactly frg_match
    pg.tenant = norm(perm.front());
    return match_impl(s, q, nq, k, &pg, out_rows, out_scores, out_accept, st, ExchangeTail());
  }
  std::vector<TcTenantGroup> groups;
  for (int32_t i = 0; i < nq;) {
    int32_t j = i + 1;
    while (j < nq && norm(perm[size_t(j)]) == norm(perm[size_t(i)])) ++j;
    TcTenantGroup g{};
    g.tenant = norm(perm[size_t(i)]); g.q0 = i; g.nq = j - i;
    groups.push_back(g);
    i = j;
  }
  DeviceGuard dg(s->device);
  if (!dg.ok) { set_error("cannot select device %d", s->device); return FRG_ERR_CUDA; }
  DeviceInfo di;
  FRG_CHECK(device_info(s->device, &di));
  std::lock_guard<std::mutex> lk(s->mu);    // one snapshot of the store for every tenant of the call
  FRG_CHECK(store_begin_read(s, st));
  const int variant = pick_variant(s, p, nq);
  const char* why = "";
  const bool grouped = (variant == FRG_VARIANT_TC_EXACT || variant == FRG_VARIANT_TC_BF16) && has_plane8(s) &&
                       s->master && p->metric == FRG_METRIC_COSINE && !(p->flags & FRG_QUERY_PRENORMALISED) &&
                       tc_supported(s->dim, p->metric, &why) && s->rows > 0 && s->rows <= 0x7fffffff;
  if (grouped) {
    struct SeqBump { ~SeqBump() { ++g_match_seq; } } bump;
    for (TcTenantGroup& g : groups) FRG_CHECK(tenant_tiles(s, g.tenant, st, &g));
    const GalleryWindow w = window_of(s, -1);
    FRG_CHECK(launch_tc_match_grouped(&w, q, perm, groups, k, p->threshold, p->row_offset, di.sm_count, out_rows,
                                      out_scores, out_accept, st));
    g_variant = "tc_exact_grouped";
    return FRG_OK;
  }
  // every other store / variant: frg_match's own path once per tenant, into tenant-sorted scratch, then scattered
  const size_t qb = (size_t(nq) * s->dim * 4 + 255) & ~size_t(255), pb = (size_t(nq) * 4 + 255) & ~size_t(255);
  const size_t rb = (size_t(nq) * k * 8 + 255) & ~size_t(255), sb = (size_t(nq) * k * 4 + 255) & ~size_t(255);
  unsigned char* ws = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), qb + pb + rb + sb + size_t(nq), st));
  float* qs = reinterpret_cast<float*>(ws);
  int32_t* dperm = reinterpret_cast<int32_t*>(ws + qb);
  int64_t* srows = reinterpret_cast<int64_t*>(ws + qb + pb);
  float* sscores = reinterpret_cast<float*>(ws + qb + pb + rb);
  uint8_t* sacc = ws + qb + pb + rb + sb;
  int rc = stage_upload(dperm, perm.data(), size_t(nq) * 4, st);
  if (rc == FRG_OK) rc = launch_gather_queries(q, dperm, nq, s->dim, qs, st);
  for (size_t i = 0; rc == FRG_OK && i < groups.size(); ++i) {
    pg.tenant = groups[i].tenant;
    const int q0 = groups[i].q0;
    rc = match_locked(s, qs + size_t(q0) * s->dim, groups[i].nq, k, &pg, srows + size_t(q0) * k,
                      sscores + size_t(q0) * k, sacc + q0, st, ExchangeTail(), di.sm_count);
  }
  const char* ran = g_variant;               // the per-tenant path that ran (the scatter does not rename it)
  if (rc == FRG_OK) rc = launch_scatter_results(srows, sscores, sacc, dperm, nq, k, out_rows, out_scores, out_accept, st);
  g_variant = ran;
  cudaError_t e = cudaFreeAsync(ws, st);
  if (rc == FRG_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync", __FILE__, __LINE__);
  return rc;
}

int frg_match_tenants(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                      const int32_t* tenants, int64_t* out_rows, float* out_scores, uint8_t* out_accept, void* stream) {
  return match_tenants_impl(s, q, nq, k, p, tenants, out_rows, out_scores, out_accept, static_cast<cudaStream_t>(stream));
}

static int check_exchange(const frg_exchange_t* x, int32_t nq, int32_t k, XPush* out) {
  if (!x || x->world < 1 || x->world > kExchangeMaxWorld || x->rank < 0 || x->rank >= x->world || !x->peer_bufs) {
    set_error("exchange: bad descriptor (world 1..%d)", kExchangeMaxWorld);
    return FRG_ERR_INVALID;
  }
  if ((x->flags & 0xffu) & ~uint32_t(FRG_XCHG_PUSH_ONLY | FRG_XCHG_MERGE_ONLY) ||
      (x->flags & FRG_XCHG_PUSH_ONLY && x->flags & FRG_XCHG_MERGE_ONLY)) {
    set_error("exchange: bad flags 0x%x", x->flags);
    return FRG_ERR_INVALID;
  }
  if (nq >= (1 << 27)) { set_error("exchange: nq too large for the hello word"); return FRG_ERR_INVALID; }
  if (x->epoch == 0) { set_error("exchange: epochs start at 1 (the buffers are zero-initialised)"); return FRG_ERR_INVALID; }
  if (x->block_cap < int64_t(nq) * k * 24 || x->block_cap % 8) { set_error("exchange: block_cap too small / unaligned"); return FRG_ERR_INVALID; }
  out->peer_bufs = reinterpret_cast<unsigned char* const*>(x->peer_bufs);
  out->rank = x->rank; out->world = x->world; out->epoch = x->epoch;
  out->block_cap = x->block_cap;
  exchange_fill_defaults(out, nq, k);
  if (x->flags >> 8) out->timeout_ns = (unsigned long long)(x->flags >> 8) * 1000000ull;    // FRG_XCHG_TIMEOUT_MS
  return FRG_OK;
}

int frg_match_exchange(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                       const frg_exchange_t* x, int64_t* local_rows, float* local_scores,
                       int64_t* out_rows, float* out_scores, uint8_t* out_accept, void* stream) {
  if (nq > 0 && (!local_rows || !local_scores)) { set_error("match_exchange: local scratch is NULL"); return FRG_ERR_INVALID; }
  if (nq < 0 || k < 1 || k > FRG_MAX_K) { set_error("match_exchange: bad nq / k"); return FRG_ERR_INVALID; }
  ExchangeTail tail;
  FRG_CHECK(check_exchange(x, nq, k, &tail.x));
  tail.active = true;
  tail.merge = !(x->flags & FRG_XCHG_PUSH_ONLY);
  tail.fin_rows = out_rows; tail.fin_scores = out_scores; tail.fin_accept = out_accept;
  if (nq > 0 && tail.merge && (!out_rows || !out_scores)) { set_error("match_exchange: bad argument"); return FRG_ERR_INVALID; }
  if (x->flags & FRG_XCHG_MERGE_ONLY) {
    // this shard's result of the call went out earlier (FRG_XCHG_PUSH_ONLY): only wait and merge
    reset_launches();
    if (!s || !p) { set_error("match_exchange: bad argument"); return FRG_ERR_INVALID; }
    if (nq == 0) return FRG_OK;
    DeviceGuard g(s->device);
    if (!g.ok) { set_error("cannot select device %d", s->device); return FRG_ERR_CUDA; }
    DeviceInfo di;
    FRG_CHECK(device_info(s->device, &di));
    return launch_exchange_merge(tail.x, nq, k, p->metric, p->threshold, di.sm_count, out_rows, out_scores,
                                 out_accept, static_cast<cudaStream_t>(stream));
  }
  // the local stage writes this shard's own top-k (global rows) into the scratch; no local decision is kept
  return match_impl(s, q, nq, k, p, local_rows, local_scores, nullptr, stream, tail);
}

// Per-thread pinned bounce buffer for results: ONE device->host copy per match instead of three, at full
// PCIe rate whether or not the caller's arrays are pinned.  Grow-only; released with the thread.
struct PinnedScratch {
  unsigned char* p = nullptr;
  size_t cap = 0;
  ~PinnedScratch() { if (p) cudaFreeHost(p); }
  unsigned char* get(size_t bytes) {
    if (bytes > cap) {
      if (p) cudaFreeHost(p);
      p = nullptr; cap = 0;
      const size_t want = (bytes + 65535) & ~size_t(65535);
      if (cudaHostAlloc(reinterpret_cast<void**>(&p), want, cudaHostAllocDefault) != cudaSuccess) { p = nullptr; return nullptr; }
      cap = want;
    }
    return p;
  }
};
static thread_local PinnedScratch g_result_bounce;

// tenants == nullptr: frg_match, else frg_match_tenants
static int match_host_impl(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                           const int32_t* tenants, int64_t* out_rows, float* out_scores, uint8_t* out_accept) {
  if (k < 1 || k > FRG_MAX_K) { set_error("match: k=%d out of range 1..%d", k, FRG_MAX_K); return FRG_ERR_INVALID; }
  if (nq == 0) return FRG_OK;
  DeviceGuard g(s->device);
  cudaStream_t st = cudaStreamPerThread;
  const size_t qb = size_t(nq) * s->dim * sizeof(float);
  const size_t rb = size_t(nq) * k * sizeof(int64_t), sb = size_t(nq) * k * sizeof(float), ab = size_t(nq);
  const size_t o_r = (qb + 255) & ~size_t(255), o_s = (o_r + rb + 255) & ~size_t(255), o_a = (o_s + sb + 255) & ~size_t(255);
  unsigned char* d = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&d), o_a + ab, st));
  int rc = FRG_OK;
  cudaError_t e = cudaMemcpyAsync(d, q, qb, cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) rc = cuda_fail(e, "H2D queries", __FILE__, __LINE__);
  if (rc == FRG_OK)
    rc = tenants ? match_tenants_impl(s, reinterpret_cast<float*>(d), nq, k, p, tenants, reinterpret_cast<int64_t*>(d + o_r),
                                      reinterpret_cast<float*>(d + o_s), d + o_a, st)
                 : frg_match(s, reinterpret_cast<float*>(d), nq, k, p, reinterpret_cast<int64_t*>(d + o_r),
                             reinterpret_cast<float*>(d + o_s), d + o_a, st);
  if (rc == FRG_OK) {
    // rows | scores | accept sit in one device range [o_r, o_a + ab): one copy into the pinned bounce
    const size_t span = o_a + ab - o_r;
    unsigned char* h = g_result_bounce.get(span);
    if (h) {
      e = cudaMemcpyAsync(h, d + o_r, span, cudaMemcpyDeviceToHost, st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);
      if (e == cudaSuccess) {
        memcpy(out_rows, h, rb);
        memcpy(out_scores, h + (o_s - o_r), sb);
        if (out_accept) memcpy(out_accept, h + (o_a - o_r), ab);
      }
    } else {
      (void)cudaGetLastError();        // no pinned memory to be had: three direct copies
      e = cudaMemcpyAsync(out_rows, d + o_r, rb, cudaMemcpyDeviceToHost, st);
      if (e == cudaSuccess) e = cudaMemcpyAsync(out_scores, d + o_s, sb, cudaMemcpyDeviceToHost, st);
      if (e == cudaSuccess && out_accept) e = cudaMemcpyAsync(out_accept, d + o_a, ab, cudaMemcpyDeviceToHost, st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (e != cudaSuccess) rc = cuda_fail(e, "D2H results", __FILE__, __LINE__);
    else rc = store_fault(s);
  }
  cudaFreeAsync(d, st);
  return rc;
}

int frg_match_host(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                   int64_t* out_rows, float* out_scores, uint8_t* out_accept) {
  if (!s || nq < 0 || (nq > 0 && (!q || !out_rows || !out_scores))) { set_error("match_host: bad argument"); return FRG_ERR_INVALID; }
  return match_host_impl(s, q, nq, k, p, nullptr, out_rows, out_scores, out_accept);
}

int frg_match_tenants_host(frg_store* s, const float* q, int32_t nq, int32_t k, const frg_match_params_t* p,
                           const int32_t* tenants, int64_t* out_rows, float* out_scores, uint8_t* out_accept) {
  if (!s || !p || nq < 0 || (nq > 0 && (!q || !out_rows || !out_scores || !tenants))) {
    set_error("match_tenants_host: bad argument");
    return FRG_ERR_INVALID;
  }
  return match_host_impl(s, q, nq, k, p, tenants, out_rows, out_scores, out_accept);
}

int frg_first_match(frg_store* s, const float* q, int32_t nq, const frg_match_params_t* p,
                    int64_t* out_rows, float* out_scores, void* stream) {
  reset_launches();
  if (!s || !p || nq < 0 || (nq > 0 && (!q || !out_rows || !out_scores))) { set_error("first_match: bad argument"); return FRG_ERR_INVALID; }
  if (p->metric != FRG_METRIC_COSINE) { set_error("first_match: cosine / dot only"); return FRG_ERR_UNSUPPORTED; }
  if (!s->master) { set_error("first_match: needs the fp32 master; this store is bf16-only"); return FRG_ERR_UNSUPPORTED; }
  if (nq == 0) return FRG_OK;
  DeviceGuard g(s->device);
  if (!g.ok) { set_error("cannot select device %d", s->device); return FRG_ERR_CUDA; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DeviceInfo di;
  FRG_CHECK(device_info(s->device, &di));
  std::lock_guard<std::mutex> lk(s->mu);
  FRG_CHECK(store_begin_read(s, st));
  const size_t qn_bytes = (size_t(nq) * s->dim * sizeof(float) + 255) & ~size_t(255);
  unsigned char* ws = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), qn_bytes + size_t(nq) * 8, st));
  float* qn = reinterpret_cast<float*>(ws);
  int rc = launch_normalise_queries(q, nq, s->dim, !(p->flags & FRG_QUERY_PRENORMALISED), qn, nullptr, nullptr,
                                    nullptr, nullptr, st);
  const GalleryWindow w = window_of(s, p->tenant);
  if (rc == FRG_OK)
    rc = launch_first_match(w.master, w.tags, w.rows, s->dim, qn, nq, p->tenant, p->threshold,
                            (p->flags & FRG_FIRST_STRICT) != 0, p->row_offset + w.row0,
                            reinterpret_cast<unsigned long long*>(ws + qn_bytes), di.sm_count, out_rows, out_scores, st);
  cudaError_t e = cudaFreeAsync(ws, st);
  if (rc == FRG_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync", __FILE__, __LINE__);
  return rc;
}

int frg_first_match_host(frg_store* s, const float* q, int32_t nq, const frg_match_params_t* p,
                         int64_t* out_rows, float* out_scores) {
  if (!s || nq < 0 || (nq > 0 && (!q || !out_rows || !out_scores))) { set_error("first_match_host: bad argument"); return FRG_ERR_INVALID; }
  if (nq == 0) return FRG_OK;
  DeviceGuard g(s->device);
  cudaStream_t st = cudaStreamPerThread;
  const size_t qb = size_t(nq) * s->dim * sizeof(float);
  const size_t o_r = (qb + 255) & ~size_t(255), o_s = o_r + ((size_t(nq) * 8 + 255) & ~size_t(255));
  unsigned char* d = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&d), o_s + size_t(nq) * 4, st));
  int rc = FRG_OK;
  cudaError_t e = cudaMemcpyAsync(d, q, qb, cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) rc = cuda_fail(e, "H2D queries", __FILE__, __LINE__);
  if (rc == FRG_OK)
    rc = frg_first_match(s, reinterpret_cast<float*>(d), nq, p, reinterpret_cast<int64_t*>(d + o_r),
                         reinterpret_cast<float*>(d + o_s), st);
  if (rc == FRG_OK) {
    e = cudaMemcpyAsync(out_rows, d + o_r, size_t(nq) * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_scores, d + o_s, size_t(nq) * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = cuda_fail(e, "D2H results", __FILE__, __LINE__);
  }
  cudaFreeAsync(d, st);
  return rc;
}

// --------------------------------------------------------------------------------------------- range search
// Tensor-core path (unit cosine stores with a plane and a covered dim): query prep (fp32 unit queries, int8 image,
// eps[q]) -> filter with the fixed floor threshold - eps[q] -> range_select_kernel -> exact range scan of the
// queries whose candidates overflowed.  Everything else: the exact range scan over all queries.
static int range_impl(frg_store* s, const float* q, int32_t nq, int32_t max_hits, const frg_match_params_t* p,
                      int64_t* out_counts, int64_t* out_rows, float* out_scores, cudaStream_t st) {
  reset_launches();
  if (!s || !p || nq < 0 || (nq > 0 && (!q || !out_counts || !out_rows || !out_scores))) {
    set_error("match_range: bad argument");
    return FRG_ERR_INVALID;
  }
  if (max_hits < 1) { set_error("match_range: max_hits=%d must be >= 1", max_hits); return FRG_ERR_INVALID; }
  if (p->metric != FRG_METRIC_COSINE && p->metric != FRG_METRIC_EUCLIDEAN) { set_error("match_range: unknown metric %d", p->metric); return FRG_ERR_INVALID; }
  if (p->variant < FRG_VARIANT_AUTO || p->variant > FRG_VARIANT_TC_BF16) { set_error("match_range: unknown variant %d", p->variant); return FRG_ERR_INVALID; }
  if (p->variant == FRG_VARIANT_TC_BF16) {
    set_error("match_range: FRG_VARIANT_TC_BF16 has no exact scores to hold against the threshold (use AUTO, TC_EXACT or SCAN_F32)");
    return FRG_ERR_UNSUPPORTED;
  }
  if (!s->master) { set_error("match_range: a bf16-only store has no fp32 master for the exact scores"); return FRG_ERR_UNSUPPORTED; }
  if (p->variant == FRG_VARIANT_TC_EXACT && p->metric == FRG_METRIC_EUCLIDEAN) {
    set_error("match_range: the Euclidean range search runs on the exact scan only (FRG_VARIANT_SCAN_F32 / AUTO)");
    return FRG_ERR_UNSUPPORTED;
  }
  const char* why = "";
  if (!range_scan_supported(s->dim, &why)) { set_error("match_range: %s", why); return FRG_ERR_UNSUPPORTED; }
  const bool unit = !(s->flags & FRG_STORE_RAW) && !(p->flags & FRG_QUERY_PRENORMALISED);
  const bool tc_ok = s->plane8 != nullptr && unit && p->metric == FRG_METRIC_COSINE && tc_supported(s->dim, p->metric, &why);
  const bool use_tc = p->variant == FRG_VARIANT_TC_EXACT || (p->variant == FRG_VARIANT_AUTO && tc_ok);
  if (use_tc && !tc_ok) {
    set_error("match_range: FRG_VARIANT_TC_EXACT needs a unit-row store with a scan plane, normalised queries and "
              "dim 128 / 256 / 512");
    return FRG_ERR_UNSUPPORTED;
  }
  if (nq == 0) return FRG_OK;
  DeviceGuard g(s->device);
  if (!g.ok) { set_error("cannot select device %d", s->device); return FRG_ERR_CUDA; }
  DeviceInfo di;
  FRG_CHECK(device_info(s->device, &di));
  std::lock_guard<std::mutex> lk(s->mu);
  FRG_CHECK(store_begin_read(s, st));
  const GalleryWindow w = window_of(s, p->tenant, use_tc);
  if (w.rows > 0x7fffffff) { set_error("match_range: more than 2^31-1 rows in one shard"); return FRG_ERR_UNSUPPORTED; }
  const int64_t row_offset = p->row_offset + w.row0;
  const bool strict = (p->flags & FRG_FIRST_STRICT) != 0;
  ScanArgs a;
  a.master = w.master; a.plane = w.plane; a.tags = w.tags; a.rows = w.rows; a.dim = w.dim;
  a.nq = nq; a.k = 1; a.metric = p->metric; a.tenant = p->tenant; a.sm_count = di.sm_count;
  const size_t qn_bytes = (size_t(nq) * w.dim * sizeof(float) + 255) & ~size_t(255);
  unsigned char* ws = nullptr;
  int rc = FRG_OK;
  if (use_tc && w.rows > 0) {
    const size_t qb_bytes = (size_t(nq) * w.dim + 255) & ~size_t(255);              // int8 image
    const size_t eps_bytes = (size_t(nq) * sizeof(float) + 255) & ~size_t(255);
    const int32_t* tile_list = nullptr;
    int n_list = 0;
    const int64_t plan_rows = tc_effective_rows(&w, nq, st, &tile_list, &n_list);
    if (plan_rows < 0) return FRG_ERR_CUDA;
    const size_t tc_bytes = tc_workspace_bytes(plan_rows, w.dim, nq, 1, di.sm_count, true, true);
    FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), qn_bytes + qb_bytes + 2 * eps_bytes + tc_bytes, st));
    float* qn = reinterpret_cast<float*>(ws);
    int8_t* qi8 = reinterpret_cast<int8_t*>(ws + qn_bytes);
    float* eps = reinterpret_cast<float*>(ws + qn_bytes + qb_bytes);
    float* qstep = reinterpret_cast<float*>(ws + qn_bytes + qb_bytes + eps_bytes);
    unsigned char* tc_ws = ws + qn_bytes + qb_bytes + 2 * eps_bytes;
    void* keys = nullptr; int* ct0 = nullptr; int* nf0 = nullptr;
    tc_workspace_init_targets(plan_rows, w.dim, nq, 1, di.sm_count, tc_ws, &keys, &ct0, &nf0, true, true);
    int* flagged = nullptr; int* n_flagged = nullptr;
    profile_begin(st, kStagePrep);
    rc = launch_prepare_queries_i8(q, nq, w.dim, qn, qi8, qstep, eps, s->gmax_bits,
                                   static_cast<unsigned long long*>(keys), ct0, nf0, st);
    profile_end(st, 1);
    if (rc == FRG_OK)
      rc = launch_tc_range(&w, qn, qi8, qstep, eps, nq, max_hits, p->tenant, p->threshold, strict, row_offset, tc_ws,
                           di.sm_count, out_counts, out_rows, out_scores, &flagged, &n_flagged, st, plan_rows,
                           tile_list, n_list);
    if (rc == FRG_OK) {
      a.qn = qn;
      profile_begin(st, kStageFallback);
      rc = launch_range_scan(a, flagged, n_flagged, max_hits, p->threshold, strict, row_offset, out_counts,
                             out_rows, out_scores, st);
      profile_end(st, 1);
    }
    g_variant = "range_tc";
  } else {
    FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), qn_bytes, st));
    float* qn = reinterpret_cast<float*>(ws);
    a.qn = qn;
    rc = launch_normalise_queries(q, nq, w.dim, p->metric == FRG_METRIC_COSINE && !(p->flags & FRG_QUERY_PRENORMALISED),
                                  qn, nullptr, nullptr, nullptr, nullptr, st);
    profile_begin(st, kStageDominant);
    if (rc == FRG_OK)
      rc = launch_range_scan(a, nullptr, nullptr, max_hits, p->threshold, strict, row_offset, out_counts, out_rows,
                             out_scores, st);
    profile_end(st, 3);
    g_variant = "range_scan";
  }
  cudaError_t e = cudaFreeAsync(ws, st);
  if (rc == FRG_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync", __FILE__, __LINE__);
  return rc;
}

int frg_match_range(frg_store* s, const float* q, int32_t nq, int32_t max_hits, const frg_match_params_t* p,
                    int64_t* out_counts, int64_t* out_rows, float* out_scores, void* stream) {
  return range_impl(s, q, nq, max_hits, p, out_counts, out_rows, out_scores, static_cast<cudaStream_t>(stream));
}

int frg_match_range_host(frg_store* s, const float* q, int32_t nq, int32_t max_hits, const frg_match_params_t* p,
                         int64_t* out_counts, int64_t* out_rows, float* out_scores) {
  if (!s || !p || nq < 0 || (nq > 0 && (!q || !out_counts || !out_rows || !out_scores)) || max_hits < 1) {
    // the device entry point names the argument
    return range_impl(s, q, nq, max_hits, p, out_counts, out_rows, out_scores, nullptr);
  }
  if (nq == 0) return range_impl(s, q, nq, max_hits, p, out_counts, out_rows, out_scores, nullptr);
  DeviceGuard g(s->device);
  cudaStream_t st = cudaStreamPerThread;
  const size_t slots = size_t(nq) * size_t(max_hits);
  const size_t qb = size_t(nq) * s->dim * sizeof(float), cb = size_t(nq) * sizeof(int64_t);
  const size_t o_c = (qb + 255) & ~size_t(255), o_r = (o_c + cb + 255) & ~size_t(255),
               o_s = (o_r + slots * sizeof(int64_t) + 255) & ~size_t(255);
  unsigned char* d = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&d), o_s + slots * sizeof(float), st));
  int rc = FRG_OK;
  cudaError_t e = cudaMemcpyAsync(d, q, qb, cudaMemcpyHostToDevice, st);
  if (e != cudaSuccess) rc = cuda_fail(e, "H2D queries", __FILE__, __LINE__);
  if (rc == FRG_OK)
    rc = range_impl(s, reinterpret_cast<float*>(d), nq, max_hits, p, reinterpret_cast<int64_t*>(d + o_c),
                    reinterpret_cast<int64_t*>(d + o_r), reinterpret_cast<float*>(d + o_s), st);
  if (rc == FRG_OK) {
    e = cudaMemcpyAsync(out_counts, d + o_c, cb, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_rows, d + o_r, slots * sizeof(int64_t), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_scores, d + o_s, slots * sizeof(float), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = cuda_fail(e, "D2H results", __FILE__, __LINE__);
    else rc = store_fault(s);
  }
  cudaFreeAsync(d, st);
  return rc;
}

// --------------------------------------------------------------------------------------------- gallery self-join
// The store's rows [row0, row0 + n) as queries against the rows after them (the upper triangle), in slabs of
// FRG_JOIN_SLAB_ROWS query rows that reuse one workspace.  Query tile u of 128 rows [R, R + 128) scans the rows from
// its own tile R / 128 to an end row: the store's last row; with p->tenant >= 0 that tenant's extent end; with
// FRG_JOIN_SAME_TAG the largest extent end among the tags whose extent overlaps the tile.  When exactly one tag's extent
// overlaps the tile, the filter masks with that tag.  A tile no live row of the rule can sit in scans nothing.
// Tensor-core path (unit store with an int8 plane and a covered dim): per slab query prep straight from the master
// rows -> floor threshold - eps[q] -> GROUPED filter -> join_select_kernel -> exact join scan of the overflowed
// queries.  SCAN_F32 (and plane-less stores): per slab query prep -> exact join scan of every query.
static_assert(FRG_JOIN_SLAB_ROWS % kTcTileRows == 0, "slabs are whole query tiles");

struct JoinTile { int32_t tenant; int32_t end_row; };

static void join_plan_tiles(const frg_store* s, int64_t row0, int64_t n, int32_t tenant, bool same_tag,
                            std::vector<JoinTile>* out) {
  const int64_t rows = s->rows;
  const int64_t nt = (n + kTcTileRows - 1) / kTcTileRows;
  out->assign(size_t(nt), JoinTile{tenant >= 0 ? tenant : -1, int32_t(rows)});
  if (!s->extents_known || (tenant < 0 && !same_tag)) return;
  if (tenant >= 0) {
    auto it = s->extents.find(tenant);
    const int64_t lo = it != s->extents.end() ? it->second.lo : 0;
    const int64_t hi = it != s->extents.end() ? (it->second.hi < rows ? it->second.hi : rows) : 0;
    for (int64_t u = 0; u < nt; ++u) {
      const int64_t R = row0 + u * kTcTileRows, Re = R + kTcTileRows < row0 + n ? R + kTcTileRows : row0 + n;
      (*out)[size_t(u)].end_row = int32_t(hi > lo && Re > lo && R < hi ? hi : R);
    }
    return;
  }
  // sweep over the query tiles (ascending) with the extents sorted by start and their ends sorted: the extents that
  // overlap [R, Re) are those starting before Re minus those ending at or before R, and the largest end among the
  // started ones, when it is past R, belongs to an overlapping extent
  struct Ext { int64_t lo, hi; int32_t tag; };
  std::vector<Ext> ext;
  std::vector<int64_t> ends;
  for (const auto& kv : s->extents) {
    const int64_t hi = kv.second.hi < rows ? kv.second.hi : rows;
    if (hi <= kv.second.lo) continue;
    ext.push_back(Ext{kv.second.lo, hi, kv.first});
    ends.push_back(hi);
  }
  std::sort(ext.begin(), ext.end(), [](const Ext& x, const Ext& y) { return x.lo < y.lo || (x.lo == y.lo && x.tag < y.tag); });
  std::sort(ends.begin(), ends.end());
  size_t i = 0, j = 0;
  int64_t max_hi = 0;
  int32_t max_tag = -1;
  for (int64_t u = 0; u < nt; ++u) {
    const int64_t R = row0 + u * kTcTileRows, Re = R + kTcTileRows < row0 + n ? R + kTcTileRows : row0 + n;
    for (; i < ext.size() && ext[i].lo < Re; ++i)
      if (ext[i].hi > max_hi) { max_hi = ext[i].hi; max_tag = ext[i].tag; }
    while (j < ends.size() && ends[j] <= R) ++j;
    const size_t overlap = i - j;
    JoinTile& t = (*out)[size_t(u)];
    t.end_row = int32_t(overlap > 0 ? max_hi : R);
    t.tenant = overlap == 1 ? max_tag : -1;
  }
}

static int self_join_impl(frg_store* s, int64_t row0, int64_t n, int32_t max_hits, const frg_match_params_t* p,
                          int64_t* out_counts, int64_t* out_rows, float* out_scores, cudaStream_t st) {
  reset_launches();
  if (!s || !p || n < 0 || row0 < 0 || (n > 0 && (!out_counts || !out_rows || !out_scores))) {
    set_error("self_join: bad argument");
    return FRG_ERR_INVALID;
  }
  if (max_hits < 1) { set_error("self_join: max_hits=%d must be >= 1", max_hits); return FRG_ERR_INVALID; }
  if (p->metric == FRG_METRIC_EUCLIDEAN) { set_error("self_join: cosine only (Euclidean stores are raw)"); return FRG_ERR_UNSUPPORTED; }
  if (p->metric != FRG_METRIC_COSINE) { set_error("self_join: unknown metric %d", p->metric); return FRG_ERR_INVALID; }
  if (p->variant < FRG_VARIANT_AUTO || p->variant > FRG_VARIANT_TC_BF16) { set_error("self_join: unknown variant %d", p->variant); return FRG_ERR_INVALID; }
  if (p->variant == FRG_VARIANT_TC_BF16) {
    set_error("self_join: FRG_VARIANT_TC_BF16 has no exact scores to hold against the threshold (use AUTO, TC_EXACT or SCAN_F32)");
    return FRG_ERR_UNSUPPORTED;
  }
  if (p->flags & ~(FRG_FIRST_STRICT | FRG_QUERY_PRENORMALISED | FRG_JOIN_SAME_TAG)) {
    set_error("self_join: unknown flags 0x%x", p->flags);
    return FRG_ERR_INVALID;
  }
  if (p->flags & FRG_QUERY_PRENORMALISED) { set_error("self_join: the queries are the store's rows (FRG_QUERY_PRENORMALISED does not apply)"); return FRG_ERR_UNSUPPORTED; }
  if (!s->master) { set_error("self_join: a bf16-only store has no fp32 master for the exact scores"); return FRG_ERR_UNSUPPORTED; }
  if (s->flags & FRG_STORE_RAW) { set_error("self_join: scores on a raw store are not symmetric (unit cosine stores only)"); return FRG_ERR_UNSUPPORTED; }
  const char* why = "";
  if (!range_scan_supported(s->dim, &why)) { set_error("self_join: %s", why); return FRG_ERR_UNSUPPORTED; }
  const bool tc_ok = s->plane8 != nullptr && tc_supported(s->dim, FRG_METRIC_COSINE, &why);
  const bool use_tc = p->variant == FRG_VARIANT_TC_EXACT || (p->variant == FRG_VARIANT_AUTO && tc_ok);
  if (use_tc && !tc_ok) {
    set_error("self_join: FRG_VARIANT_TC_EXACT needs a unit-row store with a scan plane and dim 128 / 256 / 512");
    return FRG_ERR_UNSUPPORTED;
  }
  DeviceGuard g(s->device);
  if (!g.ok) { set_error("cannot select device %d", s->device); return FRG_ERR_CUDA; }
  DeviceInfo di;
  FRG_CHECK(device_info(s->device, &di));
  std::lock_guard<std::mutex> lk(s->mu);
  if (row0 + n > s->rows) {
    set_error("self_join: rows [%lld, %lld) beyond the %lld rows in use", (long long)row0, (long long)(row0 + n), (long long)s->rows);
    return FRG_ERR_INVALID;
  }
  if (s->rows > 0x7fffffff) { set_error("self_join: more than 2^31-1 rows in one shard"); return FRG_ERR_UNSUPPORTED; }
  g_variant = use_tc ? "join_tc" : "join_scan";
  if (n == 0) return FRG_OK;
  FRG_CHECK(store_begin_read(s, st));
  const bool same_tag = (p->flags & FRG_JOIN_SAME_TAG) != 0, strict = (p->flags & FRG_FIRST_STRICT) != 0;
  const int dim = s->dim;
  std::vector<JoinTile> plan;
  join_plan_tiles(s, row0, n, p->tenant, same_tag, &plan);
  // per slab: the upload [end row of each query tile][filter descriptors] and the filter's candidate entries
  const int64_t S = n < FRG_JOIN_SLAB_ROWS ? n : FRG_JOIN_SLAB_ROWS;
  const size_t t_cta = (size_t(S / kTcTileRows + 1) * 4 + 15) & ~size_t(15);
  std::vector<std::vector<unsigned char>> tables;
  std::vector<int> ctas;
  int64_t max_cand = 1;
  size_t max_table = t_cta;
  for (int64_t s0 = 0; s0 < n; s0 += S) {
    const int64_t ns = n - s0 < S ? n - s0 : S;
    const int64_t u0 = s0 / kTcTileRows, nu = (ns + kTcTileRows - 1) / kTcTileRows;
    std::vector<TcTenantGroup> tiles;
    std::vector<unsigned char> cta_bytes;
    int n_ctas = 0;
    int64_t cand = 0;
    if (use_tc) {
      for (int64_t u = 0; u < nu; ++u) {
        const JoinTile& t = plan[size_t(u0 + u)];
        const int64_t R = row0 + (u0 + u) * kTcTileRows;
        TcTenantGroup G{};
        G.tenant = t.tenant; G.q0 = int(u * kTcTileRows); G.nq = int(ns - u * kTcTileRows < kTcTileRows ? ns - u * kTcTileRows : kTcTileRows);
        G.tile0 = int(R / kTcTileRows);
        G.n_tiles = t.end_row > R + 1 ? int((t.end_row - 1) / kTcTileRows) - G.tile0 + 1 : 0;   // b > a >= R
        G.list = nullptr;
        tiles.push_back(G);
      }
      tc_join_plan(tiles, di.sm_count, &cta_bytes, &n_ctas, &cand);
    }
    std::vector<unsigned char> table(t_cta + cta_bytes.size(), 0);
    for (int64_t u = 0; u < nu; ++u) memcpy(table.data() + u * 4, &plan[size_t(u0 + u)].end_row, 4);
    if (!cta_bytes.empty()) memcpy(table.data() + t_cta, cta_bytes.data(), cta_bytes.size());
    if (cand > max_cand) max_cand = cand;
    if (table.size() > max_table) max_table = table.size();
    tables.push_back(std::move(table));
    ctas.push_back(n_ctas);
  }
  // ---- one workspace for every slab
  ScanArgs a;
  a.master = s->master; a.tags = s->tags; a.rows = s->rows; a.dim = dim;
  a.qn = nullptr; a.nq = int(S); a.k = 1; a.metric = FRG_METRIC_COSINE; a.tenant = p->tenant; a.sm_count = di.sm_count;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  const size_t o_qn = take(size_t(S) * dim * 4), o_table = take(max_table), o_scan = take(join_scan_workspace_bytes(a));
  size_t o_qi8 = 0, o_eps = 0, o_step = 0, o_keys = 0, o_cnt = 0, o_flag = 0, o_floor = 0, o_dense = 0, o_cand = 0;
  if (use_tc) {
    o_qi8 = take(size_t(S) * dim); o_eps = take(size_t(S) * 4); o_step = take(size_t(S) * 4);
    o_keys = take(size_t(S) * 32 * 8); o_cnt = take(size_t(S) * 4); o_flag = take(size_t(S) * 4 + 12);
    o_floor = take(size_t(S) * 4); o_dense = take(size_t(S) * kRangeBudget * 8); o_cand = take(size_t(max_cand) * 8);
  }
  unsigned char* ws = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&ws), off, st));
  float* qn = reinterpret_cast<float*>(ws + o_qn);
  const int32_t* tile_end = reinterpret_cast<const int32_t*>(ws + o_table);
  a.qn = qn;
  const GalleryWindow w = window_of(s, -1);
  const int64_t row_offset = p->row_offset;
  int rc = FRG_OK;
  for (size_t i = 0; rc == FRG_OK && i < tables.size(); ++i) {
    const int64_t s0 = int64_t(i) * S, ns = n - s0 < S ? n - s0 : S, qrow0 = row0 + s0;
    int64_t* oc = out_counts + s0;
    int64_t* orow = out_rows + s0 * max_hits;
    float* osc = out_scores + s0 * max_hits;
    a.nq = int(ns);
    rc = stage_upload(ws + o_table, tables[i].data(), tables[i].size(), st);
    if (rc != FRG_OK) break;
    if (use_tc) {
      int8_t* qi8 = reinterpret_cast<int8_t*>(ws + o_qi8);
      float* eps = reinterpret_cast<float*>(ws + o_eps);
      float* qstep = reinterpret_cast<float*>(ws + o_step);
      int* cnt = reinterpret_cast<int*>(ws + o_cnt);
      int* flagged = reinterpret_cast<int*>(ws + o_flag);
      int* n_flagged = flagged + S;
      profile_begin(st, kStagePrep);
      rc = launch_prepare_queries_i8(s->master + qrow0 * dim, int(ns), dim, qn, qi8, qstep, eps, s->gmax_bits,
                                     reinterpret_cast<unsigned long long*>(ws + o_keys), cnt, n_flagged, st);
      profile_end(st, 1);
      if (rc == FRG_OK)
        rc = launch_tc_join(&w, qn, qi8, qstep, eps, int(ns), ws + o_table + t_cta, ctas[i], qrow0, p->tenant, same_tag,
                            p->threshold, strict, max_hits, row_offset, reinterpret_cast<int2*>(ws + o_cand), cnt,
                            reinterpret_cast<int2*>(ws + o_dense), reinterpret_cast<float*>(ws + o_floor), flagged,
                            n_flagged, oc, orow, osc, st);
      if (rc == FRG_OK) {
        profile_begin(st, kStageFallback);
        rc = launch_join_scan(a, qrow0, tile_end, same_tag, flagged, n_flagged, max_hits, p->threshold, strict,
                              row_offset, ws + o_scan, oc, orow, osc, st);
        profile_end(st, 3);
      }
    } else {
      profile_begin(st, kStagePrep);
      rc = launch_normalise_queries(s->master + qrow0 * dim, int(ns), dim, true, qn, nullptr, nullptr, nullptr, nullptr, st);
      profile_end(st, 1);
      if (rc == FRG_OK) {
        profile_begin(st, kStageDominant);
        rc = launch_join_scan(a, qrow0, tile_end, same_tag, nullptr, nullptr, max_hits, p->threshold, strict,
                              row_offset, ws + o_scan, oc, orow, osc, st);
        profile_end(st, 3);
      }
    }
  }
  g_variant = use_tc ? "join_tc" : "join_scan";
  cudaError_t e = cudaFreeAsync(ws, st);
  if (rc == FRG_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaFreeAsync", __FILE__, __LINE__);
  return rc;
}

int frg_self_join(frg_store* s, int64_t row0, int64_t n, int32_t max_hits, const frg_match_params_t* p,
                  int64_t* out_counts, int64_t* out_rows, float* out_scores, void* stream) {
  return self_join_impl(s, row0, n, max_hits, p, out_counts, out_rows, out_scores, static_cast<cudaStream_t>(stream));
}

int frg_self_join_host(frg_store* s, int64_t row0, int64_t n, int32_t max_hits, const frg_match_params_t* p,
                       int64_t* out_counts, int64_t* out_rows, float* out_scores) {
  if (!s || !p || n <= 0 || row0 < 0 || !out_counts || !out_rows || !out_scores || max_hits < 1) {
    // the device entry point names the argument (and takes n = 0)
    return self_join_impl(s, row0, n, max_hits, p, out_counts, out_rows, out_scores, nullptr);
  }
  DeviceGuard g(s->device);
  cudaStream_t st = cudaStreamPerThread;
  const size_t slots = size_t(n) * size_t(max_hits), cb = size_t(n) * sizeof(int64_t);
  const size_t o_r = (cb + 255) & ~size_t(255), o_s = (o_r + slots * sizeof(int64_t) + 255) & ~size_t(255);
  unsigned char* d = nullptr;
  FRG_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&d), o_s + slots * sizeof(float), st));
  int rc = self_join_impl(s, row0, n, max_hits, p, reinterpret_cast<int64_t*>(d), reinterpret_cast<int64_t*>(d + o_r),
                          reinterpret_cast<float*>(d + o_s), st);
  if (rc == FRG_OK) {
    cudaError_t e = cudaMemcpyAsync(out_counts, d, cb, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_rows, d + o_r, slots * sizeof(int64_t), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_scores, d + o_s, slots * sizeof(float), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = cuda_fail(e, "D2H results", __FILE__, __LINE__);
    else rc = store_fault(s);
  }
  cudaFreeAsync(d, st);
  return rc;
}

int frg_merge_topk(int32_t device, const float* scores, const int64_t* rows, int32_t parts,
                   int32_t nq, int32_t k, int32_t metric, float threshold,
                   int64_t* out_rows, float* out_scores, uint8_t* out_accept, void* stream) {
  reset_launches();
  if (parts < 0 || nq < 0 || (nq > 0 && (!out_rows || !out_scores)) || (parts > 0 && nq > 0 && (!scores || !rows))) {
    set_error("merge_topk: bad argument");
    return FRG_ERR_INVALID;
  }
  DeviceGuard g(device);
  if (!g.ok) { set_error("cannot select device %d", device); return FRG_ERR_CUDA; }
  return launch_merge_i64(scores, rows, parts, nq, k, k, metric, threshold, 0, false, out_rows, out_scores,
                          out_accept, static_cast<cudaStream_t>(stream));
}

int frg_merge_topk_strided(int32_t device, const float* scores, int64_t score_part_stride,
                           const int64_t* rows, int64_t row_part_stride, int32_t parts, int32_t nq, int32_t k,
                           int32_t metric, float threshold, int64_t* out_rows, float* out_scores,
                           uint8_t* out_accept, void* stream) {
  reset_launches();
  if (parts < 0 || nq < 0 || (nq > 0 && (!out_rows || !out_scores)) || (parts > 0 && nq > 0 && (!scores || !rows))) {
    set_error("merge_topk_strided: bad argument");
    return FRG_ERR_INVALID;
  }
  DeviceGuard g(device);
  if (!g.ok) { set_error("cannot select device %d", device); return FRG_ERR_CUDA; }
  return launch_merge_i64_strided(scores, score_part_stride, rows, row_part_stride, parts, nq, k, metric, threshold,
                                  out_rows, out_scores, out_accept, static_cast<cudaStream_t>(stream));
}

int frg_exchange_bytes(int32_t world, int32_t nq, int32_t k, int64_t* block_cap, int64_t* total) {
  if (world < 1 || world > kExchangeMaxWorld || nq < 0 || k < 1 || k > FRG_MAX_K || !block_cap || !total) {
    set_error("exchange_bytes: bad argument");
    return FRG_ERR_INVALID;
  }
  const int64_t cap = ((int64_t(nq) * k * 24 + 255) / 256) * 256;      // three 8-byte packets per slot
  *block_cap = cap;
  *total = kExchangeHeader + 2 * int64_t(world) * cap;
  return FRG_OK;
}

int frg_exchange_merge_topk(int32_t device, const frg_exchange_t* x, const int64_t* local_rows,
                            const float* local_scores, int32_t nq, int32_t k, int32_t metric, float threshold,
                            int64_t* out_rows, float* out_scores, uint8_t* out_accept, void* stream) {
  reset_launches();
  if (nq < 0 || k < 1 || k > FRG_MAX_K || (nq > 0 && (!local_rows || !local_scores || !out_rows || !out_scores))) {
    set_error("exchange_merge_topk: bad argument");
    return FRG_ERR_INVALID;
  }
  XPush xp;
  FRG_CHECK(check_exchange(x, nq, k, &xp));
  DeviceGuard g(device);
  if (!g.ok) { set_error("cannot select device %d", device); return FRG_ERR_CUDA; }
  DeviceInfo di;
  FRG_CHECK(device_info(device, &di));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!(x->flags & FRG_XCHG_MERGE_ONLY)) FRG_CHECK(launch_exchange_push(xp, local_rows, local_scores, nq, k, di.sm_count, st));
  if (x->flags & FRG_XCHG_PUSH_ONLY) return FRG_OK;
  return launch_exchange_merge(xp, nq, k, metric, threshold, di.sm_count, out_rows, out_scores, out_accept, st);
}

int frg_exchange_status(int32_t device, const void* own_buf, int32_t clear, void* stream, frg_exchange_status_t* out) {
  if (!own_buf || !out) { set_error("exchange_status: NULL argument"); return FRG_ERR_INVALID; }
  DeviceGuard g(device);
  if (!g.ok) { set_error("cannot select device %d", device); return FRG_ERR_CUDA; }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  XStatus h{};
  const unsigned char* rec = static_cast<const unsigned char*>(own_buf) + kExchangeStatusOff;
  FRG_CUDA(cudaMemcpyAsync(&h, rec, sizeof(h), cudaMemcpyDeviceToHost, st));
  if (clear) FRG_CUDA(cudaMemsetAsync(const_cast<unsigned char*>(rec), 0, sizeof(h), st));
  FRG_CUDA(cudaStreamSynchronize(st));
  memset(out, 0, sizeof(*out));
  out->code = int32_t(h.code); out->peer = int32_t(h.peer); out->epoch = h.epoch; out->peer_epoch = h.seen_epoch;
  out->nq = int32_t(h.want_hello >> 5); out->k = int32_t(h.want_hello & 31u);
  out->peer_nq = int32_t(h.seen_hello >> 5); out->peer_k = int32_t(h.seen_hello & 31u);
  out->slot = int32_t(h.query);
  switch (h.code) {
    case kXOk: return FRG_OK;
    case kXHelloTimeout:
      set_error("exchange: call %u (nq=%d, k=%d): rank %d never announced it (its last call on this parity: %u) - "
                "the ranks made different numbers of collective calls, or that rank is down",
                h.epoch, out->nq, out->k, out->peer, h.seen_epoch);
      break;
    case kXHelloMismatch:
      set_error("exchange: call %u: this rank passed nq=%d, k=%d but rank %d passed nq=%d, k=%d",
                h.epoch, out->nq, out->k, out->peer, out->peer_nq, out->peer_k);
      break;
    case kXDataTimeout:
      set_error("exchange: call %u (nq=%d, k=%d): slot %d of rank %d never arrived (packet epoch %u)",
                h.epoch, out->nq, out->k, out->slot, out->peer, h.seen_epoch);
      break;
    default:
      set_error("exchange: status record holds unknown code %u", h.code);
      break;
  }
  return FRG_ERR_STATE;
}

}  // extern "C"
