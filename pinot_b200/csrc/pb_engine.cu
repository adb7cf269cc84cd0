// pb_engine.cu — host runtime behind the C ABI in include/pinot_b200.h.
//
// Staging (Pinot index buffers -> HBM, once), per-query lowering of the caller's filter tree into the
// device descriptors of pb_device.cuh, table allocation, the kernel sequence, and result hand-back into
// pinned host memory.  No CPU implementation of the query path lives here: if the device cannot run a
// query the call fails with PB_ERR_UNSUPPORTED and the plan maker declines to the stock CPU plan.
#include "../../include/pinot_b200.h"
#include "pb_device.cuh"
#include "pb_filter_spec.h"

#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_set>
#include <vector>

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[1024];
static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return code;
}
extern "C" const char* pb_last_error(void) { return g_err; }

#define CU(call)                                                                                     \
  do {                                                                                               \
    cudaError_t e__ = (call);                                                                        \
    if (e__ != cudaSuccess) return fail(e__ == cudaErrorMemoryAllocation ? PB_ERR_OOM : PB_ERR_CUDA, \
                                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct PinnedBlock { void* p; size_t cap; };
#define PB_N_EVENTS 7
struct StreamSet { cudaStream_t stream = nullptr; cudaEvent_t ev[PB_N_EVENTS] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr}; };   // one per in-flight call, pooled

// One Context per device handed to pb_init (SURVEY.md §8b threading contract: every entry point selects the device of the
// handle it works on; a JVM worker thread that never called pb_init itself still runs on the right GPU).
struct Context {
  std::mutex mu;
  int device = 0;                             // CUDA device ordinal
  int index = 0;                              // position in pb_init's device_ids (the device_index of pb_segment_stage)
  int num_sms = 148;
  std::vector<PinnedBlock> scratch_free;      // large device scratch buffers (match lists), reused across calls
  std::vector<StreamSet> streams_free;        // stream + timing events of finished calls (creation costs ~10 us per call)
  cudaStream_t util_stream = nullptr;         // stream-ordered allocations / frees of staged data
  cudaStream_t copy_stream = nullptr;         // host -> HBM staging copies (queries wait on per-segment events)
  bool smem_attr_set = false;
  // segment cache accounting (hbm_cache_bytes of pb_init): staged bytes on this device and the LRU clock
  int64_t staged_bytes = 0;
  uint64_t lru_clock = 0;
  uint64_t evictions = 0;
  std::vector<struct pb_segment_s*> segments; // every live segment staged on this device (eviction candidates)
  // cross-rank merge (pb_comm_init): receive buffer of the table all-gather, grown on demand
  void* gather_buf = nullptr; size_t gather_cap = 0;
};
struct Global {
  std::mutex mu;
  bool inited = false;
  std::vector<std::unique_ptr<Context>> ctxs;
  size_t hbm_cache_bytes = 0;                 // 0 = unlimited
  std::vector<PinnedBlock> pinned_free;       // page-locked host blocks (portable: usable from every device)
};
static Global g_all;

// cudaSetDevice for the duration of one entry point (restores the caller's device)
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(const Context* c) { cudaGetDevice(&prev); if (c && prev != c->device) cudaSetDevice(c->device); else prev = -1; }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

static int init_context(Context* c) {
  CU(cudaSetDevice(c->device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, c->device));
  c->num_sms = prop.multiProcessorCount;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, c->device) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  // the aggregation kernel gathers 4-8 bytes at random docIds: fetch single 32-byte sectors from DRAM instead of
  // the default 64 (PB_L2_FETCH=64|128 restores the larger granularity for A/B measurements)
  {
    size_t gran = 32;
    if (const char* e = getenv("PB_L2_FETCH")) gran = (size_t)atoi(e);
    if (gran == 32 || gran == 64 || gran == 128) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, gran);
  }
  CU(cudaStreamCreateWithFlags(&c->util_stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  return PB_OK;
}

static int init_devices(const int* device_ids, int n_devices, size_t hbm_cache_bytes) {
  std::lock_guard<std::mutex> lk(g_all.mu);
  if (g_all.inited) {
    // a second pb_init may only restate the devices it already has (the JVM calls it once per server)
    if (n_devices > 0 && device_ids) {
      if ((size_t)n_devices != g_all.ctxs.size()) return fail(PB_ERR_STATE, "pb_init: already initialised with %zu devices", g_all.ctxs.size());
      for (int i = 0; i < n_devices; i++) if (g_all.ctxs[i]->device != device_ids[i]) return fail(PB_ERR_STATE, "pb_init: already initialised with device %d at index %d", g_all.ctxs[i]->device, i);
    }
    if (hbm_cache_bytes) g_all.hbm_cache_bytes = hbm_cache_bytes;
    return PB_OK;
  }
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) return fail(PB_ERR_CUDA, "no CUDA device: %s", cudaGetErrorString(e));
  int prev = 0;
  cudaGetDevice(&prev);
  std::vector<int> ids;
  if (n_devices > 0 && device_ids) ids.assign(device_ids, device_ids + n_devices); else ids.push_back(prev);
  for (size_t i = 0; i < ids.size(); i++) {
    if (ids[i] < 0 || ids[i] >= n) return fail(PB_ERR_INVALID, "pb_init: device %d does not exist (%d devices)", ids[i], n);
    for (size_t k = 0; k < i; k++) if (ids[k] == ids[i]) return fail(PB_ERR_INVALID, "pb_init: device %d listed twice", ids[i]);
  }
  std::vector<std::unique_ptr<Context>> ctxs;
  for (size_t i = 0; i < ids.size(); i++) {
    std::unique_ptr<Context> c(new Context());
    c->device = ids[i]; c->index = (int)i;
    int rc = init_context(c.get());
    if (rc) { cudaSetDevice(prev); return rc; }
    ctxs.push_back(std::move(c));
  }
  // one JVM driving several GPUs: the cross-device table merge reads the peers' blocks over NVLink
  for (size_t i = 0; i < ctxs.size(); i++)
    for (size_t k = 0; k < ctxs.size(); k++) {
      if (i == k) continue;
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, ctxs[i]->device, ctxs[k]->device) == cudaSuccess && can) {
        cudaSetDevice(ctxs[i]->device);
        cudaError_t pe = cudaDeviceEnablePeerAccess(ctxs[k]->device, 0);
        if (pe != cudaSuccess) cudaGetLastError();   // already enabled / unsupported: the merge falls back to copies
        // the tables live in device k's stream-ordered memory pool: pools keep their own access lists
        // (cudaDeviceEnablePeerAccess does not cover them), so device i is granted read / write access to it explicitly
        cudaMemPool_t pool_k;
        if (cudaDeviceGetDefaultMemPool(&pool_k, ctxs[k]->device) == cudaSuccess) {
          cudaMemAccessDesc desc;
          memset(&desc, 0, sizeof desc);
          desc.location.type = cudaMemLocationTypeDevice;
          desc.location.id = ctxs[i]->device;
          desc.flags = cudaMemAccessFlagsProtReadWrite;
          if (cudaMemPoolSetAccess(pool_k, &desc, 1) != cudaSuccess) cudaGetLastError();
        }
      }
    }
  cudaSetDevice(prev);
  g_all.ctxs = std::move(ctxs);
  g_all.hbm_cache_bytes = hbm_cache_bytes;
  g_all.inited = true;
  return PB_OK;
}

static int ensure_init() {
  if (g_all.inited) return PB_OK;
  return init_devices(nullptr, 0, 0);
}
static Context* ctx_at(int index) { return (index >= 0 && index < (int)g_all.ctxs.size()) ? g_all.ctxs[index].get() : nullptr; }

// staged data comes from the stream-ordered pool (release threshold = keep everything): re-staging a segment reuses
// pool memory instead of paying cudaMalloc / cudaFree (hundreds of microseconds each)
static cudaError_t dev_alloc(Context* c, void** p, size_t bytes) {
  cudaError_t e = cudaMallocAsync(p, bytes, c->util_stream);
  if (e != cudaSuccess) return e;
  return cudaStreamSynchronize(c->util_stream);
}
static void dev_free(Context* c, void* p) {
  if (p && c && c->util_stream) cudaFreeAsync(p, c->util_stream);
  else if (p) cudaFree(p);
}

extern "C" int pb_init(const int* device_ids, int n_devices, size_t hbm_cache_bytes) {
  return init_devices(device_ids, n_devices, hbm_cache_bytes);
}
static void comm_shutdown();
extern "C" int pb_shutdown(void) {
  comm_shutdown();
  std::lock_guard<std::mutex> lk(g_all.mu);
  for (auto& b : g_all.pinned_free) cudaFreeHost(b.p);
  g_all.pinned_free.clear();
  for (auto& c : g_all.ctxs) {
    DeviceGuard dg(c.get());
    std::lock_guard<std::mutex> lk2(c->mu);
    for (auto& b : c->scratch_free) cudaFree(b.p);
    c->scratch_free.clear();
    for (auto& ss : c->streams_free) { for (int i = 0; i < PB_N_EVENTS; i++) if (ss.ev[i]) cudaEventDestroy(ss.ev[i]); cudaStreamDestroy(ss.stream); }
    c->streams_free.clear();
    if (c->gather_buf) { cudaFree(c->gather_buf); c->gather_buf = nullptr; c->gather_cap = 0; }
  }
  return PB_OK;
}
extern "C" int pb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

static void* pinned_alloc(size_t bytes) {
  size_t cap = 256;
  while (cap < bytes) cap <<= 1;
  {
    std::lock_guard<std::mutex> lk(g_all.mu);
    for (size_t i = 0; i < g_all.pinned_free.size(); i++)
      if (g_all.pinned_free[i].cap == cap) {
        void* p = g_all.pinned_free[i].p;
        g_all.pinned_free.erase(g_all.pinned_free.begin() + i);
        return p;
      }
  }
  void* p = nullptr;
  if (cudaHostAlloc(&p, cap, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) return nullptr;
  return p;
}
static void pinned_free(void* p, size_t bytes) {
  if (!p) return;
  size_t cap = 256;
  while (cap < bytes) cap <<= 1;
  std::lock_guard<std::mutex> lk(g_all.mu);
  if (g_all.pinned_free.size() < 256) g_all.pinned_free.push_back({p, cap});
  else cudaFreeHost(p);
}

static int stream_set_acquire(Context* c, StreamSet* out) {
  {
    std::lock_guard<std::mutex> lk(c->mu);
    if (!c->streams_free.empty()) { *out = c->streams_free.back(); c->streams_free.pop_back(); return PB_OK; }
  }
  StreamSet s;
  CU(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
  for (int i = 0; i < PB_N_EVENTS; i++) CU(cudaEventCreate(&s.ev[i]));
  *out = s;
  return PB_OK;
}
static void stream_set_release(Context* c, const StreamSet& s) {   // the stream must be idle
  if (!s.stream) return;
  {
    std::lock_guard<std::mutex> lk(c->mu);
    if (c->streams_free.size() < 64) { c->streams_free.push_back(s); return; }
  }
  for (int i = 0; i < PB_N_EVENTS; i++) if (s.ev[i]) cudaEventDestroy(s.ev[i]);
  cudaStreamDestroy(s.stream);
}

// large device scratch (the match list): cudaMallocAsync of hundreds of MB is not free even from the pool
static void* scratch_alloc(Context* c, size_t bytes, size_t* cap_out) {
  {
    std::lock_guard<std::mutex> lk(c->mu);
    int best = -1;
    for (size_t i = 0; i < c->scratch_free.size(); i++)
      if (c->scratch_free[i].cap >= bytes && (best < 0 || c->scratch_free[i].cap < c->scratch_free[best].cap)) best = (int)i;
    if (best >= 0) {
      PinnedBlock b = c->scratch_free[best];
      c->scratch_free.erase(c->scratch_free.begin() + best);
      *cap_out = b.cap;
      return b.p;
    }
  }
  size_t cap = (bytes + ((size_t)1 << 20) - 1) & ~(((size_t)1 << 20) - 1);
  void* p = nullptr;
  if (cudaMalloc(&p, cap) != cudaSuccess) return nullptr;
  *cap_out = cap;
  return p;
}
static void scratch_free(Context* c, void* p, size_t cap) {
  if (!p) return;
  std::lock_guard<std::mutex> lk(c->mu);
  if (c->scratch_free.size() < 8) c->scratch_free.push_back({p, cap});
  else cudaFree(p);
}

// ------------------------------------------------------------------------------------------------
// segments
// ------------------------------------------------------------------------------------------------
static inline uint32_t be32(const uint8_t* p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }
static inline uint64_t be64(const uint8_t* p) { return ((uint64_t)be32(p) << 32) | be32(p + 4); }

struct Column {
  std::string name;
  int type = 0, has_dict = 0, is_sorted = 0, card = 0, bits = 0, entry_bytes = 0;
  // caller's buffers (valid until staged; Pinot keeps the mmap alive while the segment is acquired)
  const uint8_t* h_fwd = nullptr; uint64_t h_fwd_len = 0;
  const uint8_t* h_inv = nullptr; uint64_t h_inv_len = 0;
  const uint8_t* h_null = nullptr; uint64_t h_null_len = 0;   // null-value vector (a RoaringBitmap): IS [NOT] NULL leaves arrive as PB_F_BITMAP
  std::vector<uint8_t> h_dict;          // host copy of the dictionary (big-endian, as stored)
  uint64_t raw_data_start = 0;
  int raw_width = 0;
  // chunk-compressed raw forward index (ChunkCompressionType != PASS_THROUGH): decoded on the device at stage time
  int raw_codec = 0, raw_num_chunks = 0, raw_docs_per_chunk = 0, raw_offset_bytes = 4;
  uint64_t raw_header_start = 0;
  // device
  uint8_t* d_fwd = nullptr; uint64_t d_fwd_bytes = 0;     // bit-packed stream / raw values (16-byte padded)
  int32_t* d_sorted_pairs = nullptr;                       // sorted column: LE (start,end) pairs
  std::vector<int32_t> h_sorted_pairs;
  double* d_dict_f64 = nullptr;
  uint8_t* d_dict_native = nullptr;                       // native-endian entries (group-key decode on the device)
  uint8_t* d_inv = nullptr;
  // PB_Q_GATHER_IN_PLACE: device-visible alias of the caller's page-locked forward index (no HBM copy)
  const uint8_t* d_fwd_host = nullptr; uint32_t host_full_words = 0, host_tail_word = 0;
  bool fwd_staged = false, dict_staged = false, inv_staged = false, native_staged = false;
};

// A row-major copy of the dictionary columns some query gathers together (see DevKeyCol in pb_device.cuh)
struct RowGroup {
  // members: (column index, form) -- form 0: the dictId (bits wide); form 1: the DECODED dictionary value, 4 or 8 bytes,
  // stored like a raw forward index entry, for aggregation inputs (no dictionary lookup per matching row)
  std::vector<int> cols, form;
  std::vector<int> bit_off;       // field offset of each member inside a row (value fields first, 32-bit aligned)
  int stride_bits = 0;            // 64 / 128 / 256: rows never straddle a 32-byte sector
  uint8_t* d_rows = nullptr;
  uint64_t bytes = 0;
  uint64_t last_used = 0;
  int find(int col, int f) const { for (size_t i = 0; i < cols.size(); i++) if (cols[i] == col && form[i] == f) return (int)i; return -1; }
};
#define PB_MAX_ROW_GROUPS_PER_SEGMENT 4

struct pb_segment_s {
  std::string name;
  int num_docs = 0;
  Context* ctx = nullptr;                   // the device this segment is staged on (device_index of pb_segment_stage)
  std::vector<Column> cols;
  std::mutex mu;
  int64_t device_bytes = 0;
  // segment cache (hbm_cache_bytes): queries in flight pin the segment; epoch changes whenever device buffers are dropped,
  // which invalidates cached query plans that hold pointers into them
  int inflight = 0;
  uint64_t last_used = 0, epoch = 0;
  int64_t accounted_bytes = 0;              // part of device_bytes already added to the context's staged_bytes
  // staging copies run on the context's copy stream; `staged_ev` marks the last one enqueued for this segment and
  // every query that touches the segment orders its kernels after it (until it is known to have completed)
  cudaEvent_t staged_ev = nullptr;
  bool staged_pending = false, stage_dirty = false;
  std::vector<PinnedBlock> staging_bufs;   // pinned sources of in-flight dictionary uploads (freed with the segment)
  std::vector<std::unique_ptr<RowGroup>> row_groups;
};

static int find_col(const pb_segment_s* s, const char* name) {
  for (size_t i = 0; i < s->cols.size(); i++) if (s->cols[i].name == name) return (int)i;
  return -1;
}

extern "C" int pb_segment_stage(const pb_segment_desc* d, int device_index, pb_segment_handle* out) {
  // registers the buffers and validates the layouts; columns are copied to HBM on first use by a query
  // so planning-only callers never touch the device
  if (!d || !out || d->num_columns < 0 || d->num_docs < 0) return fail(PB_ERR_INVALID, "bad segment descriptor");
  // registration itself never touches the device (planning-only callers: eligibility checks, EXPLAIN); without any CUDA
  // device the handle is still valid for the host planning layer and queries on it fail with PB_ERR_CUDA
  Context* ctx = nullptr;
  if (ensure_init() == PB_OK) {
    ctx = ctx_at(device_index);
    if (!ctx) return fail(PB_ERR_INVALID, "pb_segment_stage: device_index %d is not one of the %zu devices given to pb_init", device_index, g_all.ctxs.size());
  } else if (device_index != 0) return PB_ERR_CUDA;
  std::unique_ptr<pb_segment_s> s(new pb_segment_s());
  s->ctx = ctx;
  s->name = d->segment_name ? d->segment_name : "";
  s->num_docs = d->num_docs;
  s->cols.resize(d->num_columns);
  for (int i = 0; i < d->num_columns; i++) {
    const pb_column_desc& cd = d->columns[i];
    Column& c = s->cols[i];
    if (!cd.name || !cd.forward_index) return fail(PB_ERR_INVALID, "column %d: name/forward index missing", i);
    c.name = cd.name;
    c.type = cd.stored_type; c.has_dict = cd.has_dictionary; c.is_sorted = cd.is_sorted && cd.has_dictionary;
    c.card = cd.cardinality; c.bits = cd.bits_per_element; c.entry_bytes = cd.dict_entry_bytes;
    c.h_fwd = (const uint8_t*)cd.forward_index; c.h_fwd_len = cd.forward_index_len;
    c.h_inv = (const uint8_t*)cd.inverted_index; c.h_inv_len = cd.inverted_index_len;
    c.h_null = (const uint8_t*)cd.null_value_vector; c.h_null_len = cd.null_value_vector ? cd.null_value_vector_len : 0;
    if (c.type < PB_INT || c.type > PB_STRING) return fail(PB_ERR_UNSUPPORTED, "column %s: stored type %d", cd.name, c.type);
    if (c.has_dict) {
      if (!cd.dictionary || c.card <= 0 || c.bits < 1 || c.bits > 32) return fail(PB_ERR_INVALID, "column %s: bad dictionary metadata", cd.name);
      const uint8_t* db = (const uint8_t*)cd.dictionary;
      if (c.type == PB_STRING && cd.dictionary_len >= 20 && memcmp(db, ".vl;", 4) == 0 && be32(db + 4) == 1) {
        // var-length dictionary (VarLengthValueReader, SEGL/io/util/VarLengthValueReader.java:41-96: magic, version, numValues,
        // dataSectionStartOffset, numValues + 1 offsets, bytes): kept on this side as zero-padded entries of the longest
        // value's width, the layout every later step (global dictionaries, key decode) works on
        const uint32_t nv = be32(db + 8), data0 = be32(db + 12);
        if ((int64_t)nv != (int64_t)c.card) return fail(PB_ERR_INVALID, "column %s: var-length dictionary holds %u values, metadata says %d", cd.name, nv, c.card);
        if ((uint64_t)data0 + 4ull * ((uint64_t)nv + 1) > cd.dictionary_len) return fail(PB_ERR_INVALID, "column %s: var-length dictionary offsets out of bounds", cd.name);
        uint32_t width = 1;
        for (uint32_t k = 0; k < nv; k++) {
          const uint32_t a = be32(db + data0 + 4ull * k), b = be32(db + data0 + 4ull * k + 4);
          if (b < a || b > cd.dictionary_len) return fail(PB_ERR_INVALID, "column %s: var-length dictionary entry %u out of bounds", cd.name, k);
          width = std::max(width, b - a);
        }
        if (width > (1u << 20)) return fail(PB_ERR_UNSUPPORTED, "column %s: %u-byte dictionary values", cd.name, width);
        c.entry_bytes = (int)width;
        c.h_dict.assign((size_t)nv * width, 0);
        for (uint32_t k = 0; k < nv; k++) {
          const uint32_t a = be32(db + data0 + 4ull * k), b = be32(db + data0 + 4ull * k + 4);
          memcpy(c.h_dict.data() + (size_t)k * width, db + a, b - a);
        }
      } else {
        if (c.entry_bytes <= 0) return fail(PB_ERR_INVALID, "column %s: dictionary entry width %d", cd.name, c.entry_bytes);
        uint64_t need = (uint64_t)c.card * (uint64_t)c.entry_bytes;
        if (cd.dictionary_len < need) return fail(PB_ERR_INVALID, "column %s: dictionary too short", cd.name);
        c.h_dict.assign(db, db + need);
      }
      if (c.is_sorted) {
        if (c.h_fwd_len < 8ull * c.card) return fail(PB_ERR_INVALID, "column %s: sorted index too short", cd.name);
        c.h_sorted_pairs.resize(2 * (size_t)c.card);
        for (int k = 0; k < 2 * c.card; k++) c.h_sorted_pairs[k] = (int32_t)be32(c.h_fwd + 4ull * k);
      } else if (c.h_fwd_len < ((uint64_t)s->num_docs * c.bits + 7) / 8) return fail(PB_ERR_INVALID, "column %s: forward index too short", cd.name);
    } else {
      // BaseChunkForwardIndexReader header (SEGL/segment/index/readers/forward/BaseChunkForwardIndexReader.java:61-104)
      if (c.type == PB_STRING) return fail(PB_ERR_UNSUPPORTED, "column %s: raw STRING forward index", cd.name);
      if (c.h_fwd_len < 28) return fail(PB_ERR_INVALID, "column %s: raw forward index header", cd.name);
      int version = (int)be32(c.h_fwd), num_chunks = (int)be32(c.h_fwd + 4);
      // version 1 has no compression field: always SNAPPY, chunk offsets start right after the four header ints
      int compression = version > 1 ? (int)be32(c.h_fwd + 20) : PB_CODEC_SNAPPY;
      if (compression != 0 && compression != PB_CODEC_SNAPPY && compression != PB_CODEC_LZ4 && compression != PB_CODEC_LZ4_LENGTH_PREFIXED)
        return fail(PB_ERR_UNSUPPORTED, "column %s: chunk compression %d (PASS_THROUGH, SNAPPY, LZ4 and LZ4_LENGTH_PREFIXED are decoded)", cd.name, compression);
      int data_header_start = version > 1 ? (int)be32(c.h_fwd + 24) : 16;
      c.raw_offset_bytes = version <= 2 ? 4 : 8;
      c.raw_data_start = (uint64_t)data_header_start + (uint64_t)num_chunks * (uint64_t)c.raw_offset_bytes;
      c.raw_width = (c.type == PB_INT || c.type == PB_FLOAT) ? 4 : 8;
      c.raw_codec = compression; c.raw_num_chunks = num_chunks; c.raw_docs_per_chunk = (int)be32(c.h_fwd + 8); c.raw_header_start = (uint64_t)data_header_start;
      if (num_chunks < 0 || data_header_start < 16 || c.h_fwd_len < c.raw_data_start) return fail(PB_ERR_INVALID, "column %s: raw forward index header", cd.name);
      if (compression == 0) {
        if (c.h_fwd_len < c.raw_data_start + (uint64_t)s->num_docs * c.raw_width) return fail(PB_ERR_INVALID, "column %s: raw forward index too short", cd.name);
      } else {
        if ((int)be32(c.h_fwd + 12) != c.raw_width) return fail(PB_ERR_INVALID, "column %s: raw forward index entry size %d", cd.name, (int)be32(c.h_fwd + 12));
        if (c.raw_docs_per_chunk <= 0 || (uint64_t)c.raw_docs_per_chunk * (uint64_t)c.raw_width > 0x7fffffffull ||
            (uint64_t)num_chunks != ((uint64_t)s->num_docs + (uint64_t)c.raw_docs_per_chunk - 1) / (uint64_t)c.raw_docs_per_chunk)
          return fail(PB_ERR_INVALID, "column %s: raw forward index chunking (%d chunks of %d docs for %d docs)", cd.name, num_chunks, c.raw_docs_per_chunk, s->num_docs);
      }
    }
  }
  if (ctx) { std::lock_guard<std::mutex> lk(ctx->mu); ctx->segments.push_back(s.get()); }
  *out = s.release();
  return PB_OK;
}

// stage what a query needs of one column (under the segment lock)
static void native_entry(const Column& c, int id, uint8_t* out);
// Columns that a query only GATHERS (group-by keys, aggregation inputs) can be read in place from the caller's
// page-locked, device-mapped host buffer: for a selective query that moves a few sectors per matching row over PCIe
// instead of the whole column.  Needs pb_host_register'd memory and 4-byte alignment; otherwise the column is staged.
static bool map_column_in_place(pb_segment_s* s, Column& c) {
  if (c.d_fwd_host) return true;
  if ((c.has_dict && c.is_sorted) || (!c.has_dict && c.raw_codec != 0)) return false;
  const uint8_t* src = c.has_dict ? c.h_fwd : c.h_fwd + c.raw_data_start;
  uint64_t bytes = c.has_dict ? ((uint64_t)s->num_docs * c.bits + 7) / 8 : (uint64_t)s->num_docs * c.raw_width;
  if (!src || bytes == 0 || (reinterpret_cast<uintptr_t>(src) & 3u) || bytes / 4 >= 0xFFFFFFFFull) return false;
  void* dp = nullptr;
  if (cudaHostGetDevicePointer(&dp, const_cast<uint8_t*>(src), 0) != cudaSuccess || !dp) { cudaGetLastError(); return false; }
  // the last byte must be mapped too
  void* dp_end = nullptr;
  if (cudaHostGetDevicePointer(&dp_end, const_cast<uint8_t*>(src + bytes - 1), 0) != cudaSuccess) { cudaGetLastError(); return false; }
  c.d_fwd_host = static_cast<const uint8_t*>(dp);
  c.host_full_words = (uint32_t)(bytes / 4);
  uint8_t tail[4] = {0, 0, 0, 0};
  memcpy(tail, src + (bytes & ~3ull), (size_t)(bytes & 3ull));
  memcpy(&c.host_tail_word, tail, 4);
  return true;
}

static int stage_column(pb_segment_s* s, Column& c, bool need_fwd, bool need_dict, bool need_inv, cudaStream_t st, bool need_native = false,
                        bool in_place_ok = false) {
  if (need_fwd && !c.fwd_staged && in_place_ok && map_column_in_place(s, c)) need_fwd = false;
  if (need_fwd && !c.fwd_staged) {
    if (c.has_dict && c.is_sorted) {
      // pairs -> device, then materialise the bit-packed stream on the device
      CU(dev_alloc(s->ctx, (void**)&c.d_sorted_pairs, sizeof(int32_t) * 2 * (size_t)c.card));
      CU(cudaMemcpyAsync(c.d_sorted_pairs, c.h_sorted_pairs.data(), sizeof(int32_t) * 2 * (size_t)c.card, cudaMemcpyHostToDevice, st));
      uint64_t bytes = ((uint64_t)s->num_docs * c.bits + 7) / 8;
      uint64_t padded = ((bytes + 15) & ~15ull) + 32;
      CU(dev_alloc(s->ctx, (void**)&c.d_fwd, padded));
      CU(cudaMemsetAsync(c.d_fwd, 0, padded, st));
      uint64_t n_words = (bytes + 3) / 4;
      int grid = (int)std::min<uint64_t>((n_words + 255) / 256, 4096);
      if (grid < 1) grid = 1;
      pb_sorted_to_packed_kernel<<<grid, 256, 0, st>>>(c.d_sorted_pairs, c.card, (uint32_t)s->num_docs, c.bits, (uint32_t*)c.d_fwd, n_words);
      CU(cudaGetLastError());
      c.d_fwd_bytes = padded;
      s->device_bytes += (int64_t)padded;
    } else if (!c.has_dict && c.raw_codec != 0) {
      // compressed chunks -> device, decode there into the PASS_THROUGH value area (pb_chunk_decode_kernel)
      const uint64_t bytes = (uint64_t)s->num_docs * c.raw_width;
      const uint64_t padded = ((bytes + 15) & ~15ull) + 32;
      const size_t n_chunks = (size_t)c.raw_num_chunks;
      const size_t offs_bytes = sizeof(uint64_t) * (n_chunks + 1);
      uint64_t* offs = static_cast<uint64_t*>(pinned_alloc(offs_bytes + 8));
      if (!offs) return fail(PB_ERR_OOM, "pinned host allocation failed");
      s->staging_bufs.push_back({offs, offs_bytes + 8});
      for (size_t k = 0; k <= n_chunks; k++) {
        uint64_t o = c.h_fwd_len;                                              // the last chunk ends with the buffer
        if (k < n_chunks) o = c.raw_offset_bytes == 4 ? (uint64_t)be32(c.h_fwd + c.raw_header_start + 4 * k) : be64(c.h_fwd + c.raw_header_start + 8 * k);
        if (o < c.raw_data_start || o > c.h_fwd_len || (k > 0 && o - c.raw_data_start < offs[k - 1]))
          return fail(PB_ERR_INVALID, "column %s: chunk offset %zu of the raw forward index is out of order or out of range", c.name.c_str(), k);
        offs[k] = o - c.raw_data_start;
      }
      const uint64_t comp_bytes = c.h_fwd_len - c.raw_data_start;
      uint8_t* d_comp = nullptr; uint64_t* d_offs = nullptr; uint32_t* d_err = nullptr;
      CU(dev_alloc(s->ctx, (void**)&d_comp, comp_bytes + 16));
      CU(dev_alloc(s->ctx, (void**)&d_offs, offs_bytes + 16));
      d_err = reinterpret_cast<uint32_t*>(d_offs + n_chunks + 1);
      CU(dev_alloc(s->ctx, (void**)&c.d_fwd, padded));
      offs[n_chunks + 1] = 0;                                                  // the error word rides behind the offsets
      CU(cudaMemsetAsync(c.d_fwd + (bytes & ~15ull), 0, padded - (bytes & ~15ull), st));
      CU(cudaMemcpyAsync(d_comp, c.h_fwd + c.raw_data_start, comp_bytes, cudaMemcpyHostToDevice, st));
      CU(cudaMemcpyAsync(d_offs, offs, offs_bytes + 8, cudaMemcpyHostToDevice, st));
      DevChunkDecode D;
      D.src = d_comp; D.offs = d_offs; D.dst = c.d_fwd; D.total_bytes = bytes; D.n_chunks = (uint32_t)n_chunks;
      D.chunk_bytes = (uint32_t)((uint64_t)c.raw_docs_per_chunk * (uint64_t)c.raw_width); D.codec = c.raw_codec; D.err = d_err;
      if (n_chunks > 0) {
        pb_chunk_decode_kernel<<<(unsigned)((n_chunks + 7) / 8), 256, 0, st>>>(D);
        CU(cudaGetLastError());
      }
      uint32_t* h_err = reinterpret_cast<uint32_t*>(offs + n_chunks + 1);
      CU(cudaMemcpyAsync(h_err, d_err, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      CU(cudaStreamSynchronize(st));                                           // one-time cost of a compressed column; frees the temporaries
      dev_free(s->ctx, d_comp); dev_free(s->ctx, d_offs);
      if (*h_err != 0) {
        dev_free(s->ctx, c.d_fwd); c.d_fwd = nullptr;
        return fail(PB_ERR_INVALID, "column %s: %u chunk(s) of the raw forward index do not decode (codec %d)", c.name.c_str(), *h_err, c.raw_codec);
      }
      c.d_fwd_bytes = padded;
      s->device_bytes += (int64_t)padded;
    } else {
      const uint8_t* src = c.has_dict ? c.h_fwd : c.h_fwd + c.raw_data_start;
      uint64_t bytes = c.has_dict ? ((uint64_t)s->num_docs * c.bits + 7) / 8 : (uint64_t)s->num_docs * c.raw_width;
      uint64_t padded = ((bytes + 15) & ~15ull) + 32;
      CU(dev_alloc(s->ctx, (void**)&c.d_fwd, padded));
      CU(cudaMemsetAsync(c.d_fwd + (bytes & ~15ull), 0, padded - (bytes & ~15ull), st));
      CU(cudaMemcpyAsync(c.d_fwd, src, bytes, cudaMemcpyHostToDevice, st));
      c.d_fwd_bytes = padded;
      s->device_bytes += (int64_t)padded;
    }
    c.fwd_staged = true;
    s->stage_dirty = true;
  }
  if (need_dict && !c.dict_staged && c.has_dict && c.type != PB_STRING) {
    // BaseImmutableDictionary value reads, widened to double (Dictionary.getDoubleValue)
    const size_t vbytes = sizeof(double) * (size_t)std::max(c.card, 1);
    double* v = static_cast<double*>(pinned_alloc(vbytes));       // pinned so the upload never synchronises the copy stream
    if (!v) return fail(PB_ERR_OOM, "pinned host allocation failed");
    s->staging_bufs.push_back({v, vbytes});
    for (int i = 0; i < c.card; i++) {
      const uint8_t* p = c.h_dict.data() + (size_t)i * c.entry_bytes;
      switch (c.type) {
        case PB_INT: v[i] = (double)(int32_t)be32(p); break;
        case PB_LONG: v[i] = (double)(int64_t)be64(p); break;
        case PB_FLOAT: { uint32_t u = be32(p); float f; memcpy(&f, &u, 4); v[i] = (double)f; break; }
        default: { uint64_t u = be64(p); double dd; memcpy(&dd, &u, 8); v[i] = dd; break; }
      }
    }
    CU(dev_alloc(s->ctx, (void**)&c.d_dict_f64, sizeof(double) * (size_t)c.card));
    CU(cudaMemcpyAsync(c.d_dict_f64, v, sizeof(double) * (size_t)c.card, cudaMemcpyHostToDevice, st));
    s->stage_dirty = true;
    s->device_bytes += (int64_t)sizeof(double) * c.card;
    c.dict_staged = true;
  }
  if (need_native && !c.native_staged && c.has_dict) {
    std::vector<uint8_t> v((size_t)c.card * c.entry_bytes);
    for (int i = 0; i < c.card; i++) native_entry(c, i, v.data() + (size_t)i * c.entry_bytes);
    CU(dev_alloc(s->ctx, (void**)&c.d_dict_native, v.size() + 16));
    CU(cudaMemcpy(c.d_dict_native, v.data(), v.size(), cudaMemcpyHostToDevice));
    s->device_bytes += (int64_t)v.size();
    c.native_staged = true;
  }
  if (need_inv && !c.inv_staged) {
    if (!c.h_inv) return fail(PB_ERR_INVALID, "column %s has no inverted index", c.name.c_str());
    CU(dev_alloc(s->ctx, (void**)&c.d_inv, c.h_inv_len + 16));
    CU(cudaMemcpyAsync(c.d_inv, c.h_inv, c.h_inv_len, cudaMemcpyHostToDevice, st));
    s->device_bytes += (int64_t)c.h_inv_len;
    c.inv_staged = true;
    s->stage_dirty = true;
  }
  return PB_OK;
}


// ---- segment cache (hbm_cache_bytes of pb_init): when the staged bytes of a device exceed the limit, the least recently
// used segments that no query is using lose their HBM copies (their host buffers are still the caller's mmap: the next
// query on them stages again).  Every eviction bumps the segment's epoch, which retires cached plans that point into it. ----
static void drop_device_copies(pb_segment_s* s) {     // under s->mu, inflight == 0, no staging copy pending
  for (auto& c : s->cols) {
    dev_free(s->ctx, c.d_fwd); dev_free(s->ctx, c.d_sorted_pairs); dev_free(s->ctx, c.d_dict_f64); dev_free(s->ctx, c.d_dict_native); dev_free(s->ctx, c.d_inv);
    c.d_fwd = nullptr; c.d_sorted_pairs = nullptr; c.d_dict_f64 = nullptr; c.d_dict_native = nullptr; c.d_inv = nullptr;
    c.d_fwd_bytes = 0;
    c.fwd_staged = c.dict_staged = c.inv_staged = c.native_staged = false;
  }
  for (auto& b : s->staging_bufs) pinned_free(b.p, b.cap);
  s->staging_bufs.clear();
  for (auto& rg : s->row_groups) dev_free(s->ctx, rg->d_rows);
  s->row_groups.clear();
  s->device_bytes = 0; s->accounted_bytes = 0;
  s->epoch++;
}
static void enforce_cache_limit(Context* ctx) {
  const size_t limit = g_all.hbm_cache_bytes;
  if (!limit) return;
  std::vector<pb_segment_s*> cand;
  {
    std::lock_guard<std::mutex> lk(ctx->mu);
    if ((size_t)std::max<int64_t>(ctx->staged_bytes, 0) <= limit) return;
    cand = ctx->segments;
  }
  std::sort(cand.begin(), cand.end(), [](const pb_segment_s* a, const pb_segment_s* b) { return a->last_used < b->last_used; });
  for (pb_segment_s* s : cand) {
    {
      std::lock_guard<std::mutex> lk(ctx->mu);
      if ((size_t)std::max<int64_t>(ctx->staged_bytes, 0) <= limit) return;
    }
    std::unique_lock<std::mutex> sl(s->mu, std::try_to_lock);
    if (!sl.owns_lock() || s->inflight > 0 || s->device_bytes == 0) continue;
    if (s->staged_pending) {
      if (cudaEventQuery(s->staged_ev) != cudaSuccess) { cudaGetLastError(); continue; }
      s->staged_pending = false;
    }
    const int64_t freed = s->accounted_bytes;
    drop_device_copies(s);
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->staged_bytes -= freed;
    ctx->evictions++;
  }
}


// The row group that holds every (column, form) of `want`: an existing one whose members include them, else a new one
// built on the copy stream behind the column copies it reads.  Returns nullptr when rows would not pay (a single field, more
// than 256 bits) or cannot be built.  Under s->mu.
static int field_bits(const Column& c, int form) { return form ? 8 * c.entry_bytes : c.bits; }
static const RowGroup* row_group_for(pb_segment_s* s, std::vector<std::pair<int, int>> want, cudaStream_t cs) {
  if (want.size() < 2 || want.size() > PB_ROW_MAX_COLS) return nullptr;
  int sum_bits = 0;
  for (auto& w : want) {
    const Column& c = s->cols[w.first];
    if (!c.has_dict || !c.fwd_staged) return nullptr;
    if (w.second && (!c.native_staged || (c.entry_bytes != 4 && c.entry_bytes != 8) || c.type == PB_STRING)) return nullptr;
    sum_bits += field_bits(c, w.second);
  }
  if (sum_bits > 256) return nullptr;
  const uint64_t tick = [&]() { std::lock_guard<std::mutex> lk(s->ctx->mu); return ++s->ctx->lru_clock; }();
  for (auto& rg : s->row_groups) {
    bool all = true;
    for (auto& w : want) if (rg->find(w.first, w.second) < 0) { all = false; break; }
    if (all) { rg->last_used = tick; return rg.get(); }
  }
  if (s->row_groups.size() >= PB_MAX_ROW_GROUPS_PER_SEGMENT) {
    // (a parked plan may still point into the oldest one: the epoch retires those plans)
    if (s->inflight > 1) return nullptr;          // another query of this segment is in flight and may be reading it
    size_t old = 0;
    for (size_t i = 1; i < s->row_groups.size(); i++) if (s->row_groups[i]->last_used < s->row_groups[old]->last_used) old = i;
    dev_free(s->ctx, s->row_groups[old]->d_rows);
    s->device_bytes -= (int64_t)s->row_groups[old]->bytes;
    s->row_groups.erase(s->row_groups.begin() + (long)old);
    s->epoch++;
  }
  // value fields first (8-byte ones, then 4-byte ones: all stay 32-bit aligned), then the bit-packed dictIds
  std::stable_sort(want.begin(), want.end(), [&](const std::pair<int, int>& a, const std::pair<int, int>& b) {
    const int ka = a.second ? (s->cols[a.first].entry_bytes == 8 ? 0 : 1) : 2, kb = b.second ? (s->cols[b.first].entry_bytes == 8 ? 0 : 1) : 2;
    return ka < kb;
  });
  std::unique_ptr<RowGroup> rg(new RowGroup());
  rg->stride_bits = sum_bits <= 64 ? 64 : sum_bits <= 128 ? 128 : 256;
  int off = 0;
  for (auto& w : want) { rg->cols.push_back(w.first); rg->form.push_back(w.second); rg->bit_off.push_back(off); off += field_bits(s->cols[w.first], w.second); }
  rg->bytes = (uint64_t)s->num_docs * (uint64_t)(rg->stride_bits / 8) + 32;
  if (dev_alloc(s->ctx, (void**)&rg->d_rows, rg->bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  DevRowBuild B; memset(&B, 0, sizeof B);
  B.n_cols = (int)want.size(); B.stride_words = rg->stride_bits / 32; B.num_docs = (uint32_t)s->num_docs; B.out = (uint32_t*)rg->d_rows;
  for (size_t i = 0; i < want.size(); i++) {
    const Column& c = s->cols[want[i].first];
    B.fwd[i] = c.d_fwd; B.bits[i] = c.bits; B.bit_off[i] = rg->bit_off[i];
    if (want[i].second) { B.dict_native[i] = c.d_dict_native; B.value_bytes[i] = c.entry_bytes; }
  }
  if (cudaMemsetAsync(rg->d_rows + (rg->bytes - 32), 0, 32, cs) != cudaSuccess) { cudaGetLastError(); dev_free(s->ctx, rg->d_rows); return nullptr; }
  int grid = (int)std::min<uint64_t>(((uint64_t)s->num_docs + 255) / 256, (uint64_t)s->ctx->num_sms * 16);
  if (grid < 1) grid = 1;
  pb_build_rows_kernel<<<grid, 256, 0, cs>>>(B);
  if (cudaGetLastError() != cudaSuccess) { dev_free(s->ctx, rg->d_rows); return nullptr; }
  rg->last_used = tick;
  s->device_bytes += (int64_t)rg->bytes;
  s->stage_dirty = true;                          // the query's kernels wait for the build like for a staging copy
  s->row_groups.push_back(std::move(rg));
  return s->row_groups.back().get();
}

extern "C" int pb_segment_release(pb_segment_handle s) {
  if (!s) return PB_OK;
  DeviceGuard dg(s->ctx);
  if (s->ctx) {
    std::lock_guard<std::mutex> lk(s->ctx->mu);
    auto& v = s->ctx->segments;
    v.erase(std::remove(v.begin(), v.end(), s), v.end());
    s->ctx->staged_bytes -= s->accounted_bytes;
  }
  if (s->staged_ev) { cudaEventSynchronize(s->staged_ev); cudaEventDestroy(s->staged_ev); }
  for (auto& b : s->staging_bufs) pinned_free(b.p, b.cap);
  for (auto& c : s->cols) {
    dev_free(s->ctx, c.d_fwd); dev_free(s->ctx, c.d_sorted_pairs); dev_free(s->ctx, c.d_dict_f64); dev_free(s->ctx, c.d_dict_native); dev_free(s->ctx, c.d_inv);
  }
  for (auto& rg : s->row_groups) dev_free(s->ctx, rg->d_rows);
  delete s;
  return PB_OK;
}
extern "C" int64_t pb_segment_device_bytes(pb_segment_handle s) { return s ? s->device_bytes : 0; }
extern "C" int pb_cache_stats(int device_index, int64_t* staged_bytes, int64_t* evictions) {
  Context* c = ctx_at(device_index);
  if (!c) return fail(PB_ERR_INVALID, "pb_cache_stats: no device at index %d", device_index);
  std::lock_guard<std::mutex> lk(c->mu);
  if (staged_bytes) *staged_bytes = c->staged_bytes;
  if (evictions) *evictions = (int64_t)c->evictions;
  return PB_OK;
}

// ------------------------------------------------------------------------------------------------
// segment groups and global dictionaries
// ------------------------------------------------------------------------------------------------
struct GlobalDict {
  int type = 0, entry_bytes = 0;
  int64_t n = 0;
  std::vector<uint8_t> values;                 // native-endian stored-type values / padded strings, sorted
  std::vector<std::vector<int32_t>> h_remap;   // per segment: local dictId -> global dictId
  std::vector<int32_t*> d_remap;
  uint8_t* d_values = nullptr;                 // device copy of `values`
  bool external = false;
  bool uploaded = false;                       // remaps + values are on the device                       // installed by pb_segment_group_set_global_dictionary
};

struct pb_group_s {
  std::vector<pb_segment_s*> segs;
  std::map<std::string, GlobalDict> dicts;
  std::mutex mu;
  Context* ctx = nullptr;                      // device of the segments; nullptr when they span several devices
  // segments on several devices of this process (one JVM driving N GPUs): one child group per device, in order of first
  // appearance; child_of[i] / index_in_child[i] locate segment i.  Children run the per-device part of a query and the
  // parent merges their tables over NVLink (pb_query_execute).
  std::vector<pb_group_s*> children;
  std::vector<int> child_of, index_in_child;
  std::map<std::string, uint64_t> child_dict_version;   // global dictionaries already installed in the children
  uint64_t dict_version = 0;                   // bumps whenever a global dictionary changes (cached plans depend on it)
  std::vector<pb_result_s*> plans;             // cached query plans of this group: parked results that can be replayed (plan cache)
};

// dictionary entry -> native-endian comparable form
static void native_entry(const Column& c, int id, uint8_t* out) {
  const uint8_t* p = c.h_dict.data() + (size_t)id * c.entry_bytes;
  if (c.type == PB_STRING) { memcpy(out, p, c.entry_bytes); return; }
  if (c.entry_bytes == 4) { uint32_t u = be32(p); memcpy(out, &u, 4); } else { uint64_t u = be64(p); memcpy(out, &u, 8); }
}
// Strings compare the way their dictionaries are sorted: String.compareTo, i.e. by UTF-16 code units
// (ValueReaderComparisons.compareUtf8Bytes, SEGL/io/util/ValueReaderComparisons.java:68-139).  Byte order differs from that
// only between a supplementary character (a surrogate pair) and a BMP character at or above U+E000 -- but a segment
// dictionary holding both IS sorted the Java way, and the merge walk of build_remaps relies on one order on both sides.
static void utf16_units_at(const uint8_t* p, size_t avail, uint32_t* u1, uint32_t* u2) {
  *u1 = 0xfffd; *u2 = 0xfffd;
  if (avail == 0) { *u1 = 0; return; }
  auto cont = [&](size_t k) -> uint32_t { return k < avail ? (p[k] & 0x3Fu) : 0u; };
  const uint8_t b = p[0];
  if (b < 0x80) *u1 = b;
  else if ((b & 0xF0) < 0xE0) *u1 = ((uint32_t)(b & 0x1F) << 6) | cont(1);
  else if ((b & 0xF0) == 0xE0) *u1 = ((uint32_t)(b & 0x0F) << 12) | (cont(1) << 6) | cont(2);
  else {
    const uint32_t cp = ((uint32_t)(b & 0x07) << 18) | (cont(1) << 12) | (cont(2) << 6) | cont(3);
    if (cp >= 0x10000 && cp <= 0x10FFFF) { *u1 = 0xD800 + ((cp - 0x10000) >> 10); *u2 = 0xDC00 + ((cp - 0x10000) & 0x3FF); }
  }
}
static int cmp_utf8_java_order(const uint8_t* a, const uint8_t* b, size_t n) {     // two zero-padded entries of n bytes
  size_t i = 0;
  while (i < n && a[i] == b[i]) i++;
  if (i == n) return 0;
  while (i > 0 && (b[i] & 0xC0) == 0x80) i--;
  uint32_t a1, a2, b1, b2;
  utf16_units_at(a + i, n - i, &a1, &a2);
  utf16_units_at(b + i, n - i, &b1, &b2);
  if (a1 != b1) return a1 < b1 ? -1 : 1;
  return (a2 > b2) - (a2 < b2);
}
static int cmp_entry(int type, int eb, const uint8_t* a, const uint8_t* b) {
  switch (type) {
    case PB_INT: { int32_t x, y; memcpy(&x, a, 4); memcpy(&y, b, 4); return (x > y) - (x < y); }
    case PB_LONG: { int64_t x, y; memcpy(&x, a, 8); memcpy(&y, b, 8); return (x > y) - (x < y); }
    case PB_FLOAT: { float x, y; memcpy(&x, a, 4); memcpy(&y, b, 4); return (x > y) - (x < y); }
    case PB_DOUBLE: { double x, y; memcpy(&x, a, 8); memcpy(&y, b, 8); return (x > y) - (x < y); }
    default: return cmp_utf8_java_order(a, b, (size_t)eb);
  }
}

extern "C" int pb_segment_group_create(const pb_segment_handle* segs, int n, pb_segment_group_handle* out) {
  if (!segs || n <= 0 || !out) return fail(PB_ERR_INVALID, "bad segment group");
  for (int i = 0; i < n; i++) if (!segs[i]) return fail(PB_ERR_INVALID, "segment %d of the group is null", i);
  pb_group_s* g = new pb_group_s();
  g->segs.assign(segs, segs + n);
  g->ctx = segs[0]->ctx;
  for (int i = 1; i < n; i++) if (segs[i]->ctx != g->ctx) g->ctx = nullptr;
  if (!g->ctx) {
    std::vector<Context*> order;
    std::vector<std::vector<pb_segment_s*>> parts;
    g->child_of.resize(n); g->index_in_child.resize(n);
    for (int i = 0; i < n; i++) {
      size_t k = 0;
      while (k < order.size() && order[k] != segs[i]->ctx) k++;
      if (k == order.size()) { order.push_back(segs[i]->ctx); parts.emplace_back(); }
      g->child_of[i] = (int)k; g->index_in_child[i] = (int)parts[k].size();
      parts[k].push_back(segs[i]);
    }
    for (size_t k = 0; k < order.size(); k++) {
      pb_group_s* c = new pb_group_s();
      c->segs = parts[k]; c->ctx = order[k];
      g->children.push_back(c);
    }
  }
  *out = g;
  return PB_OK;
}
static void free_plans(pb_group_s* g);
extern "C" int pb_segment_group_release(pb_segment_group_handle g) {
  if (!g) return PB_OK;
  for (auto* c : g->children) pb_segment_group_release(c);
  DeviceGuard dg(g->ctx);
  free_plans(g);
  for (auto& kv : g->dicts) { for (auto p : kv.second.d_remap) dev_free(g->ctx, p); dev_free(g->ctx, kv.second.d_values); }
  delete g;
  return PB_OK;
}

// sorted union of the segments' dictionaries (k-way by concatenate + sort + unique; dictionaries are small)
static int build_union(pb_group_s* g, const char* column, GlobalDict& gd) {
  int type = -1, eb = 0;
  for (auto* s : g->segs) {
    int ci = find_col(s, column);
    if (ci < 0) return fail(PB_ERR_INVALID, "segment %s has no column %s", s->name.c_str(), column);
    const Column& c = s->cols[ci];
    if (!c.has_dict) return fail(PB_ERR_UNSUPPORTED, "column %s has no dictionary", column);
    if (type < 0) type = c.type;
    if (type != c.type) return fail(PB_ERR_INVALID, "column %s: stored type differs across segments", column);
    eb = std::max(eb, c.entry_bytes);
  }
  std::vector<uint8_t> all;
  for (auto* s : g->segs) {
    const Column& c = s->cols[find_col(s, column)];
    size_t base = all.size();
    all.resize(base + (size_t)c.card * eb, 0);
    for (int i = 0; i < c.card; i++) native_entry(c, i, all.data() + base + (size_t)i * eb);
  }
  size_t total = all.size() / eb;
  std::vector<uint32_t> idx(total);
  for (size_t i = 0; i < total; i++) idx[i] = (uint32_t)i;
  std::sort(idx.begin(), idx.end(), [&](uint32_t a, uint32_t b) { return cmp_entry(type, eb, all.data() + (size_t)a * eb, all.data() + (size_t)b * eb) < 0; });
  gd.type = type; gd.entry_bytes = eb; gd.values.clear(); gd.n = 0;
  for (size_t k = 0; k < total; k++) {
    const uint8_t* e = all.data() + (size_t)idx[k] * eb;
    if (gd.n == 0 || cmp_entry(type, eb, gd.values.data() + (size_t)(gd.n - 1) * eb, e) != 0) {
      gd.values.insert(gd.values.end(), e, e + eb);
      gd.n++;
    }
  }
  return PB_OK;
}

static int upload_remaps(pb_group_s* g, GlobalDict& gd) {
  if (gd.uploaded) return PB_OK;
  if (!g->ctx) return fail(PB_ERR_STATE, "global dictionaries are uploaded per device group");
  for (auto p : gd.d_remap) dev_free(g->ctx, p);
  dev_free(g->ctx, gd.d_values); gd.d_values = nullptr;
  CU(dev_alloc(g->ctx, (void**)&gd.d_values, gd.values.size() + 16));
  CU(cudaMemcpy(gd.d_values, gd.values.data(), gd.values.size(), cudaMemcpyHostToDevice));
  gd.d_remap.assign(g->segs.size(), nullptr);
  for (size_t si = 0; si < g->segs.size(); si++) {
    const auto& rm = gd.h_remap[si];
    CU(dev_alloc(g->ctx, (void**)&gd.d_remap[si], sizeof(int32_t) * std::max<size_t>(rm.size(), 1)));
    CU(cudaMemcpy(gd.d_remap[si], rm.data(), sizeof(int32_t) * rm.size(), cudaMemcpyHostToDevice));
  }
  gd.uploaded = true;
  return PB_OK;
}

static int build_remaps(pb_group_s* g, const char* column, GlobalDict& gd) {
  gd.uploaded = false;
  gd.h_remap.assign(g->segs.size(), {});
  std::vector<uint8_t> tmp((size_t)gd.entry_bytes);
  for (size_t si = 0; si < g->segs.size(); si++) {
    pb_segment_s* s = g->segs[si];
    const Column& c = s->cols[find_col(s, column)];
    auto& rm = gd.h_remap[si];
    rm.resize((size_t)c.card);
    int64_t pos = 0;   // both sides are sorted: merge walk
    for (int i = 0; i < c.card; i++) {
      std::fill(tmp.begin(), tmp.end(), 0);
      native_entry(c, i, tmp.data());
      while (pos < gd.n && cmp_entry(gd.type, gd.entry_bytes, gd.values.data() + (size_t)pos * gd.entry_bytes, tmp.data()) < 0) pos++;
      if (pos >= gd.n || cmp_entry(gd.type, gd.entry_bytes, gd.values.data() + (size_t)pos * gd.entry_bytes, tmp.data()) != 0)
        return fail(PB_ERR_INVALID, "global dictionary of %s misses a value of segment %s", column, s->name.c_str());
      rm[i] = (int32_t)pos;
    }
  }
  return PB_OK;
}

static int get_global_dict(pb_group_s* g, const char* column, GlobalDict** out) {
  std::lock_guard<std::mutex> lk(g->mu);
  auto it = g->dicts.find(column);
  if (it == g->dicts.end()) {
    GlobalDict gd;
    int rc = build_union(g, column, gd);
    if (rc) return rc;
    it = g->dicts.emplace(column, std::move(gd)).first;
  }
  if (it->second.h_remap.empty()) {
    int rc = build_remaps(g, column, it->second);
    if (rc) return rc;
  }
  int rc = upload_remaps(g, it->second);
  if (rc) return rc;
  *out = &it->second;
  return PB_OK;
}

// host view of a remap (tests / multi-process agreement checks)
extern "C" int pb_segment_group_remap(pb_segment_group_handle g, const char* column, int32_t segment_index, const int32_t** remap, int32_t* n) {
  if (!g || !column || !remap || !n) return fail(PB_ERR_INVALID, "bad arguments");
  std::lock_guard<std::mutex> lk(g->mu);
  auto it = g->dicts.find(column);
  if (it == g->dicts.end()) {
    GlobalDict gd;
    int rc = build_union(g, column, gd);
    if (rc) return rc;
    it = g->dicts.emplace(column, std::move(gd)).first;
  }
  if (it->second.h_remap.empty()) { int rc = build_remaps(g, column, it->second); if (rc) return rc; }
  if (segment_index < 0 || segment_index >= (int)it->second.h_remap.size()) return fail(PB_ERR_INVALID, "segment index");
  *remap = it->second.h_remap[segment_index].data(); *n = (int32_t)it->second.h_remap[segment_index].size();
  return PB_OK;
}

extern "C" int pb_segment_group_export_dictionary(pb_segment_group_handle g, const char* column, const void** values,
                                                  int64_t* num_values, int32_t* entry_bytes) {
  if (!g || !column) return fail(PB_ERR_INVALID, "bad arguments");
  std::lock_guard<std::mutex> lk(g->mu);
  auto it = g->dicts.find(column);
  if (it == g->dicts.end()) {
    GlobalDict gd;
    int rc = build_union(g, column, gd);
    if (rc) return rc;
    it = g->dicts.emplace(column, std::move(gd)).first;
  }
  *values = it->second.values.data(); *num_values = it->second.n; *entry_bytes = it->second.entry_bytes;
  return PB_OK;
}
extern "C" int pb_segment_group_set_global_dictionary(pb_segment_group_handle g, const char* column, const void* values,
                                                      int64_t num_values, int32_t entry_bytes) {
  if (!g || !column || !values || num_values <= 0) return fail(PB_ERR_INVALID, "bad arguments");
  std::lock_guard<std::mutex> lk(g->mu);
  int ci = find_col(g->segs[0], column);
  if (ci < 0) return fail(PB_ERR_INVALID, "no column %s", column);
  for (auto* sg : g->segs) {
    int cj = find_col(sg, column);
    if (cj < 0) return fail(PB_ERR_INVALID, "segment %s has no column %s", sg->name.c_str(), column);
    // build_remaps writes each segment entry into an entry_bytes-sized buffer: a narrower global entry would overflow it
    if (!sg->cols[cj].has_dict) return fail(PB_ERR_UNSUPPORTED, "column %s has no dictionary", column);
    if (entry_bytes < sg->cols[cj].entry_bytes) return fail(PB_ERR_INVALID, "global dictionary of %s: entry_bytes %d < %d of segment %s", column, entry_bytes, sg->cols[cj].entry_bytes, sg->name.c_str());
  }
  GlobalDict& gd = g->dicts[column];
  g->dict_version++;
  gd.type = g->segs[0]->cols[ci].type;
  gd.entry_bytes = entry_bytes; gd.n = num_values; gd.external = true;
  gd.values.assign((const uint8_t*)values, (const uint8_t*)values + (size_t)num_values * entry_bytes);
  return build_remaps(g, column, gd);
}

// ------------------------------------------------------------------------------------------------
// results
// ------------------------------------------------------------------------------------------------
struct HostArr {
  void* p = nullptr; size_t bytes = 0;
  void alloc(size_t b) { bytes = b ? b : 8; p = pinned_alloc(bytes); }
  void release() { pinned_free(p, bytes); p = nullptr; }
};

struct TableMeta {
  int mode = 0;
  uint64_t capacity = 0;
  std::vector<int> seg_idx;                 // segments accumulated into this table
  std::vector<int64_t> cards;               // per group-by column (global or local)
  std::vector<int> shifts, widths;          // hash key layout
  DevTable dev;                             // device pointers (host copy of the struct)
  // finalize outputs
  int64_t num_groups = 0;
  HostArr slots, rows;
  std::vector<HostArr> dbl, lng, key_ids, key_vals, dc_off, dc_ids;
  std::vector<int> key_type, key_eb;
  std::vector<uint64_t> dset_cap;           // per aggregation: entries of the raw-column DISTINCTCOUNT value set (0 = none)
  std::vector<HostArr> dc_vals;             // ... and its value sets, materialised on demand
  pb_exec_stats stats{};
  uint64_t out_cap = 0;                     // capacity of the pinned output arrays
};

struct pb_result_s {
  pb_group_s* group = nullptr;
  cudaStream_t stream = nullptr;
  int n_gb = 0, n_aggs = 0;
  int table_mode = 0;
  bool combine = false, finalized = false;
  unsigned long long* d_seg_stats = nullptr;   // filtered aggregations: [n_segs][1 + PB_MAX_AGG_FILTERS] docs per swim-lane
  int n_agg_filters = 0;
  bool count_all = false;                   // PB_Q_NULL_HANDLING: every aggregation keeps its own (non-null) row count
  std::vector<int> agg_filter_of;
  int waves = 1;                            // launches were split into this many waves behind the staging copies
  int in_place_columns = 0;                 // (segment, column) pairs gathered from mapped host memory (PB_Q_GATHER_IN_PLACE)
  int residual_leaves = 0;                  // (segment, filter leaf) pairs tested by pb_agg_rows_kernel (DevRowLeaf)
  std::vector<int> agg_op;
  std::vector<std::string> gb_names, agg_cols;
  std::vector<TableMeta> tables;
  std::vector<void*> dev_allocs;            // freed (stream-ordered) with the result
  void* scratch = nullptr; size_t scratch_cap = 0;   // cached large scratch (match list)
  unsigned long long* d_counters = nullptr; // per table: [num_groups(u32 pair), limit flag, docs_matched, compaction counter]
  HostArr h_counters;
  int n_distinct_cols = 0;
  int n_scan_leaves_total = 0;
  std::vector<int64_t> seg_scan_leaves;     // per segment: number of scan leaves (for numEntriesScannedInFilter)
  double device_ms = 0, scan_ms = 0;
  double host_us[8] = {0};   // [0] stage+resolve [1] tables [2] descriptors [3] launches [4] finalize: count [5] gather+D2H wait [6] host decode
  int launches = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, evm = nullptr, ev2 = nullptr, ev3 = nullptr;
  StreamSet sset;
  bool match_all = false;
  double filter_ms = 0, agg_ms = 0;
  // contiguous spans of table 0 for the cross-GPU reduce: [counters .. row counts] int64 SUM, sums float64 SUM, min/max int64 MIN
  unsigned long long* span_i64 = nullptr; int64_t span_i64_n = 0;
  double* span_f64 = nullptr; int64_t span_f64_n = 0;
  long long* span_mm = nullptr; int64_t span_mm_n = 0;
  // the whole reducible state of table 0 as one block: [0, sum_off) counters + row counts (u64 SUM), [sum_off, dc_off) sums
  // (f64 SUM), [dc_off, mm_off) distinct bitsets (OR), [mm_off, bytes) min/max (i64 MIN)
  uint8_t* block = nullptr; int64_t block_bytes = 0, block_sum_off = 0, block_dc_off = 0, block_mm_off = 0;
  unsigned long long fingerprint = 0;       // of the block layout (counter cell [9])
  int merged_ranks = 1;                     // blocks summed into this one (cross-GPU merges)
  int pinned_segments = 0;                  // the first k segments of the group are pinned by this call
  // ---- everything needed to enqueue the call's kernels again without planning (a cached plan: see plan cache below) ----
  struct WaveLaunch { DevQuery dq; int seg_lo = 0, seg_hi = 0; uint64_t n_units = 0, n_docs = 0; int grid_filter = 0, grid_agg = 0; };
  struct Replay {
    std::vector<WaveLaunch> waves;
    const DevExpandItem* expand_items = nullptr; int n_expand = 0;
    int U = 2; bool u2_three = false; size_t smem_filter = 0;
    int spec_w = 0, spec_pk = 0;             // > 0: the plan-time specialised filter kernel of that width / predicate kind
    const DevRowSeg* row_segs = nullptr; int rows_rw = 0;   // agg_kind 4: pb_agg_rows_kernel<rows_rw>
    int agg_kind = 0;                        // 0 none (fused), 1 pb_agg_kernel<6>, 2 pb_agg_kernel<4>, 3 pb_agg_smem_kernel
    size_t smem_agg = 0;
    const DevLaneWeights* lane_w = nullptr; int n_lanes = 0, n_segs = 0;
    std::vector<DevFinalize> fin; std::vector<int> fin_grid; bool fin_prepared = false;
    // plan cache
    bool cacheable = false, busy = false;
    std::string sig;
    std::string host_sig;                    // key of the UNLOWERED query (host planning layer): a hit skips the lowering too
    uint64_t dict_version = 0; std::vector<uint64_t> seg_epochs;   // what the plan's pointers depend on (checked on a host-key hit)
    pb_group_s* owner = nullptr;             // group whose plan list holds this result (nullptr: not registered / orphaned)
    cudaGraphExec_t graph = nullptr;
    int uses = 0, graph_launches = 0;
    double comm_ms_sample = 0;               // cross-rank merge time of the plan's last kernel-by-kernel run (graph replays repeat it)
    uint32_t flags = 0;
  } rp;
  bool graph_replayed = false;
  struct InitArgs { uint4* zero = nullptr; uint64_t zn = 0; uint4* ff = nullptr; uint64_t fn = 0; uint4* mm = nullptr; uint64_t mn = 0;
                    uint4* aux = nullptr; uint64_t an = 0; const uint4* head = nullptr; uint64_t head_n16 = 0; int grid = 1; } init;   // pb_init_tables_kernel
  int key_words = 1;
  // ORDER BY ... LIMIT trim (pb_query_desc.order_by): per table an order-key array and the radix-select state
  pb_order_by order0{0, 0, 0}; int trim_size = 0, trim_threshold = 0;
  std::vector<unsigned long long*> d_okey; std::vector<DevSelectState*> d_sel;
  bool track_first = false; uint32_t* d_first_thr = nullptr;   // numGroupsLimit in doc order (dense per-segment tables)
  bool repair_pass = false;                 // hash tables with a reachable numGroupsLimit: conditional second aggregation pass
  bool fused = false, smem_table = false;   // how the matches reached the table (see exec_single)
  bool comm_timed = false;                  // events [5],[6] bracket the cross-rank merge
  double comm_ms = 0;
  Context* ctx = nullptr;
  std::vector<pb_result_s*> parts;          // multi-device group: the per-device results merged into this one (freed with it)
  std::vector<std::pair<int, int>> table_map;   // shell result of a multi-device per-segment query: table -> (part, table of the part)
};


// ------------------------------------------------------------------------------------------------
// Plan cache.  A dashboard sends the same query over the same segments again and again; everything pb_query_execute
// builds for it -- staged-column lookups, table layout, descriptors, device tables, pinned result arrays, launch geometry
// -- depends only on (segment group, query), not on the call.  A finished result whose plan is reusable is therefore not
// destroyed by pb_result_free but parked in its group; the next identical call takes it back and only re-enqueues the
// kernels: from its second reuse on as ONE CUDA graph launch (table init -> filter -> aggregation -> hand-back).  All the
// work of the query is redone every time -- only the planning is reused.  Keyed by the full byte image of the query (no
// hash collisions), the group's dictionary version and the segments' staging epochs.  PB_PLAN_CACHE=0 disables it,
// PB_GRAPH=0 keeps the cache but enqueues the kernels one by one.
// ------------------------------------------------------------------------------------------------
static std::mutex g_plan_mu;
#define PB_MAX_PLANS_PER_GROUP 8

static void sig_put(std::string& s, const void* p, size_t n) { s.append(static_cast<const char*>(p), n); }
template <class T> static void sig_pod(std::string& s, const T& v) { sig_put(s, &v, sizeof v); }
static void sig_str(std::string& s, const char* c) { const uint32_t n = c ? (uint32_t)strlen(c) : 0xffffffffu; sig_pod(s, n); if (c) sig_put(s, c, n); }
static void sig_nodes(std::string& s, const pb_filter_node* nodes, int n) {
  sig_pod(s, n);
  for (int i = 0; i < n; i++) {
    const pb_filter_node& f = nodes[i];
    sig_pod(s, f.kind); sig_pod(s, f.column); sig_pod(s, f.num_children); sig_pod(s, f.exclusive); sig_pod(s, f.lo); sig_pod(s, f.hi);
    sig_pod(s, f.dlo); sig_pod(s, f.dhi); sig_pod(s, f.dlo_inclusive); sig_pod(s, f.dhi_inclusive); sig_pod(s, f.num_ids); sig_pod(s, f.num_raw_values);
    sig_pod(s, f.blob_len);
    if (f.ids && f.num_ids > 0) sig_put(s, f.ids, sizeof(int32_t) * (size_t)f.num_ids * (f.kind == PB_F_SORTED ? 2 : 1));
    if (f.raw_values && f.num_raw_values > 0) sig_put(s, f.raw_values, sizeof(int64_t) * (size_t)f.num_raw_values);
    if (f.blob && f.blob_len > 0) sig_put(s, f.blob, (size_t)f.blob_len);
  }
}
static std::string plan_signature(pb_group_s* g, const pb_segment_query* sqs, const pb_query_desc* q) {
  std::string s;
  s.reserve(4096);
  sig_pod(s, q->flags); sig_pod(s, q->num_groups_limit); sig_pod(s, q->max_initial_result_holder_capacity);
  sig_pod(s, q->num_group_by);
  for (int j = 0; j < q->num_group_by; j++) sig_str(s, q->group_by_columns[j]);
  sig_pod(s, q->num_aggregations);
  for (int a = 0; a < q->num_aggregations; a++) { sig_pod(s, q->aggregations[a].op); sig_str(s, q->aggregations[a].column); }
  sig_pod(s, q->num_agg_filters);
  if (q->num_agg_filters > 0) sig_put(s, q->agg_filter_of, sizeof(int32_t) * (size_t)q->num_aggregations);
  sig_pod(s, q->num_order_by); sig_pod(s, q->trim_size); sig_pod(s, q->trim_threshold);
  if (q->num_order_by > 0 && q->order_by) sig_put(s, q->order_by, sizeof(pb_order_by) * (size_t)q->num_order_by);
  sig_pod(s, g->dict_version);
  for (size_t si = 0; si < g->segs.size(); si++) {
    sig_pod(s, g->segs[si]->epoch);
    sig_nodes(s, sqs[si].filter, sqs[si].num_filter_nodes);
    for (int f = 0; f < q->num_agg_filters; f++) sig_nodes(s, sqs[si].agg_filters[f], sqs[si].agg_filter_nodes[f]);
  }
  return s;
}
static bool plan_cache_enabled() { static const bool on = []() { const char* e = getenv("PB_PLAN_CACHE"); return !e || atoi(e) != 0; }(); return on; }
static bool plan_graph_enabled() { static const bool on = []() { const char* e = getenv("PB_GRAPH"); return !e || atoi(e) != 0; }(); return on; }

static pb_result_s* plan_take(pb_group_s* g, const std::string& sig) {
  std::lock_guard<std::mutex> lk(g_plan_mu);
  for (auto* p : g->plans)
    if (!p->rp.busy && p->rp.sig == sig) { p->rp.busy = true; return p; }
  return nullptr;
}
static void destroy_result(pb_result_s* r);
static thread_local std::string g_pending_host_key;      // set by the host planning layer around its pb_query_execute call
static void plan_register(pb_group_s* g, pb_result_s* r, std::string&& sig) {
  std::vector<pb_result_s*> evict;
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    r->rp.sig = std::move(sig); r->rp.owner = g; r->rp.busy = true;
    r->rp.host_sig = g_pending_host_key;
    r->rp.dict_version = g->dict_version;
    r->rp.seg_epochs.clear();
    for (auto* sg : g->segs) r->rp.seg_epochs.push_back(sg->epoch);
    g->plans.push_back(r);
    for (size_t i = 0; g->plans.size() > PB_MAX_PLANS_PER_GROUP && i < g->plans.size();) {      // oldest idle plans go first
      if (!g->plans[i]->rp.busy) { evict.push_back(g->plans[i]); g->plans[i]->rp.owner = nullptr; g->plans.erase(g->plans.begin() + (long)i); }
      else i++;
    }
  }
  for (auto* p : evict) destroy_result(p);
}
// group release: idle plans die with the group; a plan that is out as a live result is orphaned and dies on its pb_result_free
static void free_plans(pb_group_s* g) {
  std::vector<pb_result_s*> idle;
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    for (auto* p : g->plans) { p->rp.owner = nullptr; if (!p->rp.busy) idle.push_back(p); }
    g->plans.clear();
  }
  for (auto* p : idle) destroy_result(p);
}

// queries in flight pin their segments against eviction from the HBM segment cache; the pins are dropped when the result
// is finalized (a deferred result: when it is finalized or freed -- its group must still be alive then)
static void release_segments(pb_result_s* r) {
  if (!r->pinned_segments || !r->group) return;
  for (int i = 0; i < r->pinned_segments && i < (int)r->group->segs.size(); i++) {
    pb_segment_s* s = r->group->segs[(size_t)i];
    std::lock_guard<std::mutex> lk(s->mu);
    if (s->inflight > 0) s->inflight--;
  }
  r->pinned_segments = 0;
}
// CUDA graphs that captured NCCL collectives hold references on the communicator, and ncclCommDestroy waits until the last
// of them is gone: pb_comm_destroy therefore destroys these graphs first (their plans simply capture again later)
static std::mutex g_comm_graphs_mu;
static std::unordered_set<pb_result_s*> g_comm_graphs;
static void free_result(pb_result_s* r);
static void destroy_result(pb_result_s* r) {
  if (!r) return;
  for (auto* p : r->parts) free_result(p);
  { std::lock_guard<std::mutex> lk(g_comm_graphs_mu); g_comm_graphs.erase(r); }
  if (r->rp.graph) { cudaGraphExecDestroy(r->rp.graph); r->rp.graph = nullptr; }
  DeviceGuard dg(r->ctx);
  if (r->stream) cudaStreamSynchronize(r->stream);
  release_segments(r);
  if (r->ctx) scratch_free(r->ctx, r->scratch, r->scratch_cap);
  for (void* p : r->dev_allocs) cudaFreeAsync(p, r->stream);
  for (auto& t : r->tables) {
    t.slots.release(); t.rows.release();
    for (auto* v : {&t.dbl, &t.lng, &t.key_ids, &t.key_vals, &t.dc_off, &t.dc_ids, &t.dc_vals}) for (auto& a : *v) a.release();
  }
  r->h_counters.release();
  if (r->stream) { cudaStreamSynchronize(r->stream); stream_set_release(r->ctx, r->sset); }
  delete r;
}
// pb_result_free: a result whose plan is registered in its (still living) group is parked for the next identical query
static void free_result(pb_result_s* r) {
  if (!r) return;
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    if (r->rp.owner) {
      if (r->stream) { DeviceGuard dg(r->ctx); cudaStreamSynchronize(r->stream); }
      release_segments(r);
      r->rp.busy = false;
      return;
    }
  }
  destroy_result(r);
}
extern "C" void pb_result_free(pb_result_handle r) { free_result(r); }

// ------------------------------------------------------------------------------------------------
// query execution
// ------------------------------------------------------------------------------------------------
#define PB_DENSE_MAX (1ull << 24)
#define PB_MAX_WAVES 8            // cold segments: launches are split into waves that follow the staging copies
// u64 cells per table at the head of the table block (summed by cross-GPU merges like the row counts):
//   [0] num_groups (lo u32)  [1] limit flag (lo u32)  [2] docs matched  [3] compaction cursor (0 until finalize)
//   [4] swim-lane docs  [5] swim-lane entries scanned post filter (filtered aggregations, pb_lane_stats_kernel)
//   [6] total docs  [7] entries scanned in filter  [8] segments        (host-known; injected by pb_init_tables_kernel)
//   [9] layout fingerprint of the block: after a merge over n ranks it must read n x the local value, else the ranks
//       did not run the same query over the same global dictionaries
#define PB_COUNTERS_PER_TABLE 10

struct Arena {   // host mirror of a device allocation; pointers are handed out as device addresses
  std::vector<uint8_t> host;
  uint8_t* dev = nullptr;
  size_t cap = 0, used = 0;
  template <class T> T* put(const T* src, size_t count, T** host_view = nullptr) {
    size_t bytes = sizeof(T) * count;
    used = (used + 15) & ~(size_t)15;
    if (used + bytes > cap) return nullptr;
    if (src) memcpy(host.data() + used, src, bytes); else memset(host.data() + used, 0, bytes);
    if (host_view) *host_view = reinterpret_cast<T*>(host.data() + used);
    T* d = reinterpret_cast<T*>(dev + used);
    used += bytes;
    return d;
  }
};

// Expected fraction of a segment's docs that pass one filter leaf, from dictionary cardinalities (uniform values).
static double estimate_leaf(const pb_segment_s* s, const pb_filter_node& fn) {
  const Column* c = (fn.column >= 0 && fn.column < (int)s->cols.size()) ? &s->cols[fn.column] : nullptr;
  const double card = c && c->card > 0 ? (double)c->card : 1.0;
  auto excl = [&](double f) { return fn.exclusive ? 1.0 - f : f; };
  switch (fn.kind) {
    case PB_F_MATCH_ALL: return 1.0;
    case PB_F_EMPTY: return 0.0;
    case PB_F_SCAN_DICT_RANGE: return std::min(1.0, std::max(0.0, (double)(fn.hi - fn.lo) / card));
    case PB_F_SCAN_DICT_SET: case PB_F_INVERTED: return excl(std::min(1.0, (double)fn.num_ids / card));
    case PB_F_SORTED: {
      double docs = 0;
      for (int i = 0; i + 1 < fn.num_ids; i += 2) docs += (double)(fn.ids[i + 1] - fn.ids[i] + 1);
      return excl(std::min(1.0, docs / std::max(1, s->num_docs)));
    }
    default: return 0.5;     // raw-value predicates, serialized bitmaps: no statistics
  }
}

// Which scan leaves of a flat conjunction run on CANDIDATES instead of on the streamed column (DevLeaf::gather): leaves are
// taken most-selective first (as the kernel orders them); once the expected survivors drop to PB_GATHER_LEAF_PERMILLE
// (default 30 = 3 %), every later scan leaf costs less as one 32-byte sector read per surviving doc than as bits/8 bytes
// of stream per doc, and its column no longer occupies shared-memory stages.  cand_frac[n] = expected fraction of docs
// that reach leaf n.  (The reference does the same on the CPU: AndDocIdSet drives later scan iterators through applyAnd.)
static void plan_candidate_leaves(const pb_segment_s* s, const pb_segment_query& sq, std::vector<char>& gather, std::vector<double>& cand_frac) {
  const int nn = sq.num_filter_nodes;
  gather.assign((size_t)std::max(nn, 0), 0);
  cand_frac.assign((size_t)std::max(nn, 0), 1.0);
  static const int permille_max = []() { const char* e = getenv("PB_GATHER_LEAF_PERMILLE"); return e ? atoi(e) : 30; }();
  if (nn < 3) return;
  const pb_filter_node& root = sq.filter[nn - 1];
  if (root.kind != PB_F_AND || root.num_children != nn - 1) return;
  struct L { int n; double est; bool scan; };
  std::vector<L> ls;
  for (int n = 0; n + 1 < nn; n++) {
    const int k = sq.filter[n].kind;
    if (k == PB_F_AND || k == PB_F_OR || k == PB_F_NOT) return;
    const bool scan = k == PB_F_SCAN_DICT_RANGE || k == PB_F_SCAN_DICT_SET || k == PB_F_SCAN_RAW_RANGE || k == PB_F_SCAN_RAW_SET;
    ls.push_back({n, estimate_leaf(s, sq.filter[n]), scan});
  }
  std::stable_sort(ls.begin(), ls.end(), [](const L& a, const L& b) { return a.est < b.est; });
  double p = 1.0;
  bool have_dense = false;
  for (const L& l : ls) {
    cand_frac[l.n] = p;
    if (have_dense && l.scan && permille_max > 0 && p * 1000.0 <= (double)permille_max) gather[l.n] = 1;
    else have_dense = true;
    p *= l.est;
  }
  // a column that is streamed anyway (another leaf on it runs dense) is not gathered as well
  for (const L& l : ls)
    if (gather[l.n])
      for (const L& o : ls)
        if (!gather[o.n] && o.scan && sq.filter[o.n].column == sq.filter[l.n].column) { gather[l.n] = 0; break; }
  // shared-memory budget: every streamed column takes 2 stages x 8 warps x 1024 docs x its width.  Predicates on several wide
  // (raw LONG / DOUBLE) columns do not fit; the most selective leaves stay streamed, the rest run on the candidates whatever
  // the expected survivors (slower than streaming at low selectivity, but it runs -- and exactly the reference's applyAnd)
  const int budget_bits = 96;
  int used = 0;
  std::vector<int> streamed_cols;
  auto width_of = [&](int n) {
    const int col = sq.filter[n].column;
    if (col < 0 || col >= (int)s->cols.size()) return 0;          // (rejected later, when the leaf is lowered)
    const Column& c = s->cols[(size_t)col];
    return c.has_dict ? c.bits : 8 * c.raw_width;
  };
  for (const L& l : ls) {
    if (!l.scan || gather[l.n]) continue;
    const int col = sq.filter[l.n].column;
    if (std::find(streamed_cols.begin(), streamed_cols.end(), col) != streamed_cols.end()) continue;     // shares a streamed column
    const int w = width_of(l.n);
    if (!streamed_cols.empty() && used + w > budget_bits) { gather[l.n] = 1; continue; }
    used += w; streamed_cols.push_back(col);
  }
}

// Expected fraction of a segment's docs that pass the filter (postfix tree).  Drives the stage-or-gather choice of
// PB_Q_GATHER_IN_PLACE.
static double estimate_selectivity(const pb_segment_s* s, const pb_segment_query& sq) {
  if (sq.num_filter_nodes <= 0) return 1.0;
  std::vector<double> stk;
  for (int n = 0; n < sq.num_filter_nodes; n++) {
    const pb_filter_node& fn = sq.filter[n];
    switch (fn.kind) {
      case PB_F_AND: case PB_F_OR: {
        int k = std::min<int>(fn.num_children, (int)stk.size());
        double v = fn.kind == PB_F_AND ? 1.0 : 0.0;
        for (int i = 0; i < k; i++) { double x = stk.back(); stk.pop_back(); v = fn.kind == PB_F_AND ? v * x : v + x; }
        stk.push_back(std::min(1.0, v));
        break;
      }
      case PB_F_NOT: if (!stk.empty()) stk.back() = 1.0 - stk.back(); break;
      default: stk.push_back(estimate_leaf(s, fn)); break;
    }
  }
  return stk.empty() ? 1.0 : std::min(1.0, std::max(0.0, stk.back()));
}

static int finalize_result(pb_result_s* r);
static int enqueue_finalize(pb_result_s* r);
static int enqueue_trim(pb_result_s* r);
static int finish_finalize(pb_result_s* r);
static inline double now_us() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); }


// ------------------------------------------------------------------------------------------------
// cross-rank communicator (one process per GPU): NCCL, loaded at run time so that a single-GPU server needs no NCCL at all.
// The merge of the per-rank group tables is the device-side equivalent of GroupByCombineOperator's IndexedTable merge
// (CTR/operator/combine/GroupByCombineOperator.java:132-147) across the servers' GPUs.
// ------------------------------------------------------------------------------------------------
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*GetVersion)(int*) = nullptr;
};
struct Comm {
  std::mutex mu;
  NcclApi api;
  ncclComm_t comm = nullptr;
  int n_ranks = 1, rank = 0;
  Context* ctx = nullptr;
  int64_t checked_block_bytes = -1;      // block size the ranks last agreed on (sizes must match before an all-gather)
};
static Comm g_comm;

static int nccl_load() {
  NcclApi& a = g_comm.api;
  if (a.handle) return PB_OK;
  // (1) PB_NCCL_LIB, (2) a libnccl already mapped into the process (e.g. by torch: two NCCL copies in one process work but
  // waste memory), (3) the system library
  const char* env = getenv("PB_NCCL_LIB");
  void* h = env ? dlopen(env, RTLD_NOW | RTLD_LOCAL) : nullptr;
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL | RTLD_NOLOAD);
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_LOCAL);
  if (!h) return fail(PB_ERR_STATE, "NCCL not found (%s); set PB_NCCL_LIB", dlerror());
#define PB_NCCL_SYM(field, name)                                                                   \
  *(void**)(&a.field) = dlsym(h, name);                                                            \
  if (!a.field) { dlclose(h); return fail(PB_ERR_STATE, "NCCL symbol %s missing", name); }
  PB_NCCL_SYM(GetUniqueId, "ncclGetUniqueId") PB_NCCL_SYM(CommInitRank, "ncclCommInitRank") PB_NCCL_SYM(CommDestroy, "ncclCommDestroy")
  PB_NCCL_SYM(AllGather, "ncclAllGather") PB_NCCL_SYM(Send, "ncclSend") PB_NCCL_SYM(Recv, "ncclRecv")
  PB_NCCL_SYM(GroupStart, "ncclGroupStart") PB_NCCL_SYM(GroupEnd, "ncclGroupEnd") PB_NCCL_SYM(GetErrorString, "ncclGetErrorString")
  PB_NCCL_SYM(GetVersion, "ncclGetVersion")
#undef PB_NCCL_SYM
  a.handle = h;
  return PB_OK;
}
#define NC(call)                                                                                     \
  do {                                                                                               \
    ncclResult_t e__ = (call);                                                                       \
    if (e__ != ncclSuccess) return fail(PB_ERR_CUDA, "%s failed: %s", #call, g_comm.api.GetErrorString(e__)); \
  } while (0)

extern "C" int pb_comm_unique_id(void* out, size_t cap) {
  if (!out || cap < sizeof(ncclUniqueId)) return fail(PB_ERR_INVALID, "pb_comm_unique_id: need %zu bytes", sizeof(ncclUniqueId));
  std::lock_guard<std::mutex> lk(g_comm.mu);
  int rc = nccl_load();
  if (rc) return rc;
  ncclUniqueId id;
  NC(g_comm.api.GetUniqueId(&id));
  memcpy(out, &id, sizeof id);
  return PB_OK;
}
extern "C" int pb_comm_init(int n_ranks, int rank, const void* unique_id, size_t id_bytes) {
  if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(PB_ERR_INVALID, "pb_comm_init: rank %d of %d", rank, n_ranks);
  if (!unique_id || id_bytes < sizeof(ncclUniqueId)) return fail(PB_ERR_INVALID, "pb_comm_init: unique id of %zu bytes expected", sizeof(ncclUniqueId));
  int rc = ensure_init();
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g_comm.mu);
  if (g_comm.comm) return fail(PB_ERR_STATE, "pb_comm_init: communicator already initialised (rank %d of %d)", g_comm.rank, g_comm.n_ranks);
  if (g_all.ctxs.size() != 1) return fail(PB_ERR_UNSUPPORTED, "pb_comm_init: one device per process (this process drives %zu)", g_all.ctxs.size());
  if ((rc = nccl_load())) return rc;
  Context* ctx = g_all.ctxs[0].get();
  DeviceGuard dg(ctx);
  ncclUniqueId id;
  memcpy(&id, unique_id, sizeof id);
  NC(g_comm.api.CommInitRank(&g_comm.comm, n_ranks, id, rank));
  g_comm.n_ranks = n_ranks; g_comm.rank = rank; g_comm.ctx = ctx; g_comm.checked_block_bytes = -1;
  return PB_OK;
}
extern "C" int pb_comm_info(int* n_ranks, int* rank) {
  std::lock_guard<std::mutex> lk(g_comm.mu);
  if (n_ranks) *n_ranks = g_comm.comm ? g_comm.n_ranks : 1;
  if (rank) *rank = g_comm.comm ? g_comm.rank : 0;
  return g_comm.comm ? 1 : 0;
}
static void comm_shutdown() {
  std::lock_guard<std::mutex> lk(g_comm.mu);
  if (g_comm.comm) {
    DeviceGuard dg(g_comm.ctx);
    cudaDeviceSynchronize();
    {
      std::lock_guard<std::mutex> lk2(g_comm_graphs_mu);
      for (pb_result_s* r : g_comm_graphs) if (r->rp.graph) { cudaGraphExecDestroy(r->rp.graph); r->rp.graph = nullptr; }
      g_comm_graphs.clear();
    }
    g_comm.api.CommDestroy(g_comm.comm);
    g_comm.comm = nullptr; g_comm.n_ranks = 1; g_comm.rank = 0;
  }
}
extern "C" int pb_comm_destroy(void) { comm_shutdown(); return PB_OK; }

static int ensure_gather_buf(Context* ctx, size_t bytes, cudaStream_t st) {
  if (ctx->gather_cap >= bytes) return PB_OK;
  // the old buffer may still be read by a merge kernel in flight on another stream: let the device drain first (rare: growth only)
  if (ctx->gather_buf) { CU(cudaDeviceSynchronize()); CU(cudaFree(ctx->gather_buf)); ctx->gather_buf = nullptr; ctx->gather_cap = 0; }
  size_t cap = (bytes + ((size_t)1 << 20) - 1) & ~(((size_t)1 << 20) - 1);
  CU(cudaMalloc(&ctx->gather_buf, cap));
  ctx->gather_cap = cap;
  (void)st;
  return PB_OK;
}

static int launch_merge(pb_result_s* r, const void* gathered, int n_rows, bool base_is_dst);
static int launch_merge_rows(pb_result_s* r, const void* gathered, const DevMergePeers* peers, int n_rows, bool base_is_dst);
static int comm_merge_hash(pb_result_s* r);

// All ranks call with the same query (PB_Q_ALL_RANKS): all-gather of the table blocks + one merge kernel, on the call's own
// stream.  Every rank ends up with the merged table.
static int comm_merge(pb_result_s* r) {
  std::lock_guard<std::mutex> lk(g_comm.mu);       // collectives of one communicator must be issued in the same order on every rank
  if (!g_comm.comm) return fail(PB_ERR_STATE, "PB_Q_ALL_RANKS without pb_comm_init");
  if (g_comm.n_ranks == 1) return PB_OK;
  if (!r->combine || r->tables.size() != 1) return fail(PB_ERR_UNSUPPORTED, "PB_Q_ALL_RANKS needs PB_Q_COMBINE (one table per rank)");
  if (r->ctx != g_comm.ctx) return fail(PB_ERR_STATE, "PB_Q_ALL_RANKS: the result is not on the communicator's device");
  if (r->table_mode == T_HASH) return comm_merge_hash(r);
  const int n = g_comm.n_ranks;
  cudaStream_t st = r->stream;
  if (g_comm.checked_block_bytes != r->block_bytes) {
    // first query of this shape: the ranks compare their block sizes before anything is shipped (a size mismatch inside
    // ncclAllGather would corrupt memory or hang); same-size layouts are told apart later by the fingerprint cell
    int rc = ensure_gather_buf(r->ctx, 8 * (size_t)n + 8, st);
    if (rc) return rc;
    long long mine = r->block_bytes;
    long long* d = reinterpret_cast<long long*>(r->ctx->gather_buf);
    CU(cudaMemcpyAsync(d + n, &mine, 8, cudaMemcpyHostToDevice, st));
    NC(g_comm.api.AllGather(d + n, d, 8, ncclChar, g_comm.comm, st));
    std::vector<long long> all((size_t)n);
    CU(cudaMemcpyAsync(all.data(), d, 8 * (size_t)n, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int k = 0; k < n; k++)
      if (all[k] != mine) return fail(PB_ERR_STATE, "PB_Q_ALL_RANKS: rank %d's table block is %lld bytes, rank %d's %lld (different query or global dictionaries)", k, all[k], g_comm.rank, mine);
    g_comm.checked_block_bytes = r->block_bytes;
  }
  int rc = ensure_gather_buf(r->ctx, (size_t)n * (size_t)r->block_bytes, st);
  if (rc) return rc;
  CU(cudaEventRecord(r->sset.ev[5], st));
  NC(g_comm.api.AllGather(r->block, r->ctx->gather_buf, (size_t)r->block_bytes, ncclChar, g_comm.comm, st));
  if ((rc = launch_merge(r, r->ctx->gather_buf, n, false))) return rc;
  CU(cudaEventRecord(r->sset.ev[6], st));
  r->comm_timed = true;
  r->merged_ranks *= n;
  return PB_OK;
}


// Enqueue the call's kernels on its stream from the saved launch plan: table init -> index leaves to flat bitmaps ->
// per wave: filter (-> match list) and aggregation -> swim-lane statistics.  seg_wait (first execution of a cold query
// only): staging events the waves must wait for.
static int enqueue_all(pb_result_s* r, const std::vector<cudaEvent_t>* seg_wait) {
  cudaStream_t st = r->stream;
  const pb_result_s::Replay& rp = r->rp;
  CU(cudaEventRecord(r->ev0, st));
  pb_init_tables_kernel<<<r->init.grid, 256, 0, st>>>(r->init.zero, r->init.zn, r->init.ff, r->init.fn, r->init.mm, r->init.mn, r->init.aux, r->init.an,
                                                       r->init.head, r->init.head_n16);
  r->launches++;
  // index leaves -> flat bitmaps: one launch for every bitmap / range list of every segment
  for (int y0 = 0; y0 < rp.n_expand; y0 += 65535) {
    dim3 grid(32, (unsigned)std::min(65535, rp.n_expand - y0));
    pb_expand_kernel<<<grid, 256, 0, st>>>(rp.expand_items + y0);
    r->launches++;
  }
  CU(cudaGetLastError());
  // kernel 1: filter -> match list (or fused aggregation);  kernel 2: gather + aggregate the matching docs (per wave)
  CU(cudaEventRecord(r->ev1, st));
  for (size_t wi = 0; wi < rp.waves.size(); wi++) {
    const pb_result_s::WaveLaunch& w = rp.waves[wi];
    if (seg_wait && rp.waves.size() > 1)
      for (int si = w.seg_lo; si < w.seg_hi; si++) if ((*seg_wait)[si]) CU(cudaStreamWaitEvent(st, (*seg_wait)[si], 0));
    if (w.grid_filter > 0 && rp.spec_w > 0) {
      CU(pb_filter_spec_launch(rp.spec_w, rp.spec_pk, w.grid_filter, rp.smem_filter, st, &w.dq));
      r->launches++;
    } else if (w.grid_filter > 0) {
      if (rp.U == 1) pb_filter_kernel<1, 3><<<w.grid_filter, PB_NTHREADS, rp.smem_filter, st>>>(w.dq);
      else if (rp.u2_three) pb_filter_kernel<2, 3><<<w.grid_filter, PB_NTHREADS, rp.smem_filter, st>>>(w.dq);
      else pb_filter_kernel<2, 2><<<w.grid_filter, PB_NTHREADS, rp.smem_filter, st>>>(w.dq);
      r->launches++;
      CU(cudaGetLastError());
    }
    if (wi + 1 == rp.waves.size() || rp.waves.size() == 1) CU(cudaEventRecord(r->evm, st));   // (waves interleave: the split is only exact for one wave)
    if (w.grid_agg > 0) {
      if (rp.agg_kind == 4) {
        if (rp.rows_rw == 2) pb_agg_rows_kernel<2><<<w.grid_agg, PB_AGG_SMEM_THREADS, rp.smem_agg, st>>>(w.dq, rp.row_segs);
        else if (rp.rows_rw == 4) pb_agg_rows_kernel<4><<<w.grid_agg, PB_AGG_SMEM_THREADS, rp.smem_agg, st>>>(w.dq, rp.row_segs);
        else pb_agg_rows_kernel<8><<<w.grid_agg, PB_AGG_SMEM_THREADS, rp.smem_agg, st>>>(w.dq, rp.row_segs);
      } else if (rp.agg_kind == 3) pb_agg_smem_kernel<<<w.grid_agg, PB_AGG_SMEM_THREADS, rp.smem_agg, st>>>(w.dq);
      else if (rp.agg_kind == 2) pb_agg_kernel<4><<<w.grid_agg, PB_NTHREADS, rp.smem_agg, st>>>(w.dq);
      else pb_agg_kernel<6><<<w.grid_agg, PB_NTHREADS, rp.smem_agg, st>>>(w.dq);
      r->launches++;
      CU(cudaGetLastError());
      if (r->repair_pass && rp.waves.size() == 1 && (rp.agg_kind == 1 || rp.agg_kind == 2)) {
        // numGroupsLimit was reachable: if some key was refused (device-side check), zero the aggregates (keys and counters
        // stay) and aggregate the matches again in lookup-only mode, see pb_hash_slot
        const uint64_t skip16 = (((uint64_t)PB_COUNTERS_PER_TABLE * 8 * r->tables.size() + 255) & ~(uint64_t)255) / 16;
        pb_init_tables_kernel<<<r->init.grid, 256, 0, st>>>(r->init.zero + skip16, r->init.zn - skip16, nullptr, 0, r->init.mm, r->init.mn, nullptr, 0, nullptr, 0,
                                                             w.dq.any_limit);
        DevQuery dq2 = w.dq;
        dq2.phase = 2;
        if (rp.agg_kind == 2) pb_agg_kernel<4><<<w.grid_agg, PB_NTHREADS, rp.smem_agg, st>>>(dq2);
        else pb_agg_kernel<6><<<w.grid_agg, PB_NTHREADS, rp.smem_agg, st>>>(dq2);
        r->launches += 2;
        CU(cudaGetLastError());
      }
    }
  }
  CU(cudaEventRecord(r->ev2, st));
  if (rp.n_lanes > 1 && rp.n_segs > 0) {
    pb_lane_stats_kernel<<<(rp.n_segs + 127) / 128, 128, 0, st>>>(rp.lane_w, r->d_seg_stats, rp.n_segs, rp.n_lanes, r->d_counters, PB_COUNTERS_PER_TABLE);
    r->launches++;
    CU(cudaGetLastError());
  }
  return PB_OK;
}


// Run a cached plan again: pin the segments, re-enqueue the kernels (one graph launch from the second reuse on), hand back.
static int replay_plan(pb_result_s* r, const pb_query_desc* q) {
  pb_result_s::Replay& rp = r->rp;
  pb_group_s* g = r->group;
  Context* ctx = r->ctx;
  cudaStream_t st = r->stream;
  const double t0 = now_us();
  r->finalized = false; r->launches = 0; r->comm_timed = false; r->comm_ms = 0; r->merged_ranks = 1;
  for (int i = 0; i < 8; i++) r->host_us[i] = 0;
  for (auto& tm : r->tables) {
    tm.num_groups = 0;
    for (auto& a : tm.dc_off) a.release();        // DISTINCTCOUNT value sets of the previous run (materialised on demand)
    for (auto& a : tm.dc_ids) a.release();
    for (auto& a : tm.dc_vals) a.release();
  }
  for (size_t si = 0; si < g->segs.size(); si++) {
    pb_segment_s* sg = g->segs[si];
    std::lock_guard<std::mutex> lk(sg->mu);
    sg->inflight++; r->pinned_segments = (int)si + 1;
    std::lock_guard<std::mutex> lk2(ctx->mu);
    sg->last_used = ++ctx->lru_clock;
  }
  int rc = PB_OK;
  const bool all_ranks = (q->flags & PB_Q_ALL_RANKS) != 0;
  r->host_us[0] = now_us() - t0;
  const double t1 = now_us();
  // a collective query is captured too (NCCL collectives are graph-capturable): every rank replays the same plan the same
  // number of times, so all of them capture, sample and launch in step.  Hash tables merge with a host round trip and stay eager.
  static const bool graph_comm = []() { const char* e = getenv("PB_GRAPH_COMM"); return !e || atoi(e) != 0; }();
  const bool graph_ok = plan_graph_enabled() && (!all_ranks || (graph_comm && r->table_mode != T_HASH && g_comm.comm && g_comm.checked_block_bytes == r->block_bytes));
  if (graph_ok) {
    if (!rp.graph && rp.uses >= 1) {
      // second reuse: record the whole sequence once
      cudaGraph_t graph = nullptr;
      CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
      rc = enqueue_all(r, nullptr);
      if (!rc && all_ranks) rc = comm_merge(r);
      if (!rc) rc = enqueue_trim(r);
      if (!rc) rc = enqueue_finalize(r);
      cudaError_t e = cudaStreamEndCapture(st, &graph);
      if (rc || e != cudaSuccess || !graph) { if (graph) cudaGraphDestroy(graph); cudaGetLastError(); return rc ? rc : fail(PB_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e)); }
      e = cudaGraphInstantiate(&rp.graph, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) { rp.graph = nullptr; return fail(PB_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(e)); }
      if (all_ranks) { std::lock_guard<std::mutex> lk(g_comm_graphs_mu); g_comm_graphs.insert(r); }
      rp.graph_launches = r->launches;
      r->launches = 0;
      r->merged_ranks = 1; r->comm_timed = false;       // (the capture ran comm_merge's bookkeeping, not the collective)
    }
    // CUDA events recorded inside a graph cannot be timed: every 8th replay is enqueued kernel by kernel instead, which
    // keeps the per-kernel CUDA-event times (pb_result_phase_ms) of a cached plan live; the others report the last sample
    const bool sample = rp.graph && (rp.uses & 7) == 7;
    if (rp.graph && !sample) {
      CU(cudaGraphLaunch(rp.graph, st)); r->launches = rp.graph_launches; r->graph_replayed = true;
      if (all_ranks) { r->merged_ranks *= g_comm.n_ranks; r->comm_timed = true; r->comm_ms = rp.comm_ms_sample; }
    } else {
      r->graph_replayed = false;
      if ((rc = enqueue_all(r, nullptr))) return rc;
      if (all_ranks && (rc = comm_merge(r))) return rc;
      if ((rc = enqueue_trim(r))) return rc;
      if ((rc = enqueue_finalize(r))) return rc;
    }
  } else {
    if ((rc = enqueue_all(r, nullptr))) return rc;
    if (all_ranks && (rc = comm_merge(r))) return rc;
    if ((rc = enqueue_trim(r))) return rc;
    if ((rc = enqueue_finalize(r))) return rc;
  }
  r->host_us[3] = now_us() - t1;
  rp.uses++;
  return finish_finalize(r);
}

// One device's part of a query: every segment of `g` lives on g->ctx.  Leaves the tables on the device when
// PB_Q_DEFER_FINALIZE is set; otherwise merges across ranks (PB_Q_ALL_RANKS) and finalizes.
static int exec_single(pb_segment_group_handle g, const pb_segment_query* sqs, const pb_query_desc* q, pb_result_handle* out) {
  int rc = PB_OK;
  Context* ctx = g->ctx;
  const int n_segs = (int)g->segs.size();
  const int nG = q->num_group_by, nA = q->num_aggregations;
  if (nG < 0 || nG > PB_MAX_GROUP_BY) return fail(PB_ERR_UNSUPPORTED, "%d group-by columns (max %d)", nG, PB_MAX_GROUP_BY);
  if (nA <= 0 || nA > PB_MAX_AGGS) return fail(PB_ERR_UNSUPPORTED, "%d aggregations (max %d)", nA, PB_MAX_AGGS);
  const bool combine = (q->flags & PB_Q_COMBINE) != 0;
  const bool in_place = (q->flags & PB_Q_GATHER_IN_PLACE) != 0;
  const int n_tables = combine ? 1 : n_segs;
  const int nF = q->num_agg_filters;
  const bool count_all = (q->flags & PB_Q_NULL_HANDLING) != 0;
  if (nF < 0 || nF > PB_MAX_AGG_FILTERS) return fail(PB_ERR_UNSUPPORTED, "%d FILTER clauses (max %d)", nF, PB_MAX_AGG_FILTERS);
  if (nF > 0) {
    if (!q->agg_filter_of) return fail(PB_ERR_INVALID, "agg_filter_of missing");
    for (int a = 0; a < nA; a++) if (q->agg_filter_of[a] < -1 || q->agg_filter_of[a] >= nF) return fail(PB_ERR_INVALID, "aggregation %d: bad FILTER clause index", a);
    for (int si = 0; si < n_segs; si++) if (!sqs[si].agg_filters || !sqs[si].agg_filter_nodes) return fail(PB_ERR_INVALID, "segment %d: FILTER clause programs missing", si);
  }

  // ---- plan cache: the same query over the same segments again -> replay its parked plan ----
  std::string sig;
  const bool try_cache = plan_cache_enabled() && !(q->flags & (PB_Q_DEFER_FINALIZE | PB_Q_GATHER_IN_PLACE));
  if (try_cache) {
    sig = plan_signature(g, sqs, q);
    if (pb_result_s* p = plan_take(g, sig)) {
      if ((rc = replay_plan(p, q))) { free_result(p); return rc; }
      *out = p;
      return PB_OK;
    }
  }
  std::unique_ptr<pb_result_s, void (*)(pb_result_s*)> R(new pb_result_s(), free_result);
  pb_result_s* r = R.get();
  r->group = g; r->n_gb = nG; r->n_aggs = nA; r->combine = combine; r->ctx = ctx;
  if ((rc = stream_set_acquire(ctx, &r->sset))) return rc;
  r->stream = r->sset.stream;
  cudaStream_t st = r->stream;
  r->ev0 = r->sset.ev[0]; r->ev1 = r->sset.ev[1]; r->evm = r->sset.ev[2]; r->ev2 = r->sset.ev[3]; r->ev3 = r->sset.ev[4];
  for (int j = 0; j < nG; j++) r->gb_names.push_back(q->group_by_columns[j]);
  for (int a = 0; a < nA; a++) {
    r->agg_op.push_back(q->aggregations[a].op);
    r->agg_cols.push_back(q->aggregations[a].column ? q->aggregations[a].column : "");
    if (q->aggregations[a].op < PB_AGG_COUNT || q->aggregations[a].op > PB_AGG_DISTINCTCOUNT) return fail(PB_ERR_UNSUPPORTED, "aggregation op %d", q->aggregations[a].op);
    if (q->aggregations[a].op != PB_AGG_COUNT && !q->aggregations[a].column) return fail(PB_ERR_INVALID, "aggregation %d needs a column", a);
  }

  double t_prev = now_us();
  auto lap = [&](int i) { double t = now_us(); r->host_us[i] += t - t_prev; t_prev = t; };
  // ---- resolve columns, stage what is needed ----
  std::vector<std::vector<int>> gcol(n_segs, std::vector<int>(nG)), acol(n_segs, std::vector<int>(nA, -1));
  bool any_raw_key = false;
  cudaStream_t cs = ctx->copy_stream;
  std::vector<cudaEvent_t> seg_wait(n_segs, nullptr);   // staging events this call's kernels must wait for
  int n_pending = 0;
  static const bool row_groups_on = []() { const char* e = getenv("PB_ROW_GROUPS"); return !e || atoi(e) != 0; }();
  std::vector<const RowGroup*> seg_rg(n_segs, nullptr);  // row group the gathers of each segment read from (nullptr: the columns themselves)
  std::vector<std::vector<char>> cand_leaf(n_segs);     // per filter node: scan leaf evaluated on candidates (DevLeaf::gather)
  std::vector<std::vector<double>> cand_frac(n_segs);
  for (int si = 0; si < n_segs; si++) plan_candidate_leaves(g->segs[si], sqs[si], cand_leaf[si], cand_frac[si]);
  for (int si = 0; si < n_segs; si++) {
    pb_segment_s* s = g->segs[si];
    std::lock_guard<std::mutex> lk(s->mu);
    s->inflight++; r->pinned_segments = si + 1;
    { std::lock_guard<std::mutex> lk2(ctx->mu); s->last_used = ++ctx->lru_clock; }
    // PB_Q_GATHER_IN_PLACE, per column: a gathered value costs one 32-byte PCIe read = 32 B payload + ~24 B of TLP
    // overhead of link time (measured on B200 / PCIe Gen5: the cold query is link-bound and each in-place value costs
    // ~56 streamed bytes); copying the column costs bits/8 bytes per doc.  Gather in place only where that is cheaper:
    // expected matches x 56 B < column bytes.
    // (PB_IN_PLACE_COST overrides the 56 B; 0 = always gather: used by the tests to reach every code path.)
    const double sel = in_place ? estimate_selectivity(s, sqs[si]) : 1.0;
    double gather_cost = 56.0;
    if (in_place) if (const char* e = getenv("PB_IN_PLACE_COST")) gather_cost = atof(e);
    auto gather_ok = [&](const Column& c) {
      if (!in_place) return false;
      const double col_bytes_per_doc = c.has_dict ? c.bits / 8.0 : (double)c.raw_width;
      return sel * gather_cost < col_bytes_per_doc;
    };
    for (int j = 0; j < nG; j++) {
      int ci = find_col(s, q->group_by_columns[j]);
      if (ci < 0) return fail(PB_ERR_INVALID, "segment %s: no column %s", s->name.c_str(), q->group_by_columns[j]);
      gcol[si][j] = ci;
      Column& c = s->cols[ci];
      if (!c.has_dict) any_raw_key = true;
      if ((rc = stage_column(s, c, true, false, false, cs, !combine, gather_ok(c)))) return rc;
    }
    for (int a = 0; a < nA; a++) {
      if (q->aggregations[a].op == PB_AGG_COUNT) continue;
      int ci = find_col(s, q->aggregations[a].column);
      if (ci < 0) return fail(PB_ERR_INVALID, "segment %s: no column %s", s->name.c_str(), q->aggregations[a].column);
      acol[si][a] = ci;
      Column& c = s->cols[ci];
      if (q->aggregations[a].op == PB_AGG_DISTINCTCOUNT) {
        if (!c.has_dict && c.type == PB_STRING) return fail(PB_ERR_UNSUPPORTED, "DISTINCTCOUNT on raw STRING column %s", c.name.c_str());
        if ((rc = stage_column(s, c, true, false, false, cs, false, gather_ok(c)))) return rc;
      } else {
        if (c.type == PB_STRING) return fail(PB_ERR_UNSUPPORTED, "numeric aggregation on STRING column %s", c.name.c_str());
        if ((rc = stage_column(s, c, true, true, false, cs, false, gather_ok(c)))) return rc;
      }
    }
    const pb_segment_query& sq = sqs[si];
    if (sq.num_filter_nodes > PB_MAX_NODES) return fail(PB_ERR_UNSUPPORTED, "filter has %d nodes (max %d)", sq.num_filter_nodes, PB_MAX_NODES);
    for (int n = 0; n < sq.num_filter_nodes; n++) {
      const pb_filter_node& fn = sq.filter[n];
      if (fn.kind >= PB_F_SCAN_DICT_RANGE && fn.kind <= PB_F_INVERTED) {
        if (fn.column < 0 || fn.column >= (int)s->cols.size()) return fail(PB_ERR_INVALID, "filter node %d: bad column", n);
        Column& c = s->cols[fn.column];
        bool inv = fn.kind == PB_F_INVERTED;
        if ((fn.kind == PB_F_SCAN_DICT_RANGE || fn.kind == PB_F_SCAN_DICT_SET) && !c.has_dict) return fail(PB_ERR_INVALID, "filter node %d: dictionary scan on raw column", n);
        if ((fn.kind == PB_F_SCAN_RAW_RANGE || fn.kind == PB_F_SCAN_RAW_SET) && c.has_dict) return fail(PB_ERR_INVALID, "filter node %d: raw scan on dictionary column", n);
        // a leaf that runs on candidates only reads the rows that reach it: cold segments can leave its column in host memory
        bool leaf_in_place = false;
        if (in_place && !inv && cand_leaf[si][n]) {
          const double col_bytes_per_doc = c.has_dict ? c.bits / 8.0 : (double)c.raw_width;
          leaf_in_place = cand_frac[si][n] * gather_cost < col_bytes_per_doc;
        }
        if ((rc = stage_column(s, c, !inv, false, inv, cs, false, leaf_in_place))) return rc;
      }
    }
    // FILTER(WHERE ...) clauses: their leaves are tested per matching doc by the aggregation kernel (gathers)
    for (int f = 0; f < nF; f++) {
      if (sq.agg_filter_nodes[f] < 0 || sq.agg_filter_nodes[f] > PB_MAX_AF_NODES) return fail(PB_ERR_UNSUPPORTED, "FILTER clause %d has %d nodes (max %d)", f, sq.agg_filter_nodes[f], PB_MAX_AF_NODES);
      for (int n = 0; n < sq.agg_filter_nodes[f]; n++) {
        const pb_filter_node& fn = sq.agg_filters[f][n];
        if (fn.kind >= PB_F_SCAN_DICT_RANGE && fn.kind <= PB_F_INVERTED) {
          if (fn.column < 0 || fn.column >= (int)s->cols.size()) return fail(PB_ERR_INVALID, "FILTER clause %d node %d: bad column", f, n);
          Column& c = s->cols[fn.column];
          bool inv = fn.kind == PB_F_INVERTED;
          if ((fn.kind == PB_F_SCAN_DICT_RANGE || fn.kind == PB_F_SCAN_DICT_SET) && !c.has_dict) return fail(PB_ERR_INVALID, "FILTER clause %d node %d: dictionary scan on raw column", f, n);
          if ((fn.kind == PB_F_SCAN_RAW_RANGE || fn.kind == PB_F_SCAN_RAW_SET) && c.has_dict) return fail(PB_ERR_INVALID, "FILTER clause %d node %d: raw scan on dictionary column", f, n);
          if ((rc = stage_column(s, c, !inv, false, inv, cs, false, !inv && gather_ok(c)))) return rc;
        }
      }
    }
    // ---- row group: the dictionary columns this query gathers per matching doc, side by side in one row ----
    if (row_groups_on && !in_place) {
      const double sel_rg = estimate_selectivity(s, sq);
      if (sel_rg <= 0.5) {
        std::vector<std::pair<int, int>> want;      // (column, form): 0 = dictId, 1 = decoded value (numeric aggregation inputs)
        auto add = [&](int ci, int form) {
          if (ci < 0 || !s->cols[ci].has_dict || !s->cols[ci].fwd_staged) return;
          if (std::find(want.begin(), want.end(), std::make_pair(ci, form)) == want.end()) want.push_back({ci, form});
        };
        for (int j = 0; j < nG; j++) add(gcol[si][j], 0);
        for (int a = 0; a < nA; a++) {
          if (acol[si][a] < 0) continue;
          Column& c = s->cols[acol[si][a]];
          const bool decoded = q->aggregations[a].op != PB_AGG_DISTINCTCOUNT && c.has_dict && c.type != PB_STRING;
          if (decoded && !c.native_staged && (rc = stage_column(s, c, false, false, false, cs, true, false))) return rc;   // the build reads the native dictionary
          add(acol[si][a], decoded ? 1 : 0);
        }
        for (int n = 0; n < sq.num_filter_nodes; n++)
          if (cand_leaf[si][n] && (sq.filter[n].kind == PB_F_SCAN_DICT_RANGE || sq.filter[n].kind == PB_F_SCAN_DICT_SET)) add(sq.filter[n].column, 0);
        for (int f = 0; f < nF; f++)
          for (int n = 0; n < sq.agg_filter_nodes[f]; n++)
            if (sq.agg_filters[f][n].kind == PB_F_SCAN_DICT_RANGE || sq.agg_filters[f][n].kind == PB_F_SCAN_DICT_SET) add(sq.agg_filters[f][n].column, 0);
        std::sort(want.begin(), want.end());
        seg_rg[si] = row_group_for(s, want, cs);
      }
    }
    if (s->device_bytes != s->accounted_bytes) {
      std::lock_guard<std::mutex> lk2(ctx->mu);
      ctx->staged_bytes += s->device_bytes - s->accounted_bytes;
      s->accounted_bytes = s->device_bytes;
    }
    // order this (and every later) query's kernels after the copies just enqueued for the segment
    if (s->stage_dirty) {
      if (!s->staged_ev) CU(cudaEventCreateWithFlags(&s->staged_ev, cudaEventDisableTiming));
      CU(cudaEventRecord(s->staged_ev, cs));
      s->stage_dirty = false; s->staged_pending = true;
    }
    if (s->staged_pending) {
      if (cudaEventQuery(s->staged_ev) == cudaSuccess) s->staged_pending = false;
      else { seg_wait[si] = s->staged_ev; n_pending++; }
      cudaGetLastError();   // cudaErrorNotReady is not an error
    }
  }

  enforce_cache_limit(ctx);      // this call's segments are pinned: only others can go

  // ---- global dictionaries (combined mode) ----
  std::vector<GlobalDict*> gdict(nG, nullptr), adict(nA, nullptr);
  if (combine) {
    for (int j = 0; j < nG; j++) {
      if (!g->segs[0]->cols[gcol[0][j]].has_dict) continue;
      if ((rc = get_global_dict(g, q->group_by_columns[j], &gdict[j]))) return rc;
    }
    for (int a = 0; a < nA; a++)
      if (q->aggregations[a].op == PB_AGG_DISTINCTCOUNT && g->segs[0]->cols[acol[0][a]].has_dict &&
          (rc = get_global_dict(g, q->aggregations[a].column, &adict[a]))) return rc;
  }

  lap(0);
  // ---- table mode and layout ----
  r->tables.resize(n_tables);
  int table_mode = nG == 0 ? T_KEYLESS : T_DENSE;
  int key_words = 1;
  if (nG > 0) {
    for (int t = 0; t < n_tables; t++) {
      TableMeta& tm = r->tables[t];
      int si0 = combine ? 0 : t;
      tm.cards.resize(nG); tm.shifts.resize(nG); tm.widths.resize(nG);
      unsigned __int128 prod = 1;
      int total_bits = 0;
      for (int j = 0; j < nG; j++) {
        const Column& c = g->segs[si0]->cols[gcol[si0][j]];
        int64_t card; int width;
        if (c.has_dict) {
          card = combine ? gdict[j]->n : c.card;
          width = 1; while ((1ll << width) < card) width++;
        } else {
          card = -1;
          width = (c.type == PB_INT || c.type == PB_FLOAT) ? 32 : 64;
          if (nG == 1) width = 64;
        }
        tm.cards[j] = card; tm.widths[j] = width; tm.shifts[j] = total_bits; total_bits += width;
        if (card > 0 && prod <= ((unsigned __int128)1 << 70)) prod *= (unsigned __int128)card;
      }
      bool dense_ok = !any_raw_key && prod <= PB_DENSE_MAX;
      if (!dense_ok) {
        if (total_bits > 128) return fail(PB_ERR_UNSUPPORTED, "group key needs %d bits (> 128): decline to the CPU plan", total_bits);
        if (total_bits > 64) key_words = 2;
        table_mode = T_HASH;
      }
      tm.capacity = dense_ok ? (uint64_t)prod : 0;
    }
  }
  if (table_mode == T_HASH) {
    for (int t = 0; t < n_tables; t++) {
      TableMeta& tm = r->tables[t];
      uint64_t docs = 0;
      if (combine) for (auto* s : g->segs) docs += (uint64_t)s->num_docs; else docs = (uint64_t)g->segs[t]->num_docs;
      uint64_t want = std::min<uint64_t>((uint64_t)std::max(1, q->num_groups_limit), std::max<uint64_t>(docs, 1));
      uint64_t cap = 1024;
      while (cap < 2 * want) cap <<= 1;
      tm.capacity = cap;
    }
  }
  if (table_mode == T_KEYLESS) for (auto& tm : r->tables) tm.capacity = 1;
  r->table_mode = table_mode;
  for (int t = 0; t < n_tables; t++) {
    TableMeta& tm = r->tables[t];
    tm.mode = table_mode;
    if (combine) for (int si = 0; si < n_segs; si++) tm.seg_idx.push_back(si); else tm.seg_idx.push_back(t);
  }

  // ---- ORDER BY ... LIMIT trim requested? (first ORDER BY expression: a group-by column or a COUNT / SUM / MIN / MAX / AVG) ----
  if (q->num_order_by > 0 && q->order_by && q->trim_size > 0 && nG > 0) {
    const pb_order_by& ob = q->order_by[0];
    const bool ok = (ob.kind == 0 && ob.index >= 0 && ob.index < nG) ||
                    (ob.kind == 1 && ob.index >= 0 && ob.index < nA && q->aggregations[ob.index].op != PB_AGG_DISTINCTCOUNT);
    if (!ok) return fail(PB_ERR_UNSUPPORTED, "ORDER BY expression %d/%d cannot drive a device-side trim", ob.kind, ob.index);
    r->order0 = ob; r->trim_size = q->trim_size; r->trim_threshold = std::max(0, q->trim_threshold);
  }

  // ---- device table arenas: [zero region][0xFF region][min/max region] ----
  auto slots_of = [&](const TableMeta& tm) { return tm.capacity + (table_mode == T_HASH ? 1 : 0); };
  size_t zero_bytes = 0, ff_bytes = 0, mm_elems = 0;
  // numGroupsLimit below the key space of a dense table: the reference creates groups first come first served in doc order
  // (IntMapBasedHolder); kept exact for per-segment tables (a merged table reports the superset and the flag, DESIGN.md §4.6)
  bool track_first = false;
  if (table_mode == T_DENSE && (!combine || n_segs == 1))
    for (auto& tm : r->tables) if ((uint64_t)std::max(1, q->num_groups_limit) < tm.capacity) track_first = true;
  r->track_first = track_first;
  std::vector<uint64_t> dc_words(nA, 0);
  std::vector<char> dc_raw(nA, 0);           // DISTINCTCOUNT on a raw column: a (slot, value) set instead of a dictId bitset
  for (int a = 0; a < nA; a++)
    if (q->aggregations[a].op == PB_AGG_DISTINCTCOUNT && !g->segs[0]->cols[acol[0][a]].has_dict) dc_raw[a] = 1;
  for (int a = 0; a < nA; a++)
    if (q->aggregations[a].op == PB_AGG_DISTINCTCOUNT && !dc_raw[a]) {
      int64_t maxcard = 0;
      if (combine) maxcard = adict[a]->n; else for (int si = 0; si < n_segs; si++) maxcard = std::max<int64_t>(maxcard, g->segs[si]->cols[acol[si][a]].card);
      dc_words[a] = ((uint64_t)maxcard + 31) / 32;
    }
  for (auto& tm : r->tables) {
    uint64_t S = slots_of(tm);
    zero_bytes += 8 * S;                                     // rowcnt
    for (int a = 0; a < nA; a++) {
      int op = q->aggregations[a].op;
      if (nF > 0 && q->agg_filter_of[a] >= 0 && (op == PB_AGG_COUNT || op == PB_AGG_AVG || count_all)) zero_bytes += 8 * S;   // fcnt
      if (op == PB_AGG_SUM || op == PB_AGG_AVG) zero_bytes += 8 * S;
      if (op == PB_AGG_MIN || op == PB_AGG_MAX) mm_elems += S;
      if (op == PB_AGG_DISTINCTCOUNT && !dc_raw[a]) zero_bytes += 4 * S * dc_words[a];
      if (op == PB_AGG_DISTINCTCOUNT && dc_raw[a]) {
        zero_bytes += 8 * S;                                   // dcnt
        uint64_t docs = 0;
        for (int si : tm.seg_idx) docs += (uint64_t)g->segs[si]->num_docs;
        uint64_t cap = 1024;
        while (cap < 2 * docs) cap <<= 1;                      // at most one entry per doc
        if (cap > (1ull << 28)) return fail(PB_ERR_UNSUPPORTED, "DISTINCTCOUNT on raw column %s over %llu docs: value set too large", q->aggregations[a].column, (unsigned long long)docs);
        tm.dset_cap.resize(nA, 0); tm.dset_cap[a] = cap;
        ff_bytes += 16 * cap;
      }
    }
    zero_bytes = (zero_bytes + 255) & ~(size_t)255;
    if (table_mode == T_HASH) ff_bytes += (8 * S * (size_t)key_words + 15) & ~(size_t)15;      // (every piece of the 0xFF region starts 16-byte aligned: CAS.128)
    if (track_first) ff_bytes += (4 * S + 15) & ~(size_t)15;
  }
  const size_t seg_stats_bytes = nF > 0 ? 8 * (size_t)(1 + PB_MAX_AGG_FILTERS) * (size_t)n_segs : 0;   // swim-lane statistics per segment
  zero_bytes += 8 * PB_COUNTERS_PER_TABLE * (size_t)n_tables + 256;
  if (zero_bytes > (64ull << 30)) return fail(PB_ERR_UNSUPPORTED, "group table needs %zu bytes: decline to the CPU plan", zero_bytes);
  uint8_t *d_zero = nullptr, *d_ff = nullptr; long long* d_mm = nullptr;
  unsigned long long* d_seg_stats = nullptr;
  // one block: [zero region | min/max region] so that a cross-GPU merge can ship the whole table in one collective.  Its size
  // and layout depend on the query and the (global) dictionaries only -- never on how many segments this rank holds: the
  // per-wave match counters and per-segment swim-lane statistics live in an aux region behind it that is not shipped.
  zero_bytes = (zero_bytes + 255) & ~(size_t)255;
  const size_t mm_bytes = (8 * mm_elems + 255) & ~(size_t)255;
  const size_t any_limit_off = 8 * PB_MAX_WAVES + seg_stats_bytes;   // query-wide "a key was refused" flag (hash tables)
  const size_t thr_off = any_limit_off + 8;          // numGroupsLimit thresholds (one u32 per table), after the statistics
  const size_t aux_bytes = (thr_off + (track_first ? 4 * (size_t)n_tables : 0) + 255) & ~(size_t)255;
  CU(cudaMallocAsync((void**)&d_zero, zero_bytes + mm_bytes + aux_bytes + 16, st)); r->dev_allocs.push_back(d_zero);
  if (ff_bytes) { CU(cudaMallocAsync((void**)&d_ff, ff_bytes + 16, st)); r->dev_allocs.push_back(d_ff); }
  if (mm_elems) d_mm = reinterpret_cast<long long*>(d_zero + zero_bytes);
  uint8_t* d_aux = d_zero + zero_bytes + mm_bytes;
  r->d_first_thr = track_first ? reinterpret_cast<uint32_t*>(d_aux + thr_off) : nullptr;
  r->block = d_zero; r->block_bytes = (int64_t)(zero_bytes + 8 * mm_elems);
  r->block_mm_off = (int64_t)zero_bytes;

  {
    size_t zo = 0, fo = 0, mo = 0;
    r->d_counters = reinterpret_cast<unsigned long long*>(d_zero);
    zo += 8 * PB_COUNTERS_PER_TABLE * (size_t)n_tables;
    if (seg_stats_bytes) d_seg_stats = reinterpret_cast<unsigned long long*>(d_aux + 8 * PB_MAX_WAVES);
    r->d_seg_stats = d_seg_stats;
    zo = (zo + 255) & ~(size_t)255;
    for (int t = 0; t < n_tables; t++) {
      TableMeta& tm = r->tables[t];
      uint64_t S = slots_of(tm);
      DevTable& dt = tm.dev;
      memset(&dt, 0, sizeof dt);
      dt.mode = table_mode; dt.capacity = tm.capacity;
      dt.rowcnt = reinterpret_cast<unsigned long long*>(d_zero + zo); zo += 8 * S;
      for (int a = 0; a < nA; a++) {   // row counts of COUNT / AVG with a FILTER clause (u64, summed across GPUs with the row counts)
        int op = q->aggregations[a].op;
        if (nF > 0 && q->agg_filter_of[a] >= 0 && (op == PB_AGG_COUNT || op == PB_AGG_AVG || count_all)) { dt.fcnt[a] = reinterpret_cast<unsigned long long*>(d_zero + zo); zo += 8 * S; }
      }
      if (t == 0) { r->span_i64 = r->d_counters; r->span_i64_n = (int64_t)((d_zero + zo - (uint8_t*)r->d_counters) / 8); }
      // sums first (one contiguous float64 span for the cross-GPU reduce), then the distinct bitsets
      if (t == 0) r->span_f64 = reinterpret_cast<double*>(d_zero + zo);
      for (int a = 0; a < nA; a++) {
        int op = q->aggregations[a].op;
        if (op == PB_AGG_SUM || op == PB_AGG_AVG) { dt.sum[a] = reinterpret_cast<double*>(d_zero + zo); zo += 8 * S; }
      }
      if (t == 0) r->span_f64_n = (int64_t)((d_zero + zo - (uint8_t*)r->span_f64) / 8);
      if (t == 0) { r->block_sum_off = (int64_t)((uint8_t*)r->span_f64 - d_zero); r->block_dc_off = (int64_t)zo; }
      for (int a = 0; a < nA; a++) {
        int op = q->aggregations[a].op;
        if (op == PB_AGG_DISTINCTCOUNT && !dc_raw[a]) { dt.dc_bits[a] = reinterpret_cast<uint32_t*>(d_zero + zo); dt.dc_words[a] = dc_words[a]; zo += 4 * S * dc_words[a]; }
        if (op == PB_AGG_DISTINCTCOUNT && dc_raw[a]) { dt.dcnt[a] = reinterpret_cast<unsigned long long*>(d_zero + zo); zo += 8 * S; }
        if (op == PB_AGG_MIN || op == PB_AGG_MAX) {
          dt.mm[a] = d_mm + mo; mo += S;
        }
      }
      if (t == 0) { r->span_mm = d_mm; r->span_mm_n = (int64_t)mo; }
      zo = (zo + 255) & ~(size_t)255;
      if (table_mode == T_HASH) { dt.hkeys = reinterpret_cast<unsigned long long*>(d_ff + fo); fo += (8 * S * (size_t)key_words + 15) & ~(size_t)15; dt.key_words = key_words; }
      if (track_first) { dt.first_doc = reinterpret_cast<uint32_t*>(d_ff + fo); fo += (4 * S + 15) & ~(size_t)15; }
      for (int a = 0; a < nA; a++)
        if (dc_raw[a]) { dt.dset[a] = reinterpret_cast<unsigned long long*>(d_ff + fo); dt.dset_mask[a] = tm.dset_cap[a] - 1; fo += 16 * tm.dset_cap[a]; }
      unsigned long long* cnt = r->d_counters + (size_t)t * PB_COUNTERS_PER_TABLE;
      dt.num_groups = reinterpret_cast<unsigned int*>(cnt + 0);
      dt.limit_reached = reinterpret_cast<unsigned int*>(cnt + 1);
      dt.any_limit = reinterpret_cast<unsigned int*>(d_aux + any_limit_off);
      dt.docs_matched = cnt + 2;
      dt.num_groups_limit = (uint32_t)std::max(1, q->num_groups_limit);
      {
        uint64_t docs = 0;
        for (int si : tm.seg_idx) docs += (uint64_t)g->segs[si]->num_docs;
        dt.limit_active = (uint64_t)dt.num_groups_limit < docs ? 1u : 0u;    // groups <= docs: an unreachable limit needs no tickets
      }
    }
    CU(cudaGetLastError());
  }

  if (r->trim_size > 0) {
    for (int t = 0; t < n_tables; t++) {
      const uint64_t S = slots_of(r->tables[t]);
      unsigned long long* ok = nullptr; DevSelectState* sel = nullptr;
      CU(cudaMallocAsync((void**)&ok, 8 * S, st)); r->dev_allocs.push_back(ok);
      CU(cudaMallocAsync((void**)&sel, sizeof(DevSelectState), st)); r->dev_allocs.push_back(sel);
      CU(cudaMemsetAsync(sel, 0, sizeof(DevSelectState), st));
      r->d_okey.push_back(ok); r->d_sel.push_back(sel);
    }
  }
  lap(1);
  // ---- query arena (descriptors + leaf payloads) ----
  size_t arena_cap = (sizeof(DevQuery) + 16) * (1 + PB_MAX_WAVES) + 256 + (sizeof(DevSegQuery) + 64) * (size_t)n_segs + (sizeof(DevTable) + 64) * (size_t)n_tables
                     + 8 * PB_COUNTERS_PER_TABLE * (size_t)n_tables + 64 + (nF > 0 ? (sizeof(DevLaneWeights) + 16) * (size_t)n_segs : 0)
                     + (sizeof(DevRowSeg) + 16) * (size_t)n_segs;
  size_t bitmap_words_total = 0;
  for (int si = 0; si < n_segs; si++) {
    const pb_segment_query& sq = sqs[si];
    pb_segment_s* s = g->segs[si];
    auto account = [&](const pb_filter_node* nodes, int n_nodes) {
      for (int n = 0; n < n_nodes; n++) {
        const pb_filter_node& fn = nodes[n];
        if (fn.kind == PB_F_SCAN_DICT_SET) arena_cap += 4 * (((size_t)s->cols[fn.column].card + 31) / 32) + 32;
        if (fn.kind == PB_F_SCAN_RAW_SET) arena_cap += 8 * (size_t)fn.num_raw_values + 32;
        if (fn.kind == PB_F_INVERTED) arena_cap += (4 + sizeof(DevExpandItem)) * (size_t)std::max(fn.num_ids, 0) + 64;
        if (fn.kind == PB_F_SORTED) arena_cap += 8 * (size_t)std::max(fn.num_ids, 0) + sizeof(DevExpandItem) + 64;
        if (fn.kind == PB_F_BITMAP) {
          uint64_t bl = fn.blob ? fn.blob_len : 0;
          if (!fn.blob && fn.column >= 0 && fn.column < (int)s->cols.size()) bl = s->cols[(size_t)fn.column].h_null_len;   // the column's null-value vector
          arena_cap += bl + sizeof(DevExpandItem) + 128;
        }
        if (fn.kind == PB_F_INVERTED || fn.kind == PB_F_SORTED || fn.kind == PB_F_BITMAP) bitmap_words_total += (((size_t)s->num_docs + 2047) / 2048) * 64;
      }
    };
    account(sq.filter, sq.num_filter_nodes);
    for (int f = 0; f < nF; f++) account(sq.agg_filters[f], sq.agg_filter_nodes[f]);
  }
  Arena ar;
  ar.cap = arena_cap; ar.host.resize(arena_cap);
  CU(cudaMallocAsync((void**)&ar.dev, arena_cap, st)); r->dev_allocs.push_back(ar.dev);
  uint32_t* d_bitmaps = nullptr;
  if (bitmap_words_total) {
    CU(cudaMallocAsync((void**)&d_bitmaps, 4 * bitmap_words_total, st)); r->dev_allocs.push_back(d_bitmaps);
    CU(cudaMemsetAsync(d_bitmaps, 0, 4 * bitmap_words_total, st));
  }

  DevQuery* hq = nullptr;
  DevQuery* dq = ar.put<DevQuery>(nullptr, 1, &hq);
  DevSegQuery* hsegs = nullptr;
  DevSegQuery* dsegs = ar.put<DevSegQuery>(nullptr, (size_t)n_segs, &hsegs);
  DevTable* htabs = nullptr;
  DevTable* dtabs = ar.put<DevTable>(nullptr, (size_t)n_tables, &htabs);
  for (int t = 0; t < n_tables; t++) htabs[t] = r->tables[t].dev;

  struct PendingExpand { int kind; const uint8_t* inv; int card; const int32_t* ids; int n_ids; uint32_t* out; uint32_t num_docs; std::vector<int32_t> host_ids; };
  std::vector<PendingExpand> expands;
  int slot_bits_max[PB_MAX_SCAN_SLOTS] = {0};
  int set_cache_max = 0;
  int n_slots_max = 0;
  bool any_cand_leaf = false;
  size_t bm_off = 0;
  r->seg_scan_leaves.assign(n_segs, 0);

  // ---- plan-time specialisation of the aggregation (pb_agg_rows_kernel): a dense table, every key a dictionary column
  // and every aggregation COUNT(*) or a numeric column, all of them fields of row groups of one stride ----
  int rows_rw = 0;
  bool rows_ok = false;
  {
    static const bool rows_on = []() { const char* e = getenv("PB_AGG_ROWS"); return !e || atoi(e) != 0; }();
    rows_ok = rows_on && table_mode == T_DENSE && nF == 0 && nG > 0 && n_segs > 0;
    for (int si = 0; si < n_segs && rows_ok; si++) {
      const RowGroup* rg = seg_rg[si];
      if (!rg || (rows_rw && rows_rw != rg->stride_bits / 32)) { rows_ok = false; break; }
      rows_rw = rg->stride_bits / 32;
      for (int j = 0; j < nG && rows_ok; j++) if (rg->find(gcol[si][j], 0) < 0) rows_ok = false;
      for (int a = 0; a < nA && rows_ok; a++) {
        const int op = q->aggregations[a].op;
        if (op == PB_AGG_COUNT) continue;
        if (op == PB_AGG_DISTINCTCOUNT || rg->find(acol[si][a], 1) < 0) rows_ok = false;
      }
    }
    if (!rows_ok) rows_rw = 0;
  }
  // Residual leaves (DevRowLeaf): with the rows kernel, a dictionary leaf that would run on the filter kernel's candidates
  // and whose column is a row-group field leaves the filter program; the rows kernel tests it on the row it loads anyway.
  // (PB_AGG_RESIDUAL=0 keeps such leaves on the candidates.)
  static const bool residual_on = []() { const char* e = getenv("PB_AGG_RESIDUAL"); return !e || atoi(e) != 0; }();
  std::vector<std::vector<DevRowLeaf>> residual(n_segs);
  r->residual_leaves = 0;

  for (int si = 0; si < n_segs; si++) {
    pb_segment_s* s = g->segs[si];
    const pb_segment_query& sq = sqs[si];
    DevSegQuery& ds = hsegs[si];
    ds.num_docs = s->num_docs;
    ds.table = combine ? 0 : si;
    int n_scan = 0, set_smem_used = 0;
    int slot_of_col[PB_MAX_SCAN_SLOTS];
    std::vector<char> residual_node((size_t)std::max(sq.num_filter_nodes, 0), 0);
    // one postfix filter program -> device nodes + leaves.  force_gather: every scan leaf is tested per doc from its forward
    // index (FILTER clauses, evaluated by pb_agg_kernel); otherwise the candidate plan decides per leaf.
    auto build_program = [&](const pb_filter_node* nodes, int n_nodes, int8_t* node_kind, int8_t* node_arg, DevLeaf* leaves, int max_leaves,
                             int& n_leaves, bool force_gather) -> int {
    for (int n = 0; n < n_nodes; n++) {
      const pb_filter_node& fn = nodes[n];
      if (fn.kind == PB_F_AND || fn.kind == PB_F_OR) {
        if (fn.num_children < 1 || fn.num_children > PB_MAX_LEAVES) return fail(PB_ERR_UNSUPPORTED, "AND/OR with %d children", fn.num_children);
        node_kind[n] = fn.kind == PB_F_AND ? N_AND : N_OR; node_arg[n] = (int8_t)fn.num_children; continue;
      }
      if (fn.kind == PB_F_NOT) { node_kind[n] = N_NOT; node_arg[n] = 1; continue; }
      if (n_leaves >= max_leaves) return fail(PB_ERR_UNSUPPORTED, "more than %d filter leaves", max_leaves);
      DevLeaf& lf = leaves[n_leaves];
      memset(&lf, 0, sizeof lf);
      lf.set_smem_off = -1;
      lf.est_permille = 500;
      node_kind[n] = N_LEAF; node_arg[n] = (int8_t)n_leaves; n_leaves++;
      // row-group field of a residual leaf, -1 = the leaf stays in this program
      const int residual_field = (!force_gather && rows_ok && residual_on && cand_leaf[si][n] && residual[si].size() < PB_ROWS_MAX_LEAVES &&
                                  (fn.kind == PB_F_SCAN_DICT_RANGE || fn.kind == PB_F_SCAN_DICT_SET)) ? seg_rg[si]->find(fn.column, 0) : -1;
      auto make_residual = [&](const Column& c, const uint32_t* set) {
        DevRowLeaf rl; memset(&rl, 0, sizeof rl);
        rl.off = (uint32_t)seg_rg[si]->bit_off[(size_t)residual_field]; rl.bits = (uint32_t)c.bits;
        rl.lo = lf.lo; rl.span = lf.span; rl.set = set; rl.excl = (uint32_t)lf.exclusive;
        residual[si].push_back(rl);
        residual_node[n] = 1;
      };
      auto scan_slot = [&](const Column& c) -> int {
        if (force_gather || cand_leaf[si][n]) {          // evaluated on candidates: no stage slot, read where the column lies
          lf.gather = 1;
          lf.gfwd = c.fwd_staged ? c.d_fwd : c.d_fwd_host;
          lf.g_full_words = c.fwd_staged ? 0xFFFFFFFFu : c.host_full_words;
          lf.g_tail_word = c.fwd_staged ? 0u : c.host_tail_word;
          lf.g_stride_bits = c.bits; lf.g_bit_off = 0;
          if (!c.has_dict) lf.g_stride_bits = 8 * c.raw_width;
          if (c.has_dict && seg_rg[si] && seg_rg[si]->find(fn.column, 0) >= 0) {
            const RowGroup* rg = seg_rg[si];
            lf.gfwd = rg->d_rows; lf.g_full_words = 0xFFFFFFFFu; lf.g_tail_word = 0u;
            lf.g_stride_bits = rg->stride_bits; lf.g_bit_off = rg->bit_off[(size_t)rg->find(fn.column, 0)];
          }
          if (!c.fwd_staged) r->in_place_columns++;
          any_cand_leaf = true;
          return PB_MAX_SCAN_SLOTS;      // not a slot index (>= 0 = success)
        }
        for (int k = 0; k < n_scan; k++) if (slot_of_col[k] == fn.column) return k;
        if (n_scan >= PB_MAX_SCAN_SLOTS) return -1;
        slot_of_col[n_scan] = fn.column;
        DevScanCol& sc = ds.scan[n_scan];
        sc.base = c.d_fwd; sc.bits_per_doc = c.has_dict ? c.bits : 8 * c.raw_width; sc.bytes_total = c.d_fwd_bytes;
        slot_bits_max[n_scan] = std::max(slot_bits_max[n_scan], sc.bits_per_doc);
        return n_scan++;
      };
      switch (fn.kind) {
        case PB_F_MATCH_ALL: lf.kind = L_TRUE; break;
        case PB_F_EMPTY: lf.kind = L_FALSE; break;
        case PB_F_SCAN_DICT_RANGE: {
          const Column& c = s->cols[fn.column];
          int64_t lo = std::max<int64_t>(fn.lo, 0), hi = std::min<int64_t>(fn.hi, c.card);
          if (hi <= lo) { lf.kind = L_FALSE; break; }
          // the whole dictionary: no scan (and span == 2^bits would overflow the top-aligned compare of PredRange::test<W>)
          if (lo == 0 && hi >= c.card) { lf.kind = L_TRUE; break; }
          lf.kind = L_DICT_RANGE; lf.bits = c.bits; lf.lo = (uint32_t)lo; lf.span = (uint32_t)(hi - lo);
          lf.est_permille = (int32_t)(1000.0 * (double)(hi - lo) / (double)c.card);
          if (residual_field >= 0) make_residual(c, nullptr);
          else if ((lf.slot = scan_slot(c)) < 0) return fail(PB_ERR_UNSUPPORTED, "more than %d scanned columns", PB_MAX_SCAN_SLOTS);
          r->seg_scan_leaves[si]++;
          break;
        }
        case PB_F_SCAN_DICT_SET: {
          const Column& c = s->cols[fn.column];
          if (fn.num_ids <= 0) { lf.kind = fn.exclusive ? L_TRUE : L_FALSE; break; }
          size_t words = ((size_t)c.card + 31) / 32;
          uint32_t* hbits = nullptr;
          const uint32_t* dbits = ar.put<uint32_t>(nullptr, words, &hbits);
          if (!dbits) return fail(PB_ERR_STATE, "query arena overflow");
          for (int k = 0; k < fn.num_ids; k++) {
            int32_t id = fn.ids[k];
            if (id < 0 || id >= c.card) return fail(PB_ERR_INVALID, "filter node %d: dictId %d out of range", n, id);
            hbits[id >> 5] |= 1u << (id & 31);
          }
          lf.kind = L_DICT_SET; lf.bits = c.bits; lf.exclusive = fn.exclusive ? 1 : 0;
          lf.set_bits = dbits; lf.set_card = c.card;
          { double f = (double)fn.num_ids / (double)c.card; lf.est_permille = (int32_t)(1000.0 * (fn.exclusive ? 1.0 - f : f)); }
          if (residual_field >= 0) make_residual(c, dbits);
          else {
            if (!force_gather && set_smem_used + c.card <= PB_SET_SMEM_BYTES) { lf.set_smem_off = set_smem_used; set_smem_used += (c.card + 15) & ~15; }
            if ((lf.slot = scan_slot(c)) < 0) return fail(PB_ERR_UNSUPPORTED, "more than %d scanned columns", PB_MAX_SCAN_SLOTS);
          }
          r->seg_scan_leaves[si]++;
          break;
        }
        case PB_F_SCAN_RAW_RANGE: {
          const Column& c = s->cols[fn.column];
          lf.raw_width = c.raw_width; lf.data_type = c.type;
          if (c.type == PB_INT || c.type == PB_LONG) { lf.kind = L_RAW_RANGE_I; lf.ilo = fn.lo; lf.ihi = fn.hi; }
          else { lf.kind = L_RAW_RANGE_F; lf.dlo = fn.dlo; lf.dhi = fn.dhi; lf.dlo_incl = fn.dlo_inclusive; lf.dhi_incl = fn.dhi_inclusive; }
          if ((lf.slot = scan_slot(c)) < 0) return fail(PB_ERR_UNSUPPORTED, "more than %d scanned columns", PB_MAX_SCAN_SLOTS);
          r->seg_scan_leaves[si]++;
          break;
        }
        case PB_F_SCAN_RAW_SET: {
          const Column& c = s->cols[fn.column];
          if (fn.num_raw_values <= 0) { lf.kind = fn.exclusive ? L_TRUE : L_FALSE; break; }
          lf.kind = L_RAW_SET; lf.raw_width = c.raw_width; lf.data_type = c.type; lf.exclusive = fn.exclusive ? 1 : 0;
          lf.raw_set = ar.put<int64_t>(fn.raw_values, (size_t)fn.num_raw_values);
          lf.n_raw_set = fn.num_raw_values;
          if (!lf.raw_set) return fail(PB_ERR_STATE, "query arena overflow");
          if ((lf.slot = scan_slot(c)) < 0) return fail(PB_ERR_UNSUPPORTED, "more than %d scanned columns", PB_MAX_SCAN_SLOTS);
          r->seg_scan_leaves[si]++;
          break;
        }
        case PB_F_INVERTED: case PB_F_SORTED: case PB_F_BITMAP: {
          size_t words = (((size_t)s->num_docs + 2047) / 2048) * 64;
          uint32_t* bm = d_bitmaps + bm_off; bm_off += words;
          lf.kind = L_BITMAP; lf.bitmap = bm; lf.exclusive = fn.exclusive ? 1 : 0;
          if (fn.kind == PB_F_INVERTED) {
            const Column& c = s->cols[fn.column];
            if (fn.num_ids <= 0) { lf.kind = fn.exclusive ? L_TRUE : L_FALSE; break; }
            for (int k = 0; k < fn.num_ids; k++) if (fn.ids[k] < 0 || fn.ids[k] >= c.card) return fail(PB_ERR_INVALID, "filter node %d: dictId out of range", n);
            const int32_t* dids = ar.put<int32_t>(fn.ids, (size_t)fn.num_ids);
            if (!dids) return fail(PB_ERR_STATE, "query arena overflow");
            expands.push_back({0, c.d_inv, c.card, dids, fn.num_ids, bm, (uint32_t)s->num_docs, std::vector<int32_t>(fn.ids, fn.ids + fn.num_ids)});
          } else if (fn.kind == PB_F_SORTED) {
            lf.exclusive = 0;
            if (fn.num_ids <= 0) { lf.kind = L_FALSE; break; }
            for (int k = 0; k < fn.num_ids; k++) {
              int32_t lo = fn.ids[2 * k], hi = fn.ids[2 * k + 1];
              if (lo < 0 || hi < lo || hi >= s->num_docs) return fail(PB_ERR_INVALID, "filter node %d: bad docId range [%d,%d]", n, lo, hi);
            }
            const int32_t* dp = ar.put<int32_t>(fn.ids, 2 * (size_t)fn.num_ids);
            if (!dp) return fail(PB_ERR_STATE, "query arena overflow");
            expands.push_back({1, nullptr, 0, dp, fn.num_ids, bm, (uint32_t)s->num_docs, {}});
          } else {
            // wrap the caller's Roaring blob as a one-entry inverted index: [BE off0][BE off1][blob]
            // (no blob: the null-value vector staged with the node's column -- IS NULL / IS NOT NULL, FilterPlanNode.java:294-307)
            const uint8_t* blob = (const uint8_t*)fn.blob; uint64_t blob_len = fn.blob_len;
            if (!blob && fn.column >= 0 && fn.column < (int)s->cols.size()) { blob = s->cols[(size_t)fn.column].h_null; blob_len = s->cols[(size_t)fn.column].h_null_len; }
            if (!blob || blob_len < 8) return fail(PB_ERR_INVALID, "filter node %d: bitmap blob missing (and column %d has no null-value vector)", n, fn.column);
            std::vector<uint8_t> tmp(8 + blob_len);
            uint32_t o0 = 8, o1 = (uint32_t)(8 + blob_len);
            tmp[0] = o0 >> 24; tmp[1] = o0 >> 16; tmp[2] = o0 >> 8; tmp[3] = (uint8_t)o0;
            tmp[4] = o1 >> 24; tmp[5] = o1 >> 16; tmp[6] = o1 >> 8; tmp[7] = (uint8_t)o1;
            memcpy(tmp.data() + 8, blob, blob_len);
            const uint8_t* dblob = ar.put<uint8_t>(tmp.data(), tmp.size());
            static const int32_t zero_id = 0;
            const int32_t* dids = ar.put<int32_t>(&zero_id, 1);
            if (!dblob || !dids) return fail(PB_ERR_STATE, "query arena overflow");
            expands.push_back({0, dblob, 1, dids, 1, bm, (uint32_t)s->num_docs, std::vector<int32_t>(1, 0)});
          }
          break;
        }
        default: return fail(PB_ERR_INVALID, "filter node %d: unknown kind %d", n, fn.kind);
      }
      if (lf.gather) lf.slot = -1;
    }
    return PB_OK;
    };
    ds.n_nodes = sq.num_filter_nodes;
    {
      int nl = 0;
      if ((rc = build_program(sq.filter, sq.num_filter_nodes, ds.node_kind, ds.node_arg, ds.leaves, PB_MAX_LEAVES, nl, false))) return rc;
      if (!residual[si].empty()) {
        // the program is a flat AND (candidate leaves exist only there) whose leaf i is node i: keep the other leaves, which
        // include the streamed one, under an AND of their number
        int kept = 0;
        for (int n = 0; n + 1 < sq.num_filter_nodes; n++) {
          if (residual_node[n]) continue;
          ds.leaves[kept] = ds.leaves[ds.node_arg[n]];
          ds.node_kind[kept] = N_LEAF; ds.node_arg[kept] = (int8_t)kept;
          kept++;
        }
        ds.node_kind[kept] = N_AND; ds.node_arg[kept] = (int8_t)kept;
        ds.n_nodes = kept + 1;
        for (int l = kept; l < nl; l++) memset(&ds.leaves[l], 0, sizeof(DevLeaf));
        r->residual_leaves += (int)residual[si].size();
      }
    }
    // FILTER(WHERE ...) clauses
    ds.n_agg_filters = nF;
    {
      int nl = 0, nn = 0;
      for (int f = 0; f < nF; f++) {
        ds.af_begin[f] = nn;
        if (nn + sq.agg_filter_nodes[f] > PB_MAX_AF_NODES) return fail(PB_ERR_UNSUPPORTED, "FILTER clauses have more than %d nodes", PB_MAX_AF_NODES);
        if ((rc = build_program(sq.agg_filters[f], sq.agg_filter_nodes[f], ds.af_node_kind + nn, ds.af_node_arg + nn, ds.af_leaves, PB_MAX_AF_LEAVES, nl, true))) return rc;
        nn += sq.agg_filter_nodes[f];
      }
      for (int f = nF; f <= PB_MAX_AGG_FILTERS; f++) ds.af_begin[f] = nn;
      ds.af_docs = d_seg_stats ? d_seg_stats + (size_t)si * (1 + PB_MAX_AGG_FILTERS) : nullptr;
    }
    ds.n_scan = n_scan;
    set_cache_max = std::max(set_cache_max, set_smem_used);
    n_slots_max = std::max(n_slots_max, n_scan);
    r->n_scan_leaves_total += (int)r->seg_scan_leaves[si];

    // group-by / aggregation columns
    const TableMeta& tm = r->tables[ds.table];
    uint64_t mult = 1;
    for (int j = 0; j < nG; j++) {
      const Column& c = s->cols[gcol[si][j]];
      DevKeyCol& kc = ds.keys[j];
      kc.fwd = c.fwd_staged ? c.d_fwd : c.d_fwd_host; kc.n_full_words = c.fwd_staged ? 0xFFFFFFFFu : c.host_full_words;
      kc.tail_word = c.fwd_staged ? 0u : c.host_tail_word; if (!c.fwd_staged) r->in_place_columns++;
      kc.bits = c.bits; kc.raw_width = c.has_dict ? 0 : c.raw_width; kc.data_type = c.type;
      kc.stride_bits = c.has_dict ? c.bits : 8 * c.raw_width; kc.bit_off = 0;
      if (c.has_dict && seg_rg[si] && seg_rg[si]->find(gcol[si][j], 0) >= 0) {
        const RowGroup* rg = seg_rg[si];
        kc.fwd = rg->d_rows; kc.n_full_words = 0xFFFFFFFFu; kc.tail_word = 0u;
        kc.stride_bits = rg->stride_bits; kc.bit_off = rg->bit_off[(size_t)rg->find(gcol[si][j], 0)];
      }
      kc.remap = (combine && gdict[j]) ? gdict[j]->d_remap[si] : nullptr;
      kc.shift = tm.shifts[j];
      kc.mult = mult;
      if (tm.cards[j] > 0) mult *= (uint64_t)tm.cards[j];
      if (!c.has_dict && (c.type == PB_FLOAT) && nG > 1) return fail(PB_ERR_UNSUPPORTED, "raw FLOAT key in a multi-column group-by");
    }
    for (int a = 0; a < nA; a++) {
      if (acol[si][a] < 0) continue;
      const Column& c = s->cols[acol[si][a]];
      DevAggCol& ac = ds.aggs[a];
      ac.fwd = c.fwd_staged ? c.d_fwd : c.d_fwd_host; ac.n_full_words = c.fwd_staged ? 0xFFFFFFFFu : c.host_full_words;
      ac.tail_word = c.fwd_staged ? 0u : c.host_tail_word; if (!c.fwd_staged) r->in_place_columns++;
      ac.dict_f64 = c.d_dict_f64; ac.bits = c.bits; ac.raw_width = c.has_dict ? 0 : c.raw_width; ac.data_type = c.type;
      ac.stride_bits = c.has_dict ? c.bits : 8 * c.raw_width; ac.bit_off = 0;
      if (c.has_dict && seg_rg[si]) {
        const RowGroup* rg = seg_rg[si];
        const int fv = q->aggregations[a].op != PB_AGG_DISTINCTCOUNT ? rg->find(acol[si][a], 1) : -1, fi = rg->find(acol[si][a], 0);
        if (fv >= 0) {            // decoded value field: read like a raw column, no dictionary lookup
          ac.fwd = rg->d_rows; ac.n_full_words = 0xFFFFFFFFu; ac.tail_word = 0u;
          ac.raw_width = c.entry_bytes; ac.stride_bits = rg->stride_bits; ac.bit_off = rg->bit_off[(size_t)fv];
        } else if (fi >= 0) {
          ac.fwd = rg->d_rows; ac.n_full_words = 0xFFFFFFFFu; ac.tail_word = 0u;
          ac.stride_bits = rg->stride_bits; ac.bit_off = rg->bit_off[(size_t)fi];
        }
      }
      ac.remap = (combine && adict[a]) ? adict[a]->d_remap[si] : nullptr;
    }
  }

  // ---- the rows kernel's per-segment descriptors ----
  const DevRowSeg* d_row_segs = nullptr;
  if (rows_ok) {
    {
      DevRowSeg* h_rs = nullptr;
      d_row_segs = ar.put<DevRowSeg>(nullptr, (size_t)n_segs, &h_rs);
      if (!d_row_segs) return fail(PB_ERR_STATE, "query arena overflow");
      for (int si = 0; si < n_segs; si++) {
        const RowGroup* rg = seg_rg[si];
        const pb_segment_s* sg = g->segs[si];
        DevRowSeg& rs = h_rs[si];
        rs.rows = reinterpret_cast<const uint32_t*>(rg->d_rows);
        rs.table = hsegs[si].table;
        for (int j = 0; j < nG; j++) {
          const DevKeyCol& kc = hsegs[si].keys[j];
          rs.keys[j].off = (uint32_t)rg->bit_off[(size_t)rg->find(gcol[si][j], 0)];
          rs.keys[j].bits = (uint32_t)sg->cols[gcol[si][j]].bits;
          rs.keys[j].mult = kc.mult; rs.keys[j].remap = kc.remap;
        }
        for (int a = 0; a < nA; a++) {
          if (q->aggregations[a].op == PB_AGG_COUNT) continue;
          const Column& c = sg->cols[acol[si][a]];
          rs.aggs[a].off = (uint32_t)rg->bit_off[(size_t)rg->find(acol[si][a], 1)];
          rs.aggs[a].width = (uint32_t)c.entry_bytes; rs.aggs[a].type = (uint32_t)c.type; rs.aggs[a].exact_int = 0;
        }
        rs.n_leaves = (int32_t)residual[si].size();
        for (int k = 0; k < rs.n_leaves; k++) rs.leaves[k] = residual[si][(size_t)k];
      }
      // SUM / AVG over INT / LONG columns: when max|value| x docs < 2^53 every partial sum is an integer a double holds
      // exactly, so the CTA-private table may accumulate them as 64-bit integers with two native 32-bit shared-memory
      // atomics instead of a compare-and-swap loop on a double -- bit-identical to the reference's double accumulation,
      // whatever the order (DevRowAgg::exact_int)
      static const bool exact_on = []() { const char* e = getenv("PB_AGG_EXACT_INT"); return !e || atoi(e) != 0; }();
      uint64_t docs_all = 0;
      for (int si = 0; si < n_segs; si++) docs_all += (uint64_t)g->segs[si]->num_docs;
      for (int a = 0; a < nA && exact_on; a++) {
        const int op = q->aggregations[a].op;
        if (op != PB_AGG_SUM && op != PB_AGG_AVG) continue;
        bool exact = true;
        for (int si = 0; si < n_segs && exact; si++) {
          const Column& c = g->segs[si]->cols[acol[si][a]];
          if (!c.has_dict || c.card <= 0 || (c.type != PB_INT && c.type != PB_LONG) || c.h_dict.size() < (size_t)c.card * (size_t)c.entry_bytes) { exact = false; break; }
          // sorted dictionary: the extremes are its first and last entries
          const uint8_t* lo = c.h_dict.data(); const uint8_t* hi = c.h_dict.data() + (size_t)(c.card - 1) * (size_t)c.entry_bytes;
          const int64_t vlo = c.type == PB_INT ? (int64_t)(int32_t)be32(lo) : (int64_t)be64(lo);
          const int64_t vhi = c.type == PB_INT ? (int64_t)(int32_t)be32(hi) : (int64_t)be64(hi);
          const uint64_t alo = vlo < 0 ? (uint64_t)0 - (uint64_t)vlo : (uint64_t)vlo, ahi = vhi < 0 ? (uint64_t)0 - (uint64_t)vhi : (uint64_t)vhi;
          const uint64_t bound = std::max<uint64_t>(std::max(alo, ahi), 1);
          if (bound >= (1ull << 53) || docs_all >= (1ull << 53) / bound) exact = false;
        }
        if (exact) for (int si = 0; si < n_segs; si++) h_rs[si].aggs[a].exact_int = 1;
      }
    }
  }

  // ---- work-unit geometry: one stage = one unit (U x 1024 docs) of every scan slot, per warp ----
  int sum_bits = 0;
  for (int k = 0; k < n_slots_max; k++) sum_bits += slot_bits_max[k];
  static const int unit_env = []() { const char* e = getenv("PB_UNIT"); return e ? atoi(e) : 2; }();
  auto stage_bytes_for = [&](int U, int32_t* offs) {
    size_t b = 0;
    for (int k = 0; k < n_slots_max; k++) {
      if (offs) offs[k] = (int32_t)b;
      b += (((size_t)U * PB_CHUNK_DOCS * slot_bits_max[k] / 8 + 16) + 15) & ~(size_t)15;
    }
    return b;
  };
  // two chunks per unit halve the per-unit overhead (dispatch, TMA issue, list append) when two CTAs still fit an SM
  int U = (unit_env == 1) ? 1 : 2;
  if (U == 2 && stage_bytes_for(2, nullptr) * PB_NSTAGE * PB_NWARPS > 100 * 1024) U = 1;
  int32_t slot_offs[PB_MAX_SCAN_SLOTS] = {0};
  size_t stage_bytes = stage_bytes_for(U, slot_offs);
  if (stage_bytes * PB_NSTAGE * PB_NWARPS > 200 * 1024)
    return fail(PB_ERR_UNSUPPORTED, "scan predicates touch %d bits per row: unit stages do not fit shared memory", sum_bits);
  const uint64_t unit_docs = (uint64_t)U * PB_CHUNK_DOCS;
  uint64_t n_chunks = 0, n_docs_total = 0;
  bool match_all = true;
  for (int si = 0; si < n_segs; si++) {
    hsegs[si].unit_begin = n_chunks;
    hsegs[si].n_units = ((uint64_t)g->segs[si]->num_docs + unit_docs - 1) / unit_docs;
    hsegs[si].doc_base = n_docs_total;
    n_chunks += hsegs[si].n_units;
    n_docs_total += (uint64_t)g->segs[si]->num_docs;
    if (sqs[si].num_filter_nodes != 0) match_all = false;
  }
  if (d_row_segs) {
    DevRowSeg* h_rs = reinterpret_cast<DevRowSeg*>(ar.host.data() + (reinterpret_cast<const uint8_t*>(d_row_segs) - ar.dev));
    for (int si = 0; si < n_segs; si++) h_rs[si].doc_base = hsegs[si].doc_base;
  }
  if (n_docs_total >= (1ull << 32)) return fail(PB_ERR_UNSUPPORTED, "%llu docs in one call (match list is 32-bit): split the segment group", (unsigned long long)n_docs_total);
  // ---- how the matches reach the group table (see pb_device.cuh):
  //   smem      one dense table that fits shared memory and enough matches to amortise merging 148 private copies
  //   global    everything else: pb_agg_kernel, one thread per match, reductions straight into the global table
  // (a third way -- the filter kernel aggregating its own matches, no match list -- was measured and removed: the two
  //  kernels are bound by the same memory system and did not overlap, profiles/r2_experiments.md)
  const bool fuse = false;
  int n_acc = 0, n_fc = 0;
  for (int a = 0; a < nA; a++) {
    const int op = q->aggregations[a].op;
    if (op >= PB_AGG_SUM && op <= PB_AGG_AVG) n_acc++;
    if (nF > 0 && q->agg_filter_of[a] >= 0 && (op == PB_AGG_COUNT || op == PB_AGG_AVG || count_all)) n_fc++;
  }
  static const int smem_table_env = []() { const char* e = getenv("PB_AGG_SMEM"); return e ? atoi(e) : 1; }();
  static const size_t smem_table_budget = 200 * 1024;
  size_t st_rep_bytes = 0; int st_replicas = 0;
  if (smem_table_env && !fuse && !track_first && table_mode == T_DENSE && n_tables == 1 && r->tables[0].capacity <= (1u << 20)) {
    st_rep_bytes = pb_smem_table_bytes((uint32_t)r->tables[0].capacity, n_fc, n_acc);
    if (st_rep_bytes <= smem_table_budget) { st_replicas = 1; while (st_replicas < 32 && (size_t)(2 * st_replicas) * st_rep_bytes <= smem_table_budget) st_replicas *= 2; }
  }
  const bool use_smem_table = st_replicas > 0;
  uint32_t* d_match_list = nullptr;
  if (!match_all && !fuse && n_docs_total > 0) {
    r->scratch = scratch_alloc(ctx, 4 * (size_t)n_docs_total + 256, &r->scratch_cap);
    if (!r->scratch) return fail(PB_ERR_OOM, "match list allocation (%zu bytes) failed", 4 * (size_t)n_docs_total + 256);
    d_match_list = (uint32_t*)r->scratch;
  }
  r->match_all = match_all;
  r->n_agg_filters = nF; r->count_all = count_all;
  // ---- counter cells that the host knows up front (ExecutionStatistics; see PB_COUNTERS_PER_TABLE) ----
  unsigned long long* h_head = nullptr;
  const unsigned long long* d_head = ar.put<unsigned long long>(nullptr, (size_t)PB_COUNTERS_PER_TABLE * n_tables, &h_head);
  if (!d_head) return fail(PB_ERR_STATE, "query arena overflow");
  for (int si = 0; si < n_segs; si++) {
    unsigned long long* c = h_head + (size_t)hsegs[si].table * PB_COUNTERS_PER_TABLE;
    const unsigned long long nd = (unsigned long long)g->segs[si]->num_docs;
    if (match_all) c[2] += nd;                                   // numDocsScanned of a match-all query (no filter kernel)
    c[6] += nd;                                                  // numTotalDocs
    c[7] += (unsigned long long)r->seg_scan_leaves[si] * nd;     // every scan leaf reads every doc of the segment on the device
    c[8] += 1;
  }
  {
    // what must agree across ranks for the blocks to be mergeable element by element
    unsigned long long fp = 0xcbf29ce484222325ull;
    auto mix = [&](unsigned long long v) { fp ^= v; fp *= 0x100000001b3ull; fp ^= fp >> 29; };
    mix((unsigned long long)r->block_bytes); mix((unsigned long long)r->block_sum_off); mix((unsigned long long)r->block_dc_off); mix((unsigned long long)r->block_mm_off);
    mix((unsigned long long)table_mode); mix((unsigned long long)nG); mix((unsigned long long)nA); mix((unsigned long long)nF);
    for (int a = 0; a < nA; a++) mix((unsigned long long)q->aggregations[a].op * 131 + dc_words[a]);
    for (auto& tm : r->tables) { mix(tm.capacity); for (auto cd : tm.cards) mix((unsigned long long)cd); }
    r->fingerprint = fp >> 8;                               // head room: n_ranks x fp must not wrap
    for (int t = 0; t < n_tables; t++) h_head[(size_t)t * PB_COUNTERS_PER_TABLE + 9] = r->fingerprint;
  }
  // ---- filtered aggregations: which swim-lanes exist per segment, and how many columns each projects
  // (AggregationFunctionUtils.buildFilteredAggregationInfos :312-400; statistics are summed lane by lane,
  // FilteredGroupByOperator.java:146-149): one lane per FILTER clause over (main AND clause) -- unless the clause matches all
  // under a real main filter, then its functions join the non-filtered lane -- plus the non-filtered lane when it has
  // functions or the query groups; an empty main filter is a single lane without docs ----
  const DevLaneWeights* d_lane_w = nullptr;
  if (nF > 0) {
    r->agg_filter_of.assign(q->agg_filter_of, q->agg_filter_of + nA);
    auto classify = [](const pb_filter_node* nodes, int n) { return n == 0 ? 1 : (n == 1 && nodes[0].kind == PB_F_MATCH_ALL ? 1 : (n == 1 && nodes[0].kind == PB_F_EMPTY ? 2 : 0)); };
    auto lane_cols = [&](const std::vector<char>& in_lane) {
      std::vector<std::string> cols;
      for (auto& nme : r->gb_names) if (std::find(cols.begin(), cols.end(), nme) == cols.end()) cols.push_back(nme);
      for (int a = 0; a < nA; a++) if (in_lane[a] && !r->agg_cols[a].empty() && std::find(cols.begin(), cols.end(), r->agg_cols[a]) == cols.end()) cols.push_back(r->agg_cols[a]);
      return (int32_t)cols.size();
    };
    DevLaneWeights* h_lw = nullptr;
    d_lane_w = ar.put<DevLaneWeights>(nullptr, (size_t)n_segs, &h_lw);
    if (!d_lane_w) return fail(PB_ERR_STATE, "query arena overflow");
    for (int si = 0; si < n_segs; si++) {
      DevLaneWeights& lw = h_lw[si];
      lw.table = hsegs[si].table;
      const int main_kind = classify(sqs[si].filter, sqs[si].num_filter_nodes);
      if (main_kind == 2) continue;                        // empty main filter: no docs in any lane
      std::vector<char> in_main(nA, 0);
      bool any_main = false;
      for (int f = 0; f < nF; f++) {
        std::vector<char> in_lane(nA, 0);
        for (int a = 0; a < nA; a++) if (q->agg_filter_of[a] == f) in_lane[a] = 1;
        if (main_kind != 1 && classify(sqs[si].agg_filters[f], sqs[si].agg_filter_nodes[f]) == 1) {
          for (int a = 0; a < nA; a++) if (in_lane[a]) { in_main[a] = 1; any_main = true; }
          continue;
        }
        lw.docs_w[1 + f] = 1; lw.post_w[1 + f] = lane_cols(in_lane);
      }
      for (int a = 0; a < nA; a++) if (q->agg_filter_of[a] < 0) { in_main[a] = 1; any_main = true; }
      if (any_main || nG > 0) { lw.docs_w[0] = 1; lw.post_w[0] = lane_cols(in_main); }
    }
  }

  hq->n_segs = n_segs; hq->n_group_by = nG; hq->n_aggs = nA; hq->table_mode = table_mode;
  for (int a = 0; a < nA; a++) hq->agg_op[a] = q->aggregations[a].op;
  for (int a = 0; a < PB_MAX_AGGS; a++) hq->agg_filter_of[a] = (nF > 0 && a < nA) ? q->agg_filter_of[a] : -1;
  hq->n_agg_filters = nF;
  for (int k = 0; k < n_slots_max; k++) hq->slot_off[k] = slot_offs[k];
  hq->stage_bytes = (int32_t)stage_bytes;
  hq->set_cache_bytes = set_cache_max;
  hq->out_cap = PB_OUT_CAP; hq->cand_cap = PB_CAND_CAP;
  hq->cand_bytes = any_cand_leaf ? (int32_t)(2 * PB_CAND_CAP * PB_NWARPS) : 0;   // u16 offsets inside the unit, one list per warp
  hq->use_tma = (q->flags & PB_Q_NO_TMA) ? 0 : 1;
  hq->generic = (q->flags & PB_Q_GENERIC_KERNEL) ? 1 : 0;
  hq->n_units = n_chunks; hq->segs = dsegs; hq->tables = dtabs;
  hq->n_docs_total = n_docs_total; hq->match_all = match_all ? 1 : 0;
  hq->agg_counts_docs = r->residual_leaves > 0 ? 1 : 0;
  { static const int sm = []() { const char* e = getenv("PB_SPARSE_MAX"); return e ? atoi(e) : PB_SPARSE_MAX; }(); hq->sparse_max = sm; }
  hq->match_list = d_match_list;
  if (use_smem_table) {
    hq->st_slots = (int32_t)r->tables[0].capacity; hq->st_replicas = st_replicas;
    // merging a CTA's private table costs up to one RED per slot and aggregate: it pays once a CTA sees several matches per slot
    static const long long min_env = []() { const char* e = getenv("PB_AGG_SMEM_MIN"); return e ? atoll(e) : -1ll; }();
    hq->st_min_docs = min_env >= 0 ? (uint64_t)min_env : 4ull * (uint64_t)ctx->num_sms * r->tables[0].capacity;
  }
  r->fused = fuse; r->smem_table = use_smem_table;
  hq->match_count = reinterpret_cast<unsigned long long*>(d_aux);   // PB_MAX_WAVES zeroed cells (aux region)
  hq->any_limit = reinterpret_cast<const unsigned int*>(d_aux + any_limit_off);
  r->repair_pass = false;
  if (table_mode == T_HASH) for (auto& tm : r->tables) if (tm.dev.limit_active) r->repair_pass = true;

  // expand items (one per inverted-index bitmap / per sorted-index range list)
  int n_expand_items = 0;
  for (auto& e : expands) n_expand_items += e.kind == 0 ? e.n_ids : 1;
  const DevExpandItem* d_expand_items = nullptr;
  if (n_expand_items > 0) {
    std::vector<DevExpandItem> items;
    items.reserve((size_t)n_expand_items);
    for (auto& e : expands) {
      if (e.kind == 0) {
        for (int k = 0; k < e.n_ids; k++) {
          DevExpandItem it; memset(&it, 0, sizeof it);
          it.inv = e.inv; it.out = e.out; it.kind = 0; it.card = e.card; it.id = e.host_ids[k]; it.num_docs = e.num_docs;
          items.push_back(it);
        }
      } else {
        DevExpandItem it; memset(&it, 0, sizeof it);
        it.pairs = e.ids; it.out = e.out; it.kind = 1; it.n_pairs = e.n_ids; it.num_docs = e.num_docs;
        items.push_back(it);
      }
    }
    d_expand_items = ar.put<DevExpandItem>(items.data(), items.size());
    if (!d_expand_items) return fail(PB_ERR_STATE, "query arena overflow");
  }
  // ---- waves: when some segments are still being copied to HBM, launch per run of segments so that the kernels of
  // one wave (and its in-place gathers over PCIe) overlap the staging copies of the next ----
  struct Wave { int seg_lo, seg_hi; DevQuery dq; uint64_t n_units, n_docs; };   // the descriptor travels as a __grid_constant__ kernel parameter
  std::vector<Wave> waves;
  if (n_pending > 0 && !match_all && n_expand_items == 0 && n_segs > 1 && n_chunks > 0) {
    const int per_wave = (n_segs + PB_MAX_WAVES - 1) / PB_MAX_WAVES;
    for (int lo = 0; lo < n_segs; lo += per_wave) {
      const int hi = std::min(n_segs, lo + per_wave);
      DevQuery w = *hq;
      w.unit_lo = hsegs[lo].unit_begin;
      w.n_units = hsegs[hi - 1].unit_begin + hsegs[hi - 1].n_units - w.unit_lo;
      w.n_docs_total = hsegs[hi - 1].doc_base + (uint64_t)g->segs[hi - 1]->num_docs - hsegs[lo].doc_base;
      w.match_list = d_match_list + hsegs[lo].doc_base;
      w.match_count = hq->match_count + waves.size();
      waves.push_back({lo, hi, w, w.n_units, w.n_docs_total});
    }
  } else {
    for (int si = 0; si < n_segs; si++) if (seg_wait[si]) CU(cudaStreamWaitEvent(st, seg_wait[si], 0));
    waves.push_back({0, n_segs, *hq, n_chunks, n_docs_total});
  }
  r->waves = (int)waves.size();
  CU(cudaMemcpyAsync(ar.dev, ar.host.data(), ar.used, cudaMemcpyHostToDevice, st));
  {
    // table init: all regions are 16-byte multiples (cudaMallocAsync alignment is 256)
    const uint64_t zn = (zero_bytes + 15) / 16, fn = (ff_bytes + 15) / 16, mn = (8 * mm_elems + 15) / 16, an = (aux_bytes + 15) / 16;
    const uint64_t mx = std::max(std::max(zn, an), std::max(fn, mn));
    int grid = (int)std::min<uint64_t>((mx + 255) / 256, (uint64_t)ctx->num_sms * 8);
    if (grid < 1) grid = 1;
    r->init = {(uint4*)d_zero, zn, (uint4*)d_ff, fn, (uint4*)d_mm, mn, (uint4*)d_aux, an, reinterpret_cast<const uint4*>(d_head),
               (uint64_t)PB_COUNTERS_PER_TABLE * n_tables / 2, grid};
    r->key_words = key_words;
  }
  lap(2);

  // ---- launch geometry of the two hot kernels ----
  {
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->smem_attr_set) {
      CU(cudaFuncSetAttribute(pb_filter_kernel<1, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      CU(cudaFuncSetAttribute(pb_filter_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      CU(cudaFuncSetAttribute(pb_filter_kernel<2, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      CU(cudaFuncSetAttribute(pb_agg_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
      CU(cudaFuncSetAttribute(pb_agg_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
      CU(cudaFuncSetAttribute(pb_agg_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 16 * 1024));
      CU(cudaFuncSetAttribute(pb_agg_rows_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 32 * 1024));
      CU(cudaFuncSetAttribute(pb_agg_rows_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 32 * 1024));
      CU(cudaFuncSetAttribute(pb_agg_rows_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 32 * 1024));
      ctx->smem_attr_set = true;
    }
  }
  auto filter_smem = [&](int out_cap, int cand_cap) {
    return ((sizeof(FilterSmemHeader) + 127) & ~(size_t)127) + (((size_t)set_cache_max + 127) & ~(size_t)127) + (any_cand_leaf ? (size_t)2 * cand_cap * PB_NWARPS : 0) +
           (size_t)PB_NWARPS * out_cap * 4 + stage_bytes * PB_NSTAGE * PB_NWARPS;
  };
  size_t smem = 0;
  uint64_t max_ctas = 0;
  bool u2_three = false;
  if (!match_all && n_chunks > 0) {
    smem = filter_smem(PB_OUT_CAP, PB_CAND_CAP);
    if (smem > 227 * 1024) return fail(PB_ERR_UNSUPPORTED, "filter kernel needs %zu bytes of shared memory", smem);
    int occ = 1;
    // U = 2 comes in two register budgets: 3 CTAs/SM (80 registers) when three stages sets fit shared memory, else 2 CTAs/SM
    u2_three = U == 2 && 3 * (smem + 1024) <= 227 * 1024;
    if (U == 1) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pb_filter_kernel<1, 3>, PB_NTHREADS, smem));
    else if (u2_three) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pb_filter_kernel<2, 3>, PB_NTHREADS, smem));
    else CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pb_filter_kernel<2, 2>, PB_NTHREADS, smem));
    if (occ < 1) return fail(PB_ERR_CUDA, "filter kernel does not fit an SM (smem %zu)", smem);
    max_ctas = (uint64_t)ctx->num_sms * (uint64_t)occ;
  }
  // ---- plan-time specialisation: every segment of the launch is "one streamed dictionary leaf of the same width and
  // predicate kind + candidate leaves" -> the small kernel compiled for exactly that (pb_filter_spec.cu) ----
  int spec_w = 0, spec_pk = 0;
  {
    static const bool spec_on = []() { const char* e = getenv("PB_FILTER_SPEC"); return !e || atoi(e) != 0; }();
    if (spec_on && !match_all && n_chunks > 0 && U == 2 && u2_three && !hq->generic && hq->use_tma) {
      int w = -1, pk = -1;
      bool ok = true;
      for (int si = 0; si < n_segs && ok; si++) {
        const DevSegQuery& ds = hsegs[si];
        int nl = 0, dense = -1, n_dense = 0;
        for (int n = 0; n < ds.n_nodes && ok; n++) {
          if (ds.node_kind[n] == N_LEAF) {
            const DevLeaf& lf = ds.leaves[ds.node_arg[n]];
            if (!lf.gather) { dense = ds.node_arg[n]; n_dense++; }
            nl++;
          } else if (!(ds.node_kind[n] == N_AND && n == ds.n_nodes - 1 && ds.node_arg[n] == nl)) ok = false;
        }
        if (!ok || n_dense != 1) { ok = false; break; }
        const DevLeaf& lf = ds.leaves[dense];
        const int k = lf.kind == L_DICT_RANGE ? 0 : (lf.kind == L_DICT_SET && lf.set_smem_off >= 0) ? 1 : -1;
        if (k < 0 || (w >= 0 && (w != lf.bits || pk != k))) { ok = false; break; }
        w = lf.bits; pk = k;
      }
      if (ok && w > 0 && pb_filter_spec_available(w, pk)) {
        // the specialised kernel needs 64 registers: a fourth CTA fits an SM when its shared memory does -- halve the
        // per-warp output buffer and candidate list for that (more flushes / candidate passes, both cheap)
        size_t smem_spec = smem;
        int oc = PB_OUT_CAP, cc = PB_CAND_CAP;
        if (4 * (filter_smem(PB_OUT_CAP / 2, PB_CAND_CAP / 2) + 1024) <= 227 * 1024 && 4 * (smem + 1024) > 227 * 1024) { oc /= 2; cc /= 2; smem_spec = filter_smem(oc, cc); }
        int occ = 0;
        if (pb_filter_spec_prepare(w, pk, smem_spec, &occ) == cudaSuccess && occ >= 1) {
          spec_w = w; spec_pk = pk; max_ctas = (uint64_t)ctx->num_sms * (uint64_t)occ; smem = smem_spec;
          hq->out_cap = oc; hq->cand_cap = cc; hq->cand_bytes = any_cand_leaf ? (int32_t)(2 * cc * PB_NWARPS) : 0;
          for (auto& wv : waves) { wv.dq.out_cap = oc; wv.dq.cand_cap = cc; wv.dq.cand_bytes = hq->cand_bytes; }
        } else cudaGetLastError();
      }
    }
  }
  const size_t smem2 = table_mode == T_KEYLESS ? (nF > 0 ? 3 : 2) * sizeof(double) * (size_t)nA * PB_NTHREADS : 0;
  // more resident threads = more gathers in flight (the kernel is DRAM-latency bound); 6 CTAs/SM costs a 4-byte spill
  static const int agg_occ = []() { const char* e = getenv("PB_AGG_OCC"); int v = e ? atoi(e) : 6; return v == 4 ? 4 : 6; }();
  uint64_t max2 = 0;
  if (n_docs_total > 0 && !fuse && !use_smem_table) {
    int occ2 = 1;
    if (agg_occ == 4) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, pb_agg_kernel<4>, PB_NTHREADS, smem2));
    else CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, pb_agg_kernel<6>, PB_NTHREADS, smem2));
    if (occ2 < 1) return fail(PB_ERR_CUDA, "aggregation kernel does not fit an SM");
    max2 = (uint64_t)ctx->num_sms * (uint64_t)occ2;
  }
  {
    pb_result_s::Replay& rp = r->rp;
    rp.expand_items = d_expand_items; rp.n_expand = n_expand_items;
    rp.U = U; rp.u2_three = u2_three; rp.smem_filter = smem; rp.spec_w = spec_w; rp.spec_pk = spec_pk;
    rp.agg_kind = (fuse || n_docs_total == 0) ? 0 : d_row_segs ? 4 : use_smem_table ? 3 : agg_occ == 4 ? 2 : 1;
    rp.smem_agg = (use_smem_table && rp.agg_kind >= 3) ? (size_t)st_replicas * st_rep_bytes : rp.agg_kind == 4 ? 0 : smem2;
    rp.row_segs = d_row_segs; rp.rows_rw = rows_rw;
    rp.lane_w = d_lane_w; rp.n_lanes = 1 + nF; rp.n_segs = n_segs;
    rp.flags = q->flags;
    for (const Wave& w : waves) {
      pb_result_s::WaveLaunch wl;
      wl.dq = w.dq; wl.seg_lo = w.seg_lo; wl.seg_hi = w.seg_hi; wl.n_units = w.n_units; wl.n_docs = w.n_docs;
      // every CTA gets a contiguous range of chunks; keep at least one chunk per warp
      wl.grid_filter = (!match_all && w.n_units > 0) ? (int)std::min<uint64_t>(std::max<uint64_t>((w.n_units + PB_NWARPS - 1) / PB_NWARPS, 1), max_ctas) : 0;
      if (rp.agg_kind >= 3) wl.grid_agg = (int)std::min<uint64_t>(std::max<uint64_t>((w.n_docs + PB_AGG_SMEM_THREADS - 1) / PB_AGG_SMEM_THREADS, 1), (uint64_t)ctx->num_sms);
      else if (rp.agg_kind) wl.grid_agg = (int)std::min<uint64_t>(std::max<uint64_t>((w.n_docs + PB_NTHREADS - 1) / PB_NTHREADS, 1), max2);
      if (w.n_docs == 0) wl.grid_agg = 0;
      rp.waves.push_back(wl);
    }
    // a plan can be kept for the next identical query when nothing about it depends on this call's circumstances: all
    // segments resident (no staging waits, no in-place host reads), one wave, tables small enough for single-pass hand-back
    bool small = true;
    for (auto& tm : r->tables) if (tm.capacity + 1 > (1ull << 20)) small = false;
    rp.cacheable = n_pending == 0 && !in_place && waves.size() == 1 && small && !(q->flags & PB_Q_DEFER_FINALIZE) && r->in_place_columns == 0;
  }
  if ((rc = enqueue_all(r, &seg_wait))) return rc;
  lap(3);

  if (q->flags & PB_Q_DEFER_FINALIZE) {
    CU(cudaEventRecord(r->ev3, st));
    *out = R.release();
    return PB_OK;
  }
  if ((q->flags & PB_Q_ALL_RANKS) && (rc = comm_merge(r))) return rc;
  rc = finalize_result(r);
  if (rc) return rc;
  if (try_cache && r->rp.cacheable) plan_register(g, r, std::move(sig));
  *out = R.release();
  return PB_OK;
}

// hash tables across ranks: see comm_merge_hash further down (hash-partitioned all-to-all)

// Install the global dictionary of `column` (sorted union over ALL segments of the parent group) in every per-device child.
static int sync_child_dictionary(pb_group_s* g, const char* column) {
  std::lock_guard<std::mutex> lk(g->mu);
  auto it = g->dicts.find(column);
  if (it == g->dicts.end()) {
    GlobalDict gd;
    int rc = build_union(g, column, gd);
    if (rc) return rc;
    it = g->dicts.emplace(column, std::move(gd)).first;
    g->dict_version++;
  }
  auto ver = g->child_dict_version.find(column);
  if (ver != g->child_dict_version.end() && ver->second == g->dict_version) return PB_OK;
  const GlobalDict& gd = it->second;
  for (auto* c : g->children) {
    int rc = pb_segment_group_set_global_dictionary(c, column, gd.values.data(), gd.n, gd.entry_bytes);
    if (rc) return rc;
  }
  g->child_dict_version[column] = g->dict_version;
  return PB_OK;
}

extern "C" int pb_query_execute(pb_segment_group_handle g, const pb_segment_query* sqs, const pb_query_desc* q, pb_result_handle* out) {
  int rc = ensure_init();
  if (rc) return rc;
  if (!g || !q || !out || !sqs) return fail(PB_ERR_INVALID, "null argument");
  if (g->children.empty()) {
    if (!g->ctx) return fail(PB_ERR_STATE, "the segments of this group were registered while no CUDA device was available");
    DeviceGuard dg(g->ctx);          // SURVEY.md §8b: the calling thread may never have selected this device
    return exec_single(g, sqs, q, out);
  }
  // ---- one process driving several GPUs: every device runs its segments (asynchronously, one stream per device), then the
  // tables are merged on the first device, which reads its peers' blocks in place over NVLink.  Same role as
  // BaseCombineOperator's worker threads + the IndexedTable merge (CTR/operator/combine/BaseCombineOperator.java:97-142). ----
  const int nc = (int)g->children.size();
  const bool combine = (q->flags & PB_Q_COMBINE) != 0;
  if (nc > PB_MERGE_MAX_PEERS) return fail(PB_ERR_UNSUPPORTED, "segment group spans %d devices (max %d)", nc, PB_MERGE_MAX_PEERS);
  if (combine) {
    for (int j = 0; j < q->num_group_by; j++) {
      int ci = find_col(g->segs[0], q->group_by_columns[j]);
      if (ci < 0) return fail(PB_ERR_INVALID, "segment %s: no column %s", g->segs[0]->name.c_str(), q->group_by_columns[j]);
      if (g->segs[0]->cols[ci].has_dict && (rc = sync_child_dictionary(g, q->group_by_columns[j]))) return rc;
    }
    for (int a = 0; a < q->num_aggregations; a++)
      if (q->aggregations[a].op == PB_AGG_DISTINCTCOUNT && q->aggregations[a].column) {
        int ci = find_col(g->segs[0], q->aggregations[a].column);
        if (ci >= 0 && g->segs[0]->cols[ci].has_dict && (rc = sync_child_dictionary(g, q->aggregations[a].column))) return rc;
      }
  }
  std::vector<std::vector<pb_segment_query>> csq((size_t)nc);
  for (size_t i = 0; i < g->segs.size(); i++) csq[(size_t)g->child_of[i]].push_back(sqs[i]);
  pb_query_desc cq = *q;
  cq.flags = q->flags & ~PB_Q_ALL_RANKS;
  if (combine) cq.flags |= PB_Q_DEFER_FINALIZE;
  std::vector<pb_result_s*> parts((size_t)nc, nullptr);
  auto free_parts = [&]() { for (auto* p : parts) if (p) free_result(p); };
  for (int k = 0; k < nc; k++) {
    DeviceGuard dg(g->children[k]->ctx);
    if ((rc = exec_single(g->children[k], csq[(size_t)k].data(), &cq, &parts[(size_t)k]))) { free_parts(); return rc; }
  }
  if (!combine) {
    // one table per segment, in the caller's segment order: a shell result that maps table t to (device part, local table)
    pb_result_s* shell = new pb_result_s();
    shell->group = g; shell->n_gb = parts[0]->n_gb; shell->n_aggs = parts[0]->n_aggs; shell->agg_op = parts[0]->agg_op;
    shell->table_mode = parts[0]->table_mode; shell->finalized = true;
    for (size_t i = 0; i < g->segs.size(); i++) shell->table_map.push_back({g->child_of[i], g->index_in_child[i]});
    for (auto* p : parts) { shell->device_ms = std::max(shell->device_ms, p->device_ms); shell->scan_ms = std::max(shell->scan_ms, p->scan_ms); shell->launches += p->launches; }
    shell->parts = parts;
    *out = shell;
    return PB_OK;
  }
  pb_result_s* root = parts[0];
  {
    DeviceGuard dg(root->ctx);
    for (int k = 1; k < nc; k++) {
      if (parts[(size_t)k]->block_bytes != root->block_bytes || parts[(size_t)k]->fingerprint != root->fingerprint || root->table_mode == T_HASH) {
        free_parts();
        return fail(PB_ERR_UNSUPPORTED, root->table_mode == T_HASH ? "hash group tables are not merged across the devices of one process yet: use one process per GPU"
                                                                    : "per-device table layouts differ");
      }
    }
    // the peers' kernels must have finished before their blocks are read
    for (int k = 1; k < nc; k++) {
      cudaError_t e = cudaStreamWaitEvent(root->stream, parts[(size_t)k]->ev3, 0);
      if (e != cudaSuccess) { free_parts(); return fail(PB_ERR_CUDA, "cudaStreamWaitEvent: %s", cudaGetErrorString(e)); }
    }
    bool p2p = true;
    for (int k = 1; k < nc; k++) { int can = 0; cudaDeviceCanAccessPeer(&can, root->ctx->device, parts[(size_t)k]->ctx->device); if (!can) p2p = false; }
    if (p2p) {
      DevMergePeers peers; memset(&peers, 0, sizeof peers);
      for (int k = 1; k < nc; k++) peers.p[k - 1] = reinterpret_cast<const unsigned long long*>(parts[(size_t)k]->block);
      rc = launch_merge_rows(root, nullptr, &peers, nc - 1, true);
    } else {
      // no peer access (e.g. across PCIe switches): stage the blocks through copies
      rc = ensure_gather_buf(root->ctx, (size_t)(nc - 1) * (size_t)root->block_bytes, root->stream);
      for (int k = 1; k < nc && !rc; k++) {
        cudaError_t e = cudaMemcpyPeerAsync((uint8_t*)root->ctx->gather_buf + (size_t)(k - 1) * (size_t)root->block_bytes, root->ctx->device,
                                            parts[(size_t)k]->block, parts[(size_t)k]->ctx->device, (size_t)root->block_bytes, root->stream);
        if (e != cudaSuccess) rc = fail(PB_ERR_CUDA, "cudaMemcpyPeerAsync: %s", cudaGetErrorString(e));
      }
      if (!rc) rc = launch_merge_rows(root, root->ctx->gather_buf, nullptr, nc - 1, true);
    }
    if (rc) { free_parts(); return rc; }
    root->merged_ranks *= nc;
    for (int k = 1; k < nc; k++) { root->parts.push_back(parts[(size_t)k]); root->launches += parts[(size_t)k]->launches; }
    if ((q->flags & PB_Q_ALL_RANKS) && (rc = comm_merge(root))) { free_result(root); return rc; }
    if (!(q->flags & PB_Q_DEFER_FINALIZE) && (rc = finalize_result(root))) { free_result(root); return rc; }
  }
  *out = root;
  return PB_OK;
}

// ------------------------------------------------------------------------------------------------
// finalize: compaction of non-empty groups, device -> pinned host, key decode
// ------------------------------------------------------------------------------------------------

// ORDER BY ... LIMIT trim: order keys of every table + the grid-wide radix select of the trim_size-th best (8 digit passes)
static int enqueue_trim(pb_result_s* r) {
  if (r->trim_size <= 0 || r->table_mode == T_KEYLESS) return PB_OK;
  cudaStream_t st = r->stream;
  pb_group_s* g = r->group;
  for (size_t t = 0; t < r->tables.size(); t++) {
    TableMeta& tm = r->tables[t];
    DevOrderKey K; memset(&K, 0, sizeof K);
    K.kind = r->order0.kind; K.descending = r->order0.descending; K.mode = r->table_mode; K.key_words = tm.dev.key_words;
    K.S = tm.capacity + (r->table_mode == T_HASH ? 1 : 0); K.capacity = tm.capacity;
    K.rowcnt = tm.dev.rowcnt; K.hkeys = tm.dev.hkeys; K.okey = r->d_okey[t];
    if (K.kind == 1) {
      const int a = r->order0.index;
      K.op = r->agg_op[a]; K.sum = tm.dev.sum[a]; K.mm = tm.dev.mm[a]; K.fcnt = tm.dev.fcnt[a];
    } else {
      const int j = r->order0.index;
      const pb_segment_s* s0 = g->segs[tm.seg_idx[0]];
      const Column& c0 = s0->cols[find_col(s0, r->gb_names[j].c_str())];
      K.field_is_signed = !c0.has_dict && (c0.type == PB_INT || c0.type == PB_LONG);
      K.field_is_double = !c0.has_dict && (c0.type == PB_FLOAT || c0.type == PB_DOUBLE);
      if (r->table_mode == T_DENSE) { uint64_t div = 1; for (int k = 0; k < j; k++) div *= (uint64_t)tm.cards[k]; K.div = div; K.card = (uint64_t)tm.cards[j]; }
      else { K.shift = tm.shifts[j]; K.width = tm.widths[j]; }
    }
    const int grid = (int)std::min<uint64_t>((K.S + 255) / 256, (uint64_t)r->ctx->num_sms * 8);
    pb_order_key_kernel<<<grid, 256, 0, st>>>(K);
    for (int pass = 7; pass >= 0; pass--) {
      pb_rselect_hist_kernel<<<grid, 256, 0, st>>>(K.okey, K.rowcnt, K.S, pass, r->d_sel[t]);
      pb_rselect_pick_kernel<<<1, 32, 0, st>>>(r->d_sel[t], pass, (unsigned long long)r->trim_size, (unsigned long long)r->trim_threshold);
    }
    r->launches += 17;
  }
  CU(cudaGetLastError());
  return PB_OK;
}

// ---- result hand-back in three steps, so that a cached plan can re-enqueue step 2 without redoing step 1 ----
// (1) pinned host arrays + the finalize descriptor of every table.  Very large tables are counted first (one extra pass
//     and a synchronisation) so that the host arrays can be sized exactly; such plans are not cached.
static int prepare_finalize(pb_result_s* r) {
  pb_result_s::Replay& rp = r->rp;
  if (rp.fin_prepared) return PB_OK;
  cudaStream_t st = r->stream;
  pb_group_s* g = r->group;
  const int nT = (int)r->tables.size(), nG = r->n_gb, nA = r->n_aggs;
  const int mode = r->table_mode;
  if (!r->h_counters.p) r->h_counters.alloc(8 * PB_COUNTERS_PER_TABLE * (size_t)nT);
  unsigned long long* hc = (unsigned long long*)r->h_counters.p;
  if (!hc) return fail(PB_ERR_OOM, "pinned host allocation failed");
  const uint64_t SMALL_TABLE = 1ull << 20;
  bool any_big = false;
  for (int t = 0; t < nT; t++) {
    TableMeta& tm = r->tables[t];
    const uint64_t S = tm.capacity + (mode == T_HASH ? 1 : 0);
    if (mode != T_KEYLESS && S > SMALL_TABLE) {
      any_big = true;
      int grid = (int)std::min<uint64_t>((S + 255) / 256, 2048);
      pb_count_groups_kernel<<<grid, 256, 0, st>>>(tm.dev.rowcnt, S, r->d_counters + (size_t)t * PB_COUNTERS_PER_TABLE + 3,
                                                   r->trim_size > 0 ? r->d_okey[(size_t)t] : nullptr, r->trim_size > 0 ? &r->d_sel[(size_t)t]->thr : nullptr);
      r->launches++;
    }
  }
  if (any_big) {
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(hc, r->d_counters, 8 * PB_COUNTERS_PER_TABLE * (size_t)nT, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  rp.fin.assign((size_t)nT, DevFinalize());
  rp.fin_grid.assign((size_t)nT, 1);
  for (int t = 0; t < nT; t++) {
    TableMeta& tm = r->tables[t];
    const uint64_t S = tm.capacity + (mode == T_HASH ? 1 : 0);
    uint64_t cap = mode == T_KEYLESS ? 1 : S;
    if (mode != T_KEYLESS && S > SMALL_TABLE) {
      cap = std::max<uint64_t>(hc[(size_t)t * PB_COUNTERS_PER_TABLE + 3], 1);
      CU(cudaMemsetAsync(r->d_counters + (size_t)t * PB_COUNTERS_PER_TABLE + 3, 0, 8, st));
    }
    tm.out_cap = cap;
    tm.dbl.resize(nA); tm.lng.resize(nA); tm.dc_off.resize(nA); tm.dc_ids.resize(nA);
    tm.key_ids.resize(nG); tm.key_vals.resize(nG); tm.key_type.assign(nG, 0); tm.key_eb.assign(nG, 0);
    tm.slots.alloc(8 * cap); tm.rows.alloc(8 * cap);
    if (!tm.slots.p || !tm.rows.p) return fail(PB_ERR_OOM, "pinned host allocation failed");
    DevFinalize& F = rp.fin[(size_t)t];
    memset(&F, 0, sizeof F);
    F.mode = mode; F.n_gb = nG; F.n_aggs = nA; F.always_emit = mode == T_KEYLESS ? 1 : 0; F.count_all = r->count_all ? 1 : 0;
    F.S = mode == T_KEYLESS ? 1 : S; F.capacity = tm.capacity; F.cap_out = cap; F.key_words = tm.dev.key_words;
    F.rowcnt = tm.dev.rowcnt; F.hkeys = tm.dev.hkeys;
    if (tm.dev.first_doc) { F.first_doc = tm.dev.first_doc; F.first_thr = r->d_first_thr + t; }
    if (r->trim_size > 0 && mode != T_KEYLESS) { F.okey = r->d_okey[(size_t)t]; F.othr = &r->d_sel[(size_t)t]->thr; }
    F.cursor = r->d_counters + (size_t)t * PB_COUNTERS_PER_TABLE + 3;
    // every byte of the hand-back crosses PCIe: the slot of a row is only written when a DISTINCTCOUNT will ask for it, and
    // the long arrays of SUM / MIN / MAX (all zeros) are made on the host when somebody reads them (pb_result_long)
    bool any_dc = false;
    for (int a = 0; a < nA; a++) any_dc |= r->agg_op[a] == PB_AGG_DISTINCTCOUNT;
    F.out_slots = any_dc ? (unsigned long long*)tm.slots.p : nullptr; F.out_rows = (unsigned long long*)tm.rows.p;
    for (int a = 0; a < nA; a++) {
      tm.dbl[a].alloc(8 * cap); tm.lng[a].alloc(8 * cap);
      if (!tm.dbl[a].p || !tm.lng[a].p) return fail(PB_ERR_OOM, "pinned host allocation failed");
      F.aggs[a].op = r->agg_op[a]; F.aggs[a].sum = tm.dev.sum[a]; F.aggs[a].mm = tm.dev.mm[a]; F.aggs[a].out = (double*)tm.dbl[a].p;
      const bool lng_on_device = r->agg_op[a] == PB_AGG_COUNT || r->agg_op[a] == PB_AGG_AVG || r->agg_op[a] == PB_AGG_DISTINCTCOUNT || r->count_all;
      F.aggs[a].fcnt = tm.dev.fcnt[a]; F.aggs[a].out_cnt = lng_on_device ? (long long*)tm.lng[a].p : nullptr; F.aggs[a].dcnt = tm.dev.dcnt[a];
    }
    uint64_t div = 1;
    for (int j = 0; j < nG; j++) {
      const pb_segment_s* s0 = g->segs[tm.seg_idx[0]];
      const Column& c0 = s0->cols[find_col(s0, r->gb_names[j].c_str())];
      DevFinKey& fk = F.keys[j];
      fk.is_dict = c0.has_dict; fk.type = c0.type;
      if (c0.has_dict) {
        if (r->combine) { const GlobalDict& gd = g->dicts.at(r->gb_names[j]); fk.dict_vals = gd.d_values; fk.eb = gd.entry_bytes; }
        else { fk.dict_vals = c0.d_dict_native; fk.eb = c0.entry_bytes; }
        if (!fk.dict_vals) return fail(PB_ERR_STATE, "dictionary of %s is not staged", c0.name.c_str());
      } else fk.eb = (c0.type == PB_INT || c0.type == PB_FLOAT) ? 4 : 8;
      if (mode == T_DENSE) { fk.div = div; fk.card = (uint64_t)tm.cards[j]; div *= (uint64_t)tm.cards[j]; }
      else if (mode == T_HASH) { fk.shift = tm.shifts[j]; fk.width = tm.widths[j]; }
      tm.key_type[j] = c0.type; tm.key_eb[j] = fk.eb;
      tm.key_ids[j].alloc(4 * cap); tm.key_vals[j].alloc((size_t)fk.eb * cap);
      if (!tm.key_ids[j].p || !tm.key_vals[j].p) return fail(PB_ERR_OOM, "pinned host allocation failed");
      fk.out_ids = (int32_t*)tm.key_ids[j].p; fk.out_vals = (uint8_t*)tm.key_vals[j].p;
    }
    rp.fin_grid[(size_t)t] = (int)std::min<uint64_t>((F.S + 255) / 256, 1184);
  }
  rp.fin_prepared = true;
  return PB_OK;
}
// (2) one pass per table: compaction + aggregate extraction + key decode, written straight into pinned host memory; then the
//     counter cells
static int enqueue_finalize(pb_result_s* r) {
  cudaStream_t st = r->stream;
  const int nT = (int)r->tables.size();
  for (int t = 0; t < nT; t++) {
    const DevFinalize& F = r->rp.fin[(size_t)t];
    for (int a = 0; a < r->n_aggs; a++) {
      const DevTable& dt = r->tables[(size_t)t].dev;
      if (!dt.dset[a]) continue;
      const uint64_t cap = dt.dset_mask[a] + 1;
      pb_dset_count_kernel<<<(int)std::min<uint64_t>((cap + 255) / 256, (uint64_t)r->ctx->num_sms * 8), 256, 0, st>>>(dt.dset[a], cap, dt.dcnt[a]);
      r->launches++;
    }
    if (F.first_doc) {
      pb_select_first_kernel<<<1, 1024, 0, st>>>(F.first_doc, F.S, r->tables[(size_t)t].dev.num_groups_limit, r->d_first_thr + t);
      r->launches++;
    }
    pb_finalize_kernel<<<r->rp.fin_grid[(size_t)t], 256, 0, st>>>(F);
    r->launches++;
  }
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(r->h_counters.p, r->d_counters, 8 * PB_COUNTERS_PER_TABLE * (size_t)nT, cudaMemcpyDeviceToHost, st));
  CU(cudaEventRecord(r->ev3, st));
  return PB_OK;
}
// (3) wait, then the host side: group counts, statistics, DISTINCTCOUNT sizes
static int finish_finalize(pb_result_s* r) {
  cudaStream_t st = r->stream;
  const int nT = (int)r->tables.size(), nG = r->n_gb, nA = r->n_aggs;
  unsigned long long* hc = (unsigned long long*)r->h_counters.p;
  double t_prev = now_us();
  auto lap = [&](int i) { double t = now_us(); r->host_us[i] += t - t_prev; t_prev = t; };
  CU(cudaStreamSynchronize(st));
  lap(5);
  if (!r->graph_replayed) {      // (a graph replay keeps the times of the plan's last kernel-by-kernel run)
    float ms = 0;
    if (cudaEventElapsedTime(&ms, r->ev0, r->ev3) == cudaSuccess) r->device_ms = ms;
    if (cudaEventElapsedTime(&ms, r->ev1, r->ev2) == cudaSuccess) r->scan_ms = ms;
    if (cudaEventElapsedTime(&ms, r->ev1, r->evm) == cudaSuccess) r->filter_ms = ms;
    if (cudaEventElapsedTime(&ms, r->evm, r->ev2) == cudaSuccess) r->agg_ms = ms;
    if (r->comm_timed && cudaEventElapsedTime(&ms, r->sset.ev[5], r->sset.ev[6]) == cudaSuccess) { r->comm_ms = ms; r->rp.comm_ms_sample = ms; }
    cudaGetLastError();
  }

  // host side: counts, stats, distinct value sets
  for (int t = 0; t < nT; t++) {
    TableMeta& tm = r->tables[t];
    const int64_t ng = (int64_t)std::min<uint64_t>(hc[(size_t)t * PB_COUNTERS_PER_TABLE + 3], tm.out_cap);
    tm.num_groups = ng;
    // (COUNT / AVG counts and the zeros of the other long arrays are written by the finalize kernel)
    // DISTINCTCOUNT: the sizes now; the value sets (BaseDistinctAggregateAggregationFunction intermediate result) are
    // materialised on first access (pb_result_distinct_offsets / _dict_ids) — a merged result usually needs the sizes only
    for (int a = 0; a < nA; a++) {
      if (r->agg_op[a] != PB_AGG_DISTINCTCOUNT || !tm.dev.dc_bits[a]) continue;      // (raw columns: counted by the finalize pass)
      int64_t* L = (int64_t*)tm.lng[a].p;
      if (ng > 0) {
        int wgrid = (int)(((size_t)ng * 32 + 255) / 256);
        pb_distinct_count_kernel<<<wgrid, 256, 0, st>>>(tm.dev.dc_bits[a], tm.dev.dc_words[a], (const unsigned long long*)tm.slots.p, (uint64_t)ng, (unsigned long long*)L);
        r->launches++;
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(st));
      }
    }
    // ExecutionStatistics (GroupByOperator.java:148-153; ProjectPlanNode.java:69-78)
    std::vector<std::string> proj;
    for (auto& nme : r->gb_names) if (std::find(proj.begin(), proj.end(), nme) == proj.end()) proj.push_back(nme);
    for (auto& nme : r->agg_cols) if (!nme.empty() && std::find(proj.begin(), proj.end(), nme) == proj.end()) proj.push_back(nme);
    // every statistic is a counter cell of the table block (PB_COUNTERS_PER_TABLE): device-accumulated or injected by the
    // host at init, and summed by the cross-GPU merges -- a merged result reports the totals over all ranks' segments
    const unsigned long long* cc = hc + (size_t)t * PB_COUNTERS_PER_TABLE;
    tm.stats.num_docs_scanned = (int64_t)cc[2];
    tm.stats.num_entries_scanned_post_filter = tm.stats.num_docs_scanned * (int64_t)proj.size();
    // (PB_Q_NULL_HANDLING: the clauses are the implicit "<column> IS NOT NULL" of null-skipping functions, which the reference
    //  evaluates inside the functions, not as swim-lanes: the plain figures apply.  A query that ALSO has FILTER clauses of
    //  its own reports the plain figures too, where the reference would count its lanes)
    if (r->n_agg_filters > 0 && !r->count_all) {        // swim-lanes of filtered aggregations (pb_lane_stats_kernel)
      tm.stats.num_docs_scanned = (int64_t)cc[4];
      tm.stats.num_entries_scanned_post_filter = (int64_t)cc[5];
    }
    tm.stats.num_total_docs = (int64_t)cc[6];
    tm.stats.num_entries_scanned_in_filter = (int64_t)cc[7];
    tm.stats.num_segments = (int32_t)cc[8];
    if (cc[9] != r->fingerprint * (unsigned long long)r->merged_ranks)
      return fail(PB_ERR_STATE, "cross-GPU merge: table layouts differ across ranks (different query or global dictionaries)");
    tm.stats.num_groups_limit_reached = 0;
    if (nG > 0) {
      bool flag = (uint32_t)hc[(size_t)t * PB_COUNTERS_PER_TABLE + 1] != 0;
      tm.stats.num_groups_limit_reached = (flag || ng >= (int64_t)tm.dev.num_groups_limit) ? 1 : 0;   // GroupByOperator.java:116
    }
  }
  lap(6);
  r->finalized = true;
  release_segments(r);       // everything that reads segment data has run: the segments may be evicted or released again
  for (auto* p : r->parts) release_segments(p);
  return PB_OK;
}
static int finalize_result(pb_result_s* r) {
  if (r->finalized) return PB_OK;
  int rc;
  double t0 = now_us();
  if ((rc = enqueue_trim(r))) return rc;
  if ((rc = prepare_finalize(r))) return rc;
  r->host_us[4] += now_us() - t0;
  if ((rc = enqueue_finalize(r))) return rc;
  return finish_finalize(r);
}

extern "C" int pb_result_finalize(pb_result_handle r) {
  if (!r) return fail(PB_ERR_INVALID, "null result");
  DeviceGuard dg(r->ctx);
  return finalize_result(r);
}

// ------------------------------------------------------------------------------------------------
// accessors
// ------------------------------------------------------------------------------------------------
static TableMeta* tab_of(pb_result_s*& r, int t) {     // resolves a shell result's table to the part that owns it (r is updated)
  if (!r || t < 0 || !r->finalized) return nullptr;
  if (!r->table_map.empty()) {
    if (t >= (int)r->table_map.size()) return nullptr;
    const auto m = r->table_map[(size_t)t];
    r = r->parts[(size_t)m.first];
    t = m.second;
    if (!r->finalized) return nullptr;
  }
  return t < (int)r->tables.size() ? &r->tables[(size_t)t] : nullptr;
}
#define TAB(r, t) tab_of(r, t)
extern "C" int32_t pb_result_num_tables(pb_result_handle r) { return r ? (int32_t)(r->table_map.empty() ? r->tables.size() : r->table_map.size()) : 0; }
extern "C" int64_t pb_result_num_groups(pb_result_handle r, int32_t t) { auto* tm = TAB(r, t); return tm ? tm->num_groups : -1; }
extern "C" const int32_t* pb_result_group_dict_ids(pb_result_handle r, int32_t t, int32_t gb) {
  auto* tm = TAB(r, t); if (!tm || gb < 0 || gb >= r->n_gb) return nullptr; return (const int32_t*)tm->key_ids[gb].p;
}
extern "C" const void* pb_result_group_key_values(pb_result_handle r, int32_t t, int32_t gb, int32_t* stored_type, int32_t* entry_bytes) {
  auto* tm = TAB(r, t); if (!tm || gb < 0 || gb >= r->n_gb) return nullptr;
  if (stored_type) *stored_type = tm->key_type[gb];
  if (entry_bytes) *entry_bytes = tm->key_eb[gb];
  return tm->key_vals[gb].p;
}
extern "C" const double* pb_result_double(pb_result_handle r, int32_t t, int32_t a) { auto* tm = TAB(r, t); return (tm && a >= 0 && a < r->n_aggs) ? (const double*)tm->dbl[a].p : nullptr; }
extern "C" const int64_t* pb_result_long(pb_result_handle r, int32_t t, int32_t a) {
  auto* tm = TAB(r, t);
  if (!tm || a < 0 || a >= r->n_aggs) return nullptr;
  const int op = r->agg_op[a];
  if ((op == PB_AGG_SUM || op == PB_AGG_MIN || op == PB_AGG_MAX) && !r->count_all) memset(tm->lng[a].p, 0, 8 * (size_t)std::max<int64_t>(tm->num_groups, 1));   // not written by the device
  return (const int64_t*)tm->lng[a].p;
}
// DISTINCTCOUNT value sets, materialised on first access
static int materialize_distinct(pb_result_s* r, TableMeta& tm, int a) {
  if (tm.dc_off[a].p) return PB_OK;
  if (r->agg_op[a] != PB_AGG_DISTINCTCOUNT) return fail(PB_ERR_INVALID, "aggregation %d is not DISTINCTCOUNT", a);
  DeviceGuard dg(r->ctx);
  cudaStream_t st = r->stream;
  const int64_t ng = tm.num_groups;
  const int64_t* L = (const int64_t*)tm.lng[a].p;
  tm.dc_off[a].alloc(8 * (size_t)(ng + 1));
  int64_t* off = (int64_t*)tm.dc_off[a].p;
  off[0] = 0;
  for (int64_t k = 0; k < ng; k++) off[k + 1] = off[k] + L[k];
  const int64_t total = off[ng];
  if (tm.dev.dset[a]) {
    // raw column: scatter the (slot, value) set into per-group runs, then order each run on the host (value sets are an
    // on-demand hand-back: the merged result of a query usually needs the sizes only)
    if (tm.dc_vals.size() < (size_t)r->n_aggs) tm.dc_vals.resize((size_t)r->n_aggs);
    tm.dc_vals[a].alloc(8 * (size_t)std::max<int64_t>(total, 1));
    if (!tm.dc_vals[a].p) return fail(PB_ERR_OOM, "pinned host allocation failed");
    if (total > 0) {
      const uint64_t S = tm.capacity + (r->table_mode == T_HASH ? 1 : 0), cap = tm.dev.dset_mask[a] + 1;
      uint32_t* d_map = nullptr; unsigned long long* d_cur = nullptr;
      CU(cudaMallocAsync((void**)&d_map, 4 * S, st));
      CU(cudaMallocAsync((void**)&d_cur, 8 * (size_t)ng, st));
      CU(cudaMemsetAsync(d_map, 0xff, 4 * S, st));
      CU(cudaMemsetAsync(d_cur, 0, 8 * (size_t)ng, st));
      pb_invert_slots_kernel<<<(int)std::min<int64_t>((ng + 255) / 256, 4096), 256, 0, st>>>((const unsigned long long*)tm.slots.p, (uint64_t)ng, d_map);
      pb_dset_scatter_kernel<<<(int)std::min<uint64_t>((cap + 255) / 256, (uint64_t)r->ctx->num_sms * 8), 256, 0, st>>>(
          tm.dev.dset[a], cap, d_map, (const unsigned long long*)off, d_cur, (long long*)tm.dc_vals[a].p);
      r->launches += 2;
      CU(cudaGetLastError());
      CU(cudaFreeAsync(d_map, st)); CU(cudaFreeAsync(d_cur, st));
      CU(cudaStreamSynchronize(st));
      int64_t* v = (int64_t*)tm.dc_vals[a].p;
      for (int64_t k = 0; k < ng; k++) std::sort(v + off[k], v + off[k + 1]);
    }
    return PB_OK;
  }
  tm.dc_ids[a].alloc(4 * (size_t)std::max<int64_t>(total, 1));
  if (!tm.dc_ids[a].p) return fail(PB_ERR_OOM, "pinned host allocation failed");
  if (total > 0) {
    int wgrid = (int)(((size_t)ng * 32 + 255) / 256);
    pb_distinct_ids_kernel<<<wgrid, 256, 0, st>>>(tm.dev.dc_bits[a], tm.dev.dc_words[a], (const unsigned long long*)tm.slots.p, (uint64_t)ng,
                                                  (const unsigned long long*)off, (int32_t*)tm.dc_ids[a].p);
    r->launches++;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));
  }
  return PB_OK;
}
extern "C" const int64_t* pb_result_distinct_offsets(pb_result_handle r, int32_t t, int32_t a) {
  auto* tm = TAB(r, t);
  if (!tm || a < 0 || a >= r->n_aggs || materialize_distinct(r, *tm, a) != PB_OK) return nullptr;
  return (const int64_t*)tm->dc_off[a].p;
}
extern "C" const int64_t* pb_result_distinct_values(pb_result_handle r, int32_t t, int32_t a) {
  auto* tm = TAB(r, t);
  if (!tm || a < 0 || a >= r->n_aggs || !tm->dev.dset[a] || materialize_distinct(r, *tm, a) != PB_OK) return nullptr;
  return (const int64_t*)tm->dc_vals[a].p;
}
extern "C" const int32_t* pb_result_distinct_dict_ids(pb_result_handle r, int32_t t, int32_t a) {
  auto* tm = TAB(r, t);
  if (!tm || a < 0 || a >= r->n_aggs || tm->dev.dset[a] || materialize_distinct(r, *tm, a) != PB_OK) return nullptr;
  return (const int32_t*)tm->dc_ids[a].p;
}
extern "C" const pb_exec_stats* pb_result_stats(pb_result_handle r, int32_t t) { auto* tm = TAB(r, t); return tm ? &tm->stats : nullptr; }
extern "C" double pb_result_device_ms(pb_result_handle r) { return r ? r->device_ms : 0; }
extern "C" double pb_result_scan_kernel_ms(pb_result_handle r) {
  if (!r) return 0;
  if (!r->finalized) { float ms = 0; cudaEventSynchronize(r->ev2); cudaEventElapsedTime(&ms, r->ev1, r->ev2); return ms; }
  return r->scan_ms;
}
extern "C" int32_t pb_result_kernel_launches(pb_result_handle r) { return r ? r->launches : 0; }
extern "C" void* pb_result_stream(pb_result_handle r) { return r ? (void*)r->stream : nullptr; }


// Hash tables across ranks: every rank keeps the groups whose key hashes to it.  count -> exchange counts -> pack by
// destination -> one grouped ncclSend/ncclRecv (all-to-all) -> re-initialise the local table -> insert what arrived.  The
// statistics cells are summed over all ranks, so every rank reports the query's totals next to ITS partition of the groups;
// the union of the partitions (disjoint by construction) is the merged table.
static int comm_merge_hash(pb_result_s* r) {
  const int n = g_comm.n_ranks;
  if (n > 64) return fail(PB_ERR_UNSUPPORTED, "hash table merge over %d ranks (max 64)", n);
  TableMeta& tm = r->tables[0];
  const int nA = r->n_aggs;
  for (int a = 0; a < nA; a++) if (r->agg_op[a] == PB_AGG_DISTINCTCOUNT) return fail(PB_ERR_UNSUPPORTED, "DISTINCTCOUNT in a hash group table is not merged across ranks");
  cudaStream_t st = r->stream;
  Context* ctx = r->ctx;
  const int kw = r->key_words, T = kw + 1 + nA;
  const uint64_t S = tm.capacity + 1;
  const int grid = (int)std::min<uint64_t>((S + 255) / 256, (uint64_t)ctx->num_sms * 8);
  CU(cudaEventRecord(r->sset.ev[5], st));
  // small control block: [counts n | cursors n | offsets n | all counts n*n | counter cells n*PB_COUNTERS_PER_TABLE]
  const size_t ctl_words = (size_t)3 * n + (size_t)n * n + (size_t)n * PB_COUNTERS_PER_TABLE + 8;
  unsigned long long* d_ctl = nullptr;
  CU(cudaMallocAsync((void**)&d_ctl, 8 * ctl_words, st)); r->dev_allocs.push_back(d_ctl);
  CU(cudaMemsetAsync(d_ctl, 0, 8 * ctl_words, st));
  unsigned long long *d_counts = d_ctl, *d_cursors = d_ctl + n, *d_offsets = d_ctl + 2 * n, *d_all = d_ctl + 3 * n, *d_cells = d_ctl + 3 * n + (size_t)n * n;
  DevHashXfer X; memset(&X, 0, sizeof X);
  X.n_ranks = n; X.key_words = kw; X.n_aggs = nA; X.tuple_words = T; X.S = S; X.capacity = tm.capacity;
  X.hkeys = tm.dev.hkeys; X.rowcnt = tm.dev.rowcnt;
  for (int a = 0; a < nA; a++) { X.sum[a] = tm.dev.sum[a]; X.mm[a] = tm.dev.mm[a]; X.fcnt[a] = tm.dev.fcnt[a]; }
  X.counts = d_counts; X.cursors = d_cursors; X.offsets = d_offsets;
  pb_hash_count_kernel<<<grid, 256, 0, st>>>(X);
  r->launches++;
  CU(cudaGetLastError());
  NC(g_comm.api.AllGather(d_counts, d_all, 8 * (size_t)n, ncclChar, g_comm.comm, st));
  NC(g_comm.api.AllGather(r->d_counters, d_cells, 8 * (size_t)PB_COUNTERS_PER_TABLE, ncclChar, g_comm.comm, st));
  std::vector<unsigned long long> all((size_t)n * n);
  CU(cudaMemcpyAsync(all.data(), d_all, 8 * all.size(), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  const int me = g_comm.rank;
  std::vector<unsigned long long> soff((size_t)n + 1, 0), roff((size_t)n + 1, 0);
  for (int k = 0; k < n; k++) { soff[k + 1] = soff[k] + all[(size_t)me * n + k]; roff[k + 1] = roff[k] + all[(size_t)k * n + me]; }
  const uint64_t n_send = soff[n], n_recv = roff[n];
  unsigned long long *d_send = nullptr, *d_recv = nullptr;
  CU(cudaMallocAsync((void**)&d_send, 8 * (size_t)T * std::max<uint64_t>(n_send, 1), st)); r->dev_allocs.push_back(d_send);
  CU(cudaMallocAsync((void**)&d_recv, 8 * (size_t)T * std::max<uint64_t>(n_recv, 1), st)); r->dev_allocs.push_back(d_recv);
  CU(cudaMemcpyAsync(d_offsets, soff.data(), 8 * (size_t)n, cudaMemcpyHostToDevice, st));
  X.out = d_send;
  pb_hash_pack_kernel<<<grid, 256, 0, st>>>(X);
  r->launches++;
  CU(cudaGetLastError());
  NC(g_comm.api.GroupStart());
  for (int k = 0; k < n; k++) {
    const size_t sb = 8 * (size_t)T * (size_t)(soff[k + 1] - soff[k]), rb = 8 * (size_t)T * (size_t)(roff[k + 1] - roff[k]);
    if (sb) NC(g_comm.api.Send(d_send + (size_t)T * soff[k], sb, ncclChar, k, g_comm.comm, st));
    if (rb) NC(g_comm.api.Recv(d_recv + (size_t)T * roff[k], rb, ncclChar, k, g_comm.comm, st));
  }
  NC(g_comm.api.GroupEnd());
  // the local table starts over (its rows all travelled, this rank's own share included); the counters stay
  {
    const uint64_t skip16 = (((uint64_t)PB_COUNTERS_PER_TABLE * 8 + 255) & ~(uint64_t)255) / 16;      // counter cells of the one table
    pb_init_tables_kernel<<<r->init.grid, 256, 0, st>>>(r->init.zero + skip16, r->init.zn - skip16, r->init.ff, r->init.fn, r->init.mm, r->init.mn,
                                                         nullptr, 0, nullptr, 0);
    CU(cudaMemsetAsync(r->d_counters, 0, 8, st));     // num_groups: recounted by the inserts
    pb_sum_counters_kernel<<<1, 32, 0, st>>>(r->d_counters, d_cells, n, PB_COUNTERS_PER_TABLE);
    r->launches += 2;
  }
  if (n_recv) {
    const int mgrid = (int)std::min<uint64_t>((n_recv + 255) / 256, (uint64_t)ctx->num_sms * 8);
    pb_hash_merge_kernel<<<mgrid, 256, 0, st>>>(tm.dev, d_recv, n_recv, kw, nA, T);
    r->launches++;
  }
  CU(cudaGetLastError());
  CU(cudaEventRecord(r->sset.ev[6], st));
  r->comm_timed = true;
  r->merged_ranks *= n;
  return PB_OK;
}
static int launch_merge_rows(pb_result_s* r, const void* gathered, const DevMergePeers* peers, int n_rows, bool base_is_dst) {
  if (!r->combine || r->tables.size() != 1 || r->table_mode == T_HASH) return fail(PB_ERR_UNSUPPORTED, "merge needs a combined dense / keyless result");
  for (int a = 0; a < r->n_aggs; a++) if (r->tables[0].dev.dset[a]) return fail(PB_ERR_UNSUPPORTED, "DISTINCTCOUNT on a raw column is not merged across GPUs");
  const uint64_t n_words = (uint64_t)r->block_bytes / 8;
  int grid = (int)std::min<uint64_t>((n_words + 255) / 256, (uint64_t)r->ctx->num_sms * 8);
  DevMergePeers none; memset(&none, 0, sizeof none);
  pb_merge_blocks_kernel<<<grid, 256, 0, r->stream>>>((unsigned long long*)r->block, (const unsigned long long*)gathered, peers ? *peers : none, n_rows,
                                                      base_is_dst ? 1 : 0, n_words, (uint64_t)r->block_sum_off / 8, (uint64_t)r->block_dc_off / 8,
                                                      (uint64_t)r->block_mm_off / 8);
  r->launches++;
  CU(cudaGetLastError());
  return PB_OK;
}
static int launch_merge(pb_result_s* r, const void* gathered, int n_rows, bool base_is_dst) { return launch_merge_rows(r, gathered, nullptr, n_rows, base_is_dst); }
// merge the gathered table blocks of all ranks (rank-major copies of pb_result_device_buffer(which = 8)) into this result:
// for callers that run the collective themselves (PB_Q_DEFER_FINALIZE); PB_Q_ALL_RANKS does all of it inside the library
extern "C" int pb_result_merge_gathered(pb_result_handle r, const void* gathered, int32_t n_ranks) {
  if (!r || !gathered || n_ranks < 1) return fail(PB_ERR_INVALID, "bad arguments");
  DeviceGuard dg(r->ctx);
  int rc = launch_merge(r, gathered, n_ranks, false);
  if (rc) return rc;
  r->merged_ranks *= n_ranks;
  return PB_OK;
}
extern "C" int pb_result_phase_ms(pb_result_handle r, double* filter_ms, double* agg_ms) {
  if (!r) return fail(PB_ERR_INVALID, "null result");
  if (!r->finalized) {
    float ms = 0;
    cudaEventSynchronize(r->ev2);
    cudaEventElapsedTime(&ms, r->ev1, r->evm); r->filter_ms = ms;
    cudaEventElapsedTime(&ms, r->evm, r->ev2); r->agg_ms = ms;
  }
  if (filter_ms) *filter_ms = r->filter_ms;
  if (agg_ms) *agg_ms = r->agg_ms;
  return PB_OK;
}
extern "C" int pb_result_host_timing(pb_result_handle r, double* out8) {
  if (!r || !out8) return fail(PB_ERR_INVALID, "null argument");
  for (int i = 0; i < 8; i++) out8[i] = r->host_us[i];
  return PB_OK;
}
extern "C" int pb_result_wait(pb_result_handle r) {
  if (!r) return fail(PB_ERR_INVALID, "null result");
  for (auto* p : r->parts) if (p->stream) { DeviceGuard dgp(p->ctx); CU(cudaStreamSynchronize(p->stream)); }
  if (r->stream) { DeviceGuard dg(r->ctx); CU(cudaStreamSynchronize(r->stream)); }
  return PB_OK;
}
extern "C" int32_t pb_result_in_place_columns(pb_result_handle r) { return r ? r->in_place_columns : 0; }
extern "C" int32_t pb_result_residual_leaves(pb_result_handle r) { return r ? r->residual_leaves : 0; }
extern "C" double pb_result_comm_ms(pb_result_handle r) {
  if (!r || !r->comm_timed) return 0;
  if (r->comm_ms == 0) { float ms = 0; cudaEventSynchronize(r->sset.ev[6]); if (cudaEventElapsedTime(&ms, r->sset.ev[5], r->sset.ev[6]) == cudaSuccess) r->comm_ms = ms; }
  return r->comm_ms;
}

extern "C" int pb_host_register(const void* ptr, size_t bytes) {
  int rc = ensure_init();
  if (rc) return rc;
  DeviceGuard dg(g_all.ctxs[0].get());
  CU(cudaHostRegister(const_cast<void*>(ptr), bytes, cudaHostRegisterPortable | cudaHostRegisterMapped));
  return PB_OK;
}
extern "C" int pb_host_unregister(const void* ptr) {
  CU(cudaHostUnregister(const_cast<void*>(ptr)));
  return PB_OK;
}

extern "C" int pb_result_device_buffer(pb_result_handle r, int32_t which, int32_t agg, void** device_ptr, int64_t* num_elements) {
  if (!r || !device_ptr || !num_elements) return fail(PB_ERR_INVALID, "null argument");
  if (!r->combine || r->tables.size() != 1) return fail(PB_ERR_STATE, "device buffers are exposed for PB_Q_COMBINE results only");
  if (r->table_mode == T_HASH) return fail(PB_ERR_UNSUPPORTED, "hash tables cannot be all-reduced in place");
  TableMeta& tm = r->tables[0];
  const int64_t S = (int64_t)tm.capacity;
  switch (which) {
    case 0: *device_ptr = tm.dev.rowcnt; *num_elements = S; return PB_OK;
    case 1: if (agg < 0 || agg >= r->n_aggs || !tm.dev.sum[agg]) break; *device_ptr = tm.dev.sum[agg]; *num_elements = S; return PB_OK;
    case 2: if (agg < 0 || agg >= r->n_aggs || !tm.dev.mm[agg]) break; *device_ptr = tm.dev.mm[agg]; *num_elements = S; return PB_OK;
    case 3: if (agg < 0 || agg >= r->n_aggs || !tm.dev.dc_bits[agg]) break; *device_ptr = tm.dev.dc_bits[agg]; *num_elements = S * (int64_t)tm.dev.dc_words[agg]; return PB_OK;
    case 4: *device_ptr = r->d_counters; *num_elements = PB_COUNTERS_PER_TABLE; return PB_OK;
    case 5: *device_ptr = r->span_i64; *num_elements = r->span_i64_n; return PB_OK;
    case 6: *device_ptr = r->span_f64; *num_elements = r->span_f64_n; return PB_OK;
    case 7: *device_ptr = r->span_mm; *num_elements = r->span_mm_n; return PB_OK;
    case 8: *device_ptr = r->block; *num_elements = r->block_bytes; return PB_OK;
    default: break;
  }
  return fail(PB_ERR_INVALID, "no such device buffer (which=%d agg=%d)", which, agg);
}

// ------------------------------------------------------------------------------------------------
// internal views for the host planning layer
// ------------------------------------------------------------------------------------------------
#include "pb_internal.h"
int pbi_segment_view(pb_segment_handle s, PbSegmentView* out) {
  if (!s || !out) return fail(PB_ERR_INVALID, "null segment");
  out->name = s->name; out->num_docs = s->num_docs;
  out->cols.resize(s->cols.size());
  for (size_t i = 0; i < s->cols.size(); i++) {
    const Column& c = s->cols[i];
    PbColumnView& v = out->cols[i];
    v.name = c.name; v.type = c.type; v.has_dict = c.has_dict; v.is_sorted = c.is_sorted; v.card = c.card; v.bits = c.bits;
    v.entry_bytes = c.entry_bytes; v.dict = c.h_dict.empty() ? nullptr : c.h_dict.data();
    v.sorted_pairs = c.h_sorted_pairs.empty() ? nullptr : c.h_sorted_pairs.data();
    v.has_inverted = c.h_inv != nullptr;
    v.null_vector = c.h_null; v.null_vector_len = c.h_null_len;
  }
  return PB_OK;
}
int pbi_group_segments(pb_segment_group_handle g, std::vector<pb_segment_handle>* out) {
  if (!g || !out) return fail(PB_ERR_INVALID, "null group");
  out->assign(g->segs.begin(), g->segs.end());
  return PB_OK;
}
int pbi_fail(int code, const char* msg) { return fail(code, "%s", msg); }
void pbi_set_pending_host_key(const std::string& key) { g_pending_host_key = key; }
// Replay the parked plan of an UNLOWERED query (the host layer's key): 1 = replayed (*out set), 0 = no such plan, < 0 = error
int pbi_plan_replay(pb_segment_group_handle g, const std::string& host_key, const pb_query_desc* q, pb_result_handle* out) {
  if (!g || !plan_cache_enabled() || !g->children.empty() || !g->ctx || host_key.empty()) return 0;
  pb_result_s* p = nullptr;
  {
    std::lock_guard<std::mutex> lk(g_plan_mu);
    for (auto* c : g->plans) {
      if (c->rp.busy || c->rp.host_sig != host_key || c->rp.dict_version != g->dict_version || c->rp.seg_epochs.size() != g->segs.size()) continue;
      bool same = true;
      for (size_t i = 0; i < g->segs.size(); i++) if (c->rp.seg_epochs[i] != g->segs[i]->epoch) { same = false; break; }
      if (!same) continue;
      c->rp.busy = true; p = c;
      break;
    }
  }
  if (!p) return 0;
  DeviceGuard dg(g->ctx);
  int rc = replay_plan(p, q);
  if (rc) { free_result(p); return rc; }
  *out = p;
  return 1;
}
