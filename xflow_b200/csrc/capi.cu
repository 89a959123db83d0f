// C ABI layers 2 (parameter table) and 3 (fused worker step) of include/xflow_b200.h.
// Host orchestration only — every byte of table state lives in HBM and is touched only by the
// kernels in kernels.cu.  There is no CPU fallback anywhere in this file.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>

#include "internal.h"

// -------------------------------------------------------------------------------------------------
// errors
// -------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
void xf_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
XF_DLL const char* xf_last_error(void) { return g_err; }
XF_DLL int xf_version(void) { return 100; }
XF_DLL int xf_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int XfDevBuf::ensure(size_t bytes) {
  if (bytes <= cap) return XF_OK;
  size_t want = std::max(bytes, cap + cap / 2);
  if (p) XF_CUDA_TRY(cudaFree(p));
  p = nullptr;
  cap = 0;
  XF_CUDA_TRY(cudaMalloc(&p, want));
  cap = want;
  return XF_OK;
}
void XfDevBuf::release() {
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
}
int XfPinBuf::ensure(size_t bytes) {
  if (bytes <= cap) return XF_OK;
  size_t want = std::max(bytes, cap + cap / 2);
  if (p) XF_CUDA_TRY(cudaFreeHost(p));
  p = nullptr;
  cap = 0;
  XF_CUDA_TRY(cudaHostAlloc(&p, want, cudaHostAllocDefault));
  cap = want;
  return XF_OK;
}
void XfPinBuf::release() {
  if (p) cudaFreeHost(p);
  p = nullptr;
  cap = 0;
}

// -------------------------------------------------------------------------------------------------
// table
// -------------------------------------------------------------------------------------------------
XF_DLL int xf_table_config_default(xf_table_config* cfg) {
  if (!cfg) return XF_ERR_ARG;
  memset(cfg, 0, sizeof(*cfg));
  cfg->device = 0;
  cfg->latent_dim = 0;
  cfg->optimizer = XF_OPTIMIZER_FTRL;  // server.h:24,28
  cfg->alpha = 5e-2f;                  // ftrl.h:17
  cfg->beta = 1.0f;                    // ftrl.h:18
  cfg->lambda1 = 5e-5f;                // ftrl.h:19
  cfg->lambda2 = 10.0f;                // ftrl.h:20
  cfg->learning_rate = 0.001f;         // sgd.h:16
  cfg->v_init = XF_VINIT_DEFAULT;
  cfg->seed = 0;
  cfg->capacity = 0;
  cfg->shard_index = 0;
  cfg->num_shards = 1;
  cfg->canonical_fm = 0;
  return XF_OK;
}

static uint64_t xf_pow2_at_least(uint64_t x) {
  uint64_t p = 1024;
  while (p < x) p <<= 1;
  return p;
}

int xf_table::alloc_table(uint64_t capacity) {
  capacity = xf_pow2_at_least(capacity);
  if (capacity > (1ull << 31)) {
    xf_set_error("table capacity %llu exceeds 2^31 slots", (unsigned long long)capacity);
    return XF_ERR_FULL;
  }
  const uint32_t stride = xf_row_stride(cfg.latent_dim, cfg.optimizer, cfg.canonical_fm);
  uint8_t* base = nullptr;
  XF_CUDA_TRY(cudaMalloc(&base, capacity * (uint64_t)stride));
  view.base = base;
  view.mask = capacity - 1;
  uint32_t lg = 0;
  while ((1ull << lg) < capacity) ++lg;
  view.log2cap = lg;
  view.stride = stride;
  // probing buckets = the rows that share one 128-byte line (table.cuh: xf_probe_slot); XFLOW_BUCKET_LOG2
  // overrides (0 = plain linear probing) for A/B measurements
  uint32_t bs = 0;
  while ((stride << (bs + 1)) <= 128u) ++bs;
  const char* be = getenv("XFLOW_BUCKET_LOG2");
  if (be && *be) bs = (uint32_t)std::min(std::max(atoi(be), 0), 4);
  if (bs + 4 > lg) bs = 0;
  view.bshift = bs;
  xf_launch_fill(view, stream);
  ++launches;
  XF_CUDA_TRY(cudaGetLastError());
  return XF_OK;
}

int xf_table::check_error() {
  int e = 0;
  XF_CUDA_TRY(cudaMemcpyAsync(&e, d_error, sizeof(int), cudaMemcpyDeviceToHost, stream));
  XF_CUDA_TRY(cudaStreamSynchronize(stream));
  if (e == 2) {
    xf_set_error("internal error: a row was never opened for the batch (lazy-update protocol)");
    return XF_ERR_STATE;
  }
  if (e) {
    xf_set_error("table probe sequence overflowed (table full)");
    return XF_ERR_FULL;
  }
  return XF_OK;
}

int xf_table::grow(uint64_t new_capacity) {
  XfTableView old = view;
  const int rc = alloc_table(new_capacity);  // on failure the old table (and its size counter) stay as they are
  if (rc != XF_OK) { view = old; return rc; }
  XF_CUDA_TRY(cudaMemsetAsync(d_size, 0, sizeof(unsigned long long), stream));  // the rehash re-counts every key
  xf_launch_rehash(old, view, stream);
  ++launches;
  XF_CUDA_TRY(cudaStreamSynchronize(stream));
  XF_CUDA_TRY(cudaFree(old.base));
  return XF_OK;
}

// Lazy tables number their batches (sharded: every (step, source) pair) with `seq`; rows_by_seq[seq] is the
// divisor of that batch's pending optimizer steps.  The array is a fixed ring: when the numbers run out,
// one sweep folds every pending step into its row (xf_k_flush_pending, stream-ordered, no host sync) and
// the numbering restarts at 1 — no reallocation, and the batch tag fits the 16 bits a lazy row has for it.
int xf_table::next_seq() {
  if ((size_t)seq + 1 >= rows_cap) {
    xf_launch_flush_pending(view, stream);
    ++launches;
    XF_CUDA_TRY(cudaGetLastError());
    seq = 0;
  }
  ++seq;
  return XF_OK;
}

// The sharded step takes S numbers per round and its pushes work from looks at the rows that were stashed BEFORE
// the first of them: a restart in the middle of the round would leave stashed tags of the old numbering next to
// batch numbers of the new one.  The restart is therefore taken before the round's Pull when fewer than n numbers
// are left.
int xf_table::reserve_seqs(int n) {
  if (!view.lazy) return XF_OK;
  if ((size_t)n + 2 > rows_cap) { xf_set_error("the batch-number ring (XFLOW_SEQ_RING = %zu) is too small for %d ranks", rows_cap, n); return XF_ERR_ARG; }
  if ((size_t)seq + (size_t)n + 1 < rows_cap) return XF_OK;
  xf_launch_flush_pending(view, stream);
  ++launches;
  XF_CUDA_TRY(cudaGetLastError());
  seq = 0;
  return XF_OK;
}

int xf_table::ensure_room(uint64_t incoming) {
  const uint64_t cap = view.mask + 1;
  // --- fast path: bound from the asynchronous read-backs, no host sync
  cum_incoming += incoming;
  if (h_size_ring) {
    for (int i = 0; i < 4; ++i)
      if (size_inflight[i] && cudaEventQuery(size_ev[i]) == cudaSuccess) {
        size_inflight[i] = false;
        if (size_issued_at[i] >= known_at) { known_at = size_issued_at[i]; known_size = h_size_ring[i]; }
      }
    cudaGetLastError();  // cudaErrorNotReady from the queries is not an error
    const uint64_t bound = known_size + (cum_incoming - known_at);
    const int slot = size_next;
    if (!size_inflight[slot]) {
      // reflects every kernel enqueued so far, i.e. everything but this step's own `incoming`
      if (cudaMemcpyAsync(h_size_ring + slot, d_size, sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream) ==
              cudaSuccess && cudaEventRecord(size_ev[slot], stream) == cudaSuccess) {
        size_inflight[slot] = true;
        size_issued_at[slot] = cum_incoming - incoming;
        size_next = (slot + 1) & 3;
      }
    }
    if (bound * 4 <= cap * 3) { size_bound = bound; return XF_OK; }  // load stays <= 0.75 even in the worst case
  }
  // --- slow path: read the exact size, grow to load <= 0.5 if needed
  size_bound += incoming;
  if (!h_size_ring && size_bound * 2 <= cap) return XF_OK;
  unsigned long long actual = 0;
  XF_CUDA_TRY(cudaMemcpyAsync(&actual, d_size, sizeof(actual), cudaMemcpyDeviceToHost, stream));
  XF_CUDA_TRY(cudaStreamSynchronize(stream));
  size_bound = actual + incoming;
  known_size = actual;
  known_at = cum_incoming - incoming;
  uint64_t want = cap;
  while (size_bound * 2 > want) want <<= 1;
  if (want != cap) XF_TRY(grow(want));
  return XF_OK;
}

XF_DLL int xf_table_create(xf_table** out, const xf_table_config* cfg) {
  if (!out || !cfg) { xf_set_error("null argument"); return XF_ERR_ARG; }
  if (cfg->latent_dim < 0 || cfg->latent_dim > 1024 || cfg->num_shards < 1 || cfg->shard_index < 0 ||
      cfg->shard_index >= cfg->num_shards || (cfg->optimizer != XF_OPTIMIZER_FTRL && cfg->optimizer != XF_OPTIMIZER_SGD)) {
    xf_set_error("bad table config");
    return XF_ERR_ARG;
  }
  if (cfg->canonical_fm) {
    const int K = cfg->latent_dim;
    if (!(K == 4 || K == 8 || K == 16 || K == 32 || K == 64 || K == 128) || cfg->num_shards != 1) {
      xf_set_error("canonical_fm needs latent_dim in {4, 8, 16, 32, 64, 128} and a single shard");
      return XF_ERR_ARG;
    }
  }
  XF_CUDA_TRY(cudaSetDevice(cfg->device));
  // L2 fetch granularity = one probing bucket (LR: 4 rows = one 128-byte line), so that the collision probes of
  // a bucket find the line the first probe fetched.  It costs DRAM read traffic (ncu, headline LR batch: 340 MB at
  // 32 B, 932 MB at 128 B, DRAM 33 % busy) and buys time: 0.447 ms against 0.522 ms per batch with 32-byte fetches
  // — the kernels are bound by the request rate, not by DRAM bytes (DESIGN.md section 6).  A hint: the driver may
  // ignore it.  XFLOW_L2_FETCH = 32 / 64 / 128 overrides.
  {
    int fetch = 128;
    const char* fe = getenv("XFLOW_L2_FETCH");
    if (fe && (atoi(fe) == 32 || atoi(fe) == 64 || atoi(fe) == 128)) fetch = atoi(fe);
    if (cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)fetch) != cudaSuccess) cudaGetLastError();
  }
  xf_table* t = new xf_table;
  t->cfg = *cfg;
  memset(&t->view, 0, sizeof(t->view));
  XF_CUDA_TRY(cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking));
  XF_CUDA_TRY(cudaMalloc(&t->d_size, sizeof(unsigned long long)));
  XF_CUDA_TRY(cudaMalloc(&t->d_error, sizeof(int)));
  XF_CUDA_TRY(cudaMemsetAsync(t->d_size, 0, sizeof(unsigned long long), t->stream));
  XF_CUDA_TRY(cudaMemsetAsync(t->d_error, 0, sizeof(int), t->stream));
  XfTableView& v = t->view;
  v.K = cfg->latent_dim;
  v.opt = cfg->optimizer == XF_OPTIMIZER_FTRL ? XF_OPT_FTRL : XF_OPT_SGD;
  v.alpha = cfg->alpha; v.beta = cfg->beta; v.lambda1 = cfg->lambda1; v.lambda2 = cfg->lambda2;
  v.learning_rate = cfg->learning_rate;
  v.seed = cfg->seed;
  v.v_const = 0.001f;  // sgd.h:68-70
  if (cfg->v_init == XF_VINIT_ZERO) v.v_init = XF_INIT_ZERO;
  else if (cfg->v_init == XF_VINIT_COUNTER) v.v_init = XF_INIT_COUNTER;
  else v.v_init = (v.opt == XF_OPT_FTRL) ? XF_INIT_COUNTER : XF_INIT_DEFAULT;
  v.size = t->d_size;
  v.error = t->d_error;
  v.canon = cfg->canonical_fm ? 1 : 0;
  XF_CUDA_TRY(cudaHostAlloc(&t->h_size_ring, 4 * sizeof(unsigned long long), cudaHostAllocDefault));
  for (int i = 0; i < 4; ++i) XF_CUDA_TRY(cudaEventCreateWithFlags(&t->size_ev[i], cudaEventDisableTiming));
  // K == 0 (LR) tables fold the optimizer step into the next touch of a row (step.cu); K > 0 tables
  // keep the separate optimizer kernel.  XFLOW_EAGER=1 forces the two-kernel path (A/B measurements).
  const char* eager = getenv("XFLOW_EAGER");
  v.lazy = (v.K == 0 && !(eager && *eager == '1')) ? 1 : 0;
  v.rows_by_seq = nullptr;
  if (v.lazy) {
    // XFLOW_SEQ_RING: ring size override (tests exercise the flush with a tiny ring)
    const char* ring = getenv("XFLOW_SEQ_RING");
    t->rows_cap = (ring && atoi(ring) >= 4 && atoi(ring) <= 65535) ? (size_t)atoi(ring) : (size_t)65535;  // tags are 16 bits
    XF_CUDA_TRY(cudaMalloc(&t->d_rows_by_seq, t->rows_cap * sizeof(uint32_t)));
    XF_CUDA_TRY(cudaMemsetAsync(t->d_rows_by_seq, 0, t->rows_cap * sizeof(uint32_t), t->stream));
    v.rows_by_seq = t->d_rows_by_seq;
  }
  int r = t->alloc_table(cfg->capacity ? cfg->capacity : (1ull << 20));
  if (r != XF_OK) { delete t; return r; }
  XF_CUDA_TRY(cudaStreamSynchronize(t->stream));
  *out = t;
  return XF_OK;
}

XF_DLL int xf_table_destroy(xf_table* t) {
  if (!t) return XF_OK;
  if (--t->refs > 0) return XF_OK;  // still used by a trainer; freed when the last user lets go
  cudaSetDevice(t->cfg.device);
  cudaStreamSynchronize(t->stream);
  if (t->view.base) cudaFree(t->view.base);
  cudaFree(t->d_size);
  cudaFree(t->d_error);
  if (t->d_rows_by_seq) cudaFree(t->d_rows_by_seq);
  if (t->h_size_ring) cudaFreeHost(t->h_size_ring);
  for (int i = 0; i < 4; ++i) if (t->size_ev[i]) cudaEventDestroy(t->size_ev[i]);
  t->s_keys.release(); t->s_slots.release(); t->s_w.release(); t->s_v.release();
  t->s_nw.release(); t->s_zw.release(); t->s_nv.release(); t->s_zv.release(); t->s_present.release();
  if (t->own_stream && t->stream) cudaStreamDestroy(t->stream);
  delete t;
  return XF_OK;
}

XF_DLL int xf_table_set_stream(xf_table* t, void* cuda_stream) {
  if (!t) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaStreamSynchronize(t->stream));
  if (t->own_stream && t->stream) cudaStreamDestroy(t->stream);
  if (cuda_stream) {
    t->stream = (cudaStream_t)cuda_stream;
    t->own_stream = false;
  } else {
    XF_CUDA_TRY(cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking));
    t->own_stream = true;
  }
  return XF_OK;
}

XF_DLL int xf_table_sync(xf_table* t) {
  if (!t) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaStreamSynchronize(t->stream));
  return t->check_error();
}

XF_DLL int xf_table_size(xf_table* t, uint64_t* n_keys) {
  if (!t || !n_keys) return XF_ERR_ARG;
  unsigned long long v = 0;
  XF_CUDA_TRY(cudaMemcpyAsync(&v, t->d_size, sizeof(v), cudaMemcpyDeviceToHost, t->stream));
  XF_CUDA_TRY(cudaStreamSynchronize(t->stream));
  *n_keys = v;
  return XF_OK;
}
XF_DLL int xf_table_capacity(xf_table* t, uint64_t* n_slots) {
  if (!t || !n_slots) return XF_ERR_ARG;
  *n_slots = t->view.mask + 1;
  return XF_OK;
}
XF_DLL int xf_table_row_bytes(xf_table* t, uint32_t* bytes) {
  if (!t || !bytes) return XF_ERR_ARG;
  *bytes = t->view.stride;
  return XF_OK;
}
XF_DLL int xf_table_latent_dim(xf_table* t, int* latent_dim) {
  if (!t || !latent_dim) return XF_ERR_ARG;
  *latent_dim = t->view.K;
  return XF_OK;
}
XF_DLL int xf_table_reserve(xf_table* t, uint64_t n_keys) {
  if (!t) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaSetDevice(t->cfg.device));
  uint64_t want = xf_pow2_at_least(n_keys * 2);
  if (want > t->view.mask + 1) XF_TRY(t->grow(want));
  return XF_OK;
}

XF_DLL int xf_table_pull_device(xf_table* t, const uint64_t* d_keys, uint64_t n, float* d_w_out, float* d_v_out) {
  if (!t || (!d_keys && n)) return XF_ERR_ARG;
  if (n == 0) return XF_OK;
  XF_TRY(t->ensure_room(n));
  XF_TRY(t->s_slots.ensure(n * sizeof(uint32_t)));
  xf_launch_probe(t->view, d_keys, n, true, t->s_slots.as<uint32_t>(), d_w_out, t->stream);
  ++t->launches;
  if (d_v_out && t->view.K > 0) {
    xf_launch_gather_v(t->view, t->s_slots.as<uint32_t>(), d_keys, n, d_v_out, t->stream);
    ++t->launches;
  }
  XF_CUDA_TRY(cudaGetLastError());
  return XF_OK;
}

XF_DLL int xf_table_push_device(xf_table* t, const uint64_t* d_keys, uint64_t n, const float* d_gw, const float* d_gv) {
  if (!t || (!d_keys && n)) return XF_ERR_ARG;
  if (n == 0) return XF_OK;
  if (d_gv && t->view.K == 0) d_gv = nullptr;
  XF_TRY(t->ensure_room(n));
  XF_TRY(t->s_slots.ensure(n * sizeof(uint32_t)));
  xf_launch_probe(t->view, d_keys, n, true, t->s_slots.as<uint32_t>(), nullptr, t->stream);
  xf_launch_update_pushed(t->view, t->s_slots.as<uint32_t>(), n, d_gw, d_gv, t->stream);
  t->launches += 2;
  XF_CUDA_TRY(cudaGetLastError());
  return XF_OK;
}

XF_DLL int xf_table_pull(xf_table* t, const uint64_t* keys, uint64_t n, float* w_out, float* v_out) {
  if (!t || (!keys && n)) return XF_ERR_ARG;
  std::lock_guard<std::mutex> host_lock(t->host_mu);
  if (n == 0) return XF_OK;
  XF_CUDA_TRY(cudaSetDevice(t->cfg.device));
  const int K = t->view.K;
  XF_TRY(t->s_keys.ensure(n * 8));
  XF_TRY(t->s_w.ensure(n * 4));
  if (v_out && K) XF_TRY(t->s_v.ensure(n * 4 * (size_t)K));
  XF_CUDA_TRY(cudaMemcpyAsync(t->s_keys.p, keys, n * 8, cudaMemcpyHostToDevice, t->stream));
  XF_TRY(xf_table_pull_device(t, t->s_keys.as<uint64_t>(), n, t->s_w.as<float>(), (v_out && K) ? t->s_v.as<float>() : nullptr));
  if (w_out) XF_CUDA_TRY(cudaMemcpyAsync(w_out, t->s_w.p, n * 4, cudaMemcpyDeviceToHost, t->stream));
  if (v_out && K) XF_CUDA_TRY(cudaMemcpyAsync(v_out, t->s_v.p, n * 4 * (size_t)K, cudaMemcpyDeviceToHost, t->stream));
  return xf_table_sync(t);
}

// KVWorker::Push takes sorted, unique keys (ps-lite kv_app.h: "keys must be unique and sorted in increasing order").
// The update kernel gives every list entry its own warp lanes: the same key twice would be two unordered
// read-modify-writes of one row.  Sorted input costs one pass; anything else is checked on a sorted copy.
static int xf_check_unique_keys(const uint64_t* keys, uint64_t n) {
  bool increasing = true;
  for (uint64_t i = 1; i < n; ++i) {
    if (keys[i] > keys[i - 1]) continue;
    if (keys[i] == keys[i - 1]) { xf_set_error("push: key %llu occurs more than once", (unsigned long long)keys[i]); return XF_ERR_ARG; }
    increasing = false;
    break;
  }
  if (increasing) return XF_OK;
  try {
    std::vector<uint64_t> c(keys, keys + n);
    std::sort(c.begin(), c.end());
    const auto dup = std::adjacent_find(c.begin(), c.end());
    if (dup != c.end()) { xf_set_error("push: key %llu occurs more than once", (unsigned long long)*dup); return XF_ERR_ARG; }
  } catch (const std::exception&) {
    xf_set_error("push: out of host memory while checking %llu keys", (unsigned long long)n);
    return XF_ERR_IO;
  }
  return XF_OK;
}

XF_DLL int xf_table_push(xf_table* t, const uint64_t* keys, uint64_t n, const float* gw, const float* gv) {
  if (!t || (!keys && n)) return XF_ERR_ARG;
  std::lock_guard<std::mutex> host_lock(t->host_mu);
  if (n == 0) return XF_OK;
  XF_TRY(xf_check_unique_keys(keys, n));
  XF_CUDA_TRY(cudaSetDevice(t->cfg.device));
  const int K = t->view.K;
  XF_TRY(t->s_keys.ensure(n * 8));
  XF_CUDA_TRY(cudaMemcpyAsync(t->s_keys.p, keys, n * 8, cudaMemcpyHostToDevice, t->stream));
  if (gw) {
    XF_TRY(t->s_w.ensure(n * 4));
    XF_CUDA_TRY(cudaMemcpyAsync(t->s_w.p, gw, n * 4, cudaMemcpyHostToDevice, t->stream));
  }
  if (gv && K) {
    XF_TRY(t->s_v.ensure(n * 4 * (size_t)K));
    XF_CUDA_TRY(cudaMemcpyAsync(t->s_v.p, gv, n * 4 * (size_t)K, cudaMemcpyHostToDevice, t->stream));
  }
  XF_TRY(xf_table_push_device(t, t->s_keys.as<uint64_t>(), n, gw ? t->s_w.as<float>() : nullptr,
                              (gv && K) ? t->s_v.as<float>() : nullptr));
  return xf_table_sync(t);
}

static int xf_h2d_opt(XfDevBuf& b, const float* src, size_t count, cudaStream_t st, float** dptr) {
  *dptr = nullptr;
  if (!src || count == 0) return XF_OK;
  XF_TRY(b.ensure(count * 4));
  XF_CUDA_TRY(cudaMemcpyAsync(b.p, src, count * 4, cudaMemcpyHostToDevice, st));
  *dptr = b.as<float>();
  return XF_OK;
}

XF_DLL int xf_table_import(xf_table* t, const uint64_t* keys, uint64_t n, const float* w, const float* nw,
                           const float* zw, const float* v, const float* nv, const float* zv) {
  if (!t || (!keys && n)) return XF_ERR_ARG;
  std::lock_guard<std::mutex> host_lock(t->host_mu);
  if (n == 0) return XF_OK;
  XF_CUDA_TRY(cudaSetDevice(t->cfg.device));
  const size_t K = (size_t)t->view.K;
  XF_TRY(t->ensure_room(n));
  XF_TRY(t->s_keys.ensure(n * 8));
  XF_TRY(t->s_slots.ensure(n * 4));
  XF_CUDA_TRY(cudaMemcpyAsync(t->s_keys.p, keys, n * 8, cudaMemcpyHostToDevice, t->stream));
  float *dw, *dnw, *dzw, *dv, *dnv, *dzv;
  XF_TRY(xf_h2d_opt(t->s_w, w, n, t->stream, &dw));
  XF_TRY(xf_h2d_opt(t->s_nw, nw, n, t->stream, &dnw));
  XF_TRY(xf_h2d_opt(t->s_zw, zw, n, t->stream, &dzw));
  XF_TRY(xf_h2d_opt(t->s_v, K ? v : nullptr, n * K, t->stream, &dv));
  XF_TRY(xf_h2d_opt(t->s_nv, K ? nv : nullptr, n * K, t->stream, &dnv));
  XF_TRY(xf_h2d_opt(t->s_zv, K ? zv : nullptr, n * K, t->stream, &dzv));
  xf_launch_probe(t->view, t->s_keys.as<uint64_t>(), n, true, t->s_slots.as<uint32_t>(), nullptr, t->stream);
  xf_launch_import(t->view, t->s_slots.as<uint32_t>(), n, dw, dnw, dzw, dv, dnv, dzv, t->stream);
  t->launches += 2;
  XF_CUDA_TRY(cudaGetLastError());
  return xf_table_sync(t);
}

XF_DLL int xf_table_export(xf_table* t, const uint64_t* keys, uint64_t n, float* w, float* nw, float* zw,
                           float* v, float* nv, float* zv, uint8_t* present) {
  if (!t || (!keys && n)) return XF_ERR_ARG;
  std::lock_guard<std::mutex> host_lock(t->host_mu);
  if (n == 0) return XF_OK;
  XF_CUDA_TRY(cudaSetDevice(t->cfg.device));
  const size_t K = (size_t)t->view.K;
  XF_TRY(t->s_keys.ensure(n * 8));
  XF_TRY(t->s_slots.ensure(n * 4));
  XF_TRY(t->s_w.ensure(n * 4));
  XF_TRY(t->s_nw.ensure(n * 4));
  XF_TRY(t->s_zw.ensure(n * 4));
  XF_TRY(t->s_present.ensure(n));
  if (K) {
    XF_TRY(t->s_v.ensure(n * K * 4));
    XF_TRY(t->s_nv.ensure(n * K * 4));
    XF_TRY(t->s_zv.ensure(n * K * 4));
  }
  XF_CUDA_TRY(cudaMemcpyAsync(t->s_keys.p, keys, n * 8, cudaMemcpyHostToDevice, t->stream));
  xf_launch_probe(t->view, t->s_keys.as<uint64_t>(), n, false, t->s_slots.as<uint32_t>(), nullptr, t->stream);
  xf_launch_export(t->view, t->s_slots.as<uint32_t>(), t->s_keys.as<uint64_t>(), n, t->s_w.as<float>(),
                   t->s_nw.as<float>(), t->s_zw.as<float>(), K ? t->s_v.as<float>() : nullptr,
                   K ? t->s_nv.as<float>() : nullptr, K ? t->s_zv.as<float>() : nullptr,
                   t->s_present.as<uint8_t>(), t->stream);
  t->launches += 2;
  XF_CUDA_TRY(cudaGetLastError());
  if (w) XF_CUDA_TRY(cudaMemcpyAsync(w, t->s_w.p, n * 4, cudaMemcpyDeviceToHost, t->stream));
  if (nw) XF_CUDA_TRY(cudaMemcpyAsync(nw, t->s_nw.p, n * 4, cudaMemcpyDeviceToHost, t->stream));
  if (zw) XF_CUDA_TRY(cudaMemcpyAsync(zw, t->s_zw.p, n * 4, cudaMemcpyDeviceToHost, t->stream));
  if (present) XF_CUDA_TRY(cudaMemcpyAsync(present, t->s_present.p, n, cudaMemcpyDeviceToHost, t->stream));
  if (K && v) XF_CUDA_TRY(cudaMemcpyAsync(v, t->s_v.p, n * K * 4, cudaMemcpyDeviceToHost, t->stream));
  if (K && nv) XF_CUDA_TRY(cudaMemcpyAsync(nv, t->s_nv.p, n * K * 4, cudaMemcpyDeviceToHost, t->stream));
  if (K && zv) XF_CUDA_TRY(cudaMemcpyAsync(zv, t->s_zv.p, n * K * 4, cudaMemcpyDeviceToHost, t->stream));
  return xf_table_sync(t);
}

XF_DLL int xf_table_list_keys(xf_table* t, uint64_t* keys_out, uint64_t max_keys, uint64_t* n_out) {
  if (!t || !n_out) return XF_ERR_ARG;
  std::lock_guard<std::mutex> host_lock(t->host_mu);
  XF_CUDA_TRY(cudaSetDevice(t->cfg.device));
  XF_TRY(t->s_keys.ensure(std::max<uint64_t>(max_keys, 1) * 8));
  unsigned long long* d_count = nullptr;
  XF_CUDA_TRY(cudaMalloc(&d_count, 8));
  XF_CUDA_TRY(cudaMemsetAsync(d_count, 0, 8, t->stream));
  xf_launch_list_keys(t->view, t->s_keys.as<uint64_t>(), d_count, max_keys, t->stream);
  ++t->launches;
  unsigned long long cnt = 0;
  XF_CUDA_TRY(cudaMemcpyAsync(&cnt, d_count, 8, cudaMemcpyDeviceToHost, t->stream));
  XF_CUDA_TRY(cudaStreamSynchronize(t->stream));
  cudaFree(d_count);
  uint64_t ncopy = std::min<uint64_t>(cnt, max_keys);
  if (keys_out && ncopy) XF_CUDA_TRY(cudaMemcpy(keys_out, t->s_keys.p, ncopy * 8, cudaMemcpyDeviceToHost));
  *n_out = cnt;
  return XF_OK;
}

// checkpoint file: "XFTB" u64 n, u32 K, u32 has_nz, keys[n], w[n], (nw,zw), v[n*K], (nv,zv), present[n]
XF_DLL int xf_table_save(xf_table* t, const char* path) {
  if (!t || !path) return XF_ERR_ARG;
  uint64_t n = 0;
  XF_TRY(xf_table_size(t, &n));
  std::vector<uint64_t> keys(n ? n : 1);
  uint64_t got = 0;
  XF_TRY(xf_table_list_keys(t, keys.data(), n, &got));
  n = std::min(n, got);
  std::sort(keys.begin(), keys.begin() + n);
  const size_t K = (size_t)t->view.K;
  const uint32_t has_nz = t->view.opt == XF_OPT_FTRL ? 1 : 0;
  std::vector<float> w(n), nw(n), zw(n), v(n * K), nv(n * K), zv(n * K);
  std::vector<uint8_t> present(n);
  XF_TRY(xf_table_export(t, keys.data(), n, w.data(), nw.data(), zw.data(), K ? v.data() : nullptr,
                         K ? nv.data() : nullptr, K ? zv.data() : nullptr, present.data()));
  // written under a temporary name and renamed: a reader never sees a half-written checkpoint, and a
  // short write (ENOSPC ...) is an error, not a silently truncated file
  const std::string tmp = std::string(path) + ".tmp";
  FILE* f = fopen(tmp.c_str(), "wb");
  if (!f) { xf_set_error("cannot open %s for writing", tmp.c_str()); return XF_ERR_IO; }
  uint32_t K32 = (uint32_t)K;
  bool ok = fwrite("XFTB", 1, 4, f) == 4 && fwrite(&n, 8, 1, f) == 1 && fwrite(&K32, 4, 1, f) == 1 && fwrite(&has_nz, 4, 1, f) == 1;
  auto put = [&](const void* p, size_t sz, size_t cnt) { if (ok && cnt) ok = fwrite(p, sz, cnt, f) == cnt; };
  put(keys.data(), 8, n);
  put(w.data(), 4, n);
  if (has_nz) { put(nw.data(), 4, n); put(zw.data(), 4, n); }
  put(v.data(), 4, n * K);
  if (has_nz) { put(nv.data(), 4, n * K); put(zv.data(), 4, n * K); }
  put(present.data(), 1, n);
  if (fclose(f) != 0) ok = false;
  if (!ok || rename(tmp.c_str(), path) != 0) {
    remove(tmp.c_str());
    xf_set_error("write to %s failed", path);
    return XF_ERR_IO;
  }
  return XF_OK;
}

// text model dump (SURVEY.md section 8f-3; the reference has none): one line per key, sorted by key,
//   <key>\t<w>[\t<v_0> ... <v_{K-1}>]      weights only, %.9g (round-trips a float)
// nonzero_only drops keys whose w (and every v) is exactly 0 — what FTRL's L1 leaves behind.
XF_DLL int xf_table_dump_text(xf_table* t, const char* path, int nonzero_only, uint64_t* written) {
  if (!t || !path) return XF_ERR_ARG;
  uint64_t n = 0;
  XF_TRY(xf_table_size(t, &n));
  std::vector<uint64_t> keys(n ? n : 1);
  uint64_t got = 0;
  XF_TRY(xf_table_list_keys(t, keys.data(), n, &got));
  n = std::min(n, got);
  std::sort(keys.begin(), keys.begin() + n);
  const size_t K = (size_t)t->view.K;
  std::vector<float> w(n), v(n * K);
  XF_TRY(xf_table_export(t, keys.data(), n, w.data(), nullptr, nullptr, K ? v.data() : nullptr, nullptr, nullptr,
                         nullptr));
  FILE* f = fopen(path, "w");
  if (!f) { xf_set_error("cannot open %s for writing", path); return XF_ERR_IO; }
  uint64_t lines = 0;
  for (uint64_t i = 0; i < n; ++i) {
    if (nonzero_only) {
      bool any = w[i] != 0.0f;
      for (size_t k = 0; k < K && !any; ++k) any = v[i * K + k] != 0.0f;
      if (!any) continue;
    }
    fprintf(f, "%llu\t%.9g", (unsigned long long)keys[i], (double)w[i]);
    for (size_t k = 0; k < K; ++k) fprintf(f, "%c%.9g", k ? ' ' : '\t', (double)v[i * K + k]);
    fputc('\n', f);
    ++lines;
  }
  if (fclose(f) != 0) { xf_set_error("write to %s failed", path); return XF_ERR_IO; }
  if (written) *written = lines;
  return XF_OK;
}

XF_DLL int xf_table_load(xf_table* t, const char* path) {
  if (!t || !path) return XF_ERR_ARG;
  FILE* f = fopen(path, "rb");
  if (!f) { xf_set_error("cannot open %s", path); return XF_ERR_IO; }
  char magic[4];
  uint64_t n = 0;
  uint32_t K32 = 0, has_nz = 0;
  bool ok = fread(magic, 1, 4, f) == 4 && memcmp(magic, "XFTB", 4) == 0 && fread(&n, 8, 1, f) == 1 &&
            fread(&K32, 4, 1, f) == 1 && fread(&has_nz, 4, 1, f) == 1;
  if (!ok || (int)K32 != t->view.K) {
    fclose(f);
    xf_set_error("bad checkpoint %s (K=%u, table K=%d)", path, K32, t->view.K);
    return XF_ERR_IO;
  }
  const size_t K = K32;
  // the header's key count must agree with the file's size before anything is allocated from it
  {
    const long here = ftell(f);
    fseek(f, 0, SEEK_END);
    const long fsz = ftell(f);
    fseek(f, here, SEEK_SET);
    const unsigned long long per = 8ull + 4ull * (has_nz ? 3 : 1) + 4ull * K * (has_nz ? 3 : 1) + 1ull;
    if (here < 0 || fsz < here || n > (unsigned long long)(fsz - here) / per || (unsigned long long)(fsz - here) != n * per) {
      fclose(f);
      xf_set_error("corrupt or truncated checkpoint %s (%llu keys announced, %ld bytes of payload)", path, (unsigned long long)n, fsz - here);
      return XF_ERR_IO;
    }
  }
  std::vector<uint64_t> keys;
  std::vector<float> w, nw, zw, v, nv, zv;
  try {
    keys.resize(n); w.resize(n); nw.resize(n); zw.resize(n); v.resize(n * K); nv.resize(n * K); zv.resize(n * K);
  } catch (const std::exception&) {
    fclose(f);
    xf_set_error("checkpoint %s: not enough host memory for %llu keys", path, (unsigned long long)n);
    return XF_ERR_IO;
  }
  ok = fread(keys.data(), 8, n, f) == n && fread(w.data(), 4, n, f) == n;
  if (ok && has_nz) ok = fread(nw.data(), 4, n, f) == n && fread(zw.data(), 4, n, f) == n;
  if (ok && K) ok = fread(v.data(), 4, n * K, f) == n * K;
  if (ok && K && has_nz) ok = fread(nv.data(), 4, n * K, f) == n * K && fread(zv.data(), 4, n * K, f) == n * K;
  fclose(f);
  if (!ok) { xf_set_error("truncated checkpoint %s", path); return XF_ERR_IO; }
  return xf_table_import(t, keys.data(), n, w.data(), has_nz ? nw.data() : nullptr, has_nz ? zw.data() : nullptr,
                         K ? v.data() : nullptr, (K && has_nz) ? nv.data() : nullptr,
                         (K && has_nz) ? zv.data() : nullptr);
}

XF_DLL int xf_shard_of(uint64_t key, int num_shards) {
  if (num_shards <= 1) return 0;
  const uint64_t width = 0xFFFFFFFFFFFFFFFFull / (uint64_t)num_shards;  // postoffice.cc:138-140
  const uint64_t s = key / width;
  return (int)(s < (uint64_t)num_shards ? s : (uint64_t)num_shards - 1);
}

// -------------------------------------------------------------------------------------------------
// trainer
// -------------------------------------------------------------------------------------------------
XF_DLL int xf_trainer_create(xf_trainer** out, xf_table* table, xf_comm* comm, const xf_trainer_config* cfg) {
  if (!out || !table || !cfg) { xf_set_error("null argument"); return XF_ERR_ARG; }
  if (cfg->model == XF_MODEL_FM && table->view.K <= 0) { xf_set_error("FM needs latent_dim > 0"); return XF_ERR_ARG; }
  if (cfg->model == XF_MODEL_FM_CANONICAL && (!table->view.canon || comm)) {
    xf_set_error("XF_MODEL_FM_CANONICAL needs a table created with canonical_fm = 1 and no comm");
    return XF_ERR_ARG;
  }
  if (cfg->model == XF_MODEL_MVM && (!table->view.canon || comm || table->view.K > 32)) {
    xf_set_error("XF_MODEL_MVM needs a table created with canonical_fm = 1, latent_dim <= 32 and no comm");
    return XF_ERR_ARG;
  }
  if (cfg->model != XF_MODEL_FM_CANONICAL && cfg->model != XF_MODEL_MVM && table->view.canon) {
    xf_set_error("canonical tables serve XF_MODEL_FM_CANONICAL and XF_MODEL_MVM only");
    return XF_ERR_ARG;
  }
  if (cfg->model == XF_MODEL_LR && table->view.K != 0) { xf_set_error("LR needs latent_dim == 0"); return XF_ERR_ARG; }
  if (cfg->max_rows == 0 || cfg->max_nnz == 0) { xf_set_error("max_rows/max_nnz must be > 0"); return XF_ERR_ARG; }
  XF_CUDA_TRY(cudaSetDevice(table->cfg.device));
  xf_trainer* tr = new xf_trainer;
  tr->table = table;
  tr->comm = comm;
  tr->cfg = *cfg;
  XF_CUDA_TRY(cudaStreamCreateWithFlags(&tr->copy_stream, cudaStreamNonBlocking));
  XF_CUDA_TRY(cudaStreamCreateWithFlags(&tr->ing_stream, cudaStreamNonBlocking));
  XF_CUDA_TRY(cudaStreamCreateWithFlags(&tr->ing_copy_stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    XF_CUDA_TRY(cudaEventCreateWithFlags(&tr->ing[i].copied, cudaEventDisableTiming));
    XF_CUDA_TRY(cudaEventCreateWithFlags(&tr->ing[i].parsed, cudaEventDisableTiming));
    XF_CUDA_TRY(cudaEventCreateWithFlags(&tr->ing[i].consumed, cudaEventDisableTiming));
    XF_CUDA_TRY(cudaHostAlloc(&tr->ing[i].h_totals, 16, cudaHostAllocDefault));
    XF_CUDA_TRY(cudaEventCreateWithFlags(&tr->buf[i].copied, cudaEventDisableTiming));
    XF_CUDA_TRY(cudaEventCreateWithFlags(&tr->buf[i].consumed, cudaEventDisableTiming));
    XF_CUDA_TRY(cudaEventCreateWithFlags(&tr->buf[i].staged, cudaEventDisableTiming));
  }
  // one slot per token position + the FM hot-key cache's flush positions (grid x NC, see step.cu)
  XF_TRY(tr->touched.ensure(((size_t)cfg->max_nnz + xf_step_touched_extra(table->view.K, (int)cfg->max_rows)) * 4));
  XF_TRY(tr->loss.ensure((size_t)cfg->max_rows * 4));
  XF_TRY(tr->pctr.ensure((size_t)cfg->max_rows * 4));
  XF_CUDA_TRY(cudaMalloc(&tr->d_unique_total, sizeof(unsigned long long)));
  XF_CUDA_TRY(cudaMalloc(&tr->d_abs_loss, 2 * sizeof(float)));
  XF_CUDA_TRY(cudaHostAlloc(&tr->h_abs_loss, 2 * sizeof(float), cudaHostAllocDefault));
  XF_CUDA_TRY(cudaMemsetAsync(tr->d_unique_total, 0, sizeof(unsigned long long), table->stream));
  XF_CUDA_TRY(cudaMemsetAsync(tr->d_abs_loss, 0, 2 * sizeof(float), table->stream));
  XF_CUDA_TRY(cudaStreamSynchronize(table->stream));
  // XFLOW_MG_FORCE=1: run the sharded step even with a one-rank communicator (profiling the owner / worker
  // kernels of comm.cu under ncu, which cannot wrap a multi-rank command)
  const char* force_mg = getenv("XFLOW_MG_FORCE");
  if (comm && (xf_comm_nranks(comm) > 1 || (force_mg && *force_mg == '1'))) {
    if (table->cfg.num_shards != xf_comm_nranks(comm) || table->cfg.shard_index != xf_comm_rank(comm)) {
      xf_set_error("table shard (%d of %d) does not match comm rank (%d of %d)", table->cfg.shard_index,
                   table->cfg.num_shards, xf_comm_rank(comm), xf_comm_nranks(comm));
      delete tr;
      return XF_ERR_ARG;
    }
    int r = xf_mg_create(tr);
    if (r != XF_OK) { delete tr; return r; }
  }
  ++table->refs;
  *out = tr;
  return XF_OK;
}

XF_DLL int xf_trainer_destroy(xf_trainer* tr) {
  if (!tr) return XF_OK;
  cudaSetDevice(tr->table->cfg.device);
  cudaStreamSynchronize(tr->table->stream);
  cudaStreamSynchronize(tr->copy_stream);
  if (tr->mg) xf_mg_destroy(tr);
  for (int i = 0; i < 2; ++i) {
    XfBatchBuf& b = tr->buf[i];
    b.row_ptr.release(); b.keys.release(); b.labels.release(); b.ids.release(); b.vals.release(); b.fields.release();
    b.h_row_ptr.release(); b.h_keys.release(); b.h_labels.release();
    cudaEventDestroy(b.copied); cudaEventDestroy(b.consumed); cudaEventDestroy(b.staged);
  }
  tr->touched.release(); tr->loss.release(); tr->pctr.release();
  cudaStreamSynchronize(tr->ing_copy_stream);
  cudaStreamSynchronize(tr->ing_stream);
  for (int i = 0; i < 2; ++i) {
    xf_trainer::IngestSet& g = tr->ing[i];
    if (g.copied) cudaEventDestroy(g.copied);
    g.text.release(); g.row_ptr.release(); g.keys.release(); g.labels.release(); g.totals.release(); g.stage.release();
    if (g.h_totals) cudaFreeHost(g.h_totals);
    if (g.parsed) cudaEventDestroy(g.parsed);
    if (g.consumed) cudaEventDestroy(g.consumed);
  }
  tr->ing_scratch.release();
  cudaStreamDestroy(tr->ing_stream);
  cudaStreamDestroy(tr->ing_copy_stream);
  cudaFree(tr->d_unique_total); cudaFree(tr->d_abs_loss);
  cudaFreeHost(tr->h_abs_loss);
  cudaStreamDestroy(tr->copy_stream);
  for (cudaEvent_t e : tr->prof_events) cudaEventDestroy(e);
  xf_table* table = tr->table;
  delete tr;
  return xf_table_destroy(table);  // drop the trainer's reference
}

static int xf_check_batch(xf_trainer* tr, uint32_t rows, uint32_t nnz) {
  if (rows > tr->cfg.max_rows || nnz > tr->cfg.max_nnz) {
    xf_set_error("batch (%u rows, %u tokens) exceeds trainer limits (%u, %u)", rows, nnz, tr->cfg.max_rows,
                 tr->cfg.max_nnz);
    return XF_ERR_ARG;
  }
  return XF_OK;
}

// One batch as the step kernels read it: CSR arrays (keys, or u32 ids that are hashed to keys on the device), the
// canonical FM's feature values and the multi-view machine's field ids.  Host or device pointers, as the user says.
struct XfBatch {
  const uint32_t* row_ptr = nullptr;
  const uint64_t* keys = nullptr;
  const uint8_t* labels = nullptr;
  uint32_t rows = 0, nnz = 0;
  const float* vals = nullptr;
  const uint8_t* fields = nullptr;
  const uint32_t* ids = nullptr;
};

static void xf_count_step(xf_trainer* tr, uint32_t rows, uint32_t nnz) {
  ++tr->n_steps;
  tr->n_rows += rows;
  tr->n_nnz += nnz;
  tr->last_rows = rows;
}

// the step proper, on a device-resident batch; mode 0 = train, 1 = predict
static int xf_step_device_impl(xf_trainer* tr, const XfBatch& d, int mode, float* d_abs) {
  xf_table* t = tr->table;
  const uint32_t rows = d.rows, nnz = d.nnz;
  if (rows == 0 && !tr->mg) return XF_OK;     // sharded: an empty batch still takes part in the exchange
  if (!tr->mg) XF_TRY(t->ensure_room(nnz));  // the sharded path sizes the shard from what it receives
  cudaStream_t st = t->stream;
  const bool prof = tr->profile && mode == 0;
  cudaEvent_t* pe = nullptr;
  if (tr->mg && !prof) return xf_mg_step(tr, d.row_ptr, d.keys, d.labels, rows, nnz, mode, d_abs, nullptr);
  if (prof) {
    if (tr->prof_used + 4 > tr->prof_events.size()) {
      size_t old = tr->prof_events.size();
      tr->prof_events.resize(old + 4 * 256);
      for (size_t i = old; i < tr->prof_events.size(); ++i) XF_CUDA_TRY(cudaEventCreate(&tr->prof_events[i]));
    }
    pe = &tr->prof_events[tr->prof_used];
    tr->prof_used += 4;
    if (tr->mg) return xf_mg_step(tr, d.row_ptr, d.keys, d.labels, rows, nnz, mode, d_abs, pe);
    XF_CUDA_TRY(cudaEventRecord(pe[0], st));
  }
  // per-row outputs: the residuals when the trainer keeps them, the predictions of a forward pass
  float* loss = (mode == 0 && tr->cfg.keep_loss) ? tr->loss.as<float>() : nullptr;
  float* pctr = mode == 1 ? tr->pctr.as<float>() : nullptr;
  if (t->view.lazy) {
    // one kernel: the optimizer step of earlier batches is folded in as rows are touched
    if (mode == 0) XF_TRY(t->next_seq());
    xf_launch_step_lr_lazy(t->view, d.row_ptr, d.keys, d.labels, (int)rows, mode, t->seq, t->d_rows_by_seq, loss, pctr,
                           d_abs, tr->d_unique_total, st);
    ++tr->launches;
    if (prof) {
      XF_CUDA_TRY(cudaEventRecord(pe[1], st));
      XF_CUDA_TRY(cudaEventRecord(pe[2], st));
      XF_CUDA_TRY(cudaEventRecord(pe[3], st));
    }
    XF_CUDA_TRY(cudaGetLastError());
    return XF_OK;
  }
  const bool mvm = tr->cfg.model == XF_MODEL_MVM;
  const bool canon = tr->cfg.model == XF_MODEL_FM_CANONICAL || mvm;
  if (mvm && !d.fields && nnz) { xf_set_error("XF_MODEL_MVM steps need the tokens' field ids (xf_trainer_step_host_fields)"); return XF_ERR_ARG; }
  const uint32_t extra = canon ? 0u : xf_step_touched_extra(t->view.K, (int)rows);
  XF_TRY(tr->touched.ensure(((size_t)nnz + extra) * 4));
  if (mvm)
    xf_launch_step_mvm(t->view, d.row_ptr, d.keys, d.fields, d.vals, d.labels, (int)rows, mode, tr->touched.as<uint32_t>(),
                       loss, pctr, d_abs, st);
  else if (canon)
    xf_launch_step_fmc(t->view, d.row_ptr, d.keys, d.vals, d.labels, (int)rows, mode, tr->touched.as<uint32_t>(), loss,
                       pctr, d_abs, st);
  else
    xf_launch_step(t->view, d.row_ptr, d.keys, d.labels, (int)rows, mode, tr->touched.as<uint32_t>(), nnz, loss, pctr,
                   d_abs, st);
  ++tr->launches;
  if (prof) {
    XF_CUDA_TRY(cudaEventRecord(pe[1], st));
    XF_CUDA_TRY(cudaEventRecord(pe[2], st));
  }
  if (mode == 0) {
    // Push + server-side optimizer: one FTRL/SGD step per touched key with g / rows
    xf_launch_update_touched(t->view, tr->touched.as<uint32_t>(), (uint64_t)nnz + extra, (double)rows,
                             tr->d_unique_total, st);
    ++tr->launches;
  }
  if (prof) XF_CUDA_TRY(cudaEventRecord(pe[3], st));
  XF_CUDA_TRY(cudaGetLastError());
  return XF_OK;
}

// A training step on a batch the caller keeps on the device: nothing to upload, so no buffer set, no cudaSetDevice
// and no `consumed` event.  An empty batch is counted as a step.
static int xf_step_resident(xf_trainer* tr, const XfBatch& d) {
  XF_TRY(xf_check_batch(tr, d.rows, d.nnz));
  XF_TRY(xf_step_device_impl(tr, d, 0, nullptr));
  xf_count_step(tr, d.rows, d.nnz);
  return XF_OK;
}

static bool xf_is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// stage one host array into buffer set `b` (pinned source: DMA directly; pageable: copy through the
// set's pinned staging) and enqueue the H2D on the copy stream
static int xf_stage(xf_trainer* tr, XfDevBuf& dev, XfPinBuf& pin, const void* src, size_t bytes) {
  if (bytes == 0) return XF_OK;
  XF_TRY(dev.ensure(bytes));
  const void* from = src;
  if (!xf_is_pinned(src)) {
    XF_TRY(pin.ensure(bytes));
    memcpy(pin.p, src, bytes);
    from = pin.p;
  }
  XF_CUDA_TRY(cudaMemcpyAsync(dev.p, from, bytes, cudaMemcpyHostToDevice, tr->copy_stream));
  return XF_OK;
}

// Uploads host batch `h` into buffer set `b` and describes the device copy in *d.  Keys (and labels) go through
// xf_stage on the copy stream; u32 ids come from page-locked memory, are copied directly and hashed to keys on the
// copy stream (4 B/token instead of 8 B); values and field ids are plain copies on the table stream (a small part of
// a batch).  Field ids the MVM kernel has no room for are refused here, before any kernel runs.
static int xf_upload(xf_trainer* tr, XfBatchBuf& b, const XfBatch& h, XfBatch* d) {
  const size_t rp_bytes = ((size_t)h.rows + 1) * 4;
  // the device buffers of this set may still be read by the step issued two calls ago
  XF_CUDA_TRY(cudaStreamWaitEvent(tr->copy_stream, b.consumed, 0));
  if (h.ids) {
    XF_TRY(b.row_ptr.ensure(rp_bytes));
    XF_TRY(b.ids.ensure((size_t)h.nnz * 4));
    XF_TRY(b.keys.ensure((size_t)h.nnz * 8));
    XF_TRY(b.labels.ensure(h.rows));
    XF_CUDA_TRY(cudaMemcpyAsync(b.row_ptr.p, h.row_ptr, rp_bytes, cudaMemcpyHostToDevice, tr->copy_stream));
    XF_CUDA_TRY(cudaMemcpyAsync(b.ids.p, h.ids, (size_t)h.nnz * 4, cudaMemcpyHostToDevice, tr->copy_stream));
    XF_CUDA_TRY(cudaMemcpyAsync(b.labels.p, h.labels, h.rows, cudaMemcpyHostToDevice, tr->copy_stream));
    XF_TRY(xf_launch_hash_ids(b.ids.as<uint32_t>(), h.nnz, b.keys.as<uint64_t>(), tr->copy_stream));
    ++tr->launches;
  } else {
    // its pinned staging may still be the source of that step's H2D
    XF_CUDA_TRY(cudaEventSynchronize(b.staged));
    XF_TRY(xf_stage(tr, b.row_ptr, b.h_row_ptr, h.row_ptr, rp_bytes));
    XF_TRY(xf_stage(tr, b.keys, b.h_keys, h.keys, (size_t)h.nnz * 8));
    if (h.labels) XF_TRY(xf_stage(tr, b.labels, b.h_labels, h.labels, (size_t)h.rows));
    XF_CUDA_TRY(cudaEventRecord(b.staged, tr->copy_stream));
  }
  XF_CUDA_TRY(cudaEventRecord(b.copied, tr->copy_stream));
  XF_CUDA_TRY(cudaStreamWaitEvent(tr->table->stream, b.copied, 0));
  tr->input_ready = b.copied;  // the sharded path starts its dedup on another stream
  if (!h.labels) XF_TRY(b.labels.ensure((size_t)h.rows + 1));  // unused by mode 1 but must be a valid pointer
  *d = XfBatch{b.row_ptr.as<uint32_t>(), b.keys.as<uint64_t>(), b.labels.as<uint8_t>(), h.rows, h.nnz};
  if (h.vals && h.nnz) {
    XF_TRY(b.vals.ensure((size_t)h.nnz * 4));
    XF_CUDA_TRY(cudaMemcpyAsync(b.vals.p, h.vals, (size_t)h.nnz * 4, cudaMemcpyHostToDevice, tr->table->stream));
    d->vals = b.vals.as<float>();
  }
  if (h.fields && h.nnz) {
    for (uint32_t j = 0; j < h.nnz; ++j)
      if (h.fields[j] >= XF_MVM_FIELDS) { xf_set_error("field id %u of token %u: XF_MODEL_MVM takes field ids below %d", (unsigned)h.fields[j], j, XF_MVM_FIELDS); return XF_ERR_ARG; }
    XF_TRY(b.fields.ensure((size_t)h.nnz));
    XF_CUDA_TRY(cudaMemcpyAsync(b.fields.p, h.fields, (size_t)h.nnz, cudaMemcpyHostToDevice, tr->table->stream));
    d->fields = b.fields.as<uint8_t>();
  }
  return XF_OK;
}

// What an entry point that takes a host batch hands back once the step is enqueued.
struct XfHostReturn {
  enum { NO_WAIT, WAIT, WAIT_CHECKED } wait;  // synchronise on the table stream (and check the table's error word)
  float* mean_abs_loss;      // mode 0, after the wait: the mean |loss| of the batch (0 for an empty batch)
  float* pctr_out;           // mode 1: the predictions, copied before the wait
  float* pinned_loss_sum;    // mode 0, no wait: the loss sum, copied asynchronously into this page-locked float
  const char* page_locked;   // the entry point's name if every host array must be page-locked
};

// A host batch through one of the two buffer sets: upload, step, release the set, count, read back.
static int xf_step_host_batch(xf_trainer* tr, const XfBatch& h, int mode, const XfHostReturn& r) {
  XF_TRY(xf_check_batch(tr, h.rows, h.nnz));
  if (h.rows == 0 && !tr->mg) {
    if (r.mean_abs_loss) *r.mean_abs_loss = 0.f;
    return XF_OK;
  }
  if (r.page_locked && (!xf_is_pinned(h.row_ptr) || !xf_is_pinned(h.ids ? (const void*)h.ids : h.keys) ||
                        !xf_is_pinned(h.labels) || (r.pinned_loss_sum && !xf_is_pinned(r.pinned_loss_sum)))) {
    xf_set_error("%s needs page-locked host buffers", r.page_locked);
    return XF_ERR_ARG;
  }
  XF_CUDA_TRY(cudaSetDevice(tr->table->cfg.device));
  const int slot = (int)(tr->step_index & 1);
  XfBatchBuf& b = tr->buf[slot];
  ++tr->step_index;
  XfBatch d;
  XF_TRY(xf_upload(tr, b, h, &d));
  cudaStream_t st = tr->table->stream;
  float* d_abs = mode == 0 ? tr->d_abs_loss + slot : nullptr;
  if (d_abs) XF_CUDA_TRY(cudaMemsetAsync(d_abs, 0, sizeof(float), st));
  XF_TRY(xf_step_device_impl(tr, d, mode, d_abs));
  XF_CUDA_TRY(cudaEventRecord(b.consumed, st));
  if (mode == 0) xf_count_step(tr, h.rows, h.nnz);
  if (r.pinned_loss_sum)
    XF_CUDA_TRY(cudaMemcpyAsync(r.pinned_loss_sum, d_abs, sizeof(float), cudaMemcpyDeviceToHost, st));
  if (r.wait == XfHostReturn::NO_WAIT) return XF_OK;
  if (mode == 0)
    XF_CUDA_TRY(cudaMemcpyAsync(tr->h_abs_loss + slot, d_abs, sizeof(float), cudaMemcpyDeviceToHost, st));
  else
    XF_CUDA_TRY(cudaMemcpyAsync(r.pctr_out, tr->pctr.p, (size_t)h.rows * 4, cudaMemcpyDeviceToHost, st));
  XF_CUDA_TRY(cudaStreamSynchronize(st));  // also: the caller may reuse its arrays (values, field ids) now
  if (r.mean_abs_loss) *r.mean_abs_loss = h.rows ? tr->h_abs_loss[slot] / (float)h.rows : 0.f;
  return r.wait == XfHostReturn::WAIT_CHECKED ? tr->table->check_error() : XF_OK;
}

XF_DLL int xf_trainer_step_device(xf_trainer* tr, const uint32_t* d_row_ptr, const uint64_t* d_keys,
                                  const uint8_t* d_labels, uint32_t rows, uint32_t nnz) {
  if (!tr || !d_row_ptr || !d_keys || !d_labels) return XF_ERR_ARG;
  return xf_step_resident(tr, {d_row_ptr, d_keys, d_labels, rows, nnz});
}

XF_DLL int xf_trainer_step_host(xf_trainer* tr, const uint32_t* row_ptr, const uint64_t* keys,
                                const uint8_t* labels, uint32_t rows, uint32_t nnz, float* mean_abs_loss) {
  if (!tr || !row_ptr || (!keys && nnz) || !labels) return XF_ERR_ARG;
  return xf_step_host_batch(tr, {row_ptr, keys, labels, rows, nnz}, 0,
                            {mean_abs_loss ? XfHostReturn::WAIT : XfHostReturn::NO_WAIT, mean_abs_loss});
}

XF_DLL int xf_trainer_predict_host(xf_trainer* tr, const uint32_t* row_ptr, const uint64_t* keys, uint32_t rows,
                                   uint32_t nnz, float* pctr_out) {
  if (!tr || !row_ptr || (!keys && nnz) || !pctr_out) return XF_ERR_ARG;
  return xf_step_host_batch(tr, {row_ptr, keys, nullptr, rows, nnz}, 1, {XfHostReturn::WAIT_CHECKED, nullptr, pctr_out});
}

// ---- the same entry points with feature values (XF_MODEL_FM_CANONICAL, step_fmc.cu)
XF_DLL int xf_trainer_step_device_values(xf_trainer* tr, const uint32_t* d_row_ptr, const uint64_t* d_keys,
                                         const float* d_vals, const uint8_t* d_labels, uint32_t rows, uint32_t nnz) {
  if (!tr || !d_row_ptr || !d_keys || !d_labels) return XF_ERR_ARG;
  if (tr->cfg.model != XF_MODEL_FM_CANONICAL) { xf_set_error("feature values need XF_MODEL_FM_CANONICAL"); return XF_ERR_ARG; }
  return xf_step_resident(tr, {d_row_ptr, d_keys, d_labels, rows, nnz, d_vals});
}

XF_DLL int xf_trainer_step_host_values(xf_trainer* tr, const uint32_t* row_ptr, const uint64_t* keys, const float* vals,
                                       const uint8_t* labels, uint32_t rows, uint32_t nnz, float* mean_abs_loss) {
  if (!tr || !row_ptr || (!keys && nnz) || !labels) return XF_ERR_ARG;
  if (tr->cfg.model != XF_MODEL_FM_CANONICAL) { xf_set_error("feature values need XF_MODEL_FM_CANONICAL"); return XF_ERR_ARG; }
  return xf_step_host_batch(tr, {row_ptr, keys, labels, rows, nnz, vals}, 0, {XfHostReturn::WAIT_CHECKED, mean_abs_loss});
}

XF_DLL int xf_trainer_predict_host_values(xf_trainer* tr, const uint32_t* row_ptr, const uint64_t* keys, const float* vals,
                                          uint32_t rows, uint32_t nnz, float* pctr_out) {
  if (!tr || !row_ptr || (!keys && nnz) || !pctr_out) return XF_ERR_ARG;
  if (tr->cfg.model != XF_MODEL_FM_CANONICAL) { xf_set_error("feature values need XF_MODEL_FM_CANONICAL"); return XF_ERR_ARG; }
  return xf_step_host_batch(tr, {row_ptr, keys, nullptr, rows, nnz, vals}, 1,
                            {XfHostReturn::WAIT_CHECKED, nullptr, pctr_out});
}

// ---- the defined multi-view machine (XF_MODEL_MVM, step_mvm.cu): the batch with the tokens' field ids
XF_DLL int xf_trainer_step_host_fields(xf_trainer* tr, const uint32_t* row_ptr, const uint64_t* keys, const uint8_t* fields,
                                       const float* vals, const uint8_t* labels, uint32_t rows, uint32_t nnz,
                                       float* mean_abs_loss) {
  if (!tr || !row_ptr || (!keys && nnz) || (!fields && nnz) || !labels) return XF_ERR_ARG;
  if (tr->cfg.model != XF_MODEL_MVM) { xf_set_error("field ids need XF_MODEL_MVM"); return XF_ERR_ARG; }
  return xf_step_host_batch(tr, {row_ptr, keys, labels, rows, nnz, vals, fields}, 0,
                            {XfHostReturn::WAIT_CHECKED, mean_abs_loss});
}

XF_DLL int xf_trainer_predict_host_fields(xf_trainer* tr, const uint32_t* row_ptr, const uint64_t* keys,
                                          const uint8_t* fields, const float* vals, uint32_t rows, uint32_t nnz,
                                          float* pctr_out) {
  if (!tr || !row_ptr || (!keys && nnz) || (!fields && nnz) || !pctr_out) return XF_ERR_ARG;
  if (tr->cfg.model != XF_MODEL_MVM) { xf_set_error("field ids need XF_MODEL_MVM"); return XF_ERR_ARG; }
  return xf_step_host_batch(tr, {row_ptr, keys, nullptr, rows, nnz, vals, fields}, 1,
                            {XfHostReturn::WAIT_CHECKED, nullptr, pctr_out});
}

XF_DLL int xf_trainer_init_push(xf_trainer* tr) {
  if (!tr) return XF_ERR_ARG;
  xf_table* t = tr->table;
  // Every worker pushes key 0 with a zero gradient once (lr_worker.cc:180-182, fm_worker.cc:248-252).
  // Key 0 belongs to shard 0; other shards have nothing to do.
  if (xf_shard_of(0, t->cfg.num_shards) != t->cfg.shard_index) return XF_OK;
  uint64_t key = 0;
  float gw = 0.f;
  std::vector<float> gv((size_t)std::max(t->view.K, 1), 0.f);
  int reps = tr->comm ? xf_comm_nranks(tr->comm) : 1;  // one init push per worker rank
  for (int r = 0; r < reps; ++r) XF_TRY(xf_table_push(t, &key, 1, &gw, t->view.K ? gv.data() : nullptr));
  return XF_OK;
}

XF_DLL int xf_trainer_get_loss(xf_trainer* tr, float* loss_out, uint32_t rows) {
  if (!tr || !loss_out) return XF_ERR_ARG;
  if (!tr->cfg.keep_loss) { xf_set_error("trainer created with keep_loss = 0"); return XF_ERR_STATE; }
  if (rows > tr->cfg.max_rows) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaMemcpyAsync(loss_out, tr->loss.p, (size_t)rows * 4, cudaMemcpyDeviceToHost, tr->table->stream));
  XF_CUDA_TRY(cudaStreamSynchronize(tr->table->stream));
  return XF_OK;
}

XF_DLL int xf_trainer_stats(xf_trainer* tr, uint64_t* steps, uint64_t* rows, uint64_t* nnz, uint64_t* unique_keys) {
  if (!tr) return XF_ERR_ARG;
  if (steps) *steps = tr->n_steps;
  if (rows) *rows = tr->n_rows;
  if (nnz) *nnz = tr->n_nnz;
  if (unique_keys) {
    unsigned long long u = 0;
    XF_CUDA_TRY(cudaMemcpyAsync(&u, tr->d_unique_total, sizeof(u), cudaMemcpyDeviceToHost, tr->table->stream));
    XF_CUDA_TRY(cudaStreamSynchronize(tr->table->stream));
    unsigned long long remote = 0;  // sharded: counted by the owners of this rank's keys
    if (tr->mg) XF_TRY(xf_mg_unique(tr, &remote));
    *unique_keys = u + remote;
  }
  return XF_OK;
}

XF_DLL int xf_trainer_launches(xf_trainer* tr, uint64_t* launches) {
  if (!tr || !launches) return XF_ERR_ARG;
  *launches = tr->launches + tr->table->launches;
  return XF_OK;
}

XF_DLL int xf_trainer_sync(xf_trainer* tr) {
  if (!tr) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaStreamSynchronize(tr->copy_stream));
  return xf_table_sync(tr->table);
}

XF_DLL int xf_trainer_wait_uploads(xf_trainer* tr) {
  if (!tr) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaStreamSynchronize(tr->copy_stream));
  return XF_OK;
}

XF_DLL int xf_trainer_step_host_async(xf_trainer* tr, const uint32_t* row_ptr, const uint64_t* keys,
                                      const uint8_t* labels, uint32_t rows, uint32_t nnz,
                                      float* pinned_abs_loss_sum) {
  if (!tr || !row_ptr || (!keys && nnz) || !labels) return XF_ERR_ARG;
  return xf_step_host_batch(tr, {row_ptr, keys, labels, rows, nnz}, 0,
                            {XfHostReturn::NO_WAIT, nullptr, nullptr, pinned_abs_loss_sum, "xf_trainer_step_host_async"});
}

XF_DLL int xf_trainer_step_host_ids_async(xf_trainer* tr, const uint32_t* row_ptr, const uint32_t* ids,
                                          const uint8_t* labels, uint32_t rows, uint32_t nnz,
                                          float* pinned_abs_loss_sum) {
  if (!tr || !row_ptr || (!ids && nnz) || !labels) return XF_ERR_ARG;
  XfBatch h{row_ptr, nullptr, labels, rows, nnz};
  h.ids = ids;
  return xf_step_host_batch(tr, h, 0, {XfHostReturn::NO_WAIT, nullptr, nullptr, pinned_abs_loss_sum,
                                       "xf_trainer_step_host_ids_async"});
}

// Two-phase ingest.  _begin copies the block to the device and parses it on the trainer's ingest streams
// into the set that is NOT being trained on, and returns at once; _end waits for that parse only, makes
// the set current and reports its size: read, H2D and parse of block i+1 overlap the step of block i
// (WorkerBase::run_blocks, worker.cc).
// A SECOND _begin may be issued before the first one's _end.  It targets the set that is being trained on:
// its text buffer is free (only the parsed arrays are read by the steps), so the copy starts at once on the
// copy stream and runs beside the first block's parse; its parse is launched by the _end that retires the
// set.  With the loop  begin(i+2); step(i); end(i+1)  the H2D of one block, the parse of the previous one and
// the training step of the one before that all run at the same time.
static int xf_ingest_launch_parse(xf_trainer* tr, xf_trainer::IngestSet& g) {
  cudaStream_t is = tr->ing_stream;
  // the steps that read this set (two blocks ago) must have finished before it is overwritten
  XF_CUDA_TRY(cudaStreamWaitEvent(is, g.consumed, 0));
  XF_CUDA_TRY(cudaStreamWaitEvent(is, g.copied, 0));
  const uint64_t len = g.len;
  // upper bounds for a block of `len` bytes: shortest row "0\n" = 2 bytes, shortest token "a:b:c " ~ 4 bytes
  g.max_rows = (uint32_t)std::min<uint64_t>(len / 2 + 2, tr->cfg.max_rows);
  g.max_tok = (uint32_t)std::min<uint64_t>(len / 4 + 2, tr->cfg.max_nnz);
  XF_TRY(g.row_ptr.ensure(((size_t)g.max_rows + 2) * 4));
  XF_TRY(g.keys.ensure(((size_t)g.max_tok + 1) * 8));
  XF_TRY(g.labels.ensure((size_t)g.max_rows + 1));
  XF_TRY(g.totals.ensure(16));
  // totals = {rows, tokens, parse error}; the parser's error word is its own, not the table's sticky one
  XF_CUDA_TRY(cudaMemsetAsync(g.totals.p, 0, 16, is));
  XF_TRY(xf_launch_parse(g.text.as<char>(), len, tr->ing_scratch, g.row_ptr.as<uint32_t>(), g.keys.as<uint64_t>(),
                         g.labels.as<uint8_t>(), g.max_rows, g.max_tok, g.totals.as<uint32_t>(), g.totals.as<int>() + 2, is));
  tr->launches += 5;
  XF_CUDA_TRY(cudaMemcpyAsync(g.h_totals, g.totals.p, 12, cudaMemcpyDeviceToHost, is));
  XF_CUDA_TRY(cudaEventRecord(g.parsed, is));
  return XF_OK;
}

XF_DLL int xf_trainer_ingest_begin(xf_trainer* tr, const char* text, uint64_t len) {
  if (!tr || (!text && len)) return XF_ERR_ARG;
  if (tr->ing_pending >= 2) { xf_set_error("ingest: at most two xf_trainer_ingest_begin calls may be outstanding"); return XF_ERR_STATE; }
  if (len >= 0xFFFFFFF0ull) { xf_set_error("ingest: a block must be smaller than 4 GiB (u32 token offsets)"); return XF_ERR_ARG; }
  XF_CUDA_TRY(cudaSetDevice(tr->table->cfg.device));
  // first outstanding block -> the idle set; second -> the set being trained on (text only, for now)
  xf_trainer::IngestSet& g = tr->ing[tr->ing_pending == 0 ? (tr->ing_cur ^ 1) : tr->ing_cur];
  // the set's previous text was consumed by its parse, which the _end that made the set current (or retired it)
  // has waited for; a set that was never used has nothing outstanding
  XF_CUDA_TRY(cudaEventSynchronize(g.parsed));
  XF_TRY(g.text.ensure(len + 16));
  const void* src = text;
  if (len && !xf_is_pinned(text)) {
    XF_TRY(g.stage.ensure(len));
    memcpy(g.stage.p, text, len);
    src = g.stage.p;
  }
  if (len) XF_CUDA_TRY(cudaMemcpyAsync(g.text.p, src, len, cudaMemcpyHostToDevice, tr->ing_copy_stream));
  XF_CUDA_TRY(cudaEventRecord(g.copied, tr->ing_copy_stream));
  g.len = len;
  if (tr->ing_pending == 0) XF_TRY(xf_ingest_launch_parse(tr, g));
  ++tr->ing_pending;
  return XF_OK;
}

XF_DLL int xf_trainer_ingest_end(xf_trainer* tr, uint32_t* rows, uint32_t* nnz) {
  if (!tr || !rows || !nnz) return XF_ERR_ARG;
  if (tr->ing_pending == 0) { xf_set_error("ingest: xf_trainer_ingest_end without xf_trainer_ingest_begin"); return XF_ERR_STATE; }
  XF_CUDA_TRY(cudaSetDevice(tr->table->cfg.device));
  xf_trainer::IngestSet& g = tr->ing[tr->ing_cur ^ 1];
  --tr->ing_pending;
  XF_CUDA_TRY(cudaEventSynchronize(g.parsed));
  const uint32_t* tot = g.h_totals;
  const int e = (int)tot[2];
  g.rows = g.nnz = 0;
  int rc = XF_OK;
  if (e == 4) { xf_set_error("ingest: token without three ':'-separated fields"); rc = XF_ERR_IO; }
  else if (e == 3 || tot[0] > g.max_rows || tot[1] > g.max_tok) {
    xf_set_error("ingest: block (%u rows, %u tokens) exceeds trainer limits (%u, %u)", tot[0], tot[1],
                 tr->cfg.max_rows, tr->cfg.max_nnz);
    rc = XF_ERR_ARG;
  }
  if (rc != XF_OK) {
    // the failed block is dropped; a second outstanding block (text already copied into the current set) becomes
    // the first: it cannot be parsed there, so it is dropped as well and the caller starts over
    if (tr->ing_pending) { cudaStreamSynchronize(tr->ing_copy_stream); tr->ing_pending = 0; }
    return rc;
  }
  g.rows = tot[0];
  g.nnz = tot[1];
  tr->ing_cur ^= 1;
  tr->ing_rows = g.rows;
  tr->ing_nnz = g.nnz;
  // everything the table stream does with this set comes after its parse
  XF_CUDA_TRY(cudaStreamWaitEvent(tr->table->stream, g.parsed, 0));
  *rows = g.rows;
  *nnz = g.nnz;
  // the set that was current until now is retired (the caller has issued its last step on it): a second
  // outstanding block, whose text is already on its way into that set, can be parsed there now
  if (tr->ing_pending) XF_TRY(xf_ingest_launch_parse(tr, tr->ing[tr->ing_cur ^ 1]));
  return XF_OK;
}

XF_DLL int xf_trainer_ingest_text(xf_trainer* tr, const char* text, uint64_t len, uint32_t* rows, uint32_t* nnz) {
  if (!tr || (!text && len) || !rows || !nnz) return XF_ERR_ARG;
  if (tr->ing_pending) { xf_set_error("ingest: xf_trainer_ingest_text while a two-phase ingest is outstanding"); return XF_ERR_STATE; }
  tr->ing_rows = tr->ing_nnz = 0;
  XF_TRY(xf_trainer_ingest_begin(tr, text, len));
  return xf_trainer_ingest_end(tr, rows, nnz);
}

static int xf_ingested_range(xf_trainer* tr, uint32_t row_start, uint32_t row_end) {
  if (!tr) return XF_ERR_ARG;
  if (row_start > row_end || row_end > tr->ing_rows) { xf_set_error("row range outside the ingested block"); return XF_ERR_ARG; }
  if (tr->mg && (row_start != 0 || row_end != tr->ing_rows)) {
    xf_set_error("sharded trainers step whole ingested blocks (core_num = 1)");
    return XF_ERR_ARG;
  }
  return XF_OK;
}

// A row slice of the current ingested block through the step kernels.  row_ptr holds absolute token offsets, so a
// slice is just a shifted row_ptr / labels pointer.  A forward pass (mode 1) appends its predictions and labels to
// the metric `m` and / or copies them to pctr_out / labels_out; `wait` synchronises and checks the table.
int xf_step_ingested_slice(xf_trainer* tr, uint32_t row_start, uint32_t row_end, int mode, xf_metric* m,
                           float* pctr_out, uint8_t* labels_out, bool wait) {
  XF_TRY(xf_ingested_range(tr, row_start, row_end));
  const uint32_t rows = row_end - row_start;
  if (rows == 0 && !tr->mg) return XF_OK;
  if (mode == 1 && !m && !pctr_out) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaSetDevice(tr->table->cfg.device));
  xf_trainer::IngestSet& g = tr->ing[tr->ing_cur];
  cudaStream_t st = tr->table->stream;
  // the per-token scratch (FM: touched[]) is indexed by absolute position and must not keep stale slices
  if (mode == 0 && !tr->table->view.lazy && !tr->mg)
    XF_CUDA_TRY(cudaMemsetAsync(tr->touched.p, 0xFF, (size_t)tr->ing_nnz * 4, st));
  const uint8_t* labels = g.labels.as<uint8_t>() + row_start;
  XF_TRY(xf_step_device_impl(tr, {g.row_ptr.as<uint32_t>() + row_start, g.keys.as<uint64_t>(), labels, rows, tr->ing_nnz},
                             mode, nullptr));
  if (rows) {
    if (m) XF_TRY(xf_metric_add_device(m, tr->pctr.as<float>(), labels, rows, st));
    if (pctr_out) XF_CUDA_TRY(cudaMemcpyAsync(pctr_out, tr->pctr.p, (size_t)rows * 4, cudaMemcpyDeviceToHost, st));
    if (labels_out) XF_CUDA_TRY(cudaMemcpyAsync(labels_out, labels, rows, cudaMemcpyDeviceToHost, st));
  }
  XF_CUDA_TRY(cudaEventRecord(g.consumed, st));
  if (mode == 0) xf_count_step(tr, rows, 0);  // counts the slice's rows; its tokens are not counted
  if (!wait) return XF_OK;
  XF_CUDA_TRY(cudaStreamSynchronize(st));
  return tr->table->check_error();
}

XF_DLL int xf_trainer_step_ingested(xf_trainer* tr, uint32_t row_start, uint32_t row_end) {
  return xf_step_ingested_slice(tr, row_start, row_end, 0, nullptr, nullptr, nullptr, false);
}

XF_DLL int xf_trainer_ingested_export(xf_trainer* tr, uint32_t* row_ptr_out, uint64_t* keys_out, uint8_t* labels_out) {
  if (!tr) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaSetDevice(tr->table->cfg.device));
  XF_CUDA_TRY(cudaStreamSynchronize(tr->table->stream));
  xf_trainer::IngestSet& g = tr->ing[tr->ing_cur];
  if (row_ptr_out)
    XF_CUDA_TRY(cudaMemcpy(row_ptr_out, g.row_ptr.p, ((size_t)tr->ing_rows + 1) * 4, cudaMemcpyDeviceToHost));
  if (keys_out && tr->ing_nnz)
    XF_CUDA_TRY(cudaMemcpy(keys_out, g.keys.p, (size_t)tr->ing_nnz * 8, cudaMemcpyDeviceToHost));
  if (labels_out && tr->ing_rows)
    XF_CUDA_TRY(cudaMemcpy(labels_out, g.labels.p, (size_t)tr->ing_rows, cudaMemcpyDeviceToHost));
  return XF_OK;
}

XF_DLL int xf_trainer_predict_ingested(xf_trainer* tr, uint32_t row_start, uint32_t row_end, float* pctr_out,
                                       uint8_t* labels_out) {
  return xf_step_ingested_slice(tr, row_start, row_end, 1, nullptr, pctr_out, labels_out, true);
}

XF_DLL int xf_trainer_set_profile(xf_trainer* tr, int on) {
  if (!tr) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaStreamSynchronize(tr->table->stream));
  tr->profile = on != 0;
  tr->prof_used = 0;
  if (tr->profile && tr->prof_events.empty()) {
    // the first 256 steps' marks are created here, not inside the first profiled (and usually timed) step
    XF_CUDA_TRY(cudaSetDevice(tr->table->cfg.device));
    tr->prof_events.resize(4 * 256);
    for (cudaEvent_t& e : tr->prof_events) XF_CUDA_TRY(cudaEventCreate(&e));
  }
  return XF_OK;
}

XF_DLL int xf_trainer_profile(xf_trainer* tr, double ms[2], uint64_t* steps) {
  if (!tr || !ms) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaStreamSynchronize(tr->table->stream));
  ms[0] = ms[1] = 0.0;
  for (size_t i = 0; i + 4 <= tr->prof_used; i += 4) {
    float a = 0.f, b = 0.f;
    XF_CUDA_TRY(cudaEventElapsedTime(&a, tr->prof_events[i], tr->prof_events[i + 1]));
    XF_CUDA_TRY(cudaEventElapsedTime(&b, tr->prof_events[i + 2], tr->prof_events[i + 3]));
    ms[0] += a;
    ms[1] += b;
  }
  if (steps) *steps = tr->prof_used / 4;
  tr->prof_used = 0;
  return XF_OK;
}

XF_DLL int xf_host_alloc(void** out, uint64_t bytes) {
  if (!out) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
  return XF_OK;
}
XF_DLL int xf_host_free(void* p) {
  if (p) XF_CUDA_TRY(cudaFreeHost(p));
  return XF_OK;
}
