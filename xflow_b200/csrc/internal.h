// Internal host-side structures shared by capi.cu / comm.cu / worker.cc.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>
#include <string>
#include <vector>

#include "../../include/xflow_b200.h"
#include "kernels.h"
#include "table.cuh"

void xf_set_error(const char* fmt, ...);

#define XF_CUDA_TRY(expr)                                                              \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      xf_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__, __LINE__, \
                   cudaGetErrorString(_e));                                            \
      return XF_ERR_CUDA;                                                              \
    }                                                                                  \
  } while (0)

#define XF_TRY(expr)            \
  do {                          \
    int _r = (expr);            \
    if (_r != XF_OK) return _r; \
  } while (0)

// growable device buffer
struct XfDevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes);
  void release();
  template <typename T> T* as() { return reinterpret_cast<T*>(p); }
};

// growable pinned host buffer
struct XfPinBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t bytes);
  void release();
  template <typename T> T* as() { return reinterpret_cast<T*>(p); }
};

struct xf_table {
  xf_table_config cfg;
  XfTableView view;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  unsigned long long* d_size = nullptr;
  int* d_error = nullptr;
  uint64_t size_bound = 0;   // host-side upper bound on the number of live keys (sync path)
  // asynchronous size read-back (no host sync in steady state): the device counter is copied to a
  // pinned ring after every step; bound = last completed reading + keys submitted since it was issued
  unsigned long long* h_size_ring = nullptr;
  cudaEvent_t size_ev[4] = {nullptr, nullptr, nullptr, nullptr};
  uint64_t size_issued_at[4] = {0, 0, 0, 0};
  bool size_inflight[4] = {false, false, false, false};
  int size_next = 0;
  uint64_t cum_incoming = 0, known_size = 0, known_at = 0;
  uint64_t launches = 0;
  int refs = 1;              // the creator + every trainer bound to the table (destroy order is free)
  // lazy ("update on next touch") tables: batch sequence number and the per-batch row counts
  uint32_t seq = 0;
  uint32_t* d_rows_by_seq = nullptr;
  size_t rows_cap = 0;
  int next_seq();            // advances seq; flushes all pending steps and restarts when the ring is used up
  int reserve_seqs(int n);   // makes sure the next n numbers come without a restart (flushes now if they would not)
  // scratch for the host-pointer API (pull/push/import/export on host arrays); like KVWorker::Push/Pull
  // (kv_app.h:110-165) those entry points may be called from several threads: serialised by this mutex
  std::mutex host_mu;
  XfDevBuf s_keys, s_slots, s_w, s_v, s_nw, s_zw, s_nv, s_zv, s_present;

  int alloc_table(uint64_t capacity);
  int ensure_room(uint64_t incoming_keys);
  int grow(uint64_t new_capacity);
  int check_error();
};

struct XfBatchBuf {
  XfDevBuf row_ptr, keys, labels, ids, vals, fields;
  XfPinBuf h_row_ptr, h_keys, h_labels;
  cudaEvent_t copied = nullptr;   // H2D of this buffer finished (copy stream)
  cudaEvent_t consumed = nullptr; // kernels reading this buffer finished (compute stream)
  cudaEvent_t staged = nullptr;   // H2D out of the pinned staging finished
};

struct xf_trainer {
  xf_table* table = nullptr;
  xf_comm* comm = nullptr;
  xf_trainer_config cfg;
  cudaStream_t copy_stream = nullptr;
  XfBatchBuf buf[2];
  uint64_t step_index = 0;
  XfDevBuf touched, loss, pctr;
  unsigned long long* d_unique_total = nullptr;
  float* d_abs_loss = nullptr;          // 2 slots
  float* h_abs_loss = nullptr;          // pinned, 2 slots
  uint64_t n_steps = 0, n_rows = 0, n_nnz = 0;
  uint32_t last_rows = 0;
  uint64_t launches = 0;
  // device-side ingest (xf_trainer_ingest_begin / _end): two sets of {raw text, the block's CSR}, so that
  // block i+1 is copied and parsed on the ingest stream while block i is being trained on the table stream
  struct IngestSet {
    XfDevBuf text, row_ptr, keys, labels, totals;
    XfPinBuf stage;                 // page-locked copy of a pageable source
    uint32_t* h_totals = nullptr;   // pinned {rows, tokens, parse error}
    cudaEvent_t parsed = nullptr;   // H2D + parse of this set finished (ingest stream)
    cudaEvent_t copied = nullptr;   // the block's text has arrived in `text` (ingest copy stream)
    uint64_t len = 0;               // bytes of the block whose text is in `text`
    cudaEvent_t consumed = nullptr; // the last step that reads this set finished (table stream)
    uint32_t rows = 0, nnz = 0, max_rows = 0, max_tok = 0;
  };
  IngestSet ing[2];
  XfDevBuf ing_scratch;
  cudaStream_t ing_stream = nullptr;       // parses
  cudaStream_t ing_copy_stream = nullptr;  // H2D of the blocks' text: the copy of block i+2 runs beside the parse of i+1
  int ing_cur = 0;                  // the set xf_trainer_step_ingested works on
  int ing_pending = 0;              // xf_trainer_ingest_begin calls not yet matched by _end (0..2); the second one
                                    // targets the set being trained: its text is copied at once, its parse is
                                    // launched by the _end that frees the set
  uint32_t ing_rows = 0, ing_nnz = 0;
  void* mg = nullptr;                   // multi-GPU exchange state (comm.cu)
  cudaEvent_t input_ready = nullptr;    // set by the host-batch paths: H2D of the batch about to be stepped
  // optional per-kernel timing (xf_trainer_set_profile): events around the kernels of each step
  bool profile = false;
  std::vector<cudaEvent_t> prof_events;  // 4 marks per step: step kernel [0,1], optimizer kernel(s) [2,3]
  size_t prof_used = 0;
};

// ingest.cu
int xf_launch_parse(const char* d_text, uint64_t len, XfDevBuf& scratch, uint32_t* d_row_ptr, uint64_t* d_keys,
                    uint8_t* d_labels, uint32_t max_rows, uint32_t max_tok, uint32_t* d_totals, int* d_error,
                    cudaStream_t st);
int xf_launch_hash_ids(const uint32_t* d_ids, uint32_t n, uint64_t* d_keys, cudaStream_t st);

// capi.cu: train on (mode 0) or predict (mode 1) rows [row_start, row_end) of the current ingested block
int xf_step_ingested_slice(xf_trainer* tr, uint32_t row_start, uint32_t row_end, int mode, xf_metric* m,
                           float* pctr_out, uint8_t* labels_out, bool wait);

// multi-GPU pieces implemented in comm.cu
int xf_mg_create(xf_trainer* tr);
void xf_mg_destroy(xf_trainer* tr);
int xf_mg_step(xf_trainer* tr, const uint32_t* d_row_ptr, const uint64_t* d_keys, const uint8_t* d_labels,
               uint32_t rows, uint32_t nnz, int mode, float* d_abs_loss, cudaEvent_t* prof_marks);
int xf_mg_unique(xf_trainer* tr, unsigned long long* out);
int xf_comm_nranks(xf_comm* c);
int xf_comm_rank(xf_comm* c);
