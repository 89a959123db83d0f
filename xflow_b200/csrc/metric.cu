// Test-set metric ON THE DEVICE (SURVEY.md section 8f-2): Base::calculate_auc (src/base/base.h:84-110) without
// copying the predictions back and sorting them on one host core.
//
//   predictions + labels of every forward block are appended to a device buffer (xf_metric_add_device, or
//   xf_trainer_predict_ingested_metric which runs the forward pass and appends, all asynchronous);
//   xf_metric_finish sorts them by descending prediction (CUB radix sort, stable: ties keep their input order),
//   takes the running count of positives (CUB scan) and reduces:
//     out[0]  the reference's logloss: mean of  y log2 p + (1-y) log2(1-p)  (base 2, NOT negated), the positive term
//             through float log2 like the reference's expression (base.h:97-98), accumulated in double
//     out[1]  the reference's AUC: sum over negatives of the positives ranked before them / (P N), as 64-bit
//             integers (the reference accumulates it in a float, which stops counting at 2^24)
//     out[2]  positives   out[3]  negatives
//     out[4]  mean negative natural-log likelihood, probabilities clamped to [1e-15, 1 - 1e-15]
//     out[5]  AUC with ties counted 1/2 (Mann-Whitney U / (P N)), integer arithmetic
//   (out[4], out[5] = what xf_auc_logloss_exact computes on the host.)
// Sorting and scanning are library code (CUB, part of the CUDA toolkit); the reductions are kernels of this file.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include <cub/cub.cuh>

#include "internal.h"

struct xf_metric {
  int device = 0;
  cudaStream_t stream = nullptr;
  XfDevBuf pctr, lab;                 // appended inputs
  XfDevBuf s_pctr, s_lab, psum, start, tmp, acc;
  uint64_t n = 0;
};

XF_DLL int xf_metric_create(xf_metric** out, int device) {
  if (!out) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaSetDevice(device));
  xf_metric* m = new xf_metric;
  m->device = device;
  XF_CUDA_TRY(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
  *out = m;
  return XF_OK;
}

XF_DLL int xf_metric_destroy(xf_metric* m) {
  if (!m) return XF_OK;
  cudaSetDevice(m->device);
  cudaStreamSynchronize(m->stream);
  XfDevBuf* bufs[] = {&m->pctr, &m->lab, &m->s_pctr, &m->s_lab, &m->psum, &m->start, &m->tmp, &m->acc};
  for (XfDevBuf* b : bufs) b->release();
  cudaStreamDestroy(m->stream);
  delete m;
  return XF_OK;
}

XF_DLL int xf_metric_reset(xf_metric* m) {
  if (!m) return XF_ERR_ARG;
  m->n = 0;
  return XF_OK;
}

// grow a buffer keeping its first `used` bytes (stream-ordered after everything queued on `st`)
static int xf_grow_keep(XfDevBuf& b, size_t used, size_t want, cudaStream_t st) {
  if (want <= b.cap) return XF_OK;
  size_t ncap = std::max(want, b.cap * 2);
  void* np = nullptr;
  XF_CUDA_TRY(cudaMalloc(&np, ncap));
  if (used) XF_CUDA_TRY(cudaMemcpyAsync(np, b.p, used, cudaMemcpyDeviceToDevice, st));
  XF_CUDA_TRY(cudaStreamSynchronize(st));
  if (b.p) XF_CUDA_TRY(cudaFree(b.p));
  b.p = np;
  b.cap = ncap;
  return XF_OK;
}

// append n predictions / labels that live in device memory; the copies run on `cuda_stream` (the stream that
// produced them), so no synchronisation is needed by the caller
XF_DLL int xf_metric_add_device(xf_metric* m, const float* d_pctr, const uint8_t* d_labels, uint64_t n, void* cuda_stream) {
  if (!m || ((!d_pctr || !d_labels) && n)) return XF_ERR_ARG;
  if (n == 0) return XF_OK;
  XF_CUDA_TRY(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  XF_TRY(xf_grow_keep(m->pctr, m->n * 4, (m->n + n) * 4, st));
  XF_TRY(xf_grow_keep(m->lab, m->n, m->n + n, st));
  XF_CUDA_TRY(cudaMemcpyAsync(m->pctr.as<float>() + m->n, d_pctr, n * 4, cudaMemcpyDeviceToDevice, st));
  XF_CUDA_TRY(cudaMemcpyAsync(m->lab.as<uint8_t>() + m->n, d_labels, n, cudaMemcpyDeviceToDevice, st));
  m->n += n;
  return XF_OK;
}

struct XfMaxU32 {
  __host__ __device__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};

// head[i] = i if element i starts a group of equal predictions, else 0 ; lab32[i] = label as u32
__global__ void xf_k_metric_prepare(const float* __restrict__ p, const uint8_t* __restrict__ lab, uint64_t n,
                                    uint32_t* __restrict__ lab32, uint32_t* __restrict__ head) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    lab32[i] = lab[i] == 1 ? 1u : 0u;
    head[i] = (i == 0 || p[i] != p[i - 1]) ? (uint32_t)i : 0u;
  }
}

// acc[0] (double) sum of the reference's log2 terms ; acc[1] (double) sum of -ln likelihood ;
// acc[2] (u64) sum over negatives of positives ranked before ; acc[3] (u64) twice the tie-aware U statistic
__global__ void xf_k_metric_reduce(const float* __restrict__ p, const uint8_t* __restrict__ lab,
                                   const uint32_t* __restrict__ psum, const uint32_t* __restrict__ start, uint64_t n,
                                   double* acc_d, unsigned long long* acc_u) {
  double ll2 = 0.0, lln = 0.0;
  unsigned long long area = 0ull, twice_u = 0ull;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const float pi = p[i];
    const int y = lab[i] == 1 ? 1 : 0;
    // label * log2(float) + (1.0 - label) * log2(1.0 - double(p))      base.h:97-98
    ll2 += (double)((float)y * log2f(pi)) + (1.0 - (double)y) * log2(1.0 - (double)pi);
    const double pc = fmin(fmax((double)pi, 1e-15), 1.0 - 1e-15);
    lln -= y ? log(pc) : log(1.0 - pc);
    if (!y) area += psum[i];  // positives ranked before this negative (inclusive sum; this element adds none)
    if (i + 1 == n || p[i + 1] != pi) {
      // last element of a group of equal predictions [s, i]: its negatives see the positives before the group
      // plus half of the group's own
      const uint64_t s = start[i];
      const uint64_t pb = s ? psum[s - 1] : 0u, pa = psum[i];
      const uint64_t gp = pa - pb, gn = (i - s + 1) - gp;
      twice_u += gn * (pb + pa);
    }
  }
  typedef cub::BlockReduce<double, 256> RD;
  typedef cub::BlockReduce<unsigned long long, 256> RU;
  __shared__ union { typename RD::TempStorage d; typename RU::TempStorage u; } tmp;
  const double a = RD(tmp.d).Sum(ll2);
  __syncthreads();
  const double b = RD(tmp.d).Sum(lln);
  __syncthreads();
  const unsigned long long c = RU(tmp.u).Sum(area);
  __syncthreads();
  const unsigned long long d = RU(tmp.u).Sum(twice_u);
  if (threadIdx.x == 0) {
    atomicAdd(acc_d, a);
    atomicAdd(acc_d + 1, b);
    atomicAdd(acc_u, c);
    atomicAdd(acc_u + 1, d);
  }
}

XF_DLL int xf_metric_finish(xf_metric* m, void* cuda_stream, double out[6]) {
  if (!m || !out) return XF_ERR_ARG;
  XF_CUDA_TRY(cudaSetDevice(m->device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  const uint64_t n = m->n;
  for (int i = 0; i < 6; ++i) out[i] = 0.0;
  if (n == 0) { out[0] = out[1] = out[4] = out[5] = NAN; return XF_OK; }
  if (n >= 0x7FFFFFFFull) { xf_set_error("metric: more than 2^31 predictions"); return XF_ERR_ARG; }
  XF_TRY(m->s_pctr.ensure(n * 4));
  XF_TRY(m->s_lab.ensure(n));
  XF_TRY(m->psum.ensure(n * 4));
  XF_TRY(m->start.ensure(n * 4));
  XF_TRY(m->acc.ensure(32));
  // descending by prediction, labels as payload (stable: equal predictions keep their input order)
  size_t need = 0, need2 = 0, need3 = 0;
  cub::DeviceRadixSort::SortPairsDescending(nullptr, need, m->pctr.as<float>(), m->s_pctr.as<float>(), m->lab.as<uint8_t>(),
                                            m->s_lab.as<uint8_t>(), (int)n, 0, 32, st);
  cub::DeviceScan::InclusiveSum(nullptr, need2, m->psum.as<uint32_t>(), m->psum.as<uint32_t>(), (int)n, st);
  cub::DeviceScan::InclusiveScan(nullptr, need3, m->start.as<uint32_t>(), m->start.as<uint32_t>(), XfMaxU32(), (int)n, st);
  XF_TRY(m->tmp.ensure(std::max(need, std::max(need2, need3)) + 16));
  size_t tb = m->tmp.cap;
  XF_CUDA_TRY(cub::DeviceRadixSort::SortPairsDescending(m->tmp.p, tb, m->pctr.as<float>(), m->s_pctr.as<float>(),
                                                        m->lab.as<uint8_t>(), m->s_lab.as<uint8_t>(), (int)n, 0, 32, st));
  const int grid = xf_grid_for(n, 256, 4);
  xf_k_metric_prepare<<<grid, 256, 0, st>>>(m->s_pctr.as<float>(), m->s_lab.as<uint8_t>(), n, m->psum.as<uint32_t>(),
                                            m->start.as<uint32_t>());
  tb = m->tmp.cap;
  XF_CUDA_TRY(cub::DeviceScan::InclusiveSum(m->tmp.p, tb, m->psum.as<uint32_t>(), m->psum.as<uint32_t>(), (int)n, st));
  tb = m->tmp.cap;
  XF_CUDA_TRY(cub::DeviceScan::InclusiveScan(m->tmp.p, tb, m->start.as<uint32_t>(), m->start.as<uint32_t>(), XfMaxU32(), (int)n, st));
  XF_CUDA_TRY(cudaMemsetAsync(m->acc.p, 0, 32, st));
  xf_k_metric_reduce<<<grid, 256, 0, st>>>(m->s_pctr.as<float>(), m->s_lab.as<uint8_t>(), m->psum.as<uint32_t>(),
                                           m->start.as<uint32_t>(), n, m->acc.as<double>(),
                                           reinterpret_cast<unsigned long long*>(m->acc.as<double>() + 2));
  XF_CUDA_TRY(cudaGetLastError());
  struct { double d[2]; unsigned long long u[2]; } h;
  uint32_t positives = 0;
  XF_CUDA_TRY(cudaMemcpyAsync(&h, m->acc.p, 32, cudaMemcpyDeviceToHost, st));
  XF_CUDA_TRY(cudaMemcpyAsync(&positives, m->psum.as<uint32_t>() + (n - 1), 4, cudaMemcpyDeviceToHost, st));
  XF_CUDA_TRY(cudaStreamSynchronize(st));
  const double P = (double)positives, N = (double)(n - positives);
  out[0] = h.d[0] / (double)n;
  out[2] = P;
  out[3] = N;
  out[4] = h.d[1] / (double)n;
  if (positives == 0 || positives == n) {
    out[1] = out[5] = NAN;
  } else {
    out[1] = (double)h.u[0] / (P * N);
    out[5] = (double)h.u[1] / (2.0 * P * N);
  }
  return XF_OK;
}

// one-shot convenience on device arrays
XF_DLL int xf_auc_logloss_device(const float* d_pctr, const uint8_t* d_labels, uint64_t n, int device, void* cuda_stream,
                                 double out[6]) {
  xf_metric* m = nullptr;
  XF_TRY(xf_metric_create(&m, device));
  int rc = xf_metric_add_device(m, d_pctr, d_labels, n, cuda_stream);
  if (rc == XF_OK) rc = xf_metric_finish(m, cuda_stream, out);
  xf_metric_destroy(m);
  return rc;
}

// forward pass over a row range of the current ingested block, predictions and labels appended to `m` on the
// device (lr_worker.cc:25-71 without the per-row vector push and the host sort).  pctr_out / labels_out
// (optional, host): the same values for a caller that also writes them out (pred_<rank>_<block>.txt); the call is
// asynchronous unless they are given.
XF_DLL int xf_trainer_predict_ingested_metric(xf_trainer* tr, uint32_t row_start, uint32_t row_end, xf_metric* m,
                                              float* pctr_out, uint8_t* labels_out) {
  if (!tr || !m) return XF_ERR_ARG;
  return xf_step_ingested_slice(tr, row_start, row_end, 1, m, pctr_out, labels_out, pctr_out || labels_out);
}
