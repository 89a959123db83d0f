// The textbook factorisation machine with feature values — NOT the reference's model (which ignores `val` and
// collapses the interaction over k, fm_worker.cc:177-196; that is XF_MODEL_FM in step.cu), offered as the
// non-parity option SURVEY.md section 8f-4 names:
//     y = sum_i w_i x_i + 1/2 sum_k [ (sum_i v_ik x_i)^2 - sum_i (v_ik x_i)^2 ]
//     dL/dw_i = r x_i ,  dL/dv_ik = r x_i (S_k - v_ik x_i) = r x_i S_k - v_ik r x_i^2        r = sigmoid(y) - label
// Per key the batch therefore needs G = sum r x, L2 = sum r x^2 (doubles, in the row's g / L slots) and
// A_k = sum r x S_k (K floats behind the optimizer state, canonical tables only): gv_k = A_k - v_k L2.
//
// One warp per row, C = K/4 lanes per token (each holds 4 latent coordinates = one 16-byte piece of the row: the
// C lanes of a token read its latent row with ONE instruction), 32/C tokens per pass.  Pass 1: pull + per-k sums;
// warp reductions; sigmoid.  Pass 2: the per-key sums with L2 atomics (one float4 RED per lane for A, two f64
// atomics per token for G / L2); the token that finds G untouched records the slot for xf_k_update.
#include <cuda_runtime.h>
#include <stdint.h>

#include "kernels.h"
#include "table.cuh"

#define XF_NO_SLOT 0xFFFFFFFFu

__global__ void __launch_bounds__(256)
xf_k_step_fmc(XfTableView t, const uint32_t* __restrict__ row_ptr, const uint64_t* __restrict__ keys,
              const float* __restrict__ vals, const uint8_t* __restrict__ labels, int B, int mode,
              uint32_t* __restrict__ touched, float* __restrict__ loss_out, float* __restrict__ pctr_out,
              float* __restrict__ abs_loss_sum) {
  __shared__ float s_abs[8];
  float abs_acc = 0.f;
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  const int gwarp = blockIdx.x * wpb + (threadIdx.x >> 5);
  const int nwarps = gridDim.x * wpb;
  const int K = t.K;
  const int C = K >> 2;          // lanes per token (power of two, <= 32)
  const int T = 32 / C;          // tokens per pass
  const int c = lane & (C - 1);  // which 4 coordinates
  const int tg = lane / C;       // which token of the pass
  const int lead = lane & ~(C - 1);

  for (int row = gwarp; row < B; row += nwarps) {
    const uint32_t beg = __ldg(row_ptr + row), end = __ldg(row_ptr + row + 1);
    float S[4] = {0.f, 0.f, 0.f, 0.f};
    float Q = 0.f, wx = 0.f;
    // ---------------- pass 1: pull, per-k sums
    for (uint32_t j0 = beg; j0 < end; j0 += (uint32_t)T) {
      const uint32_t j = j0 + (uint32_t)tg;
      const bool live = j < end;
      uint32_t slot = XF_NO_SLOT, flags = 0;
      uint64_t key = 0;
      float w = 0.f;
      if (live && c == 0) {
        key = __ldcs(keys + j);
        XfHead h;
        const int64_t r = xf_probe<true>(t, key, &h);
        if (r >= 0) { slot = (uint32_t)r; flags = h.flags; w = h.w; }
        touched[j] = slot;  // remembered for pass 2 (overwritten there with the first-touch marker)
      }
      slot = __shfl_sync(0xffffffffu, slot, lead);
      flags = __shfl_sync(0xffffffffu, flags, lead);
      key = __shfl_sync(0xffffffffu, (unsigned long long)key, lead);
      if (!live || slot == XF_NO_SLOT) continue;
      const float x = vals ? __ldg(vals + j) : 1.0f;
      float4 v;
      if (flags & XF_FLAG_V_READY) v = __ldcg(reinterpret_cast<const float4*>(xf_row(t, slot) + 32) + c);
      else v = make_float4(xf_v_init(t, key, 4 * c), xf_v_init(t, key, 4 * c + 1), xf_v_init(t, key, 4 * c + 2), xf_v_init(t, key, 4 * c + 3));
      const float a0 = v.x * x, a1 = v.y * x, a2 = v.z * x, a3 = v.w * x;
      S[0] += a0; S[1] += a1; S[2] += a2; S[3] += a3;
      Q += a0 * a0 + a1 * a1 + a2 * a2 + a3 * a3;
      if (c == 0) wx += w * x;
    }
    // S_k over the tokens (lanes with the same c), sum_k S_k^2 over the c's, Q and wx over the warp
#pragma unroll
    for (int e = 0; e < 4; ++e)
      for (int o = C; o < 32; o <<= 1) S[e] += __shfl_xor_sync(0xffffffffu, S[e], o);
    float s2 = S[0] * S[0] + S[1] * S[1] + S[2] * S[2] + S[3] * S[3];
    for (int o = 1; o < C; o <<= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    Q = xf_warp_sum(Q);
    wx = xf_warp_sum(wx);
    const float pctr = xf_sigmoid(wx + 0.5f * (s2 - Q));
    if (mode == 1) {
      if (lane == 0 && pctr_out) pctr_out[row] = pctr;
      continue;
    }
    const float loss = pctr - (float)labels[row];
    if (lane == 0 && loss_out) loss_out[row] = loss;
    abs_acc += fabsf(loss);
    // ---------------- pass 2: per-key sums
    for (uint32_t j0 = beg; j0 < end; j0 += (uint32_t)T) {
      const uint32_t j = j0 + (uint32_t)tg;
      const bool live = j < end;
      uint32_t slot = XF_NO_SLOT;
      if (live && c == 0) slot = touched[j];
      slot = __shfl_sync(0xffffffffu, slot, lead);
      if (!live || slot == XF_NO_SLOT) continue;
      const float x = vals ? __ldg(vals + j) : 1.0f;
      uint8_t* rowp = xf_row(t, slot);
      const float rx = loss * x;
      atomicAdd(reinterpret_cast<float4*>(xf_row_ca(t, rowp)) + c, make_float4(rx * S[0], rx * S[1], rx * S[2], rx * S[3]));
      if (c == 0) {
        // + 0.0 turns a -0.0 term (x = 0 with a negative residual) into +0.0: it must not leave the "untouched"
        // marker in place, or a later token of the key would list the row in touched[] a second time
        const double old = atomicAdd(xf_row_g(rowp), __dadd_rn((double)loss * (double)x, 0.0));
        atomicAdd(xf_row_acc(rowp, K), (double)loss * (double)x * (double)x);
        touched[j] = ((unsigned long long)__double_as_longlong(old) == XF_NEG_ZERO_BITS64) ? slot : XF_NO_SLOT;
      }
    }
  }
  if (abs_loss_sum != nullptr && mode == 0) {
    if (lane == 0) s_abs[threadIdx.x >> 5] = abs_acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      float tot = 0.f;
      for (int w = 0; w < wpb; ++w) tot += s_abs[w];
      atomicAdd(abs_loss_sum, tot);
    }
  }
}

void xf_launch_step_fmc(const XfTableView& t, const uint32_t* row_ptr, const uint64_t* keys, const float* vals,
                        const uint8_t* labels, int B, int mode, uint32_t* touched, float* loss_out, float* pctr_out,
                        float* abs_loss_sum, cudaStream_t st) {
  if (B <= 0) return;
  xf_k_step_fmc<<<xf_grid_for((uint64_t)B * 32, 256, 8), 256, 0, st>>>(t, row_ptr, keys, vals, labels, B, mode, touched,
                                                                        loss_out, pctr_out, abs_loss_sum);
}
