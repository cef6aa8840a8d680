// Loss kernels (K3): row-wise pieces of the in-batch softmax cross-entropy (reference src/models/two_tower.py:453-479),
// the explicit-negative cross-entropy (:406-451) and compute_similarity (:380-404).  HBM/L2-bound; fp32 throughout,
// warp-level reductions, coalesced along the embedding / column dimension.
#include <cfloat>
#include "host_util.h"
#include "tc_common.cuh"
#include "../../include/b200rec.h"

namespace b200 {

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(FULL_MASK, v, o));
  return v;
}
__device__ __forceinline__ float warp_add(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  return v;
}

// one 256-thread block per row of a logits chunk S[rows, cols]:  lse[r] = logsumexp_j(scale*S[r,j]),
// pos[r] = scale*S[r, diag0 + r]
__global__ void __launch_bounds__(256)
lse_rows_kernel(const float* __restrict__ S, int64_t ld, int64_t cols, float scale, int64_t diag0,
                float* __restrict__ lse, float* __restrict__ pos) {
  __shared__ float red[8];
  const int64_t r = blockIdx.x;
  const float* row = S + r * ld;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float m = -INFINITY;
  for (int64_t j = tid; j < cols; j += 256) m = fmaxf(m, __ldg(row + j) * scale);
  m = warp_max(m);
  if (lane == 0) red[warp] = m;
  __syncthreads();
  m = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
  __syncthreads();
  float s = 0.f;
  for (int64_t j = tid; j < cols; j += 256) s += expf(__ldg(row + j) * scale - m);
  s = warp_add(s);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  if (tid == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w];
    lse[r] = m + logf(t);
    if (pos) pos[r] = __ldg(row + diag0 + r) * scale;
  }
}

// G[r,j] = coef * (exp(scale*S[r,j] - lse[r]) - [j == diag0 + r])     (in place allowed)
__global__ void __launch_bounds__(256)
softmax_grad_kernel(const float* __restrict__ S, int64_t ld, int64_t rows, int64_t cols, float scale,
                    const float* __restrict__ lse, int64_t diag0, float coef, const float* __restrict__ coef_dev,
                    float* __restrict__ G, int64_t ldg) {
  const int64_t total = rows * cols;
  if (coef_dev) coef *= __ldg(coef_dev);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols, j = i - r * cols;
    float p = expf(S[r * ld + j] * scale - __ldg(lse + r));
    if (j == diag0 + r) p -= 1.f;
    G[r * ldg + j] = p * coef;
  }
}

// sum_r (lse[r] - pos[r]) added to *acc (fp32; one block, deterministic order)
__global__ void __launch_bounds__(256)
ce_sum_kernel(const float* __restrict__ lse, const float* __restrict__ pos, int64_t n, float* __restrict__ acc) {
  __shared__ double red[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double s = 0.0;
  for (int64_t i = tid; i < n; i += 256) s += (double)lse[i] - (pos ? (double)pos[i] : 0.0);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(FULL_MASK, s, o);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += red[w];
    *acc += (float)t;
  }
}

// Explicit-negative cross-entropy, one warp per sample b:
//   logit0 = <u,p>/T + bias_sum,  logit_{1+j} = <u, n_{b,j}>/T  (no bias on negatives, two_tower.py:437-438)
//   loss_b = logsumexp(logits) - logit0 ; per-row losses are written to row_loss[b]
//   gradients (when dU != null), scaled by grad_scale:  dlogit = softmax - onehot(0)
//   dU = sum_j dlogit_j * x_j / T,  dP = dlogit_0 * u / T,  dN_j = dlogit_{1+j} * u / T,  row_dbias[b] = dlogit_0
__global__ void __launch_bounds__(256)
explicit_ce_kernel(const float* __restrict__ U, const float* __restrict__ P, const float* __restrict__ Nn, int64_t B,
                   int R, int64_t E, float inv_t, const float* __restrict__ ub, const float* __restrict__ ib, float* __restrict__ row_loss,
                   float grad_scale, const float* __restrict__ grad_scale_dev, float* __restrict__ dU,
                   float* __restrict__ dP, float* __restrict__ dN, float* __restrict__ row_dbias) {
  extern __shared__ float sm_logits[];  // [warps][R+1]
  if (grad_scale_dev) grad_scale *= __ldg(grad_scale_dev);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* logits = sm_logits + warp * (R + 1);
  const float bias_sum = (ub ? ub[0] : 0.f) + (ib ? ib[0] : 0.f);
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp; b < B; b += warps) {
    const float* u = U + b * E;
    for (int j = 0; j <= R; ++j) {
      const float* x = (j == 0) ? (P + b * E) : (Nn + (b * R + (j - 1)) * E);
      float d = 0.f;
      for (int64_t c = lane; c < E; c += 32) d = fmaf(__ldg(u + c), __ldg(x + c), d);
      d = warp_add(d);
      if (lane == 0) logits[j] = d * inv_t + (j == 0 ? bias_sum : 0.f);
    }
    __syncwarp();
    float m = -INFINITY;
    for (int j = lane; j <= R; j += 32) m = fmaxf(m, logits[j]);
    m = warp_max(m);
    float s = 0.f;
    for (int j = lane; j <= R; j += 32) s += expf(logits[j] - m);
    s = warp_add(s);
    const float lse = m + logf(s);
    if (lane == 0) row_loss[b] = lse - logits[0];
    if (dU != nullptr) {
      // overwrite logits with dlogit * grad_scale
      __syncwarp();
      for (int j = lane; j <= R; j += 32) {
        float g = expf(logits[j] - lse);
        if (j == 0) g -= 1.f;
        logits[j] = g * grad_scale;
      }
      __syncwarp();
      if (lane == 0 && row_dbias) row_dbias[b] = logits[0];
      for (int64_t c = lane; c < E; c += 32) {
        const float uc = __ldg(u + c);
        float acc = logits[0] * __ldg(P + b * E + c);
        dP[b * E + c] = logits[0] * uc * inv_t;
        for (int j = 1; j <= R; ++j) {
          const int64_t off = (b * R + (j - 1)) * E + c;
          acc = fmaf(logits[j], __ldg(Nn + off), acc);
          dN[off] = logits[j] * uc * inv_t;
        }
        dU[b * E + c] = acc * inv_t;
      }
    }
    __syncwarp();
  }
}

// out[b] = <u_b, i_b> * scale + bias_sum  (compute_similarity)
__global__ void __launch_bounds__(256)
rowdot_kernel(const float* __restrict__ U, const float* __restrict__ I, int64_t B, int64_t E, float scale,
              const float* __restrict__ ub, const float* __restrict__ ib, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const float bias_sum = (ub ? ub[0] : 0.f) + (ib ? ib[0] : 0.f);
  const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); b < B; b += warps) {
    float d = 0.f;
    for (int64_t c = lane; c < E; c += 32) d = fmaf(__ldg(U + b * E + c), __ldg(I + b * E + c), d);
    d = warp_add(d);
    if (lane == 0) out[b] = d * scale + bias_sum;
  }
}
// dU[b,:] = g[b]*scale*I[b,:], dI[b,:] = g[b]*scale*U[b,:]
__global__ void __launch_bounds__(256)
rowdot_bwd_kernel(const float* __restrict__ g, const float* __restrict__ U, const float* __restrict__ I, int64_t B,
                  int64_t E, float scale, float* __restrict__ dU, float* __restrict__ dI) {
  const int64_t total = B * E;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const float gs = __ldg(g + i / E) * scale;
    dU[i] = gs * __ldg(I + i);
    dI[i] = gs * __ldg(U + i);
  }
}

static int warp_rows_grid(int64_t rows) {
  const int64_t blocks = (rows + 7) / 8;
  const int64_t cap = (int64_t)num_sms() * 16;
  return (int)(blocks < cap ? (blocks < 1 ? 1 : blocks) : cap);
}

}  // namespace b200

using namespace b200;

extern "C" int b200rec_lse_rows(const float* S, int64_t ld, int64_t rows, int64_t cols, float scale, int64_t diag0,
                                float* lse, float* pos, void* stream) {
  if (!S || !lse) return fail("lse_rows: null pointer");
  if (rows <= 0 || cols <= 0) return fail("lse_rows: empty input");
  if (pos && (diag0 < 0 || diag0 + rows > cols)) return fail("lse_rows: diagonal outside the chunk");
  lse_rows_kernel<<<(unsigned)rows, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(S, ld, cols, scale, diag0, lse, pos);
  B200_LAUNCH_OK("lse_rows_kernel");
  return 0;
}

extern "C" int b200rec_softmax_grad(const float* S, int64_t ld, int64_t rows, int64_t cols, float scale,
                                    const float* lse, int64_t diag0, float coef, const float* coef_dev, float* G,
                                    int64_t ldg, void* stream) {
  if (!S || !lse || !G) return fail("softmax_grad: null pointer");
  if (rows <= 0 || cols <= 0) return fail("softmax_grad: empty input");
  int64_t g = (rows * cols + 255) / 256;
  const int64_t cap = (int64_t)num_sms() * 32;
  if (g > cap) g = cap;
  softmax_grad_kernel<<<(unsigned)g, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(S, ld, rows, cols, scale, lse,
                                                                                      diag0, coef, coef_dev, G, ldg);
  B200_LAUNCH_OK("softmax_grad_kernel");
  return 0;
}

extern "C" int b200rec_ce_sum(const float* lse, const float* pos, int64_t n, float* acc, void* stream) {
  if (!lse || !acc) return fail("ce_sum: null pointer");
  if (n <= 0) return fail("ce_sum: empty input");
  ce_sum_kernel<<<1, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(lse, pos, n, acc);
  B200_LAUNCH_OK("ce_sum_kernel");
  return 0;
}

extern "C" int b200rec_explicit_ce(const float* U, const float* P, const float* Nn, int64_t B, int64_t R, int64_t E,
                                   float inv_temperature, const float* user_bias, const float* item_bias, float* row_loss, float grad_scale,
                                   const float* grad_scale_dev, float* dU, float* dP, float* dN, float* row_dbias,
                                   void* stream) {
  if (!U || !P || !Nn || !row_loss) return fail("explicit_ce: null pointer");
  if (B <= 0 || R <= 0 || E <= 0) return fail("explicit_ce: empty input");
  if (R > 4095) return fail("explicit_ce: at most 4095 negatives per sample");
  if (dU && (!dP || !dN)) return fail("explicit_ce: gradient outputs must be given together");
  // one row of R + 1 logits per warp: above the 48 KB default (R >= 1536) the kernel has to opt in, up to 128 KB at
  // R = 4095.  Set per launch, not once per process: the attribute belongs to the current device.
  const size_t smem = 8 * (size_t)(R + 1) * sizeof(float);
  if (smem > 48 * 1024)
    B200_CUDA_OK(cudaFuncSetAttribute(explicit_ce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  explicit_ce_kernel<<<warp_rows_grid(B), 256, smem, reinterpret_cast<cudaStream_t>(stream)>>>(
      U, P, Nn, B, (int)R, E, inv_temperature, user_bias, item_bias, row_loss, grad_scale, grad_scale_dev, dU, dP, dN,
      row_dbias);
  B200_LAUNCH_OK("explicit_ce_kernel");
  return 0;
}

extern "C" int b200rec_rowdot(const float* U, const float* I, int64_t B, int64_t E, float scale, const float* user_bias,
                              const float* item_bias, float* out, void* stream) {
  if (!U || !I || !out) return fail("rowdot: null pointer");
  if (B <= 0 || E <= 0) return fail("rowdot: empty input");
  rowdot_kernel<<<warp_rows_grid(B), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(U, I, B, E, scale, user_bias, item_bias, out);
  B200_LAUNCH_OK("rowdot_kernel");
  return 0;
}

extern "C" int b200rec_rowdot_bwd(const float* g, const float* U, const float* I, int64_t B, int64_t E, float scale,
                                  float* dU, float* dI, void* stream) {
  if (!g || !U || !I || !dU || !dI) return fail("rowdot_bwd: null pointer");
  if (B <= 0 || E <= 0) return fail("rowdot_bwd: empty input");
  int64_t gr = (B * E + 255) / 256;
  const int64_t cap = (int64_t)num_sms() * 16;
  if (gr > cap) gr = cap;
  rowdot_bwd_kernel<<<(unsigned)gr, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(g, U, I, B, E, scale, dU, dI);
  B200_LAUNCH_OK("rowdot_bwd_kernel");
  return 0;
}
