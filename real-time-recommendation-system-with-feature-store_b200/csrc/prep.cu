// Operand preparation: fp32 -> bf16 tensor-core operands (optionally L2-normalised, optionally transposed,
// optionally expanded into split-bf16 terms so that a bf16 GEMM reproduces fp32 products).
//   x = h + m + l exactly, h = bf16(x), m = bf16(x-h), l = bf16(x-h-m)
//   terms 1: left [h]            right [h]
//   terms 3: left [h m h]        right [m h h]          (products h.m, m.h, h.h: error ~2^-17 per product)
//   terms 6: left [m l h m h h]  right [m h l h m h]    (drops only m*l, l*m, l*l: ~2^-24, i.e. fp32 grade)
// Each block is kpad columns wide (zero padded), so left . right^T over K = terms*kpad is the fp32 product sum.
// Blocks are ordered SMALLEST piece product first: a tcgen05 accumulator chain adds with truncation, so every add made
// while the partial sum is still ~2^-8 (or 2^-16) of the final value costs nothing, and only the last h.h blocks
// truncate at full magnitude (E = 128, 6 terms: 8 full-magnitude adds instead of 48; the bias of a logit fell 6x).
// HBM-bound elementwise kernels: one warp per row, coalesced loads, 2-byte stores coalesced along the row.
#include "host_util.h"
#include "tc_common.cuh"
#include "../../include/b200rec.h"

namespace b200 {

__device__ __forceinline__ void split3(float x, __nv_bfloat16& h, __nv_bfloat16& m, __nv_bfloat16& l) {
  h = __float2bfloat16_rn(x);
  const float r1 = x - __bfloat162float(h);
  m = __float2bfloat16_rn(r1);
  const float r2 = r1 - __bfloat162float(m);
  l = __float2bfloat16_rn(r2);
}

// which part (0=h,1=m/lo,2=l) goes into block t for (terms, side)
__device__ __forceinline__ int part_of(int terms, int side, int t) {
  if (terms == 1) return 0;
  if (terms == 3) {
    const int L[3] = {0, 1, 0}, R[3] = {1, 0, 0};
    return side == 0 ? L[t] : R[t];
  }
  const int L6[6] = {1, 2, 0, 1, 0, 0}, R6[6] = {1, 0, 2, 0, 1, 0};
  return side == 0 ? L6[t] : R6[t];
}

__device__ __forceinline__ void store_terms(__nv_bfloat16* drow, int64_t c, int64_t kpad, int terms, int side,
                                            float x) {
  __nv_bfloat16 p[3];
  split3(x, p[0], p[1], p[2]);
#pragma unroll
  for (int t = 0; t < 6; ++t)
    if (t < terms) drow[t * kpad + c] = p[part_of(terms, side, t)];
}

__device__ __forceinline__ uint32_t pack2(__nv_bfloat16 a, __nv_bfloat16 b) {
  return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL_MASK, v, o);
  return v;
}

// one warp per row.  dst_rows (nullable): source row r is written to destination row dst_rows[r] of dst_f32 / dst_bf16
// (rows outside [0, n_dst) are skipped) and, when live_bits is given, that row's bit is set (in-place catalogue updates,
// csrc/mutate.cu); norms_out stays indexed by the source row
__global__ void __launch_bounds__(256)
prep_rows_kernel(const float* __restrict__ src, int64_t rows, int64_t cols, int64_t ld_src, int normalize,
                 int faiss_zero_rule, float* __restrict__ dst_f32, int64_t ld_dst, float* __restrict__ norms_out,
                 __nv_bfloat16* __restrict__ dst_bf16, int64_t kpad, int terms, int side,
                 const int64_t* __restrict__ dst_rows, int64_t n_dst, uint32_t* __restrict__ live_bits) {
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
  const bool vec_ok = ((ld_src & 3) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0) &&
                      ((reinterpret_cast<uintptr_t>(dst_bf16) & 15) == 0) && ((kpad & 7) == 0);
  for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < rows; r += warps_total) {
    const float* srow = src + r * ld_src;
    const int64_t dr = dst_rows ? __ldg(dst_rows + r) : r;
    if (dst_rows && (dr < 0 || dr >= n_dst)) continue;
    if (live_bits && lane == 0) atomicOr(live_bits + (dr >> 5), 1u << (dr & 31));
    float scale = 1.0f, denom = 1.0f;
    if (normalize) {
      float ss = 0.f;
      for (int64_t c = lane; c < cols; c += 32) {
        const float x = __ldg(srow + c);
        ss = fmaf(x, x, ss);
      }
      ss = warp_sum(ss);
      float nrm = sqrtf(ss);
      if (faiss_zero_rule) {
        // faiss::fvec_renorm_L2: x *= 1/sqrt(sum x^2) when the norm is > 0  (retrieval.py:86,167,214)
        scale = (ss > 0.f) ? (1.0f / nrm) : 1.0f;
        if (norms_out && lane == 0) norms_out[r] = nrm;
      } else {
        // F.normalize(p=2, eps=1e-12): x / max(||x||, eps)  (two_tower.py:132,279)
        nrm = fmaxf(nrm, 1e-12f);
        denom = nrm;
        if (norms_out && lane == 0) norms_out[r] = nrm;
      }
    }
    __nv_bfloat16* drow = dst_bf16 ? dst_bf16 + dr * terms * kpad : nullptr;
    if (drow && vec_ok) {
      // 8 columns per lane: two 128-bit loads, one 128-bit store per term block (2-byte stores ran at 1 TB/s)
      for (int64_t c = (int64_t)lane * 8; c < kpad; c += 256) {
        float x[8];
        if (c + 8 <= cols) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(srow + c));
          const float4 b = __ldg(reinterpret_cast<const float4*>(srow + c + 4));
          x[0] = a.x, x[1] = a.y, x[2] = a.z, x[3] = a.w, x[4] = b.x, x[5] = b.y, x[6] = b.z, x[7] = b.w;
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) x[j] = (c + j < cols) ? __ldg(srow + c + j) : 0.f;
        }
        __nv_bfloat16 p[3][8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (normalize) x[j] = faiss_zero_rule ? x[j] * scale : x[j] / denom;
          if (dst_f32 && c + j < cols) dst_f32[dr * ld_dst + c + j] = x[j];
          split3(x[j], p[0][j], p[1][j], p[2][j]);
        }
#pragma unroll
        for (int t = 0; t < 6; ++t) {
          if (t < terms) {
            const int part = part_of(terms, side, t);
            uint4 o;
            const __nv_bfloat16* q = part == 0 ? p[0] : (part == 1 ? p[1] : p[2]);
            o.x = pack2(q[0], q[1]), o.y = pack2(q[2], q[3]), o.z = pack2(q[4], q[5]), o.w = pack2(q[6], q[7]);
            *reinterpret_cast<uint4*>(drow + t * kpad + c) = o;
          }
        }
      }
      continue;
    }
    const int64_t cmax = dst_bf16 ? kpad : cols;
    for (int64_t c = lane; c < cmax; c += 32) {
      float x = 0.f;
      if (c < cols) {
        x = __ldg(srow + c);
        if (normalize) x = faiss_zero_rule ? x * scale : x / denom;
        if (dst_f32) dst_f32[dr * ld_dst + c] = x;
      }
      if (drow) store_terms(drow, c, kpad, terms, side, x);
    }
  }
}

// dst[r, c] = src[c, r]   (src has `cols` rows of `rows` floats).  One block = 32 dst rows x 128 dst columns: the source
// tile is transposed on its way into shared memory (row stride 132 floats keeps the rows 16-byte aligned), every lane
// then reads four consecutive columns with one 128-bit shared load and stores them as one 8-byte bf16x4 per term block:
// 256 B per warp and store instead of 64-128 B.
__global__ void __launch_bounds__(256)
prep_transpose_kernel(const float* __restrict__ src, int64_t rows, int64_t cols, int64_t ld_src,
                      __nv_bfloat16* __restrict__ dst, int64_t kpad, int terms, int side) {
  __shared__ __align__(16) float tile[32][132];
  const int64_t r0 = (int64_t)blockIdx.y * 32;   // dst rows   = src columns
  const int64_t c0 = (int64_t)blockIdx.x * 128;  // dst cols   = src rows
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
#pragma unroll 4
  for (int i = ty; i < 128; i += 8) {
    const int64_t sr = c0 + i, sc = r0 + tx;
    tile[tx][i] = (sr < cols && sc < rows) ? __ldg(src + sr * ld_src + sc) : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int i = ty; i < 32; i += 8) {
    const int64_t r = r0 + i, c = c0 + 4 * tx;
    if (r < rows && c < kpad) {   // kpad is a multiple of 8 and c of 4: c + 3 < kpad
      const float4 x = *reinterpret_cast<const float4*>(&tile[i][4 * tx]);
      __nv_bfloat16 p0[3], p1[3], p2[3], p3[3];
      split3(x.x, p0[0], p0[1], p0[2]);
      split3(x.y, p1[0], p1[1], p1[2]);
      split3(x.z, p2[0], p2[1], p2[2]);
      split3(x.w, p3[0], p3[1], p3[2]);
      __nv_bfloat16* drow = dst + r * terms * kpad;
#pragma unroll
      for (int t = 0; t < 6; ++t) {
        if (t < terms) {
          const int part = part_of(terms, side, t);
          uint2 o;
          o.x = pack2(p0[part], p1[part]);
          o.y = pack2(p2[part], p3[part]);
          *reinterpret_cast<uint2*>(drow + t * kpad + c) = o;
        }
      }
    }
  }
}

static int check_terms(int terms, int side) {
  if (terms != 1 && terms != 3 && terms != 6) return fail("terms must be 1, 3 or 6 (got %d)", terms);
  if (side != 0 && side != 1) return fail("side must be 0 (left) or 1 (right)");
  return 0;
}

// the row pass of b200rec_normalize_rows with a destination row list (b200rec_update_rows, csrc/mutate.cu)
int launch_prep_rows(const float* src, int64_t rows, int64_t cols, int64_t ld_src, int normalize, int faiss_zero_rule,
                     float* dst_f32, int64_t ld_dst, float* norms_out, void* dst_bf16, int64_t kpad, int terms, int side,
                     const int64_t* dst_rows, int64_t n_dst, uint32_t* live_bits, cudaStream_t st) {
  if (dst_bf16) {
    if (kpad < cols || (kpad % 8)) return fail("normalize_rows: kpad must be >= cols and a multiple of 8");
    if (check_terms(terms, side)) return 1;
  }
  const int64_t blocks = (rows + 7) / 8;
  const int grid = (int)(blocks < (int64_t)num_sms() * 16 ? blocks : (int64_t)num_sms() * 16);
  prep_rows_kernel<<<grid, 256, 0, st>>>(src, rows, cols, ld_src, normalize, faiss_zero_rule, dst_f32, ld_dst,
                                         norms_out, reinterpret_cast<__nv_bfloat16*>(dst_bf16), kpad, terms, side,
                                         dst_rows, n_dst, live_bits);
  B200_LAUNCH_OK("prep_rows_kernel");
  return 0;
}

}  // namespace b200

extern "C" int b200rec_split_bf16(const float* src, int64_t rows, int64_t cols, int64_t ld_src, int transpose,
                                  void* dst, int64_t kpad, int terms, int side, void* stream) {
  using namespace b200;
  if (!src || !dst) return fail("split_bf16: null pointer");
  if (rows <= 0 || cols <= 0) return fail("split_bf16: empty input");
  if (kpad < cols || (kpad % 8)) return fail("split_bf16: kpad must be >= cols and a multiple of 8");
  if (check_terms(terms, side)) return 1;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (!transpose) {
    const int64_t blocks = (rows + 7) / 8;
    const int grid = (int)(blocks < (int64_t)num_sms() * 16 ? blocks : (int64_t)num_sms() * 16);
    prep_rows_kernel<<<grid, 256, 0, st>>>(src, rows, cols, ld_src, 0, 0, nullptr, 0, nullptr,
                                           reinterpret_cast<__nv_bfloat16*>(dst), kpad, terms, side, nullptr, 0, nullptr);
    B200_LAUNCH_OK("prep_rows_kernel");
  } else {
    dim3 grid((unsigned)((kpad + 127) / 128), (unsigned)((rows + 31) / 32));
    if (grid.y > 65535) return fail("split_bf16(transpose): too many rows (%lld)", (long long)rows);
    prep_transpose_kernel<<<grid, 256, 0, st>>>(src, rows, cols, ld_src, reinterpret_cast<__nv_bfloat16*>(dst), kpad,
                                                terms, side);
    B200_LAUNCH_OK("prep_transpose_kernel");
  }
  return 0;
}

extern "C" int b200rec_normalize_rows(const float* src, int64_t rows, int64_t cols, int64_t ld_src, int normalize,
                                      int faiss_zero_rule, float* dst_f32, int64_t ld_dst, float* norms_out,
                                      void* dst_bf16, int64_t kpad, int terms, int side, void* stream) {
  using namespace b200;
  if (!src) return fail("normalize_rows: null src");
  if (rows <= 0 || cols <= 0) return fail("normalize_rows: empty input");
  return launch_prep_rows(src, rows, cols, ld_src, normalize, faiss_zero_rule, dst_f32, ld_dst, norms_out, dst_bf16,
                          kpad, terms, side, nullptr, 0, nullptr, reinterpret_cast<cudaStream_t>(stream));
}
