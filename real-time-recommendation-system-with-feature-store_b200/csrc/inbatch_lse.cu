// In-batch softmax cross-entropy forward (K3): logits GEMM on tcgen05 fused with temperature scaling and an online
// log-sum-exp, so the B x NI logits matrix never leaves TMEM (reference src/models/two_tower.py:467-479 materialises
// it through matmul + div + F.cross_entropy).  Same streaming skeleton as the top-K kernel: 128*NQ user rows resident
// in shared memory, item rows streamed by TMA, one epilogue thread per user row keeps (running max, running sum) in
// registers in the log2 domain.  A CTA that covers only part of the item rows publishes a partial (m, s) pair; a tiny
// kernel merges the partials.  fp32-grade logits come from the split-bf16 operands of prep.cu (terms 3 or 6).
#include <cfloat>
#include "stream_scores.cuh"
#include "../../include/b200rec.h"

namespace b200 {

__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

struct LseEpi {
  static constexpr bool kDbg = false;
  static constexpr int SCRATCH_BYTES = 64;
  struct Args {
    float* part_m;  // [S][max_parts][128*NQ]  running max (log2 domain)
    float* part_s;  // [S][max_parts][128*NQ]  running sum of 2^(x - m)
    float scale2;   // inv_temperature * log2(e)
  };
  float m[2], s[2];

  static __device__ __forceinline__ void init_scratch(uint32_t*, int) {}
  static __device__ __forceinline__ void epilogue_exit(uint32_t*, int) {}
  template <int SLOTS, int EPI_WARPS>
  static __device__ __forceinline__ void helper(const Args&, const StreamGeom&, int, int, uint32_t*) {}

  template <int SLOTS, int QPT>
  __device__ __forceinline__ void begin_segment(const Args&, const StreamGeom&, int, int, const long long (&)[QPT],
                                                const int (&)[QPT], int, uint32_t*) {
#pragma unroll
    for (int a = 0; a < QPT; ++a) m[a] = -INFINITY, s[a] = 0.f;
  }
  template <int BN, int QPT>
  __device__ __forceinline__ void pre_tile(const Args&, const StreamGeom&, const int (&)[QPT], int, uint32_t*) {}

  template <int BN>
  __device__ __forceinline__ void tile(const Args& ea, const StreamGeom& g, int a, uint32_t taddr,
                                       unsigned long long row0) {
    const long long remaining = g.N - (long long)row0;
    const int nvalid = remaining >= BN ? BN : (int)remaining;
    const float sc = ea.scale2;
#pragma unroll 1
    for (int c = 0; c < BN; c += 32) {
      if (c >= nvalid) break;  // warp-uniform: rows beyond N are TMA zero fill, not logits
      uint32_t v[32];
      tmem_ld_32x32(taddr + c, v);
      tmem_ld_wait();
      const int lim = nvalid - c;
      float mn, acc;
      if (lim >= 32 && sc > 0.f) {
        // full group (warp-uniform): max of the raw logits with 3-input maxima (scaling by sc > 0 is monotone), then one
        // FFMA + MUFU.EX2 + FADD per logit on four independent partial sums
        float c0 = fmax3(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]));
        float c1 = fmax3(__uint_as_float(v[3]), __uint_as_float(v[4]), __uint_as_float(v[5]));
#pragma unroll
        for (int i = 6; i < 30; i += 6) {
          c0 = fmax3(c0, __uint_as_float(v[i]), __uint_as_float(v[i + 1]));
          c1 = fmax3(c1, __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
          c0 = fmaxf(c0, __uint_as_float(v[i + 4]));
          c1 = fmaxf(c1, __uint_as_float(v[i + 5]));
        }
        c0 = fmax3(c0, __uint_as_float(v[30]), __uint_as_float(v[31]));
        mn = fmaxf(m[a], fmaxf(c0, c1) * sc);
        const float nmn = -mn;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          a0 += ex2_fast(fmaf(__uint_as_float(v[i]), sc, nmn));
          a1 += ex2_fast(fmaf(__uint_as_float(v[i + 1]), sc, nmn));
          a2 += ex2_fast(fmaf(__uint_as_float(v[i + 2]), sc, nmn));
          a3 += ex2_fast(fmaf(__uint_as_float(v[i + 3]), sc, nmn));
        }
        acc = (a0 + a1) + (a2 + a3);
      } else {
        float cm = -INFINITY;
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i < lim) cm = fmaxf(cm, __uint_as_float(v[i]) * sc);
        mn = fmaxf(m[a], cm);
        acc = 0.f;
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i < lim) acc += exp2f(fmaf(__uint_as_float(v[i]), sc, -mn));
      }
      s[a] = s[a] * exp2f(m[a] - mn) + acc;
      m[a] = mn;
    }
  }

  template <int SLOTS, int QPT>
  __device__ __forceinline__ void end_segment(const Args& ea, const StreamGeom& g, int sidx, int part,
                                              const int (&qslot)[QPT], int, uint32_t*, bool) {
#pragma unroll
    for (int a = 0; a < QPT; ++a) {
      const size_t o = ((size_t)sidx * g.max_parts + part) * SLOTS + qslot[a];
      ea.part_m[o] = m[a];
      ea.part_s[o] = s[a];
    }
  }
};

template <int NQ>
__global__ void lse_merge_kernel(const StreamGeom g, const float* __restrict__ part_m, const float* __restrict__ part_s,
                                 float* __restrict__ lse) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= g.Q) return;
  const int sidx = q / (128 * NQ), slot = q - sidx * 128 * NQ;
  const int nparts = geom_last_cta(g, sidx) - geom_first_cta(g, sidx) + 1;
  float M = -INFINITY;
  for (int p = 0; p < nparts; ++p) M = fmaxf(M, part_m[((size_t)sidx * g.max_parts + p) * (128 * NQ) + slot]);
  float S = 0.f;
  for (int p = 0; p < nparts; ++p) {
    const size_t o = ((size_t)sidx * g.max_parts + p) * (128 * NQ) + slot;
    S += part_s[o] * exp2f(part_m[o] - M);
  }
  lse[q] = (M + log2f(S)) * 0.69314718055994530942f;
}

struct LsePlan {
  int nq, bn;
  StreamGeom g;
  size_t part_bytes;
};

static int plan_lse(LsePlan& p, int64_t B, int64_t NI, int64_t ld) {
  if (B <= 0 || NI <= 0) return fail("inbatch_lse: empty input");
  if (B > INT32_MAX / 2 || NI > INT32_MAX / 2) return fail("inbatch_lse: batch too large");
  if (ld <= 0 || (ld % 64)) return fail("inbatch_lse: operand leading dimension must be a multiple of 64 (got %lld)", (long long)ld);
  const int KB = (int)(ld / 64);
  const int sms = num_sms();
  bool ok = false;
  if (B > 128 && stream_geom<2, 128>(p.g, NI, (int)B, KB, sms, LseEpi::SCRATCH_BYTES) && p.g.stages >= 3) {
    p.nq = 2, p.bn = 128, ok = true;
  } else if (stream_geom<1, 256>(p.g, NI, (int)B, KB, sms, LseEpi::SCRATCH_BYTES) && p.g.stages >= 3) {
    p.nq = 1, p.bn = 256, ok = true;
  } else if (stream_geom<1, 64>(p.g, NI, (int)B, KB, sms, LseEpi::SCRATCH_BYTES) && p.g.stages >= 2) {
    p.nq = 1, p.bn = 64, ok = true;
  }
  if (!ok) return fail("inbatch_lse: operand too wide for the resident tile (ld=%lld); use fewer split terms", (long long)ld);
  p.part_bytes = (size_t)p.g.S * p.g.max_parts * 128 * p.nq * sizeof(float);
  return 0;
}

// plan_lse's choice for b200rec_debug_loss_plan: nq, bn, stages, grid, S, T, W, max_parts; all 0 when there is no fused
// plan (b200rec_inbatch_lse_workspace_bytes returns 0 and the caller takes the GEMM + lse_rows fallback)
void lse_plan_fields(int64_t B, int64_t NI, int64_t ld, long long (&v)[LSE_PLAN_FIELDS]) {
  LsePlan p;
  if (plan_lse(p, B, NI, ld)) {
    for (long long& x : v) x = 0;
    return;
  }
  const long long f[LSE_PLAN_FIELDS] = {p.nq, p.bn, p.g.stages, p.g.grid, p.g.S, p.g.T, p.g.W, p.g.max_parts};
  for (int i = 0; i < LSE_PLAN_FIELDS; ++i) v[i] = f[i];
}

template <int NQ, int BN>
static int launch_lse(const LsePlan& p, const void* U, const void* I, int64_t ld, int64_t B, int64_t NI, float inv_t,
                      float* lse, void* workspace, cudaStream_t st) {
  CUtensorMap tq, tx;
  if (make_tmap_bf16_2d(&tq, U, (uint64_t)B, (uint64_t)ld, (uint64_t)ld, 128)) return 1;
  if (make_tmap_bf16_2d(&tx, I, (uint64_t)NI, (uint64_t)ld, (uint64_t)ld, BN)) return 1;
  LseEpi::Args ea;
  ea.part_m = reinterpret_cast<float*>(workspace);
  ea.part_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + p.part_bytes);
  ea.scale2 = inv_t * 1.44269504088896340736f;
  auto kern = stream_scores_kernel<NQ, BN, LseEpi>;
  static bool attr = false;
  if (!attr) {
    B200_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, ST_SMEM_LIMIT));
    attr = true;
  }
  kern<<<p.g.grid, ST_THREADS, p.g.smem_bytes, st>>>(tq, tx, p.g, ea);
  B200_LAUNCH_OK("stream_scores_kernel<lse>");
  lse_merge_kernel<NQ><<<(unsigned)((B + 255) / 256), 256, 0, st>>>(p.g, ea.part_m, ea.part_s, lse);
  B200_LAUNCH_OK("lse_merge_kernel");
  return 0;
}

}  // namespace b200

using namespace b200;

extern "C" size_t b200rec_inbatch_lse_workspace_bytes(int64_t B, int64_t NI, int64_t ld) {
  LsePlan p;
  if (plan_lse(p, B, NI, ld)) return 0;
  return 2 * p.part_bytes;
}

extern "C" int b200rec_inbatch_lse(const void* U_op, const void* I_op, int64_t ld, int64_t B, int64_t NI,
                                   float inv_temperature, float* lse_out, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  if (!U_op || !I_op || !lse_out || !workspace) return fail("inbatch_lse: null pointer");
  LsePlan p;
  if (plan_lse(p, B, NI, ld)) return 1;
  if (workspace_bytes < 2 * p.part_bytes) return fail("inbatch_lse: workspace too small");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (p.nq == 2) return launch_lse<2, 128>(p, U_op, I_op, ld, B, NI, inv_temperature, lse_out, workspace, st);
  if (p.bn == 256) return launch_lse<1, 256>(p, U_op, I_op, ld, B, NI, inv_temperature, lse_out, workspace, st);
  return launch_lse<1, 64>(p, U_op, I_op, ld, B, NI, inv_temperature, lse_out, workspace, st);
}
