// Host-side helpers shared by the C-ABI translation units: error string, launch counter, TMA descriptors.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdint>

namespace b200 {

extern thread_local char g_err[512];
extern std::atomic<long long> g_launches;

inline int fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}

#define B200_CUDA_OK(expr)                                                                     \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) return b200::fail("%s failed: %s", #expr, cudaGetErrorString(_e));  \
  } while (0)

#define B200_LAUNCH_OK(name)                                                                   \
  do {                                                                                         \
    b200::g_launches.fetch_add(1, std::memory_order_relaxed);                                  \
    cudaError_t _e = cudaGetLastError();                                                       \
    if (_e != cudaSuccess) return b200::fail("launch %s failed: %s", name, cudaGetErrorString(_e)); \
  } while (0)

inline int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// 2-D bf16 row-major tensor [rows, cols] with leading dimension ld (elements); box = [box_rows, 64 cols],
// 128-byte swizzle — the layout the UMMA K-major SW128 descriptors in tc_common.cuh expect.
// Out-of-bounds rows/cols are zero-filled by the TMA unit.
int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_rows);

// the fused in-batch log-sum-exp plan of (B, NI, ld), for the loss plan query (inbatch_lse.cu)
constexpr int LSE_PLAN_FIELDS = 8;
void lse_plan_fields(int64_t B, int64_t NI, int64_t ld, long long (&v)[LSE_PLAN_FIELDS]);

// launchers shared across translation units: the row pass of prep.cu (dst_rows / live_bits nullable) and the row-bit
// kernel of filter.cu (set = 1 sets, 0 clears); both validate nothing beyond what their C-ABI callers checked
int launch_prep_rows(const float* src, int64_t rows, int64_t cols, int64_t ld_src, int normalize, int faiss_zero_rule,
                     float* dst_f32, int64_t ld_dst, float* norms_out, void* dst_bf16, int64_t kpad, int terms, int side,
                     const int64_t* dst_rows, int64_t n_dst, uint32_t* live_bits, cudaStream_t st);
int launch_row_bits(const int64_t* rows, int64_t n, int64_t n_bits, uint32_t* bits, int set, cudaStream_t st);

}  // namespace b200
