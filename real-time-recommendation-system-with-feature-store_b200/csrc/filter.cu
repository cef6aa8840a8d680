// Row filters of the flat index (filtered exact top-K, csrc/topk.cu).
//   rows_to_bitmap : set of LOCAL rows -> bitmap in faiss' IDSelectorBitmap layout (bit r = bit r&7 of byte r>>3, i.e.
//                    bit r&31 of little-endian word r>>5); rows outside [0, n_bits) are ignored, duplicates are harmless
//   remap_ids      : ids of a search over a compacted catalogue (row j = catalogue row rows[j]) -> catalogue ids; the row
//                    list is increasing, so the (score desc, row asc) order of the compact search is kept
#include "host_util.h"
#include "../../include/b200rec.h"

namespace b200 {

__global__ void __launch_bounds__(256)
rows_to_bitmap_kernel(const int64_t* __restrict__ rows, int64_t n, int64_t n_bits, uint32_t* __restrict__ bits) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = __ldg(rows + i);
    if (r >= 0 && r < n_bits) atomicOr(bits + (r >> 5), 1u << (r & 31));
  }
}

__global__ void __launch_bounds__(256)
remap_ids_kernel(const int64_t* ids, int64_t n, const int64_t* __restrict__ rows, int64_t n_rows, int64_t row_offset,
                 int64_t* out) {  // ids may alias out
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = ids[i];
    out[i] = (j >= 0 && j < n_rows) ? __ldg(rows + j) + row_offset : -1;
  }
}

static int grid_for(int64_t n) {
  const int64_t blocks = (n + 255) / 256;
  const int64_t cap = (int64_t)num_sms() * 8;
  return (int)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
}

}  // namespace b200

extern "C" int b200rec_rows_to_bitmap(const int64_t* rows, int64_t n, int64_t n_bits, uint32_t* bits, void* stream) {
  using namespace b200;
  if (!bits || (!rows && n > 0)) return fail("rows_to_bitmap: null pointer");
  if (n < 0 || n_bits <= 0) return fail("rows_to_bitmap: n must be >= 0 and n_bits > 0");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  B200_CUDA_OK(cudaMemsetAsync(bits, 0, (size_t)((n_bits + 31) / 32) * sizeof(uint32_t), st));
  if (n == 0) return 0;
  rows_to_bitmap_kernel<<<grid_for(n), 256, 0, st>>>(rows, n, n_bits, bits);
  B200_LAUNCH_OK("rows_to_bitmap_kernel");
  return 0;
}

extern "C" int b200rec_remap_ids(const int64_t* ids, int64_t n, const int64_t* rows, int64_t n_rows, int64_t row_offset,
                                 int64_t* out, void* stream) {
  using namespace b200;
  if (!ids || !rows || !out) return fail("remap_ids: null pointer");
  if (n <= 0 || n_rows <= 0) return fail("remap_ids: empty input");
  remap_ids_kernel<<<grid_for(n), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(ids, n, rows, n_rows, row_offset, out);
  B200_LAUNCH_OK("remap_ids_kernel");
  return 0;
}
