// In-place mutation of the flat index (FlatIPDeviceIndex.update_rows / remove_rows).  Row slots never move: a removal
// clears the slot's bit in the index's live-row bitmap (IDSelectorBitmap layout, the one the filtered top-K tests), an
// update overwrites the slot and sets its bit again.
//   update_rows      : the row pass of b200rec_normalize_rows (prep.cu) with a destination row list and the live bits set
//                      in the same launch
//   clear_row_bits   : the row-bit kernel of b200rec_rows_to_bitmap (filter.cu), clearing instead of setting, in place
//   patch_compacted  : keeps a row filter's compacted operand (one row per allowed row, rows ascending) in step with the
//                      index: every changed row is looked up in the filter's row list; found, an update copies the new
//                      operand row into the compact row and sets its compact live bit, a removal clears that bit
#include "host_util.h"
#include "tc_common.cuh"
#include "../../include/b200rec.h"

namespace b200 {

// one warp per changed row: binary search (every lane the same probes, no shuffle) then a 16-byte-vector row copy
__global__ void __launch_bounds__(256)
patch_compacted_kernel(const int64_t* __restrict__ changed, int64_t n_changed, const int64_t* __restrict__ frows,
                       int64_t n_filter, const uint4* __restrict__ operand, int64_t row_vec, uint4* __restrict__ compact,
                       uint32_t* __restrict__ bits, int update) {
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < n_changed; i += warps_total) {
    const int64_t r = __ldg(changed + i);
    int64_t lo = 0, hi = n_filter;
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (__ldg(frows + mid) < r) lo = mid + 1;
      else hi = mid;
    }
    if (lo >= n_filter || __ldg(frows + lo) != r) continue;
    if (update) {
      const uint4* s = operand + r * row_vec;
      uint4* d = compact + lo * row_vec;
      for (int64_t c = lane; c < row_vec; c += 32) d[c] = __ldg(s + c);
      if (bits && lane == 0) atomicOr(bits + (lo >> 5), 1u << (lo & 31));
    } else if (lane == 0) {
      atomicAnd(bits + (lo >> 5), ~(1u << (lo & 31)));
    }
  }
}

}  // namespace b200

extern "C" int b200rec_update_rows(const float* src, int64_t rows, int64_t cols, int64_t ld_src, int normalize,
                                   const int64_t* dst_rows, int64_t n_slots, float* dst_f32, int64_t ld_f32,
                                   void* dst_bf16, int64_t kpad, int terms, int side, uint32_t* live_bits,
                                   void* stream) {
  using namespace b200;
  if (!src || !dst_rows || !dst_bf16) return fail("update_rows: null pointer");
  if (rows <= 0 || cols <= 0) return fail("update_rows: empty input");
  if (n_slots <= 0) return fail("update_rows: n_slots must be > 0");
  if (ld_src < cols || (dst_f32 && ld_f32 < cols)) return fail("update_rows: leading dimensions must be >= cols");
  return launch_prep_rows(src, rows, cols, ld_src, normalize, 1, dst_f32, ld_f32, nullptr, dst_bf16, kpad, terms, side,
                          dst_rows, n_slots, live_bits, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int b200rec_clear_row_bits(const int64_t* rows, int64_t n, int64_t n_bits, uint32_t* bits, void* stream) {
  using namespace b200;
  if (!rows || !bits) return fail("clear_row_bits: null pointer");
  if (n < 0 || n_bits <= 0) return fail("clear_row_bits: n must be >= 0 and n_bits > 0");
  if (n == 0) return 0;
  return launch_row_bits(rows, n, n_bits, bits, 0, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int b200rec_patch_compacted(const int64_t* changed_rows, int64_t n_changed, const int64_t* filter_rows,
                                       int64_t n_filter, const void* operand, int64_t ld, void* compact,
                                       uint32_t* compact_bits, int update, void* stream) {
  using namespace b200;
  if (!changed_rows || !filter_rows) return fail("patch_compacted: null pointer");
  if (update ? (!operand || !compact) : !compact_bits)
    return fail("patch_compacted: null pointer (an update needs both operands, a removal the compact bitmap)");
  if (n_changed < 0 || n_filter <= 0) return fail("patch_compacted: n_changed must be >= 0 and n_filter > 0");
  if (update && (ld <= 0 || ld % 8)) return fail("patch_compacted: ld must be a positive multiple of 8");
  if (n_changed == 0) return 0;
  const int64_t blocks = (n_changed + 7) / 8;
  const int grid = (int)(blocks < (int64_t)num_sms() * 16 ? blocks : (int64_t)num_sms() * 16);
  patch_compacted_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      changed_rows, n_changed, filter_rows, n_filter, reinterpret_cast<const uint4*>(operand), ld / 8,
      reinterpret_cast<uint4*>(compact), compact_bits, update);
  B200_LAUNCH_OK("patch_compacted_kernel");
  return 0;
}
