// Fused backward of the in-batch negative loss (K3, reference src/models/two_tower.py:453-479: S = U.V^T / T,
// CE(S, arange) — what torch autograd turns into softmax(S) - onehot followed by two GEMMs).  Flash-style: the logits
// tile is RECOMPUTED on the tensor cores (tcgen05, accumulator in TMEM), turned into G = coef * (exp(S/T - lse) - onehot)
// in registers, written back to TENSOR MEMORY as split-bf16 pieces (tcgen05.st) and contracted from there — as the TMEM
// A operand of a tcgen05.mma — with the other side's embeddings into the gradient accumulator (also TMEM).  Neither S,
// nor the probabilities, nor G ever reach HBM or shared memory: the kernel reads 2 x (B + NI) x E operand pieces and
// writes the two [rows, E] gradients.
//
//   out[r, :] = sum_c G[r, c] * Y[c, :]      rows r from X (a 128-row tile resident in shared memory), columns c from Y
//   mode U: X = U, Y = V, lse indexed by row,    one-hot at c == r + diag0          ->  dU
//   mode V: X = V, Y = U, lse indexed by column, one-hot at c == r - diag0          ->  dV
// Both modes run in ONE launch (work units of equal length: a 128-row X tile x a range of 64-column Y tiles; when a
// tile's columns are split over several units — data parallel: 8192 local users x 65536 gathered items — the partial
// gradients are combined with fp32 atomics into a pre-zeroed output).
//
// Per CTA: warp 0 TMA producer, warp 1 MMA issuer (one elected lane), warp 2 TMEM allocator, warps 4-19 epilogue in two
// groups of 8 (group = tile parity; warp = TMEM lane quarter x 32-column half of the logits tile).  Pipeline per Y tile t:
//   TMA: Y operand pieces -> stage t % NST (the SAME tile feeds both GEMMs)                          full / empty
//   MMA: S(t+2) = X . Y(t+2)^T  (split-bf16 products h.h + m.h + h.m [+ l.h + h.l + m.m]), B K-major  s_full / s_empty
//   epi: S(t) -> G(t) pieces (h, m) -> TMEM columns of G buffer t % 2 (tcgen05.st)                   g_full / g_empty
//   MMA: OUT[t % NACC] += G(t) . Y(t)   A = G from TMEM (TS form), B = the Y tile read MN-major (N = E contiguous,
//        K = tile rows); NACC accumulators: tcgen05 adds with truncation, short chains stay exact
// Everything the MMA-issuing warp computes per tile is a compile-time constant of IgCfg<E, NPS, NPG>.
// fp32-grade numerics as everywhere in this library: operands are exact sums of bf16 pieces, products of pieces are
// exact in the tensor core, only the dropped piece products (<= 2^-17 relative for 3 products) and fp32 accumulation
// remain.  History and ncu evidence: profiles/r02_inbatch_grad_history.md.
#include "host_util.h"
#include "tc_common.cuh"
#include "../../include/b200rec.h"

namespace b200 {

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// D[tmem] (+)= A[tmem] * B[smem]: the A operand (128 lanes x K bf16, two per 32-bit column) comes from tensor memory
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 32 lanes x 8 consecutive 32-bit columns: thread t of the warp writes TMEM lane (base_lane + t)
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

constexpr int IG_EPI_WARPS = 16;                 // epilogue warps: 4 per TMEM lane quarter, 16 logit columns each
constexpr int IG_THREADS = (4 + IG_EPI_WARPS) * 32;
constexpr int IG_BM = 128;        // X rows per unit
constexpr int IG_BN = 64;         // Y rows (logit columns) per tile
constexpr int IG_MAX_UNIT_TILES = 128;   // <= 8192 columns per unit: bounds the accumulator chains (see NACC)
constexpr int IG_SMEM_LIMIT = 232448;

struct IgSide {
  int rows;            // rows of X in this mode
  int ycols;           // rows of Y (= logit columns)
  int x_tiles;         // ceil(rows / 128)
  int splits;          // units per X tile
  int tiles_per_unit;  // Y tiles per unit
  int dshift;          // one-hot column = global row + dshift
  int lse_by_col;
  int xp[3];           // 64-column block index of pieces h, m, l inside X's operand rows
  int yp[3];           // same for Y's operand rows
  float* out;
  long long ld_out;
};

struct IgArgs {
  IgSide side[2];
  int units_u;         // units of mode U come first
  int atomic_u, atomic_v;
  float scale_log2;    // inv_t * log2(e)
  float coef;          // inv_t / total_rows (times *coef_dev when given)
  const float* coef_dev;
  const float* lse;    // [B] fp32 (natural log)
};

// Compile-time geometry of one instantiation: E = embedding width, NPS / NPG = piece products of the logits recompute
// and of the gradient GEMM.  Everything the MMA-issuing warp touches per tile (stage offsets, descriptors, piece
// products, ring sizes) is an immediate: with run-time ring sizes and product tables that single warp needed ~370
// instructions (integer divisions, constant-table loads) per tile and paced the whole CTA at ~3200 cycles per tile for
// 770 cycles of tensor work.
template <int E, int NPS, int NPG>
struct IgCfg {
  static constexpr int KB = E / 64;
  static constexpr int PS = NPS == 1 ? 1 : (NPS == 3 ? 2 : 3);   // pieces held for the logits GEMM
  static constexpr int PG = NPG == 1 ? 1 : 2;                    // pieces of G / Y^T
  static constexpr int X_BYTES = PS * KB * IG_BM * 128;
  static constexpr int YS_BYTES = PS * KB * IG_BN * 128;          // Y pieces of one stage
  static constexpr int STAGE = YS_BYTES;   // the gradient GEMM reads the same Y pieces as an MN-major operand (no Y^T copy)
  static constexpr int NL_BYTES = IG_MAX_UNIT_TILES * IG_BN * 4;   // -lse * log2e of the unit's columns (mode V)
  static constexpr int FIXED = 1024 + 256 + NL_BYTES + X_BYTES;
  static constexpr int NG = 2;                  // G buffers (tensor memory: PG pieces x 32 columns each)
  static constexpr int G_COLS = PG * (IG_BN / 2);
  static constexpr int NST_RAW = (IG_SMEM_LIMIT - FIXED) / STAGE;
  static constexpr int NST = NST_RAW > 4 ? 4 : NST_RAW;
  static constexpr bool OK = NST >= 2 && PS >= PG;
  static constexpr int LOOKAHEAD = NST >= 3 ? 2 : 1;   // logits tiles issued ahead of the gradient GEMM (< NST: a stage is
                                                       // only refilled after the gradient GEMM of its tile)
  // TMEM columns: S0 [0,64) | S1 [64,128) | G buffers [128, 128 + NG*G_COLS) | OUT accumulators [256, 256 + NACC*E)
  static constexpr int G_COL0 = 2 * IG_BN;
  static constexpr int OUT_COL0 = 256;
  static constexpr int NACC = (512 - OUT_COL0) / E > 4 ? 4 : (512 - OUT_COL0) / E;
  static constexpr int SMEM = FIXED + NST * STAGE;
};

template <int E, int NPS, int NPG>
__global__ void __launch_bounds__(IG_THREADS, 1)
inbatch_grad_kernel(const __grid_constant__ CUtensorMap tm_ux, const __grid_constant__ CUtensorMap tm_uy,
                    const __grid_constant__ CUtensorMap tm_vx, const __grid_constant__ CUtensorMap tm_vy, const IgArgs a) {
  using C = IgCfg<E, NPS, NPG>;
  constexpr int KB = C::KB, PS = C::PS, PG = C::PG, NST = C::NST, NG = C::NG, NACC = C::NACC;
  constexpr int STAGE = C::STAGE, G_COLS = C::G_COLS;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // keeps the shared address space (LDS / STS)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int mode = (int)blockIdx.x >= a.units_u ? 1 : 0;
  const IgSide& sd = a.side[mode];
  const int unit = mode ? (int)blockIdx.x - a.units_u : (int)blockIdx.x;
  const int x_tile = unit / sd.splits, split = unit - x_tile * sd.splits;
  const int y_tiles_total = (sd.ycols + IG_BN - 1) / IG_BN;
  const int t_begin = split * sd.tiles_per_unit;
  int T = y_tiles_total - t_begin;
  if (T > sd.tiles_per_unit) T = sd.tiles_per_unit;
  const CUtensorMap* tmx = mode ? &tm_vx : &tm_ux;   // X operand, box 128 rows
  const CUtensorMap* tmy = mode ? &tm_uy : &tm_vy;   // Y operand, box 64 rows

  uint8_t* x_smem = smem;
  uint8_t* st_smem = x_smem + C::X_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(st_smem + NST * STAGE);
  uint64_t* full_bar = bars;            // [4]
  uint64_t* empty_bar = bars + 4;       // [4]
  uint64_t* s_full = bars + 8;          // [2]
  uint64_t* s_empty = bars + 10;        // [2]
  uint64_t* g_full = bars + 12;         // [2]
  uint64_t* g_empty = bars + 14;        // [2]
  uint64_t* x_full = bars + 16;
  uint64_t* out_full = bars + 17;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);
  float* s_nl = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 256);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(tmx);
    tma_prefetch_desc(tmy);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < 4; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&s_full[b], 1);
      mbar_init(&s_empty[b], IG_EPI_WARPS / 2);   // the epilogue warps work in two groups, one per tile parity
      mbar_init(&g_full[b], IG_EPI_WARPS / 2);
      mbar_init(&g_empty[b], 1);
    }
    mbar_init(x_full, 1);
    mbar_init(out_full, 1);
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  if (sd.lse_by_col) {   // mode V: the log-sum-exp belongs to the COLUMN (a user): stage this unit's slice once, prescaled
    for (int i = threadIdx.x; i < T * IG_BN; i += IG_THREADS) {
      const int c = t_begin * IG_BN + i;
      s_nl[i] = c < sd.ycols ? -__ldg(a.lse + c) * 1.4426950408889634f : 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  constexpr uint32_t OUT_COL = C::OUT_COL0, G_COL = C::G_COL0;

  if (T > 0) {
    if (warp == 0) {
      // ---------------------------------------------------------------- TMA producer
      if (elect_one()) {
        mbar_arrive_expect_tx(x_full, C::X_BYTES);
#pragma unroll
        for (int p = 0; p < PS; ++p)
#pragma unroll
          for (int kb = 0; kb < KB; ++kb)
            tma_load_2d(x_smem + (p * KB + kb) * (IG_BM * 128), tmx, x_full, (sd.xp[p] * KB + kb) * 64, x_tile * IG_BM);
      }
      __syncwarp();
      int st = 0;
      uint32_t eph = 1;
      for (int t = 0; t < T; ++t) {
        mbar_wait(&empty_bar[st], eph);
        if (elect_one()) {
          uint8_t* dst = st_smem + st * STAGE;
          const int yrow = (t_begin + t) * IG_BN;
          mbar_arrive_expect_tx(&full_bar[st], STAGE);
#pragma unroll
          for (int p = 0; p < PS; ++p)
#pragma unroll
            for (int kb = 0; kb < KB; ++kb)
              tma_load_2d(dst + (p * KB + kb) * (IG_BN * 128), tmy, &full_bar[st], (sd.yp[p] * KB + kb) * 64, yrow);
        }
        __syncwarp();
        if (++st == NST) st = 0, eph ^= 1;
      }
    } else if (warp == 1) {
      // ---------------------------------------------------------------- MMA issuer (warp-uniform loop, elected lane)
      constexpr uint32_t idesc_s = (1u << 4) | (1u << 7) | (1u << 10) | ((IG_BN >> 3) << 17) | ((IG_BM >> 4) << 24);
      // gradient GEMM: OUT[128, E] += G[128, 64] . Y[64, E]; B = the Y tile as loaded for the logits GEMM ([64 rows][128 B
      // of E], SW128), read as an MN-major operand: N = E contiguous, K = the tile's rows 128 B apart (8-row groups 1024 B
      // = SBO), 64-wide E blocks one piece block apart (LBO)
      constexpr uint32_t idesc_o = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((E >> 3) << 17) | ((IG_BM >> 4) << 24);
      // piece products, smallest first (they are added in this order): (x piece, y piece)
      constexpr int PX[6] = {1, 2, 0, 1, 0, 0}, PY[6] = {1, 0, 2, 0, 1, 0};
      constexpr int P0 = 6 - NPS;   // first product used: 6 -> 0, 3 -> 3, 1 -> 5
      const uint64_t x_desc = umma_desc_k_sw128(smem_u32(x_smem));
      const uint64_t st_desc = umma_desc_k_sw128(smem_u32(st_smem));
      const uint64_t yt_desc = umma_desc_mn_sw128(smem_u32(st_smem), IG_BN * 128, 1024);
      mbar_wait(x_full, 0);
      tc_fence_after();
      int s_st = 0, o_st = 0, o_acc = 0;       // stage of the next logits tile / of the next gradient tile, accumulator
      uint32_t s_ph = 0;                        // parity of full_bar[s_st]
      auto issue_s = [&](int t) {
        const int buf = t & 1;
        mbar_wait(&full_bar[s_st], s_ph);
        mbar_wait(&s_empty[buf], ((t >> 1) & 1) ^ 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t d_addr = tmem_base + buf * IG_BN;
          const uint64_t b_base = st_desc + static_cast<uint64_t>((s_st * STAGE) >> 4);
#pragma unroll
          for (int pr = P0; pr < 6; ++pr) {
#pragma unroll
            for (int kb = 0; kb < KB; ++kb) {
              const uint64_t a_desc = x_desc + (((PX[pr] * KB + kb) * (IG_BM * 128)) >> 4);
              const uint64_t b_desc = b_base + (((PY[pr] * KB + kb) * (IG_BN * 128)) >> 4);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_bf16(d_addr, a_desc + 2 * k, b_desc + 2 * k, idesc_s, (pr == P0 && kb == 0 && k == 0) ? 0u : 1u);
            }
          }
          umma_commit(&s_full[buf]);
        }
        __syncwarp();
        if (++s_st == NST) s_st = 0, s_ph ^= 1;
      };
      auto issue_o = [&](int t) {
        const int gb = t & (NG - 1);
        mbar_wait(&g_full[gb], (NG == 2 ? (t >> 1) : t) & 1);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t d_addr = tmem_base + OUT_COL + o_acc * E;
          const uint32_t a_base = tmem_base + G_COL + gb * G_COLS;   // G(t) pieces h | m, 32 columns each, in TMEM
          const uint64_t b_base = yt_desc + static_cast<uint64_t>((o_st * STAGE) >> 4);
          const uint32_t keep = t >= NACC ? 1u : 0u;
          // products (G piece, Y piece): m.h, h.m, h.h  (or h.h alone); one MMA contracts 16 tile rows = 2048 B
#pragma unroll
          for (int pr = (NPG == 3 ? 0 : 2); pr < 3; ++pr) {
            const uint32_t a_addr = a_base + (pr == 0 ? 1 : 0) * (IG_BN / 2);
            const uint64_t b_desc = b_base + (((pr == 1 ? 1 : 0) * KB * (IG_BN * 128)) >> 4);
#pragma unroll
            for (int k = 0; k < 4; ++k)   // 16 contraction indices = 8 TMEM columns of A, 16 tile rows of B
              umma_bf16_ts(d_addr, a_addr + 8 * k, b_desc + 128 * k, idesc_o, (pr == (NPG == 3 ? 0 : 2) && k == 0) ? keep : 1u);
          }
          umma_commit(&g_empty[gb]);
          umma_commit(&empty_bar[o_st]);
          if (t == T - 1) umma_commit(out_full);
        }
        __syncwarp();
        if (++o_st == NST) o_st = 0;
        if (++o_acc == NACC) o_acc = 0;
      };
      // logits tiles run LOOKAHEAD ahead of the gradient GEMM: S(t + 2) is issued as soon as the epilogue has read S(t)
      // out of its TMEM buffer, so the epilogue of tile t + 1 never waits for the tensor core or for this warp
      constexpr int LA = C::LOOKAHEAD;
      for (int t = 0; t < LA && t < T; ++t) issue_s(t);
      for (int t = 0; t < T; ++t) {
        if (t + LA < T) issue_s(t + LA);
        issue_o(t);
      }
    } else if (warp >= 4) {
      // ---------------------------------------------------------------- epilogue: logits -> G pieces -> gradient rows
      // Two groups of 8 warps: group g turns the logits tiles t = g, g + 2, ... into G (S buffer g, G buffer g), so two
      // tiles are in flight and the groups' phases (TMEM load, MUFU, pack, TMEM store) interleave on every scheduler.
      // Within a group: warp = TMEM lane quarter x 32-column half of the 64-column tile.
      const int ew = warp - 4;
      const int quarter = warp & 3;          // TMEM lanes 32*quarter .. +31 are accessible to this warp
      const int grp = ew >> 3;
      const int half = (ew >> 2) & 1;
      const int part = ew >> 2;              // output stage: E/4 columns of the gradient rows per warp
      const int row_l = quarter * 32 + lane;
      const long long row_g = (long long)x_tile * IG_BM + row_l;
      const bool row_ok = row_g < sd.rows;
      const float LOG2E = 1.4426950408889634f;
      float coef = a.coef;
      if (a.coef_dev != nullptr) coef *= __ldg(a.coef_dev);
      const float nl_row = (!sd.lse_by_col && row_ok) ? -__ldg(a.lse + row_g) * LOG2E : 0.f;
      // this row's positive sits at global column row_g + dshift (possibly outside [0, ycols)); all index math is int32
      // (rows, ycols < 2^30).  Rows beyond sd.rows need no masking: row r of G only feeds row r of OUT, which is not
      // stored; columns beyond ycols are masked in the (warp-uniform) tail tile only.
      const int hot = (int)row_g + sd.dshift;
      const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16);
      for (int t = grp; t < T; t += 2) {
        const int buf = grp;                                       // == t & 1
        const uint32_t par = (t >> 1) & 1;
        const int cb = (t_begin + t) * IG_BN + half * 32;          // first global column of this warp's 32
        mbar_wait(&s_full[buf], par);
        tc_fence_after();
        uint32_t v[2][16];
        tmem_ld_32x16(lane_base + buf * IG_BN + half * 32, v[0]);
        tmem_ld_32x16(lane_base + buf * IG_BN + half * 32 + 16, v[1]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&s_empty[buf]);
        const uint32_t gaddr = lane_base + G_COL + buf * G_COLS + half * 16;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const int c0 = cb + hh * 16;
          // G = coef * (2^(S * scale - lse * log2e) - onehot): one FFMA, one MUFU.EX2 and one FMUL per element
          float gv[16];
          if (sd.lse_by_col) {
            const float4* nl4 = reinterpret_cast<const float4*>(s_nl + (c0 - t_begin * IG_BN));
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 n4 = nl4[j];
              gv[4 * j] = coef * ex2_approx(fmaf(__uint_as_float(v[hh][4 * j]), a.scale_log2, n4.x));
              gv[4 * j + 1] = coef * ex2_approx(fmaf(__uint_as_float(v[hh][4 * j + 1]), a.scale_log2, n4.y));
              gv[4 * j + 2] = coef * ex2_approx(fmaf(__uint_as_float(v[hh][4 * j + 2]), a.scale_log2, n4.z));
              gv[4 * j + 3] = coef * ex2_approx(fmaf(__uint_as_float(v[hh][4 * j + 3]), a.scale_log2, n4.w));
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) gv[i] = coef * ex2_approx(fmaf(__uint_as_float(v[hh][i]), a.scale_log2, nl_row));
          }
          const int d = hot - c0;                                  // position of the positive inside these 16 columns
          if (__any_sync(0xffffffffu, static_cast<unsigned>(d) < 16u)) {
#pragma unroll
            for (int i = 0; i < 16; ++i) gv[i] -= (i == d) ? coef : 0.f;
          }
          if (c0 + 16 > sd.ycols) {                                // warp-uniform: tail tile
#pragma unroll
            for (int i = 0; i < 16; ++i) gv[i] = (c0 + i < sd.ycols) ? gv[i] : 0.f;
          }
          // G(t) -> tensor memory as the A operand of the gradient GEMM: lane = row, two bf16 per 32-bit column, piece h
          // in columns [0,32) of the buffer, piece m in [32,64); 16 logit columns = 8 TMEM columns of each piece
          uint32_t hw[8], mw[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {   // x = h + m: h = rn_bf16(x), m = rn_bf16(x - h) (the subtraction is exact)
            const float f0 = gv[2 * j], f1 = gv[2 * j + 1];
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(f0, f1);
            hw[j] = *reinterpret_cast<const uint32_t*>(&h2);
            if constexpr (PG == 2) {
              const __nv_bfloat162 m2 = __floats2bfloat162_rn(f0 - __uint_as_float(hw[j] << 16),
                                                              f1 - __uint_as_float(hw[j] & 0xFFFF0000u));
              mw[j] = *reinterpret_cast<const uint32_t*>(&m2);
            }
          }
          if (hh == 0) {   // the gradient GEMM of tile t - 2 must have consumed this G buffer
            mbar_wait(&g_empty[buf], par ^ 1);
            tc_fence_after();
          }
          tmem_st_32x8(gaddr + hh * 8, hw);
          if constexpr (PG == 2) tmem_st_32x8(gaddr + IG_BN / 2 + hh * 8, mw);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&g_full[buf]);
      }
      // gradient rows: sum the NACC accumulators with round-to-nearest adds, store (or add when the tile was split)
      mbar_wait(out_full, 0);
      tc_fence_after();
      constexpr int ncol = E / 4;   // columns of OUT per thread (16 or 32)
      const int used = T < NACC ? T : NACC;
      const bool atomic = mode ? a.atomic_v != 0 : a.atomic_u != 0;
      float* orow = sd.out + row_g * sd.ld_out + part * ncol;
#pragma unroll 1
      for (int c = 0; c < ncol; c += 16) {
        uint32_t o[16];
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + OUT_COL + part * ncol + c;
        tmem_ld_32x16(taddr, o);
        tmem_ld_wait();
        for (int ac = 1; ac < used; ++ac) {
          uint32_t w[16];
          tmem_ld_32x16(taddr + ac * E, w);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) o[j] = __float_as_uint(__uint_as_float(o[j]) + __uint_as_float(w[j]));
        }
        if (row_ok) {
          if (atomic) {
#pragma unroll
            for (int j = 0; j < 16; ++j) atomicAdd(orow + c + j, __uint_as_float(o[j]));
          } else {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              *reinterpret_cast<float4*>(orow + c + j) = make_float4(__uint_as_float(o[j]), __uint_as_float(o[j + 1]),
                                                                     __uint_as_float(o[j + 2]), __uint_as_float(o[j + 3]));
          }
        }
      }
      tc_fence_before();
    }
  }
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ring sizes / shared memory of the instantiation that serves (E, nprod_s, nprod_g); false when none fits
template <int E, int NPS, int NPG>
static bool ig_cfg_get(int& smem, int& nst) {
  smem = IgCfg<E, NPS, NPG>::SMEM;
  nst = IgCfg<E, NPS, NPG>::NST;
  return IgCfg<E, NPS, NPG>::OK;
}

static bool ig_cfg(int E, int nps, int npg, int& smem, int& nst) {
  if (E == 64) {
    if (nps == 1 && npg == 1) return ig_cfg_get<64, 1, 1>(smem, nst);
    if (nps == 3 && npg == 3) return ig_cfg_get<64, 3, 3>(smem, nst);
    if (nps == 6 && npg == 3) return ig_cfg_get<64, 6, 3>(smem, nst);
  } else if (E == 128) {
    if (nps == 1 && npg == 1) return ig_cfg_get<128, 1, 1>(smem, nst);
    if (nps == 3 && npg == 3) return ig_cfg_get<128, 3, 3>(smem, nst);
    if (nps == 6 && npg == 3) return ig_cfg_get<128, 6, 3>(smem, nst);
  }
  return false;
}

static int ig_plan(IgArgs& a, int64_t B, int64_t NI, int E, int nprod_s, int nprod_g, int& smem_bytes, int& nst) {
  if (E != 64 && E != 128) return fail("inbatch_grad: fused path needs E = 64 or 128 (got %d)", E);
  if (!((nprod_s == 1 && nprod_g == 1) || (nprod_s == 3 && nprod_g == 3) || (nprod_s == 6 && nprod_g == 3)))
    return fail("inbatch_grad: piece products (logits, gradient) must be (1,1), (3,3) or (6,3)");
  if (!ig_cfg(E, nprod_s, nprod_g, smem_bytes, nst))
    return fail("inbatch_grad: E = %d with %d piece products does not fit the resident tile", E, nprod_s);
  // units of equal length: L = tiles of the shorter column range, capped (accumulator chains, tail balance)
  const int64_t tu = (NI + IG_BN - 1) / IG_BN, tv = (B + IG_BN - 1) / IG_BN;
  int64_t L = tu < tv ? tu : tv;
  if (L > IG_MAX_UNIT_TILES) L = IG_MAX_UNIT_TILES;
  if (L < 1) L = 1;
  IgSide& su = a.side[0];
  IgSide& sv = a.side[1];
  su.rows = (int)B, su.ycols = (int)NI, su.x_tiles = (int)((B + IG_BM - 1) / IG_BM);
  su.splits = (int)((tu + L - 1) / L), su.tiles_per_unit = (int)((tu + su.splits - 1) / su.splits);
  sv.rows = (int)NI, sv.ycols = (int)B, sv.x_tiles = (int)((NI + IG_BM - 1) / IG_BM);
  sv.splits = (int)((tv + L - 1) / L), sv.tiles_per_unit = (int)((tv + sv.splits - 1) / sv.splits);
  a.units_u = su.x_tiles * su.splits;
  a.atomic_u = su.splits > 1;
  a.atomic_v = sv.splits > 1;
  return 0;
}

template <int E, int NPS, int NPG>
static int ig_launch(int units, int smem, cudaStream_t st, const CUtensorMap& ux, const CUtensorMap& uy,
                     const CUtensorMap& vx, const CUtensorMap& vy, const IgArgs& a) {
  if constexpr (IgCfg<E, NPS, NPG>::OK) {
    auto kern = inbatch_grad_kernel<E, NPS, NPG>;
    static bool attr = false;
    if (!attr) {
      B200_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, IG_SMEM_LIMIT));
      attr = true;
    }
    kern<<<units, IG_THREADS, smem, st>>>(ux, uy, vx, vy, a);
    B200_LAUNCH_OK("inbatch_grad_kernel");
    return 0;
  } else {
    return fail("inbatch_grad: configuration not instantiated");
  }
}

}  // namespace b200

using namespace b200;

extern "C" int b200rec_inbatch_grad_supported(int64_t B, int64_t NI, int E, int nprod_s, int nprod_g) {
  IgArgs a;
  int smem = 0, nst = 0;
  if (B <= 0 || NI <= 0 || B > INT32_MAX / 2 || NI > INT32_MAX / 2) return 0;
  return ig_plan(a, B, NI, E, nprod_s, nprod_g, smem, nst) == 0 ? 1 : 0;
}

// The plans the in-batch loss runs with, without launching anything (no GPU needed): out[0..n_out) = sms, then the
// forward log-sum-exp of (B, NI, ld) -- nq, bn, stages, grid, S, T, W, max_parts, all 0 when the operand is too wide
// and the forward takes the GEMM + lse_rows fallback -- then the fused backward of (B, NI, E, nprod_s, nprod_g) --
// supported, smem, NST, units_u, splits_u, splits_v, atomic_u, atomic_v, all 0 when the backward takes the chunked
// path.  Tests use it to prove which kernel instantiation and work split a shape reaches.
extern "C" int b200rec_debug_loss_plan(int64_t B, int64_t NI, int64_t ld, int E, int nprod_s, int nprod_g,
                                       long long* out, int n_out) {
  if (out == nullptr || n_out < 0) return fail("loss_plan: null output");
  if (B <= 0 || NI <= 0) return fail("loss_plan: empty input");
  long long v[1 + LSE_PLAN_FIELDS + 8] = {num_sms()};
  long long lse[LSE_PLAN_FIELDS];
  lse_plan_fields(B, NI, ld, lse);
  for (int i = 0; i < LSE_PLAN_FIELDS; ++i) v[1 + i] = lse[i];
  IgArgs a;
  int smem = 0, nst = 0;
  if (b200rec_inbatch_grad_supported(B, NI, E, nprod_s, nprod_g) && ig_plan(a, B, NI, E, nprod_s, nprod_g, smem, nst) == 0) {
    const long long g[8] = {1, smem, nst, a.units_u, a.side[0].splits, a.side[1].splits, a.atomic_u, a.atomic_v};
    for (int i = 0; i < 8; ++i) v[1 + LSE_PLAN_FIELDS + i] = g[i];
  }
  for (int i = 0; i < n_out && i < (int)(sizeof(v) / sizeof(v[0])); ++i) out[i] = v[i];
  return 0;
}

extern "C" int b200rec_inbatch_grad(const void* u_op, int64_t ld_u, const int32_t* u_pieces_host, const void* v_op,
                                    int64_t ld_v, const int32_t* v_pieces_host, const void* ut_op, int64_t ld_ut,
                                    const int32_t* ut_pieces_host, const void* vt_op, int64_t ld_vt,
                                    const int32_t* vt_pieces_host, int64_t B, int64_t NI, int E, int nprod_s, int nprod_g,
                                    float inv_t, const float* lse, int64_t diag0, float coef, const float* coef_dev,
                                    float* dU, int64_t ld_du, float* dV, int64_t ld_dv, void* stream) {
  // ut_op / vt_op (transposed operands) are no longer read: the gradient GEMM takes the row operands as MN-major tiles.
  (void)ut_op, (void)ld_ut, (void)ut_pieces_host, (void)vt_op, (void)ld_vt, (void)vt_pieces_host;
  if (!u_op || !v_op || !lse || !dU || !dV) return fail("inbatch_grad: null pointer");
  if (!u_pieces_host || !v_pieces_host) return fail("inbatch_grad: null piece table");
  if (B <= 0 || NI <= 0 || B > INT32_MAX / 2 || NI > INT32_MAX / 2) return fail("inbatch_grad: bad sizes");
  if (diag0 < 0 || diag0 + B > NI) return fail("inbatch_grad: positives [diag0, diag0 + B) must lie inside the item rows");
  if ((ld_du & 3) || (ld_dv & 3) || (reinterpret_cast<uintptr_t>(dU) & 15) || (reinterpret_cast<uintptr_t>(dV) & 15))
    return fail("inbatch_grad: gradient rows must be 16-byte aligned");
  IgArgs a;
  int smem = 0, nst = 0;
  if (ig_plan(a, B, NI, E, nprod_s, nprod_g, smem, nst)) return 1;
  const int KB = E / 64;
  const int ps = nprod_s == 1 ? 1 : (nprod_s == 3 ? 2 : 3), pg = nprod_g == 1 ? 1 : 2;
  IgSide& su = a.side[0];
  IgSide& sv = a.side[1];
  int max_u = 0, max_v = 0;
  for (int p = 0; p < 3; ++p) {   // pieces h, m, l of the row operands (the gradient GEMM uses h, m of the same blocks)
    su.xp[p] = sv.yp[p] = p < ps ? u_pieces_host[p] : 0;
    su.yp[p] = sv.xp[p] = p < ps ? v_pieces_host[p] : 0;
    if (p < ps) max_u = max_u > u_pieces_host[p] ? max_u : u_pieces_host[p], max_v = max_v > v_pieces_host[p] ? max_v : v_pieces_host[p];
  }
  if (pg > ps) return fail("inbatch_grad: the gradient GEMM needs the m piece of the row operands");
  if ((max_u + 1) * KB * 64 > ld_u || (max_v + 1) * KB * 64 > ld_v) return fail("inbatch_grad: piece block outside the operand row");
  su.dshift = (int)diag0, sv.dshift = -(int)diag0;
  su.lse_by_col = 0, sv.lse_by_col = 1;
  su.out = dU, su.ld_out = ld_du, sv.out = dV, sv.ld_out = ld_dv;
  a.scale_log2 = inv_t * 1.4426950408889634f;
  a.coef = coef;
  a.coef_dev = coef_dev;
  a.lse = lse;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  CUtensorMap ux, uy, vx, vy;
  if (make_tmap_bf16_2d(&ux, u_op, (uint64_t)B, (uint64_t)ld_u, (uint64_t)ld_u, IG_BM)) return 1;
  if (make_tmap_bf16_2d(&uy, u_op, (uint64_t)B, (uint64_t)ld_u, (uint64_t)ld_u, IG_BN)) return 1;
  if (make_tmap_bf16_2d(&vx, v_op, (uint64_t)NI, (uint64_t)ld_v, (uint64_t)ld_v, IG_BM)) return 1;
  if (make_tmap_bf16_2d(&vy, v_op, (uint64_t)NI, (uint64_t)ld_v, (uint64_t)ld_v, IG_BN)) return 1;
  if (a.atomic_u) B200_CUDA_OK(cudaMemset2DAsync(dU, sizeof(float) * (size_t)ld_du, 0, sizeof(float) * (size_t)E, (size_t)B, st));
  if (a.atomic_v) B200_CUDA_OK(cudaMemset2DAsync(dV, sizeof(float) * (size_t)ld_dv, 0, sizeof(float) * (size_t)E, (size_t)NI, st));
  const int units = a.units_u + sv.x_tiles * sv.splits;
#define IG_CASE(EE, S, G) if (E == EE && nprod_s == S && nprod_g == G) return ig_launch<EE, S, G>(units, smem, st, ux, uy, vx, vy, a)
  IG_CASE(64, 1, 1);
  IG_CASE(64, 3, 3);
  IG_CASE(64, 6, 3);
  IG_CASE(128, 1, 1);
  IG_CASE(128, 3, 3);
  IG_CASE(128, 6, 3);
#undef IG_CASE
  return fail("inbatch_grad: unsupported configuration");
}
