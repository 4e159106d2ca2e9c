// CTA-pair (tcgen05 cta_group::2) kernels for the contrastive hot path -- the main path for d % 128 == 0, d <= 768.
//
// Why pairs.  With one CTA per SM the logits MMA is 128 x BLOCK_I x 16 with BLOCK_I <= 128 resident rows (shared
// memory) and the backward's TMEM budget caps BLOCK_I at 64: every MMA then pulls 6 KiB of operands through the
// 128 B/clk shared-memory port for 32 clk of tensor work (measured 63 % of peak for N = 64, tools/umma_probe.cu).
// A pair splits BOTH operands of one instruction between two SMs, so N = 256 instructions fit:
//
//   forward   S[i, j]  M = 256 (128 resident rows per CTA), N = 256 (128 streamed rows per CTA)    64 B/clk operands
//   backward  S[i, j]  M = 128 ( 64 resident rows per CTA), N = 256                                96 B/clk
//             dXhat[i, d] += G[i, j] Y[j, d]   M = 128, N = 256 (d chunk), K = j                   96 B/clk
//
// Orientation is NOT transposed here: TMEM lane <-> resident row i, TMEM column <-> streamed column j.  Per-row
// quantities (rinv_x, u_i, the row sum) are thread-local scalars for the whole sweep; per-column quantities are
// staged per step in shared memory and read as broadcast float4.  In the backward every epilogue thread owns one row
// and 64 consecutive columns: the bf16 gradient row is exactly one 128-byte swizzled row of the K-major A operand of
// the gradient MMA (eight conflict-free 16-byte stores).  The gradient MMA reads the streamed rows Y[j, :] directly
// as an MN-major B operand (N = d contiguous, K = j), so no transposed copy of the embeddings exists in HBM.
//
// M = 128 over a pair uses the "2x2" accumulator layout (validated in tools/umma_probe.cu): each CTA holds 64 rows;
// TMEM lane l, column c  <->  row l % 64, column c + (N/2) * (l / 64).
//
// Barrier protocol (all mbarriers live at the same offset in both CTAs):
//   FULL_A/B[s]   leader only: armed by the leader's producer for the bytes of BOTH CTAs; each CTA's TMA
//                 (.cta_group::2) completes its bytes on the leader's barrier
//   EMPTY_A/B[s]  both: tcgen05.commit multicast from the leader after the MMAs that read stage s
//   SFULL[b]      both: commit multicast (logits buffer b complete)         SEMPTY[b]  leader: one arrival per
//                 epilogue warp of both CTAs (remote mbarrier.arrive, CTA-scope release -- see ptx::mbar_arrive_cluster)
//   GFULL[kc]     leader: the 2 warps per CTA that wrote gradient box kc     GEMPTY[kc] both: commit multicast
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include "kernels_tc.cuh"
#include "ptx.cuh"

namespace pair {

constexpr int STEP_J = 256;            // streamed columns per step (128 TMA rows per CTA)
constexpr int STAGE_BYTES = 16384;     // one ring stage: [128 rows][64 k] or 2 x [64 j][64 d]
constexpr int MAX_STAGES = 6;
constexpr int MAX_SPLIT = 16;         // work items per row block (column-sweep split)
constexpr int SMEM_LIMIT = 232448;
constexpr int TMEM_COLS = 512;
constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;

// barrier slots (8 bytes each)
constexpr int B_FULL_A = 0, B_EMPTY_A = MAX_STAGES, B_FULL_B = 2 * MAX_STAGES, B_EMPTY_B = 3 * MAX_STAGES,
              B_XFULL = 4 * MAX_STAGES, B_SFULL = B_XFULL + 1, B_SEMPTY = B_SFULL + 2, B_GFULL = B_SEMPTY + 2,
              B_GEMPTY = B_GFULL + 4, B_ACCFULL = B_GEMPTY + 4, B_COUNT = B_ACCFULL + 1;
static_assert(B_COUNT * 8 <= 512, "barrier block");

__device__ __forceinline__ float ex2(float x) { return tc::ex2(x); }
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
// order-preserving float <-> int key (for atomicMax on scores of either sign)
__device__ __forceinline__ int float_key(float f) {
  const int b = __float_as_int(f);
  return b >= 0 ? b : b ^ 0x7fffffff;
}
__device__ __forceinline__ float key_float(int k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// Several independent (X, Y) problems of equal shape in ONE launch (the tri-modal model's three pairs -- and, for the
// backward, both sides of each: tf_clip_codes (1).ipynb:13152-13165).  All operands are members of one stacked matrix
// [n_members][n_pad, d]; the launch sweeps a block-diagonal VIRTUAL problem: problem k owns the virtual rows and columns
// [k n_pad, k n_pad + n_valid), its row blocks visit its own column steps only.  Statistics and gradients are indexed by
// virtual row / column; operand rows (and their 1/norms) by virtual index + shift.
constexpr int MAX_GROUP = 8;
struct Group {
  int n_prob;            // 0: one problem, plain indexing
  int pairs_per_prob;    // row blocks (CTA pairs) per problem
  int steps_per_prob;    // 256-column steps per problem: n_pad / 256
  int n_valid;           // rows (= columns) of every problem
  int xshift[MAX_GROUP];   // stack row of the resident operand minus virtual row
  int yshift[MAX_GROUP];   // stack row of the streamed operand minus virtual column
  int cshift[MAX_GROUP];   // backward: index of a column's statistics minus virtual column
  const float* gscale;     // backward: optional DEVICE [n_prob] upstream gradient per problem (problem k reads gscale[k % gmod])
  int gmod;
  int stack_rows;          // host: rows of the stacked operand matrix (extent of the tensor maps)
};
struct GroupView {   // what one work item needs of it
  int t_lo, t_hi, xs, ys, cs, n_rows, n_cols, k;
};
__device__ __forceinline__ GroupView group_view(const Group& g, int pair_block, int n_steps, int n_rows, int n_cols) {
  GroupView v;
  if (g.n_prob == 0) {
    v.t_lo = 0; v.t_hi = n_steps; v.xs = v.ys = v.cs = 0; v.n_rows = n_rows; v.n_cols = n_cols; v.k = 0;
  } else {
    v.k = pair_block / g.pairs_per_prob;
    v.t_lo = v.k * g.steps_per_prob;
    v.t_hi = v.t_lo + g.steps_per_prob;
    v.xs = g.xshift[v.k]; v.ys = g.yshift[v.k]; v.cs = g.cshift[v.k];
    v.n_rows = v.n_cols = v.t_lo * STEP_J + g.n_valid;
  }
  return v;
}

// ===================================================================================================== backward
constexpr int BWD_EPI_WARPS = 8;
constexpr int BWD_THREADS = 32 * (4 + BWD_EPI_WARPS);
constexpr int BWD_ROWS = 64;                       // resident rows per CTA (128 per pair)
constexpr int BWD_X_CHUNK = BWD_ROWS * 128;        // [64 rows][64 k] bf16
constexpr int BWD_G_BYTES = 4 * 8192;              // gradient tile [64 i][256 j] bf16 = four K-major boxes
constexpr int BWD_SMALL = 10240;                   // barriers (512) | tmem ptr | column vectors 2 x 4 x 256 f32 at +1024

struct BwdParams {
  int n_rows, n_cols, d;
  int nkc;        // ceil(d / 64)
  int nq2;        // ceil(d / 256): accumulator chunks (TMEM slots of 128 columns)
  int n_steps;    // ceil(n_cols / 256)
  int stages_a, stages_b, nsbuf;
  int n_pairs;      // row blocks
  int split_steps;  // steps per work item (column-sweep split, see FwdParams); item s accumulates into dx + s n_rows d
  long long diag_offset;
  float scale, diag_w, grad_out;
  const float* scale_dev;  // optional DEVICE scalar s: read instead of `scale` (no host read of the logit scale per step)
  const float* rinv_x;
  const float* rinv_y;
  const float* row_m_in;
  const float* row_w;
  const float* col_m_in;   // or nullptr (with col_w)
  const float* col_w;
  float* dx;               // [n_split][n_rows, d] f32 (summed over the splits by aux::sum_splits when n_split > 1)
  Group grp;               // several problems in one launch (n_prob = 0: one)
};

__host__ __device__ constexpr int bwd_smem_bytes(int nkc, int stages) {
  return nkc * BWD_X_CHUNK + BWD_G_BYTES + stages * STAGE_BYTES + BWD_SMALL;
}

// TWO_EXP = false: the fixed-shift form, ONE ex2 per logit -- exp(S - s) (u_i + v_j) with u, v carrying exp(s - m).
// TWO_EXP = true: exp(S - m_i) w_i + exp(S - m_j) w_j with the (shift, sum) pairs as they are, two ex2 per logit: valid
// for ANY logit range (s up to the clamp at 100, un-normalised queue rows), because every exponent is <= 0 by
// construction of the shifts (true maxima, or s where |S| <= s).
template <bool TWO_EXP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(BWD_THREADS, 1)
bwd_kernel(const __grid_constant__ CUtensorMap tmap_x,    // X  box {64 k, 64 rows}
           const __grid_constant__ CUtensorMap tmap_y,    // Y  box {64 k, 128 rows}   (logits operand, K-major)
           const __grid_constant__ CUtensorMap tmap_yg,   // Y  box {64 d, 64 rows}    (gradient operand, MN-major)
           const BwdParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t base = ptx::smem_u32(smem);
  if ((base & 1023u) != 0) __trap();
  const uint32_t rank = ptx::cluster_ctarank() & 1u;   // CTA within its pair
  const bool leader = rank == 0;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int item = blockIdx.x >> 1;
  const int split = item / p.n_pairs;
  const int i0 = (item % p.n_pairs) * (2 * BWD_ROWS) + (int)rank * BWD_ROWS;   // first resident row of this CTA
  const GroupView gv = group_view(p.grp, item % p.n_pairs, p.n_steps, p.n_rows, p.n_cols);
  const int t_begin = gv.t_lo + split * p.split_steps;
  const int n_t = min(gv.t_hi, t_begin + p.split_steps) - t_begin;            // steps of this work item

  const uint32_t x_smem = base;
  const uint32_t g_smem = x_smem + p.nkc * BWD_X_CHUNK;
  const uint32_t ring_a = g_smem + BWD_G_BYTES;
  const uint32_t ring_b = ring_a + p.stages_a * STAGE_BYTES;
  const uint32_t small_off = (ring_b - base) + p.stages_b * STAGE_BYTES;
  const uint32_t bars = base + small_off;
  auto bar = [&](int i) -> uint32_t { return bars + 8u * i; };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + small_off + 512);
  float* const colv = reinterpret_cast<float*>(smem + small_off + 1024);   // [2][4][256]

  const int S_COL0 = TMEM_COLS - 128 * p.nsbuf;
  const float sc = p.scale_dev != nullptr ? __ldg(p.scale_dev) : p.scale;   // s
  const float k2 = sc * LOG2E;                                                // s log2(e)
  const float out_scale = p.grad_out * sc * (p.grp.gscale != nullptr ? __ldg(p.grp.gscale + gv.k % p.grp.gmod) : 1.f);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_x);
    ptx::prefetch_tmap(&tmap_y);
    ptx::prefetch_tmap(&tmap_yg);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < MAX_STAGES; ++s) {
      ptx::mbar_init(bar(B_FULL_A + s), 1);
      ptx::mbar_init(bar(B_EMPTY_A + s), 1);
      ptx::mbar_init(bar(B_FULL_B + s), 1);
      ptx::mbar_init(bar(B_EMPTY_B + s), 1);
    }
    ptx::mbar_init(bar(B_XFULL), 1);
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(bar(B_SFULL + b), 1);
      ptx::mbar_init(bar(B_SEMPTY + b), 2 * BWD_EPI_WARPS);
    }
    for (int k = 0; k < 4; ++k) {
      ptx::mbar_init(bar(B_GFULL + k), 4);
      ptx::mbar_init(bar(B_GEMPTY + k), 1);
    }
    ptx::mbar_init(bar(B_ACCFULL), 1);
    ptx::fence_mbar_init();
  }
  if (warp == 2) ptx::tmem_alloc_pair(ptx::smem_u32(const_cast<uint32_t*>(tmem_ptr_smem)), TMEM_COLS);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  const uint32_t desc_hi_k = static_cast<uint32_t>(ptx::smem_desc_k_sw128(0) >> 32);
  const uint32_t desc_hi_mn = static_cast<uint32_t>(ptx::smem_desc_mn_sw128(0, 8192) >> 32);
  auto desc_lo = [&](uint32_t addr, uint32_t lbo16) -> uint32_t { return ((addr & 0x3FFFFu) >> 4) | (lbo16 << 16); };
  auto mk = [&](uint32_t hi, uint32_t lo) -> uint64_t { return (static_cast<uint64_t>(hi) << 32) | lo; };

  if (warp == 0) {
    // ================================================================= producer A: resident X, then Y rows (K-major)
    if (ptx::elect_one()) {
      if (leader) ptx::mbar_arrive_expect_tx(bar(B_XFULL), 2 * p.nkc * BWD_X_CHUNK);
      for (int kc = 0; kc < p.nkc; ++kc)
        ptx::tma_load_2d_pair(x_smem + kc * BWD_X_CHUNK, &tmap_x, bar(B_XFULL), kc * 64, i0 + gv.xs);
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < n_t; ++t) {
        for (int g = 0; g < p.nkc; ++g) {
          ptx::mbar_wait(bar(B_EMPTY_A + stage), phase ^ 1u);
          if (leader) ptx::mbar_arrive_expect_tx(bar(B_FULL_A + stage), 2 * STAGE_BYTES);
          ptx::tma_load_2d_pair(ring_a + stage * STAGE_BYTES, &tmap_y, bar(B_FULL_A + stage), g * 64,
                                (t_begin + t) * STEP_J + (int)rank * 128 + gv.ys);
          if (++stage == p.stages_a) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 2) {
    // ================================================================= producer B: Y[j, d slice] boxes (MN-major)
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int t = 0; t < n_t; ++t) {
        for (int kc = 0; kc < 4; ++kc) {
          for (int q = 0; q < p.nq2; ++q) {
            const int wq = min(256, p.d - 256 * q);   // 128 or 256 (d % 128 == 0)
            const int half = wq >> 1;                 // d columns this CTA supplies
            const int ngr = half >> 6;                // 64-wide MN groups
            ptx::mbar_wait(bar(B_EMPTY_B + stage), phase ^ 1u);
            if (leader) ptx::mbar_arrive_expect_tx(bar(B_FULL_B + stage), 2 * ngr * 8192);
            for (int gi = 0; gi < ngr; ++gi)
              ptx::tma_load_2d_pair(ring_b + stage * STAGE_BYTES + gi * 8192, &tmap_yg, bar(B_FULL_B + stage),
                                    256 * q + half * (int)rank + 64 * gi, (t_begin + t) * STEP_J + 64 * kc + gv.ys);
            if (++stage == p.stages_b) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================================================= logits MMA issuer (leader)
    if (leader && ptx::elect_one()) {
      constexpr uint32_t idesc_s = ptx::idesc_bf16_f32_major(2 * BWD_ROWS, STEP_J, 0, 0);
      const uint32_t x_lo0 = desc_lo(x_smem, 1), a_lo0 = desc_lo(ring_a, 1);
      int stage = 0;
      uint32_t phase = 0, ready = 0;
      ptx::mbar_wait(bar(B_XFULL), 0);
      for (int t = 0; t < n_t; ++t) {
        const int sb = t % p.nsbuf;
        ptx::mbar_wait(bar(B_SEMPTY + sb), ((t / p.nsbuf) & 1) ^ 1u);
        const uint32_t d_tmem = tmem_base + S_COL0 + sb * 128;
        for (int g = 0; g < p.nkc; ++g) {
          if (!ready) ptx::mbar_wait(bar(B_FULL_A + stage), phase);
          ptx::tc_fence_after();
          int ns = stage + 1;
          uint32_t np = phase;
          if (ns == p.stages_a) { ns = 0; np ^= 1u; }
          ready = ptx::mma_box_pair(d_tmem, mk(desc_hi_k, x_lo0 + g * (BWD_X_CHUNK >> 4)),
                                    mk(desc_hi_k, a_lo0 + stage * (STAGE_BYTES >> 4)), 2, 2, idesc_s, g != 0,
                                    bar(B_FULL_A + ns), np);
          ptx::mma_commit_pair(bar(B_EMPTY_A + stage));
          if (g == p.nkc - 1) ptx::mma_commit_pair(bar(B_SFULL + sb));
          stage = ns;
          phase = np;
        }
      }
    }
    __syncwarp();
  } else if (warp == 3) {
    // ================================================================= gradient MMA issuer (leader)
    if (leader && ptx::elect_one()) {
      const uint32_t g_lo0 = desc_lo(g_smem, 1), b_lo0 = desc_lo(ring_b, 8192 >> 4);
      int stage = 0;
      uint32_t phase = 0, ready = 0;
      for (int t = 0; t < n_t; ++t) {
        for (int kc = 0; kc < 4; ++kc) {
          ptx::mbar_wait(bar(B_GFULL + kc), t & 1);   // both CTAs wrote gradient box kc of step t
          for (int q = 0; q < p.nq2; ++q) {
            const int wq = min(256, p.d - 256 * q);
            const uint32_t idesc_g = ptx::idesc_bf16_f32_major(2 * BWD_ROWS, wq, 0, 1);
            if (!ready) ptx::mbar_wait(bar(B_FULL_B + stage), phase);
            ptx::tc_fence_after();
            int ns = stage + 1;
            uint32_t np = phase;
            if (ns == p.stages_b) { ns = 0; np ^= 1u; }
            ready = ptx::mma_box_pair(tmem_base + 128 * q, mk(desc_hi_k, g_lo0 + kc * (8192 >> 4)),
                                      mk(desc_hi_mn, b_lo0 + stage * (STAGE_BYTES >> 4)), 2, 2048 >> 4, idesc_g,
                                      (t | kc) != 0, bar(B_FULL_B + ns), np);
            ptx::mma_commit_pair(bar(B_EMPTY_B + stage));
            stage = ns;
            phase = np;
          }
          ptx::mma_commit_pair(bar(B_GEMPTY + kc));
        }
      }
      ptx::mma_commit_pair(bar(B_ACCFULL));
    }
    __syncwarp();
  } else {
    // ================================================================= epilogue: S tile -> bf16 gradient tile
    const int e = warp - 4;            // 0..7
    const int q = warp & 3;            // TMEM lane quarter
    const int h = e >> 2;              // which 64 of this quarter's 128 TMEM columns
    const int jh = q >> 1;             // 2x2 layout: lanes 64..127 hold columns 128..255 of the step
    const int i_local = 32 * (q & 1) + lane;
    const long long i_glob = (long long)i0 + i_local;
    const bool row_ok = i_glob < gv.n_rows;
    const int te = threadIdx.x - 128;  // 0..255: the step column this thread stages
    const int jl0 = 128 * jh + 64 * h; // first step-local column of this thread == 64 * kc
    const int kc = 2 * jh + h;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float rx = row_ok ? p.rinv_x[i_glob + gv.xs] : 0.f;
    // u_i = row_w_i exp(s - row_m_i): exp(S - s) u_i = exp(S - row_m_i) row_w_i from ONE ex2 per logit
    const float u = (!TWO_EXP && row_ok) ? p.row_w[i_glob] * ex2((sc - p.row_m_in[i_glob]) * LOG2E) : 0.f;
    const float rm2 = (TWO_EXP && row_ok) ? p.row_m_in[i_glob] * LOG2E : 0.f;   // TWO_EXP: exp(S - m_i) w_i directly
    const float rw = (TWO_EXP && row_ok) ? p.row_w[i_glob] : 0.f;
    const uint32_t g_row = g_smem + kc * 8192 + (i_local >> 3) * 1024 + (i_local & 7) * 128;
    const uint32_t sw = i_local & 7;
    const uint32_t sempty_leader = ptx::mapa(bar(B_SEMPTY), 0);
    const uint32_t gfull_leader = ptx::mapa(bar(B_GFULL + kc), 0);
    const long long dcol0 = i_glob + p.diag_offset;   // column of this row's positive

    auto load_col = [&](int t, float& cw, float& cm, float& ry) {   // t: step local to this work item
      const long long jn = (long long)(t_begin + t) * STEP_J + te;
      const bool ok = t < n_t && jn < gv.n_cols;
      cw = (ok && p.col_w != nullptr) ? p.col_w[jn + gv.cs] : 0.f;
      cm = (ok && p.col_w != nullptr) ? p.col_m_in[jn + gv.cs] : (TWO_EXP ? 0.f : sc);
      ry = ok ? p.rinv_y[jn + gv.ys] : 0.f;
      if (TWO_EXP && !(cw > 0.f)) cm = 0.f;   // weight 0 (extra negative columns: sum = +inf): keep the exponent finite
    };
    float cw_n, cm_n, ry_n;
    load_col(0, cw_n, cm_n, ry_n);

    for (int t = 0; t < n_t; ++t) {
      const int sb = t % p.nsbuf;
      float* const cv = colv + (t & 1) * 1024;
      {
        const float vj = TWO_EXP ? cw_n : cw_n * ex2((sc - cm_n) * LOG2E);
        cv[te] = ry_n * k2;          // S_ij log2(e) = acc * rinv_x[i] * cj
        cv[256 + te] = vj * ry_n;      // G is contracted against the RAW y_j -> fold rinv_y[j] into it
        cv[512 + te] = ry_n;
        if (TWO_EXP) cv[768 + te] = cm_n * LOG2E;
      }
      load_col(t + 1, cw_n, cm_n, ry_n);
      named_bar_sync(1, BWD_EPI_WARPS * 32);
      const long long dl = dcol0 - ((long long)(t_begin + t) * STEP_J + jl0);   // step-local index of the positive, if in [0, 64)
      const bool has_diag = row_ok && dl >= 0 && dl < 64;

      ptx::mbar_wait(bar(B_SFULL + sb), (t / p.nsbuf) & 1);
      ptx::tc_fence_after();
      uint32_t pk[32];   // 64 bf16 of this thread's gradient row
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(t_lane + S_COL0 + sb * 128 + 64 * h + 32 * c, r);
        ptx::tmem_ld_wait();
        if (c == 1) {   // the whole S buffer share of this warp is in registers: the next logits tile may land
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_cluster(sempty_leader + 8u * sb);
        }
        const float* const cjp = cv + jl0 + 32 * c;
#pragma unroll
        for (int x4 = 0; x4 < 8; ++x4) {
          const float4 cj4 = *reinterpret_cast<const float4*>(cjp + 4 * x4);
          const float4 vr4 = *reinterpret_cast<const float4*>(cjp + 256 + 4 * x4);
          const float4 ry4 = *reinterpret_cast<const float4*>(cjp + 512 + 4 * x4);
          const float cjv[4] = {cj4.x, cj4.y, cj4.z, cj4.w};
          const float vrv[4] = {vr4.x, vr4.y, vr4.z, vr4.w};
          const float ryv[4] = {ry4.x, ry4.y, ry4.z, ry4.w};
          float g[4];
          if constexpr (TWO_EXP) {
            const float4 cm4 = *reinterpret_cast<const float4*>(cjp + 768 + 4 * x4);
            const float cmv[4] = {cm4.x, cm4.y, cm4.z, cm4.w};
#pragma unroll
            for (int xx = 0; xx < 4; ++xx) {
              const float y = __uint_as_float(r[4 * x4 + xx]) * rx;
              const float er = ex2(fmaf(y, cjv[xx], -rm2)) * rw;        // exp(S_ij - m_i) w_i
              const float ec = ex2(fmaf(y, cjv[xx], -cmv[xx]));         // exp(S_ij - m_j)
              g[xx] = fmaf(er, ryv[xx], ec * vrv[xx]);                    // (...) rinv_y[j]
            }
          } else {
#pragma unroll
            for (int xx = 0; xx < 4; ++xx) {
              const float y = __uint_as_float(r[4 * x4 + xx]) * rx;
              const float ev = ex2(fmaf(y, cjv[xx], -k2));              // exp(S_ij - s)
              g[xx] = ev * fmaf(u, ryv[xx], vrv[xx]);                     // (u_i + v_j) rinv_y[j]
            }
          }
          if (has_diag) {
#pragma unroll
            for (int xx = 0; xx < 4; ++xx)
              if (dl == 32 * c + 4 * x4 + xx) g[xx] -= p.diag_w * ryv[xx];
          }
          const __nv_bfloat162 p0 = __floats2bfloat162_rn(g[0], g[1]);
          const __nv_bfloat162 p1 = __floats2bfloat162_rn(g[2], g[3]);
          pk[16 * c + 2 * x4] = *reinterpret_cast<const uint32_t*>(&p0);
          pk[16 * c + 2 * x4 + 1] = *reinterpret_cast<const uint32_t*>(&p1);
        }
      }
      ptx::mbar_wait(bar(B_GEMPTY + kc), (t & 1) ^ 1u);   // gradient MMAs of step t-1 have read this box
#pragma unroll
      for (int ch = 0; ch < 8; ++ch)   // 16-byte chunk ch of the 128-byte row, XOR-swizzled by the row index
        st_shared_v4(g_row + ((static_cast<uint32_t>(ch) ^ sw) << 4), pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2],
                     pk[4 * ch + 3]);
      ptx::fence_proxy_async_smem();   // generic-proxy stores -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive_cluster(gfull_leader);
    }

    // accumulators complete: slot q2 holds dXhat[i, 256 q2 + ...] in the 2x2 layout
    ptx::mbar_wait(bar(B_ACCFULL), 0);
    ptx::tc_fence_after();
    for (int q2 = 0; q2 < p.nq2; ++q2) {
      const int halfw = min(256, p.d - 256 * q2) >> 1;   // columns of the slot in use: 128 or 64
      if (64 * h < halfw) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          uint32_t r[32];
          ptx::tmem_ld_32x32b_x32(t_lane + 128 * q2 + 64 * h + 32 * c, r);
          ptx::tmem_ld_wait();
          if (row_ok) {
            float* const dst = p.dx + ((long long)split * p.n_rows + i_glob) * p.d + 256 * q2 + halfw * jh + 64 * h + 32 * c;
#pragma unroll
            for (int x4 = 0; x4 < 8; ++x4)
              *reinterpret_cast<float4*>(dst + 4 * x4) =
                  make_float4(__uint_as_float(r[4 * x4]) * out_scale, __uint_as_float(r[4 * x4 + 1]) * out_scale,
                              __uint_as_float(r[4 * x4 + 2]) * out_scale, __uint_as_float(r[4 * x4 + 3]) * out_scale);
          }
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();   // the peer's shared memory / TMEM stay alive until every MMA of the pair has drained
  if (warp == 2) ptx::tmem_dealloc_pair(tmem_base, TMEM_COLS);
}

// ===================================================================================================== forward
constexpr int FWD_EPI_WARPS = 16;
constexpr int FWD_THREADS = 32 * (4 + FWD_EPI_WARPS);
constexpr int FWD_SMALL = 16384;   // barriers (512) | tmem ptr | +1024: column vectors 2 x 2 x 256 f32 (4 KiB)
                                   // | +5120: column partials 2 x 4 x 256 f32 (8 KiB) | +13312: row partials 16 x 32 f32

struct FwdParams {
  int n_rows, n_cols, d;
  int nkc, n_steps, stages;
  int n_pairs;        // row blocks (pairs of CTAs)
  int split_steps;    // steps per work item: the column sweep is cut into ceil(n_steps / split_steps) work items per
                      // row block so that the grid fills whole waves of CTA pairs
  long long diag_offset;
  float scale;
  const float* scale_dev;  // optional DEVICE scalar s (see BwdParams)
  const float* rinv_x;
  const float* rinv_y;
  float* row_part;    // [n_split][n_rows] partial sum_j exp(S_ij - s) over the item's columns (MODE 2: sum_j exp(S_ij - m))
  float* row_part_m;  // MODE 2: [n_split][n_rows] the item's running row maximum m (natural-log units)
  float* col_part;    // [gridDim.x][col_ld] partial sum_i exp(S_ij - s) over this CTA's rows
  long long col_ld;   // n_steps * 256
  float* diag;        // [n_rows]
  // retrieval (MODE 1): per work item and column group, every row's K best columns
  float* cand_score;  // [n_split * 4][n_rows][KT]   rinv_x[i] rinv_y[j] <x_i, y_j>  (cosine similarity)
  int* cand_idx;      // same shape: col_offset + j, or -1
  int* row_thr;       // [n_rows] order-preserving int key of a lower bound on each row's final K-th best score, shared
                      // by all work items of the row through atomicMax (initialised to a very negative key)
  long long col_offset;
  Group grp;          // MODE 0 / 2: several problems in one launch (n_prob = 0: one); the column-partial matrix then has
                      // 2 * pairs_per_prob rows (the problems own disjoint column ranges)
  // Row-sharded step with the gather of the columns running BESIDE this sweep (MODE 0, clipnce_forward_gathered): the
  // columns are the row blocks of `n_src` ranks, steps_per_src steps each; the copy engines of the peers deliver them
  // while the sweep runs and raise src_flags[q] (>= *src_epoch) behind block q.  The sweep visits the steps ROTATED by
  // rot_steps -- the local block first, then the blocks in the order the peers send them -- and waits for a block's
  // flag before its first TMA load / rinv read.  src_flags = nullptr: everything is there, no rotation.
  const uint32_t* src_flags;
  const uint32_t* src_epoch;
  int rot_steps, steps_per_src, self_src;
  unsigned long long wait_timeout_ns;
  float shift_off;    // MODE 0: the sums are taken relative to the fixed shift s - shift_off (0: the plain fixed shift s)
  const int* gate;    // optional DEVICE flag: the launch does nothing unless *gate != 0 (the exact fallback sweeps of the
                      // speculative large-scale forward, clipnce_api.cu)
};

// wait until the peer that owns source block `src` has delivered it (see FwdParams::src_flags); bounded: a lost rank traps
__device__ __forceinline__ void wait_src_block(const uint32_t* flags, uint32_t epoch, int src, unsigned long long timeout_ns) {
  const uint32_t* f = flags + src;
  if ((int32_t)(ptx::ld_acquire_sys(f) - epoch) >= 0) return;
  const unsigned long long t0 = ptx::globaltimer_ns();
  while ((int32_t)(ptx::ld_acquire_sys(f) - epoch) < 0) {
    __nanosleep(100);
    if (ptx::globaltimer_ns() - t0 > timeout_ns) __trap();
  }
}

__host__ __device__ constexpr int fwd_smem_bytes(int rows, int nkc, int stages) {
  return nkc * rows * 128 + stages * STAGE_BYTES + FWD_SMALL;
}

// ROWS = resident rows per CTA: 128 (M = 256, lane = row) for d <= 512, else 64 (M = 128, 2x2 layout).
// MODE 0: InfoNCE forward statistics.  MODE 1 (ROWS = 128 only): retrieval -- the same similarity sweep with a running
// top-KT per row instead of the soft-max sums (run1/full.py:152 argmax, :157 cosine_similarity; BASELINE config 5).
// MODE 2: ROW statistics only, with a true running maximum (online soft-max): for logit scales beyond the fixed shift's
// range -- exp().clamp(max=100) of old/clip_opt.py:100, run1/full.py:76 -- and for un-normalised queue rows
// (tong/utils/losses.py:10-14), where |S_ij| <= s does not hold.  The column statistics come from a second launch with
// the operands swapped (thread = row makes the row maximum a thread-local scalar; a column maximum would need a
// cross-lane reduction per tile).
template <int ROWS, int MODE = 0, int KT = 1>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(FWD_THREADS, 1)
fwd_kernel(const __grid_constant__ CUtensorMap tmap_x,   // X box {64 k, ROWS rows}
           const __grid_constant__ CUtensorMap tmap_y,   // Y box {64 k, 128 rows}
           const FwdParams p) {
  static_assert(ROWS == 64 || ROWS == 128, "ROWS");
  static_assert(MODE != 1 || ROWS == 128, "retrieval uses the 128-row variant");
  constexpr int X_CHUNK = ROWS * 128;
  constexpr int SBUF_COLS = ROWS == 128 ? 256 : 128;       // TMEM columns of one logits buffer
  constexpr int NCH = ROWS == 128 ? 2 : 1;                 // 32-column chunks per warp per step
  constexpr int NSLOT = ROWS == 128 ? 4 : 2;               // warps (lane quarters) that share a column
  constexpr int EPI_THREADS = FWD_EPI_WARPS * 32;

  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t base = ptx::smem_u32(smem);
  if ((base & 1023u) != 0) __trap();
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int item = blockIdx.x >> 1;
  const int split = item / p.n_pairs;
  const int i0 = (item % p.n_pairs) * (2 * ROWS) + (int)rank * ROWS;
  const GroupView gv = group_view(p.grp, item % p.n_pairs, p.n_steps, p.n_rows, p.n_cols);
  const int t_begin = gv.t_lo + split * p.split_steps;
  const int t_end = min(gv.t_hi, t_begin + p.split_steps);
  // this CTA's row of the column-partial matrix
  const int col_row = 2 * (p.grp.n_prob ? (item % p.n_pairs) % p.grp.pairs_per_prob : item % p.n_pairs) + (int)rank;
  if (p.gate != nullptr && __ldg(p.gate) == 0) return;   // uniform over the grid: before any barrier / TMEM allocation
  const float k2 = (p.scale_dev != nullptr ? __ldg(p.scale_dev) : p.scale) * LOG2E;
  // loop steps are ROTATED steps; act() gives the step's place in the column order of the operands and statistics
  const bool gathered = p.src_flags != nullptr;
  const uint32_t src_epoch = gathered ? __ldg(p.src_epoch) : 0u;
  auto act = [&](int t) -> int {
    if (!gathered) return t;
    const int ta = t + p.rot_steps;
    return ta >= p.n_steps ? ta - p.n_steps : ta;
  };

  const uint32_t x_smem = base;
  const uint32_t ring_a = x_smem + p.nkc * X_CHUNK;
  const uint32_t small_off = (ring_a - base) + p.stages * STAGE_BYTES;
  const uint32_t bars = base + small_off;
  auto bar = [&](int i) -> uint32_t { return bars + 8u * i; };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + small_off + 512);
  float* const colv = reinterpret_cast<float*>(smem + small_off + 1024);     // [2][2][256]: cj, c0
  float* const colred = reinterpret_cast<float*>(smem + small_off + 5120);   // [2][4][256]
  float* const rowred = reinterpret_cast<float*>(smem + small_off + 13312);  // [16][32]

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_x);
    ptx::prefetch_tmap(&tmap_y);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < MAX_STAGES; ++s) {
      ptx::mbar_init(bar(B_FULL_A + s), 1);
      ptx::mbar_init(bar(B_EMPTY_A + s), 1);
    }
    ptx::mbar_init(bar(B_XFULL), 1);
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(bar(B_SFULL + b), 1);
      ptx::mbar_init(bar(B_SEMPTY + b), 2 * FWD_EPI_WARPS);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 2) ptx::tmem_alloc_pair(ptx::smem_u32(const_cast<uint32_t*>(tmem_ptr_smem)), TMEM_COLS);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ================================================================= producer: resident X, then Y rows
    if (ptx::elect_one()) {
      if (leader) ptx::mbar_arrive_expect_tx(bar(B_XFULL), 2 * p.nkc * X_CHUNK);
      for (int kc = 0; kc < p.nkc; ++kc)
        ptx::tma_load_2d_pair(x_smem + kc * X_CHUNK, &tmap_x, bar(B_XFULL), kc * 64, i0 + gv.xs);
      int stage = 0;
      uint32_t phase = 0;
      int cur_src = p.self_src;
      for (int t = t_begin; t < t_end; ++t) {
        const int ta = act(t);
        if (gathered) {
          const int src = ta / p.steps_per_src;
          if (src != cur_src) {   // first tile of a block another rank delivers: its flag, then generic -> async proxy
            if (src != p.self_src) {
              wait_src_block(p.src_flags, src_epoch, src, p.wait_timeout_ns);
              ptx::fence_proxy_async_all();
            }
            cur_src = src;
          }
        }
        for (int g = 0; g < p.nkc; ++g) {
          ptx::mbar_wait(bar(B_EMPTY_A + stage), phase ^ 1u);
          if (leader) ptx::mbar_arrive_expect_tx(bar(B_FULL_A + stage), 2 * STAGE_BYTES);
          ptx::tma_load_2d_pair(ring_a + stage * STAGE_BYTES, &tmap_y, bar(B_FULL_A + stage), g * 64,
                                ta * STEP_J + (int)rank * 128 + gv.ys);
          if (++stage == p.stages) { stage = 0; phase ^= 1u; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================================================= logits MMA issuer (leader)
    if (leader && ptx::elect_one()) {
      constexpr uint32_t idesc_s = ptx::idesc_bf16_f32_major(2 * ROWS, STEP_J, 0, 0);
      const uint32_t desc_hi = static_cast<uint32_t>(ptx::smem_desc_k_sw128(0) >> 32);
      auto desc = [&](uint32_t addr) -> uint64_t {
        return (static_cast<uint64_t>(desc_hi) << 32) | (((addr & 0x3FFFFu) >> 4) | (1u << 16));
      };
      int stage = 0;
      uint32_t phase = 0, ready = 0;
      ptx::mbar_wait(bar(B_XFULL), 0);
      for (int t = 0; t < t_end - t_begin; ++t) {
        const int sb = t & 1;
        ptx::mbar_wait(bar(B_SEMPTY + sb), ((t >> 1) & 1) ^ 1u);
        const uint32_t d_tmem = tmem_base + sb * SBUF_COLS;
        for (int g = 0; g < p.nkc; ++g) {
          if (!ready) ptx::mbar_wait(bar(B_FULL_A + stage), phase);
          ptx::tc_fence_after();
          int ns = stage + 1;
          uint32_t np = phase;
          if (ns == p.stages) { ns = 0; np ^= 1u; }
          ready = ptx::mma_box_pair(d_tmem, desc(x_smem + g * X_CHUNK), desc(ring_a + stage * STAGE_BYTES), 2, 2, idesc_s,
                                    g != 0, bar(B_FULL_A + ns), np);
          ptx::mma_commit_pair(bar(B_EMPTY_A + stage));
          if (g == p.nkc - 1) ptx::mma_commit_pair(bar(B_SFULL + sb));
          stage = ns;
          phase = np;
        }
      }
    }
    __syncwarp();
  } else if (warp >= 4 && MODE == 1) {
    // ================================================================= epilogue (retrieval): running top-KT per row
    const int e = warp - 4;
    const int q = warp & 3;
    const int cgp = e >> 2;
    const int i_local = 32 * q + lane;
    const long long i_glob = (long long)i0 + i_local;
    const bool row_ok = i_glob < p.n_rows;
    const int col0 = 64 * cgp;
    const int te = threadIdx.x - 128;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t sempty_leader = ptx::mapa(bar(B_SEMPTY), 0);
    float bv[KT];   // descending; ties keep the earlier (lower) column
    int bi[KT];
#pragma unroll
    for (int k = 0; k < KT; ++k) { bv[k] = -INFINITY; bi[k] = -1; }
    // Shared threshold.  Every thread's K-th best is a lower bound on its row's final K-th best, so the maximum over
    // all threads that ever worked on the row (other column groups, other work items, earlier waves) is one too:
    // columns strictly below it can be skipped without changing the result (ties are kept: >=).  Work items that start
    // after the first wave begin with a warm threshold and insert almost nothing -- the sorted insertion, executed by
    // the whole warp whenever one lane needs it, was 55 % of the sweep time with cold lists (k = 10, 125 k-row shard).
    // Lists hold the UNSCALED score acc * rinv_y[j]; the shared key is of the scaled score (* rinv_x[i] > 0).
    const float rxp = row_ok ? p.rinv_x[i_glob] : 1.f;
    const float rxp_inv = 1.f / fmaxf(rxp, 1e-30f);
    auto shared_bound = [&]() -> float {   // the row's published bound in list units, nudged DOWN past every rounding
      const float u = key_float(__ldcg(p.row_thr + i_glob)) * rxp_inv;
      return u - (fabsf(u) * 4e-7f + 1e-37f);
    };
    float thr = row_ok ? shared_bound() : INFINITY;   // rows past the end: skip all
    float published = -INFINITY;

    float ry_n = 0.f;
    if (te < STEP_J) {
      const long long j = (long long)t_begin * STEP_J + te;
      ry_n = (j < p.n_cols) ? p.rinv_y[j] : -1.f;
    }
    for (int t = t_begin; t < t_end; ++t) {
      const int tl = t - t_begin;
      const int sb = tl & 1;
      float* const cv = colv + (tl & 1) * 512;
      if (te < STEP_J) {
        cv[te] = ry_n < 0.f ? 0.f : ry_n;                  // score / rinv_x[i] = acc * rinv_y[j]
        cv[256 + te] = ry_n < 0.f ? -INFINITY : 0.f;       // columns past the end never enter a list
        const long long jn = (long long)(t + 1) * STEP_J + te;
        ry_n = (t + 1 < t_end && jn < p.n_cols) ? p.rinv_y[jn] : -1.f;
      }
      if ((tl & 3) == 3 && row_ok) {   // every 4 steps: publish this thread's bound, pick up everybody else's
        if (bv[KT - 1] > published) {
          published = bv[KT - 1];
          atomicMax(p.row_thr + i_glob, float_key(published * rxp));
        }
        thr = fmaxf(thr, shared_bound());
      }
      named_bar_sync(1, EPI_THREADS);
      ptx::mbar_wait(bar(B_SFULL + sb), (tl >> 1) & 1);
      ptx::tc_fence_after();
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(t_lane + sb * SBUF_COLS + col0 + 32 * c, r);
        ptx::tmem_ld_wait();
        if (c == 1) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_cluster(sempty_leader + 8u * sb);
        }
        const float* const cjp = cv + col0 + 32 * c;
        const int jbase = t * STEP_J + col0 + 32 * c;
#pragma unroll
        for (int x4 = 0; x4 < 8; ++x4) {
          const float4 ry4 = *reinterpret_cast<const float4*>(cjp + 4 * x4);
          const float4 c04 = *reinterpret_cast<const float4*>(cjp + 256 + 4 * x4);
          const float ryv[4] = {ry4.x, ry4.y, ry4.z, ry4.w};
          const float c0v[4] = {c04.x, c04.y, c04.z, c04.w};
          float v4[4];
#pragma unroll
          for (int xx = 0; xx < 4; ++xx) v4[xx] = fmaf(__uint_as_float(r[4 * x4 + xx]), ryv[xx], c0v[xx]);
          // one test per four columns: insertions are rare once the threshold is warm
          const float cut = fmaxf(bv[KT - 1], thr);
          if (fmaxf(fmaxf(v4[0], v4[1]), fmaxf(v4[2], v4[3])) >= cut) {
#pragma unroll
            for (int xx = 0; xx < 4; ++xx) {
              const float v = v4[xx];
              if (v > bv[KT - 1] && v >= thr) {
                const int j = jbase + 4 * x4 + xx;
#pragma unroll
                for (int k = KT - 1; k > 0; --k) {
                  const bool up = v > bv[k - 1];
                  const bool here = v > bv[k];
                  bi[k] = up ? bi[k - 1] : (here ? j : bi[k]);
                  bv[k] = up ? bv[k - 1] : (here ? v : bv[k]);
                }
                if (v > bv[0]) { bv[0] = v; bi[0] = j; }
              }
            }
          }
        }
      }
    }
    if (row_ok && bv[KT - 1] > published) atomicMax(p.row_thr + i_glob, float_key(bv[KT - 1] * rxp));
    if (row_ok) {
      const float rx = p.rinv_x[i_glob];
      const long long o = (((long long)split * 4 + cgp) * p.n_rows + i_glob) * KT;
#pragma unroll
      for (int k = 0; k < KT; ++k) {
        p.cand_score[o + k] = bv[k] * rx;
        p.cand_idx[o + k] = bi[k] < 0 ? -1 : (int)(p.col_offset + bi[k]);
      }
    }
  } else if (warp >= 4 && MODE == 2) {
    // ================================================================= epilogue (online soft-max): row (max, sum), diagonal
    const int e = warp - 4;
    const int q = warp & 3;
    const int cgp = e >> 2;
    const int i_local = ROWS == 128 ? 32 * q + lane : 32 * (q & 1) + lane;
    const long long i_glob = (long long)i0 + i_local;
    const bool row_ok = i_glob < gv.n_rows;
    const int col0 = (ROWS == 128 ? 64 : 32) * cgp;
    const int jl0 = (ROWS == 128 ? 0 : 128 * (q >> 1)) + col0;
    const int te = threadIdx.x - 128;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float rx = row_ok ? p.rinv_x[i_glob + gv.xs] : 0.f;
    const uint32_t sempty_leader = ptx::mapa(bar(B_SEMPTY), 0);
    const long long dcol0 = i_glob + p.diag_offset;
    float m_run = -1e30f, l_run = 0.f;   // base-2 units: S log2(e)

    float ry_n = 0.f;
    if (te < STEP_J) {
      const long long j = (long long)t_begin * STEP_J + te;
      ry_n = (j < gv.n_cols) ? p.rinv_y[j + gv.ys] : -1.f;
    }
    for (int t = t_begin; t < t_end; ++t) {
      const int tl = t - t_begin;
      const int sb = tl & 1;
      float* const cv = colv + (tl & 1) * 512;
      if (te < STEP_J) {
        cv[te] = ry_n < 0.f ? 0.f : ry_n * k2;
        cv[256 + te] = ry_n < 0.f ? -INFINITY : 0.f;   // columns past the end never enter a maximum or a sum
        const long long jn = (long long)(t + 1) * STEP_J + te;
        ry_n = (t + 1 < t_end && jn < gv.n_cols) ? p.rinv_y[jn + gv.ys] : -1.f;
      }
      named_bar_sync(1, EPI_THREADS);
      ptx::mbar_wait(bar(B_SFULL + sb), (tl >> 1) & 1);
      ptx::tc_fence_after();
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(t_lane + sb * SBUF_COLS + col0 + 32 * c, r);
        ptx::tmem_ld_wait();
        if (c == NCH - 1) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_cluster(sempty_leader + 8u * sb);
        }
        const float* const cjp = cv + jl0 + 32 * c;
        const long long dl = dcol0 - ((long long)t * STEP_J + jl0 + 32 * c);
        if (p.diag != nullptr && row_ok && dl >= 0 && dl < 32) {
#pragma unroll
          for (int x = 0; x < 32; ++x)
            if (dl == x) p.diag[i_glob] = __uint_as_float(r[x]) * rx * cjp[x] * LN2;
        }
        float y[32];
        float tmax = -INFINITY;
#pragma unroll
        for (int x4 = 0; x4 < 8; ++x4) {
          const float4 cj4 = *reinterpret_cast<const float4*>(cjp + 4 * x4);
          const float4 c04 = *reinterpret_cast<const float4*>(cjp + 256 + 4 * x4);
          const float cjv[4] = {cj4.x, cj4.y, cj4.z, cj4.w};
          const float c0v[4] = {c04.x, c04.y, c04.z, c04.w};
#pragma unroll
          for (int xx = 0; xx < 4; ++xx) {
            y[4 * x4 + xx] = fmaf(__uint_as_float(r[4 * x4 + xx]) * rx, cjv[xx], c0v[xx]);
            tmax = fmaxf(tmax, y[4 * x4 + xx]);
          }
        }
        const float nm = fmaxf(m_run, tmax);
        float r4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int x = 0; x < 32; ++x) r4[x & 3] += ex2(y[x] - nm);
        l_run = fmaf(l_run, ex2(m_run - nm), (r4[0] + r4[1]) + (r4[2] + r4[3]));
        m_run = nm;
      }
    }
    // combine the warps that share a row (column groups; for the 2x2 layout both column halves) in fixed order
    float* const rowred_m = colred;          // [16][32]   (the column-partial staging is unused in this mode)
    rowred_m[e * 32 + lane] = m_run;
    rowred[e * 32 + lane] = l_run;
    named_bar_sync(1, EPI_THREADS);
    if (te < ROWS) {
      const int rq = te >> 5, rl = te & 31;
      float mm = -1e30f;
#pragma unroll
      for (int w = 0; w < FWD_EPI_WARPS; ++w) {
        const bool mine = ROWS == 128 ? ((w & 3) == rq) : ((w & 1) == rq);
        if (mine) mm = fmaxf(mm, rowred_m[w * 32 + rl]);
      }
      float tot = 0.f;
#pragma unroll
      for (int w = 0; w < FWD_EPI_WARPS; ++w) {
        const bool mine = ROWS == 128 ? ((w & 3) == rq) : ((w & 1) == rq);
        if (mine) tot += rowred[w * 32 + rl] * ex2(rowred_m[w * 32 + rl] - mm);
      }
      if ((long long)i0 + te < gv.n_rows) {
        p.row_part_m[(long long)split * p.n_rows + i0 + te] = mm * LN2;
        p.row_part[(long long)split * p.n_rows + i0 + te] = tot;
      }
    }
  } else if (warp >= 4) {
    // ================================================================= epilogue: row sums, column partials, diagonal
    const int e = warp - 4;            // 0..15
    const int q = warp & 3;            // TMEM lane quarter
    const int cgp = e >> 2;            // column group of this warp
    const int i_local = ROWS == 128 ? 32 * q + lane : 32 * (q & 1) + lane;
    const long long i_glob = (long long)i0 + i_local;
    const bool row_ok = i_glob < gv.n_rows;
    const bool warp_rows_ok = (long long)i0 + (i_local - lane) + 32 <= gv.n_rows;   // warp-uniform
    const int col0 = (ROWS == 128 ? 64 : 32) * cgp;                 // first TMEM column of this warp
    const int jl0 = (ROWS == 128 ? 0 : 128 * (q >> 1)) + col0;      // its step-local column
    const int slot = ROWS == 128 ? q : (q & 1);
    const int te = threadIdx.x - 128;  // 0..511
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float rx = row_ok ? p.rinv_x[i_glob + gv.xs] : 0.f;
    const uint32_t sempty_leader = ptx::mapa(bar(B_SEMPTY), 0);
    const long long dcol0 = i_glob + p.diag_offset;
    float rsum = 0.f;

    auto flush_cols = [&](int t) {   // column partials of step t: sum the lane quarters in fixed order
      if (te < STEP_J) {
        const float* cr = colred + ((t - t_begin) & 1) * 1024 + te;
        float s = cr[0] + cr[256];
        if (NSLOT == 4) s = (s + cr[512]) + cr[768];
        p.col_part[(long long)col_row * p.col_ld + (long long)act(t) * STEP_J + te] = s;
      }
    };
    // 1/norm of the columns of (rotated) step t; gathered: a block's values are read only behind its owner's flag
    int cur_src = p.self_src;
    auto load_ry = [&](int t) -> float {
      const int ta = act(t);
      if (gathered) {
        const int src = ta / p.steps_per_src;
        if (src != cur_src) {
          if (src != p.self_src) wait_src_block(p.src_flags, src_epoch, src, p.wait_timeout_ns);
          cur_src = src;
        }
      }
      const long long j = (long long)ta * STEP_J + te;
      return (j < gv.n_cols) ? p.rinv_y[j + gv.ys] : -1.f;   // -1 marks a column past the end
    };

    float ry_n = 0.f;
    if (te < STEP_J) ry_n = load_ry(t_begin);
    for (int t = t_begin; t < t_end; ++t) {
      const int tl = t - t_begin;
      const int sb = tl & 1;
      const int ta = act(t);
      float* const cv = colv + (tl & 1) * 512;
      if (te < STEP_J) {
        cv[te] = ry_n < 0.f ? 0.f : ry_n * k2;
        cv[256 + te] = ry_n < 0.f ? -10000.f : p.shift_off * LOG2E - k2;   // invalid column: exp2(-10000) = 0 leaves every sum untouched
        ry_n = t + 1 < t_end ? load_ry(t + 1) : -1.f;
      }
      named_bar_sync(1, EPI_THREADS);
      if (t > t_begin) flush_cols(t - 1);

      ptx::mbar_wait(bar(B_SFULL + sb), (tl >> 1) & 1);
      ptx::tc_fence_after();
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(t_lane + sb * SBUF_COLS + col0 + 32 * c, r);
        ptx::tmem_ld_wait();
        if (c == NCH - 1) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_cluster(sempty_leader + 8u * sb);
        }
        const float* const cjp = cv + jl0 + 32 * c;
        const long long dl = dcol0 - ((long long)ta * STEP_J + jl0 + 32 * c);
        if (row_ok && dl >= 0 && dl < 32) {
#pragma unroll
          for (int x = 0; x < 32; ++x)
            if (dl == x) p.diag[i_glob] = __uint_as_float(r[x]) * rx * cjp[x] * LN2;   // S_ii = acc rx ry s
        }
        float ev[32];
#pragma unroll
        for (int x4 = 0; x4 < 8; ++x4) {
          const float4 cj4 = *reinterpret_cast<const float4*>(cjp + 4 * x4);
          const float4 c04 = *reinterpret_cast<const float4*>(cjp + 256 + 4 * x4);
          const float cjv[4] = {cj4.x, cj4.y, cj4.z, cj4.w};
          const float c0v[4] = {c04.x, c04.y, c04.z, c04.w};
#pragma unroll
          for (int xx = 0; xx < 4; ++xx)
            ev[4 * x4 + xx] = ex2(fmaf(__uint_as_float(r[4 * x4 + xx]) * rx, cjv[xx], c0v[xx]));
        }
        if (!warp_rows_ok) {
#pragma unroll
          for (int x = 0; x < 32; ++x) ev[x] = row_ok ? ev[x] : 0.f;   // rows past the end: TMA zero-filled operands
        }
        float r4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int x = 0; x < 32; ++x) r4[x & 3] += ev[x];
        rsum += (r4[0] + r4[1]) + (r4[2] + r4[3]);
        tc::warp_transpose_reduce<32>(ev, lane);   // lane L: sum over this warp's 32 rows of column L
        colred[(tl & 1) * 1024 + slot * 256 + jl0 + 32 * c + lane] = ev[0];
      }
    }
    named_bar_sync(1, EPI_THREADS);
    if (t_end > t_begin) flush_cols(t_end - 1);

    // row sums: combine the warps that share a row (column groups, and for the 2x2 layout both column halves)
    rowred[e * 32 + lane] = rsum;
    named_bar_sync(1, EPI_THREADS);
    if (te < ROWS) {
      const int rq = te >> 5, rl = te & 31;
      float tot = 0.f;
#pragma unroll
      for (int w = 0; w < FWD_EPI_WARPS; ++w) {
        const bool mine = ROWS == 128 ? ((w & 3) == rq) : ((w & 1) == rq);
        if (mine) tot += rowred[w * 32 + rl];
      }
      if ((long long)i0 + te < gv.n_rows) p.row_part[(long long)split * p.n_rows + i0 + te] = tot;
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  if (warp == 2) ptx::tmem_dealloc_pair(tmem_base, TMEM_COLS);
}

}  // namespace pair
