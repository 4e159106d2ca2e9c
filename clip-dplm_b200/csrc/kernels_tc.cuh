// tcgen05 / TMEM / TMA kernels for the contrastive hot path (sm_100a only).
//
// One kernel template, two modes, both sweeping the logits S_ij = s rinv_x[i] rinv_y[j] <x_i, y_j>
// tile by tile without ever writing S (or its gradient G) to HBM:
//
//   MODE 0  forward statistics   row sums  sum_j exp(S_ij - s),  column partial sums, diagonal
//   MODE 1  backward, one side   dXhat = s * G Yhat,  G_ij = exp(S_ij - s)(u_i + v_j) - w [j == i+off]
//
// Orientation.  A CTA owns BLOCK_I rows of X (resident in shared memory for the whole sweep) and
// streams 128-row tiles of Y.  The logits tile is computed TRANSPOSED,
//       St[j (128 TMEM lanes), i (BLOCK_I TMEM columns)] = Y_J . X_I^T               (UMMA 128 x BLOCK_I x 16)
// so that epilogue thread <-> lane <-> column j of S:  per-column quantities (rinv_y[j], v_j, the
// column partial sum) are thread-local scalars, per-row quantities (rinv_x[i], u_i, the row sums) are
// indexed by the TMEM column, accumulated thread-locally over the whole sweep and reduced across
// lanes once per CTA.  No shuffle in the per-element path.  The normalise is fused here: the tensor
// cores see the caller's raw bf16 rows and rinv_x[i] * rinv_y[j] scales the fp32 accumulator.
//
// In MODE 1 the gradient tile is rounded to bf16, written to shared memory as the K-major B operand
// of a second MMA and contracted against the TRANSPOSED streamed operand:
//       dXhat^T[d (128 lanes, nq chunks), i (BLOCK_I columns)] += Y^T[d, j] . G^T[j, i]  (UMMA 128 x BLOCK_I x 16)
// The accumulators (nq * BLOCK_I TMEM columns) stay resident for the whole sweep; two S buffers use
// the remaining columns: BLOCK_I = 64 (6 x 64 + 2 x 64 = 512 columns at d = 768).  Every MMA
// operand is the same canonical layout: K-major, 128-byte rows, SWIZZLE_128B (what a TMA box
// {64 elems, R rows} writes), so one descriptor builder serves all of them.
//
// What bounds it (ncu, profiles/): with 128 x BLOCK_I x 16 instructions the operands stream through
// shared memory faster than they are consumed per byte -- TMA writes + UMMA operand reads saturate the
// 128 B/clk shared-memory port before the tensor pipe fills.  Hence the largest BLOCK_I that TMEM
// allows, separate issue warps (a single issuing thread was the first limiter), and K = 128 stages.
//
// Warp roles (384 threads): warp 0 TMA producer A (X panel, Y boxes), warp 1 logits-MMA issuer,
// warp 2 TMEM allocator + TMA producer B (Y^T boxes), warp 3 gradient-MMA issuer, warps 4-11 epilogue
// (two warps per TMEM lane quarter, each taking half of the tile's columns).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>
#include "ptx.cuh"

namespace tc {

constexpr int BLOCK_J = 128;                         // streamed rows per tile == UMMA M == TMEM lanes
constexpr int BLOCK_K = 64;                          // 64 bf16 = 128 B = one swizzle row
constexpr int UMMA_K = 16;
constexpr int BOX_BYTES = BLOCK_J * BLOCK_K * 2;     // one TMA box [128 rows][64 elems] = 16 KiB
constexpr int MAX_STAGES = 5;                        // per ring (one 16 KiB box per stage)
// epilogue warps: MODE 0 gives every warp 32 TMEM columns (BLOCK_I / 32 warps per lane quarter: ex2-bound, it wants
// many warps and few registers each); MODE 1 splits the tile's columns between two warps per lane quarter
__host__ __device__ constexpr int num_epi_warps(int mode, int block_i) { return mode == 0 ? 4 * (block_i / 32) : 8; }
__host__ __device__ constexpr int num_threads(int mode, int block_i) { return 32 * (4 + num_epi_warps(mode, block_i)); }
constexpr int TMEM_COLS = 512;
constexpr int SMEM_LIMIT = 232448;                   // 227 KiB opt-in maximum per CTA
constexpr float LOG2E = 1.4426950408889634f;
constexpr float LN2 = 0.6931471805599453f;
__host__ __device__ constexpr int small_bytes(int mode) { return mode == 1 ? 1536 : 3584; }  // barriers, tmem ptr, u/rinv, scratch
__host__ __device__ constexpr int g_bytes(int block_i) { return block_i * BLOCK_J * 2; }     // bf16 gradient tile [i][128 j]

struct Params {
  int n_rows, n_cols, d;
  int nkc;         // ceil(d / 64)   K boxes per logits tile
  int nq;          // ceil(d / 128)  accumulator chunks of the gradient MMA
  int n_jt;        // ceil(n_cols / 128)
  int stages_a;    // ring A (16 KiB stages): streamed Y boxes for the logits MMA
  int stages_b;    // ring B: streamed Y^T boxes for the gradient MMA (MODE 1)
  long long diag_offset;
  float scale;     // s
  float k2;        // s * log2(e)   (host copies; the kernel recomputes both when scale_dev is set)
  const float* scale_dev;   // optional DEVICE scalar s
  float grad_out;
  const float* rinv_x;   // [n_rows]  1 / |x_i|   (the normalise, applied to the fp32 accumulator)
  const float* rinv_y;   // [n_cols]
  // MODE 0 outputs
  float* row_m;        // [n_rows]           = s (the fixed shift)
  float* row_l;        // [n_rows]           sum_j exp(S_ij - s)
  float* col_part;     // [2 * gridDim.x][col_ld]  partial sum_i exp(S_ij - s)
  long long col_ld;
  float* diag;         // [n_rows]
  // MODE 1 inputs / outputs
  const float* row_m_in;  // [n_rows]  G_ij = exp(S_ij - row_m_i) row_w_i + exp(S_ij - col_m_j) col_w_j - ...
  const float* row_w;     // [n_rows]
  const float* col_m_in;  // [n_cols] or nullptr
  const float* col_w;     // [n_cols] or nullptr
  float diag_w;
  float out_scale;     // grad_out * s
  float* dx;           // [n_rows, d] f32
  float* ds_part;      // [gridDim.x]  sum G.S of this CTA
};

__host__ __device__ constexpr int smem_bytes(int mode, int block_i, int nkc, int ring_boxes) {
  return nkc * block_i * 128 + ring_boxes * BOX_BYTES + (mode == 1 ? 2 * g_bytes(block_i) : 0) + small_bytes(mode);
}

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// exp2 on the FMA/ALU pipes: range reduction by the 1.5*2^23 rounding trick, degree-5 minimax polynomial for 2^f on
// [-0.5, 0.5] (max relative error 2.4e-7, the same class as MUFU.EX2), exponent spliced in with an integer add.  Valid
// for x in [-125, 1]; the tensor-core path guarantees x >= -2 s log2(e) >= -124.1.  These single-CTA kernels split the
// exponentials 1:3 between MUFU and this polynomial; tools/umma_probe.cu later measured MUFU.EX2 at 16 results/clk/SM
// against 11.7 for the polynomial (issue-bound), so the pair kernels (kernels_pair.cuh) simply use MUFU.
__device__ __forceinline__ float ex2_poly(float x) {
  const float t = x + 12582912.0f;
  const float f = x - (t - 12582912.0f);
  float q = 0.001327646430581808f;
  q = fmaf(q, f, 0.009675540961325169f);
  q = fmaf(q, f, 0.05550713464617729f);
  q = fmaf(q, f, 0.24022120237350464f);
  q = fmaf(q, f, 0.6931469440460205f);
  q = fmaf(q, f, 1.0000001192092896f);
  return __int_as_float(__float_as_int(q) + (__float_as_int(t) << 23));
}
// One logit in MUFU_EVERY goes to the MUFU, the others to the polynomial: both pipes stay busy.
constexpr int MUFU_EVERY = 4;
template <int X>
__device__ __forceinline__ float ex2_mix(float x) { return (X % MUFU_EVERY == 0) ? ex2(x) : ex2_poly(x); }

template <int THREADS>
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(THREADS) : "memory"); }

// Transposing butterfly: every lane holds N partial sums v[0..N); afterwards lane L holds, in
// v[0..N/32), the totals over the warp of entries (N/32)*L + {0..N/32-1}.
template <int N>
__device__ __forceinline__ void warp_transpose_reduce(float (&v)[N], int lane) {
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const int mask = 16 >> s;
    const int half = (N / 2) >> s;
    const bool upper = (lane & mask) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float keep = upper ? v[i + half] : v[i];
      const float send = upper ? v[i] : v[i + half];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, mask);
    }
  }
}

template <int MODE, int BLOCK_I>
__global__ void __launch_bounds__(num_threads(MODE, BLOCK_I), 1)
clip_tc_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_y,
               const __grid_constant__ CUtensorMap tmap_yt, const Params p) {
  static_assert(BLOCK_I == 64 || BLOCK_I == 128, "BLOCK_I");
  static_assert(MODE == 0 || BLOCK_I == 64, "backward: accumulators + logits must fit 512 TMEM columns");
  constexpr int X_CHUNK = BLOCK_I * 128;        // bytes of one [BLOCK_I rows x 64 k] chunk of the resident panel
  constexpr int HALF = BLOCK_I / 2;             // TMEM columns per epilogue warp
  constexpr int NSBUF = 2;
  constexpr int S_COL0 = (MODE == 0) ? 0 : TMEM_COLS - NSBUF * BLOCK_I;
  constexpr int G_BYTES = g_bytes(BLOCK_I);
  constexpr int NUM_EPI_WARPS = num_epi_warps(MODE, BLOCK_I);

  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t base = ptx::smem_u32(smem);
  if ((base & 1023u) != 0) __trap();   // SWIZZLE_128B operands need 1 KiB alignment (dynamic smem starts at 1 KiB)

  const uint32_t x_smem = base;
  const uint32_t ring_a = x_smem + p.nkc * X_CHUNK;
  const uint32_t ring_b = ring_a + p.stages_a * BOX_BYTES;
  const uint32_t g_smem = ring_b + (MODE == 1 ? p.stages_b : 0) * BOX_BYTES;
  const uint32_t small_off = (g_smem - base) + (MODE == 1 ? 2 * G_BYTES : 0);
  const uint32_t bars = base + small_off;
  auto bar = [&](int i) -> uint32_t { return bars + 8u * i; };
  constexpr int B_FULL_A = 0, B_EMPTY_A = MAX_STAGES, B_FULL_B = 2 * MAX_STAGES, B_EMPTY_B = 3 * MAX_STAGES,
                B_XFULL = 4 * MAX_STAGES, B_SFULL = B_XFULL + 1, B_SEMPTY = B_SFULL + 2, B_GFULL = B_SEMPTY + 2,
                B_GEMPTY = B_GFULL + 2, B_ACCFULL = B_GEMPTY + 2;
  static_assert((B_ACCFULL + 1) * 8 <= 256, "barrier block");
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + small_off + 256);
  float* const rx_s = reinterpret_cast<float*>(smem + small_off + 512);                            // [BLOCK_I] rinv_x
  float* const u_s = reinterpret_cast<float*>(smem + small_off + 512 + BLOCK_I * 4);               // [BLOCK_I] (MODE 1)
  float* const red = reinterpret_cast<float*>(smem + small_off + (MODE == 1 ? 512 + BLOCK_I * 8 : 1536));  // [8] / [8][64]
  static_assert(MODE == 0 || 512 + BLOCK_I * 8 + 64 <= small_bytes(1), "small block");

  const int warp = threadIdx.x >> 5;   // warp-uniform
  const int lane = threadIdx.x & 31;
  const int i0 = blockIdx.x * BLOCK_I;
  const float sc = p.scale_dev != nullptr ? __ldg(p.scale_dev) : p.scale;
  const float k2 = sc * LOG2E;
  const float out_scale = p.scale_dev != nullptr ? p.grad_out * sc : p.out_scale;
  const int nga = p.nkc;                             // ring-A boxes per tile (K chunks of the logits MMA)
  const int ngb = 2 * p.nq;                          // ring-B boxes per tile ((d chunk, j half) of the gradient MMA)

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_x);
    ptx::prefetch_tmap(&tmap_y);
    if (MODE == 1) ptx::prefetch_tmap(&tmap_yt);
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
      ptx::mbar_init(bar(B_SEMPTY + b), NUM_EPI_WARPS);
      ptx::mbar_init(bar(B_GFULL + b), NUM_EPI_WARPS);
      ptx::mbar_init(bar(B_GEMPTY + b), 1);
    }
    ptx::mbar_init(bar(B_ACCFULL), 1);
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(ptx::smem_u32(const_cast<uint32_t*>(tmem_ptr_smem)), TMEM_COLS);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // Issue-side design (each step measured, see DESIGN.md section 5.1 and tools/umma_bench.cu).
  //  * One ELECTED lane runs each issuing role's whole loop, waits included.  Issuing from inside an
  //    `if (lane == 0)` region makes ptxas wrap every UTCHMMA/UTMALDG in a waterfall loop; electing per
  //    iteration costs a reconvergence (~100 clk) per four MMAs.
  //  * mbarrier.try_wait takes ~170 clk even on a completed phase -- longer than issuing the four MMAs of a box --
  //    so the wait for stage s+1 is started before stage s is issued (ptx::mma_box_prefetch / tma_box_prefetch).
  //  * Logits MMAs and gradient MMAs are issued by two different warps from two different rings.
  const uint32_t desc_hi = static_cast<uint32_t>(ptx::smem_desc_k_sw128(0) >> 32);   // SBO, version, swizzle mode
  auto desc = [&](uint32_t lo) -> uint64_t { return (static_cast<uint64_t>(desc_hi) << 32) | lo; };
  auto desc_lo = [&](uint32_t addr) -> uint32_t { return ((addr & 0x3FFFFu) >> 4) | (1u << 16); };

  if (warp == 0) {
    // ======================================================================= producer A: X panel, then Y boxes
    if (ptx::elect_one()) {
      ptx::mbar_arrive_expect_tx(bar(B_XFULL), p.nkc * X_CHUNK);
      for (int kc = 0; kc < p.nkc; ++kc)
        ptx::tma_load_2d(x_smem + kc * X_CHUNK, &tmap_x, bar(B_XFULL), kc * BLOCK_K, i0);
      int stage = 0;
      uint32_t phase = 0, ready = 1;   // every stage starts free
      for (int t = 0; t < p.n_jt; ++t) {
        for (int g = 0; g < nga; ++g) {
          if (!ready) ptx::mbar_wait(bar(B_EMPTY_A + stage), phase ^ 1u);
          int ns = stage + 1;
          uint32_t np = phase;
          if (ns == p.stages_a) { ns = 0; np ^= 1u; }
          ready = ptx::tma_box_prefetch(ring_a + stage * BOX_BYTES, &tmap_y, bar(B_FULL_A + stage), BOX_BYTES,
                                        g * BLOCK_K, t * BLOCK_J, bar(B_EMPTY_A + ns), np ^ 1u);
          stage = ns;
          phase = np;
        }
      }
    }
    __syncwarp();
  } else if (warp == 2 && MODE == 1) {
    // ======================================================================= producer B: Y^T boxes [128 d][64 j]
    if (ptx::elect_one()) {
      int stage = 0;
      uint32_t phase = 0, ready = 1;
      for (int t = 0; t < p.n_jt; ++t) {
        for (int g = 0; g < ngb; ++g) {   // (d chunk g >> 1, j half g & 1)
          if (!ready) ptx::mbar_wait(bar(B_EMPTY_B + stage), phase ^ 1u);
          int ns = stage + 1;
          uint32_t np = phase;
          if (ns == p.stages_b) { ns = 0; np ^= 1u; }
          ready = ptx::tma_box_prefetch(ring_b + stage * BOX_BYTES, &tmap_yt, bar(B_FULL_B + stage), BOX_BYTES,
                                        t * BLOCK_J + (g & 1) * BLOCK_K, (g >> 1) * 128, bar(B_EMPTY_B + ns), np ^ 1u);
          stage = ns;
          phase = np;
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ======================================================================= logits MMA issuer
    if (ptx::elect_one()) {
      constexpr uint32_t idesc_s = ptx::idesc_bf16_f32(BLOCK_J, BLOCK_I);
      const uint32_t a_lo0 = desc_lo(ring_a), x_lo0 = desc_lo(x_smem);
      int stage = 0;
      uint32_t phase = 0, ready = 0;
      ptx::mbar_wait(bar(B_XFULL), 0);
      for (int t = 0; t < p.n_jt; ++t) {
        const int sb = t % NSBUF;
        ptx::mbar_wait(bar(B_SEMPTY + sb), ((t / NSBUF) & 1) ^ 1u);   // epilogue drained this S buffer
        const uint32_t d_tmem = tmem_base + S_COL0 + sb * BLOCK_I;
        for (int g = 0; g < nga; ++g) {
          if (!ready) ptx::mbar_wait(bar(B_FULL_A + stage), phase);
          ptx::tc_fence_after();
          int ns = stage + 1;
          uint32_t np = phase;
          if (ns == p.stages_a) { ns = 0; np ^= 1u; }
          ready = ptx::mma_box_prefetch(d_tmem, desc(a_lo0 + stage * (BOX_BYTES >> 4)), desc(x_lo0 + g * (X_CHUNK >> 4)),
                                        idesc_s, g != 0, bar(B_FULL_A + ns), np);
          ptx::mma_commit(bar(B_EMPTY_A + stage));
          if (g == nga - 1) ptx::mma_commit(bar(B_SFULL + sb));
          stage = ns;
          phase = np;
        }
      }
    }
    __syncwarp();
  } else if (warp == 3 && MODE == 1) {
    // ======================================================================= gradient MMA issuer
    if (ptx::elect_one()) {
      constexpr uint32_t idesc_g = ptx::idesc_bf16_f32(BLOCK_J, BLOCK_I);
      const uint32_t a_lo0 = desc_lo(ring_b), g_lo0 = desc_lo(g_smem);
      int stage = 0;
      uint32_t phase = 0, ready = 0;
      for (int t = 0; t < p.n_jt; ++t) {
        const int gb = t & 1;
        ptx::mbar_wait(bar(B_GFULL + gb), (t >> 1) & 1);            // epilogue wrote the bf16 gradient tile t
        const uint32_t b_lo = g_lo0 + gb * (G_BYTES >> 4);            // G chunks [BLOCK_I i][64 j] x 2
        for (int g = 0; g < ngb; ++g) {
          if (!ready) ptx::mbar_wait(bar(B_FULL_B + stage), phase);
          ptx::tc_fence_after();
          int ns = stage + 1;
          uint32_t np = phase;
          if (ns == p.stages_b) { ns = 0; np ^= 1u; }
          const int q = g >> 1, kk = g & 1;
          ready = ptx::mma_box_prefetch(tmem_base + q * BLOCK_I, desc(a_lo0 + stage * (BOX_BYTES >> 4)),
                                        desc(b_lo + kk * (G_BYTES >> 5)), idesc_g, (t | kk) != 0, bar(B_FULL_B + ns), np);
          ptx::mma_commit(bar(B_EMPTY_B + stage));
          if (g == ngb - 1) {
            ptx::mma_commit(bar(B_GEMPTY + gb));
            if (t == p.n_jt - 1) ptx::mma_commit(bar(B_ACCFULL));
          }
          stage = ns;
          phase = np;
        }
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ======================================================================= epilogue
    const int e = warp - 4;        // 0..7
    const int q = warp & 3;        // TMEM lane quarter this warp may read
    const int h = e >> 2;          // which half of the tile's columns
    const int j_local = q * 32 + lane;
    const int te = threadIdx.x - 128;
    const int i_valid = max(0, min(BLOCK_I, p.n_rows - i0));
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const long long dcol0 = (long long)i0 + p.diag_offset;   // column of the positive of block row 0

    if (te < BLOCK_I) {
      rx_s[te] = (te < i_valid) ? p.rinv_x[i0 + te] : 0.f;
      // u_i = row_w_i exp(s - row_m_i): exp(S - s) u_i = exp(S - row_m_i) row_w_i from ONE ex2 per logit
      // (row_m_i == s when the statistics come from the MODE 0 kernel, so u_i = row_w_i exactly)
      if (MODE == 1) u_s[te] = (te < i_valid) ? p.row_w[i0 + te] * ex2((sc - p.row_m_in[i0 + te]) * LOG2E) : 0.f;
    }
    epi_bar_sync<NUM_EPI_WARPS * 32>();

    if (MODE == 0) {
      // warp (quarter q, column group cg): lanes j = q*32.., TMEM columns i = cg*32.. -- 32 logits per thread per tile
      const int cg = e >> 2;
      const int ibase = cg * 32;
      float racc[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) racc[i] = 0.f;
      float ry_n = (j_local < p.n_cols) ? p.rinv_y[j_local] : 0.f;   // fetched one tile ahead
      for (int t = 0; t < p.n_jt; ++t) {
        const int b = t & 1;
        const long long jg = (long long)t * BLOCK_J + j_local;
        const bool jvalid = jg < p.n_cols;
        const bool diag_tile = dcol0 < (long long)(t + 1) * BLOCK_J && dcol0 + BLOCK_I > (long long)t * BLOCK_J;
        const float ryj = ry_n;
        ry_n = (t + 1 < p.n_jt && jg + BLOCK_J < p.n_cols) ? p.rinv_y[jg + BLOCK_J] : 0.f;
        const float cj = ryj * k2;          // S_ij log2(e) = acc * rinv_x[i] * cj
        ptx::mbar_wait(bar(B_SFULL + b), (t >> 1) & 1);
        ptx::tc_fence_after();
        uint32_t r[32];
        ptx::tmem_ld_32x32b_x32(t_lane + S_COL0 + b * BLOCK_I + ibase, r);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();   // S buffer drained by this warp -> let the MMA warp overwrite it
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(bar(B_SEMPTY + b));
        if (jvalid) {
          float cs[4] = {0.f, 0.f, 0.f, 0.f};   // four partial column sums: no 32-long dependent FADD chain
          if (i_valid == BLOCK_I) {
#pragma unroll
            for (int x4 = 0; x4 < 8; ++x4) {
              const float4 rx4 = *reinterpret_cast<const float4*>(rx_s + ibase + x4 * 4);
              const float rxv[4] = {rx4.x, rx4.y, rx4.z, rx4.w};
#pragma unroll
              for (int xx = 0; xx < 4; ++xx) {
                const int x = x4 * 4 + xx;
                const float xv = fmaf(__uint_as_float(r[x]) * rxv[xx], cj, -k2);
                const float ev = (xx == 0) ? ex2(xv) : ex2_poly(xv);     // 1 in 4 on the MUFU
                racc[x] += ev;
                cs[xx] += ev;
              }
            }
          } else {
#pragma unroll
            for (int x = 0; x < 32; ++x) {
              const float ev = (ibase + x < i_valid) ? ex2(fmaf(__uint_as_float(r[x]) * rx_s[ibase + x], cj, -k2)) : 0.f;
              racc[x] += ev;
              cs[x & 3] += ev;
            }
          }
          if (diag_tile) {
            const long long id = jg - dcol0 - ibase;   // TMEM column (within this load) holding S_{i,i+off}
#pragma unroll
            for (int x = 0; x < 32; ++x)
              if (id == x && ibase + x < i_valid)
                p.diag[i0 + ibase + x] = __uint_as_float(r[x]) * rx_s[ibase + x] * ryj * sc;
          }
          p.col_part[(long long)(blockIdx.x * (BLOCK_I / 32) + cg) * p.col_ld + jg] = (cs[0] + cs[1]) + (cs[2] + cs[3]);
        }
      }
      // row sums: reduce the per-lane partials over the 128 lanes (4 warps) that share column group cg
      warp_transpose_reduce<32>(racc, lane);
      red[e * 32 + lane] = racc[0];
      epi_bar_sync<NUM_EPI_WARPS * 32>();
      if (te < BLOCK_I) {
        const int cgi = te >> 5, ii = te & 31;
        const float tot = (red[(cgi * 4 + 0) * 32 + ii] + red[(cgi * 4 + 1) * 32 + ii]) +
                          (red[(cgi * 4 + 2) * 32 + ii] + red[(cgi * 4 + 3) * 32 + ii]);
        if (te < i_valid) {
          p.row_m[i0 + te] = sc;
          p.row_l[i0 + te] = tot;
        }
      }
    } else {
      // This thread owns column j of the logits tile and HALF consecutive rows i (TMEM columns), handled in
      // groups of 16.  The element loops are straight-line code (the rare diagonal / ragged tiles take a
      // separate masked loop): independent chains the scheduler interleaves, one ex2 per logit.
      constexpr int NG = HALF / 16;
      float ds = 0.f;
      const int jj = j_local & 63;
      uint32_t row_off[8];   // byte offset of (row i, column jj) inside an 8-row swizzle group, i & 7 = k
#pragma unroll
      for (int k = 0; k < 8; ++k) row_off[k] = k * 128 + (((jj >> 3) ^ k) << 4) + (jj & 7) * 2;
      uint8_t* const g_gen = smem + (g_smem - base) + (j_local >> 6) * (G_BYTES / 2) + (h * HALF / 8) * 1024;
      const float* const rx_h = rx_s + h * HALF;
      const float* const u_h = u_s + h * HALF;
      // per-column scalars are fetched one tile ahead so their L2 latency never sits on the S -> G critical path
      auto load_col = [&](int t, float& cw, float& cm, float& ry) {
        const long long jn = (long long)t * BLOCK_J + j_local;
        const bool ok = t < p.n_jt && jn < p.n_cols;
        cw = (ok && p.col_w != nullptr) ? p.col_w[jn] : 0.f;
        cm = (ok && p.col_w != nullptr) ? p.col_m_in[jn] : sc;
        ry = ok ? p.rinv_y[jn] : 0.f;
      };
      float cw_n, cm_n, ry_n;
      load_col(0, cw_n, cm_n, ry_n);
      for (int t = 0; t < p.n_jt; ++t) {
        const int sb = t % NSBUF, gb = t & 1;
        const long long jg = (long long)t * BLOCK_J + j_local;
        const bool jvalid = jg < p.n_cols;
        const float vj = cw_n * ex2((sc - cm_n) * LOG2E);
        const float ryj = ry_n;
        const float cj = ryj * k2;
        load_col(t + 1, cw_n, cm_n, ry_n);
        const bool diag_tile = dcol0 < (long long)(t + 1) * BLOCK_J && dcol0 + BLOCK_I > (long long)t * BLOCK_J;
        const bool plain = (i_valid == BLOCK_I) && !diag_tile && (long long)(t + 1) * BLOCK_J <= p.n_cols;  // warp-uniform

        ptx::mbar_wait(bar(B_SFULL + sb), (t / NSBUF) & 1);
        ptx::tc_fence_after();
        uint32_t r[NG][16];
#pragma unroll
        for (int gq = 0; gq < NG; ++gq) ptx::tmem_ld_32x32b_x16(t_lane + S_COL0 + sb * BLOCK_I + h * HALF + gq * 16, r[gq]);
        ptx::tmem_ld_wait();
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(bar(B_SEMPTY + sb));   // S buffer is in registers: the next logits tile may land

        uint32_t gpk[NG][8];   // bf16 pairs are NOT adjacent in memory (K-major [i][j]); pack only to save registers
#pragma unroll
        for (int gq = 0; gq < NG; ++gq) {
          float g[16];
          if (plain) {
#pragma unroll
            for (int x4 = 0; x4 < 4; ++x4) {
              const float4 rx4 = *reinterpret_cast<const float4*>(rx_h + gq * 16 + x4 * 4);
              const float4 u4 = *reinterpret_cast<const float4*>(u_h + gq * 16 + x4 * 4);
              const float rxv[4] = {rx4.x, rx4.y, rx4.z, rx4.w};
              const float uv[4] = {u4.x, u4.y, u4.z, u4.w};
#pragma unroll
              for (int xx = 0; xx < 4; ++xx) {
                const int x = x4 * 4 + xx;
                const float y = __uint_as_float(r[gq][x]) * rxv[xx] * cj;      // S_ij * log2(e)
                const float ev = (xx == 0) ? ex2(y - k2) : ex2_poly(y - k2);   // 1 in 4 on the MUFU
                g[x] = ev * (uv[xx] + vj);
                ds = fmaf(g[x], y, ds);
              }
            }
          } else {
            const long long id = jg - dcol0 - h * HALF - gq * 16;
#pragma unroll
            for (int x = 0; x < 16; ++x) {
              const float y = __uint_as_float(r[gq][x]) * rx_h[gq * 16 + x] * cj;
              float gv = ex2(y - k2) * (u_h[gq * 16 + x] + vj);
              if (id == x) gv -= p.diag_w;
              if (!(jvalid && h * HALF + gq * 16 + x < i_valid)) gv = 0.f;
              g[x] = gv;
              ds = fmaf(gv, y, ds);
            }
          }
#pragma unroll
          for (int x = 0; x < 8; ++x) {   // contracted against the RAW y_j -> fold rinv_y[j] into G
            const __nv_bfloat162 pr = __floats2bfloat162_rn(g[2 * x] * ryj, g[2 * x + 1] * ryj);
            gpk[gq][x] = *reinterpret_cast<const uint32_t*>(&pr);
          }
        }
        ptx::mbar_wait(bar(B_GEMPTY + gb), ((t >> 1) & 1) ^ 1u);   // gradient MMA of tile t-2 has read this buffer
        uint8_t* const gb_base = g_gen + gb * G_BYTES;
#pragma unroll
        for (int gq = 0; gq < NG; ++gq)
#pragma unroll
          for (int x = 0; x < 16; ++x) {
            const int il = gq * 16 + x;   // row within this warp's half
            const uint16_t v = static_cast<uint16_t>((x & 1) ? (gpk[gq][x >> 1] >> 16) : (gpk[gq][x >> 1] & 0xFFFFu));
            *reinterpret_cast<uint16_t*>(gb_base + (il >> 3) * 1024 + row_off[il & 7]) = v;
          }
        ptx::fence_proxy_async_smem();   // generic-proxy stores -> visible to the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(bar(B_GFULL + gb));
      }
      // accumulators complete: dXhat^T[d = qc*128 + lane_global, i]  ->  dx[i][d]
      ptx::mbar_wait(bar(B_ACCFULL), 0);
      ptx::tc_fence_after();
      for (int qc = 0; qc < p.nq; ++qc) {
        const int dd = qc * 128 + j_local;
#pragma unroll
        for (int gq = 0; gq < NG; ++gq) {
          uint32_t r[16];
          ptx::tmem_ld_32x32b_x16(t_lane + qc * BLOCK_I + h * HALF + gq * 16, r);
          ptx::tmem_ld_wait();
          if (dd < p.d) {
#pragma unroll
            for (int x = 0; x < 16; ++x) {
              const int i = h * HALF + gq * 16 + x;
              if (i < i_valid) p.dx[(long long)(i0 + i) * p.d + dd] = __uint_as_float(r[x]) * out_scale;
            }
          }
        }
      }
      if (p.ds_part != nullptr) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ds += __shfl_xor_sync(0xffffffffu, ds, o);
        if (lane == 0) red[e] = ds;
        epi_bar_sync<NUM_EPI_WARPS * 32>();
        if (te == 0) {
          float tot = 0.f;
#pragma unroll
          for (int w = 0; w < NUM_EPI_WARPS; ++w) tot += red[w];
          p.ds_part[blockIdx.x] = tot * LN2;
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, TMEM_COLS);
}

}  // namespace tc
