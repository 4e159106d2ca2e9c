// Two-sided backward: ONE sweep over the logits tiles emits both dA_hat and dB_hat (8 N^2 d executed per step instead of
// the 10 N^2 d of two pair::bwd_kernel launches) -- loss.backward() of current/rna_clip_codes.ipynb:2074,
// run1/full.py:134, old/clip_opt.py:167.
//
// Why it is not "one CTA pair keeps two accumulators".  A pair's TMEM holds 128 K floats.  With d = 512 the stationary
// gradient of 128 resident rows already takes half of it and two logits buffers the other half; a second, per-column-block
// accumulator [256 x 512] does not fit, and flushing one per step would cost 1/(1.5 R) B per FLOP of fp32 reduction
// traffic (R = 128 rows: ~7 TB/s).  So the second gradient is formed by OTHER SMs, and what travels between them is the
// bf16 gradient tile the producer has in shared memory anyway:
//
//   producer pairs (P of the 74)   exactly pair::bwd_kernel's sweep -- 128 resident rows of X, S = X Y^T per 256-column
//                                  step, G'' = (exp(S - s)(u_i + v_j) - diag) / (|x_i| |y_j|), dX += G'' Y stationary in
//                                  TMEM -- plus a TMA store of every G'' tile [128 x 256] bf16 into a ring in global
//                                  memory (L2-resident)
//   consumer pairs (Q = 74 - P)    dY[J_t, d half] += sum over the round's producers G''_p^T X_p : a plain GEMM,
//                                  M = 256 columns j, N = 256 (d half), K = the rows of the round (<= P x 128), both
//                                  operands MN-major straight from TMA boxes; flushed once per task
//
// ONE tile serves both sides because it carries BOTH 1/norm factors: dXhat_i = (s |x_i|) sum_j G''_ij y_j and
// dYhat_j = (s |y_j|) sum_i G''_ij x_i contract it against the RAW rows; the per-row factor is applied when an accumulator
// is drained.  The logits come from the raw rows scaled in fp32, exactly as in the forward.
//
// Work items.  A producer's unit of work is (row block, column segment): the column sweep is cut into n_seg segments of
// seg_steps steps, items are numbered segment-major and dealt out in rounds of P (item r P + p goes to producer p in
// round r), so P need not divide the number of row blocks and the rounds stay full; an item's gradient goes to slab `seg`
// of dX (summed by aux::finish_rows).  All producers of a round advance in lock step, so the tiles in flight belong to a
// window of ~Q/2 + 2 steps: the ring holds `depth` steps x P tiles x 64 KiB.  A round may straddle segment boundaries:
// its producers then split into runs of equal segment ("subs"), and every (sub, step, d half) is one consumer task.
// Consumer tasks are assigned by (column step, d half) only, so every contribution to one block of dY is accumulated by
// the same threads in program order: no atomics, bit-reproducible.
//
// Row-sharded global batch (SURVEY.md section 8e): X = the rank's A rows, Y = all ranks' B rows, segment s = the columns
// owned by rank s.  The LAST contribution to a block of segment s is not written locally but stored straight into rank
// s's slot for this rank in NVLink peer memory: the kernel is the contraction AND the reduce-scatter of the partial dB
// (what the reference's all_gather formulation leaves to autograd + DDP, old/clip_opt.py:102-112); the owner sums the
// world slots in fixed order (aux::finish_rows).
//
// Flags (global memory, zeroed per launch): ready[g] counts the CTAs whose four G boxes of global step
// g = round * seg_steps + tau have landed (2 per producer pair), done[g] the consumer tasks that finished reading them.  A
// producer stores step g only after done[g - depth] is complete.  TMA stores are published by
// cp.async.bulk.wait_group -> fence.proxy.async -> red.release.gpu; consumers ld.acquire.gpu -> fence.proxy.async -> TMA
// loads.  Liveness: the smallest incomplete step's consumers never wait on anything but producers, and producers only
// wait on steps `depth` behind them.  All pairs must be co-resident (persistent grid, checked by the host).
#pragma once
#include "kernels_pair.cuh"

namespace pair2 {

using pair::LOG2E;
using pair::STAGE_BYTES;
using pair::STEP_J;
using pair::TMEM_COLS;

constexpr int THREADS = 416;                 // 4 service warps + 8 epilogue warps + the ring-store warp
constexpr int STORE_WARP = 12;
constexpr int EPI_WARPS = 8;
constexpr int ROWS = 64;                     // resident rows per producer CTA (128 per pair)
constexpr int X_CHUNK = ROWS * 128;          // [64 rows][64 k] bf16
constexpr int G_BYTES = 4 * 8192;            // [64 i][256 j] bf16 = four K-major boxes
constexpr int SMALL = 10240;                 // barriers (1000) | tmem ptr at +1016 | column vectors 2 x 4 x 256 f32 at +1024
constexpr int C_STAGE = 32768;               // consumer stage: A = 2 boxes G^T [64 i][64 j], B = 2 boxes X [64 i][64 d]
constexpr int MAXS = 6;
constexpr int RING_DEPTH = 16;               // steps of G tiles the ring holds
constexpr int MAX_WORLD = 16;

constexpr int B_FULL_A = 0, B_EMPTY_A = MAXS, B_FULL_B = 2 * MAXS, B_EMPTY_B = 3 * MAXS, B_XFULL = 4 * MAXS,
              B_XEMPTY = B_XFULL + 1, B_SFULL = B_XEMPTY + 1, B_SEMPTY = B_SFULL + 2, B_GFULL = B_SEMPTY + 2,
              B_GEMPTY = B_GFULL + 4, B_ACCFULL = B_GEMPTY + 4, B_ACCEMPTY = B_ACCFULL + 2, B_GSFULL = B_ACCEMPTY + 2,
              B_GSTORED = B_GSFULL + 4, B_COUNT = B_GSTORED + 4;      // G barriers: one per box
static_assert(B_COUNT * 8 <= 1000, "barrier block");

struct Params {
  int n_rows, n_cols, d;      // n_rows % 128 == 0, n_cols % (256 n_seg) == 0, d % 128 == 0, d <= 768
  int nsbuf;                  // producer logits buffers: 2 (d <= 512), 1 beyond (384 accumulator columns + 128)
  int nkc, nq2, n_half;
  int n_rb, n_seg, seg_steps, n_items, n_rounds;
  int P, Q, depth;
  int stages_a, stages_b, stages_c;
  long long diag_offset;      // column of row i's positive = i + diag_offset
  float scale, diag_w;
  const float* scale_dev;
  const float* rinv_x;
  const float* rinv_y;
  const float* row_m;
  const float* row_w;
  const float* col_m;
  const float* col_w;
  float* dx;                  // [n_seg][n_rows, d] f32: per-segment partials of s sum_j G_ij yhat_j
  float* dy;                  // [n_cols, d] f32: s sum_i G_ij xhat_i over the LOCAL rows (partial / result)
  // row-sharded step: the last contribution to segment s is stored at dy_peer[s] (this rank's slot in rank s's peer
  // memory, [seg_steps * 256, d] f32) instead of dy; world == 0: everything stays in dy
  float* dy_peer[MAX_WORLD];
  int world;
  uint32_t* ready;            // [n_rounds * seg_steps]
  uint32_t* done;             // [n_rounds * seg_steps]
};

__host__ __device__ constexpr int producer_smem(int nkc, int stages) {
  return nkc * X_CHUNK + G_BYTES + stages * STAGE_BYTES + SMALL;
}
constexpr int FLUSH_BYTES = EPI_WARPS * 4096;   // consumer epilogue: one [32 rows][32 f32] transposing scratch per warp
__host__ __device__ constexpr int consumer_smem(int stages) { return stages * C_STAGE + FLUSH_BYTES + SMALL; }
__device__ __forceinline__ float4 ld_shared_v4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

__device__ __forceinline__ void publish(uint32_t* flag) {   // TMA stores of this thread (already waited for) -> visible, then count
  ptx::fence_proxy_async_all();
  ptx::red_release_gpu_add(flag, 1u);
}

// The runs of equal segment ("subs") among the items of round r.
struct Sub {
  int seg, p_lo, p_hi, rb_lo;   // producers [p_lo, p_hi) of the round work on segment seg, row blocks rb_lo + (p - p_lo)
  bool first, last;             // the run holds the segment's first / last row block
};
__device__ __forceinline__ int round_items(const Params& p, int r) { return min(p.P, p.n_items - r * p.P); }
__device__ __forceinline__ int round_subs(const Params& p, int r) {
  const int lo = r * p.P, hi = lo + round_items(p, r);
  return (hi - 1) / p.n_rb - lo / p.n_rb + 1;
}
__device__ __forceinline__ Sub round_sub(const Params& p, int r, int k) {
  const int lo = r * p.P, hi = lo + round_items(p, r);
  Sub s;
  s.seg = lo / p.n_rb + k;
  const int a = max(lo, s.seg * p.n_rb), b = min(hi, (s.seg + 1) * p.n_rb);
  s.p_lo = a - lo;
  s.p_hi = b - lo;
  s.rb_lo = a - s.seg * p.n_rb;
  s.first = a == s.seg * p.n_rb;
  s.last = b == (s.seg + 1) * p.n_rb;
  return s;
}

// TWO_EXP: the producers form G from the (shift, sum) pairs as they are -- exp(S - m_i) w_i + exp(S - m_j) w_j, two ex2 per
// logit, every exponent <= 0 -- instead of the fixed shift's single exp(S - s) (u_i + v_j): kernel family 2, logit scales up
// to the reference's clamp(max=100) (old/clip_opt.py:100, run1/full.py:76), as in pair::bwd_kernel<true>.
template <bool TWO_EXP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
bwd2_kernel(const __grid_constant__ CUtensorMap tmap_x,    // X  box {64, 64 rows}     resident rows (K-major) / dY operand (MN-major)
            const __grid_constant__ CUtensorMap tmap_y,    // Y  box {64 k, 128 rows}  logits B operand, K-major
            const __grid_constant__ CUtensorMap tmap_yg,   // Y  box {64 d, 64 rows}   dX gradient B operand, MN-major
            const __grid_constant__ CUtensorMap tmap_g,    // G ring [depth * P * 128, 256] bf16, box {64 j, 64 i}
            const Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const uint32_t base = ptx::smem_u32(smem);
  if ((base & 1023u) != 0) __trap();
  const uint32_t rank = ptx::cluster_ctarank();
  const bool leader = rank == 0;
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int pair_id = blockIdx.x >> 1;
  const bool is_producer = pair_id < p.P;

  // the small block sits at the same offset for both roles: behind the larger of the two layouts
  const int body = max(producer_smem(p.nkc, p.stages_a + p.stages_b), consumer_smem(p.stages_c)) - SMALL;
  const uint32_t bars = base + body;
  auto bar = [&](int i) -> uint32_t { return bars + 8u * i; };
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem + body + 1016);
  float* const colv = reinterpret_cast<float*>(smem + body + 1024);   // [2][4][256]

  const float sc = p.scale_dev != nullptr ? __ldg(p.scale_dev) : p.scale;
  const float k2 = sc * LOG2E;

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmap_x);
    ptx::prefetch_tmap(&tmap_y);
    ptx::prefetch_tmap(&tmap_yg);
    ptx::prefetch_tmap(&tmap_g);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < MAXS; ++s) {
      ptx::mbar_init(bar(B_FULL_A + s), 1);
      ptx::mbar_init(bar(B_EMPTY_A + s), 1);
      ptx::mbar_init(bar(B_FULL_B + s), 1);
      ptx::mbar_init(bar(B_EMPTY_B + s), 1);
    }
    ptx::mbar_init(bar(B_XFULL), 1);
    ptx::mbar_init(bar(B_XEMPTY), 1);
    for (int b = 0; b < 2; ++b) {
      ptx::mbar_init(bar(B_SFULL + b), 1);
      ptx::mbar_init(bar(B_SEMPTY + b), 2 * EPI_WARPS);
      ptx::mbar_init(bar(B_ACCFULL + b), 1);
      ptx::mbar_init(bar(B_ACCEMPTY + b), 2 * EPI_WARPS);
    }
    for (int k = 0; k < 4; ++k) {
      ptx::mbar_init(bar(B_GFULL + k), 4);
      ptx::mbar_init(bar(B_GEMPTY + k), 1);
      ptx::mbar_init(bar(B_GSFULL + k), 2);     // the two epilogue warps of THIS CTA that wrote box k
      ptx::mbar_init(bar(B_GSTORED + k), 1);    // the ring store has read box k out of shared memory
    }
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

  if (is_producer) {
    // =========================================================================================== PRODUCER PAIR
    // item of round r: i = r P + pair_id  ->  segment i / n_rb, row block i % n_rb, column steps seg * seg_steps + tau
    const uint32_t x_smem = base;
    const uint32_t g_smem = x_smem + p.nkc * X_CHUNK;
    const uint32_t ring_a = g_smem + G_BYTES;
    const uint32_t ring_b = ring_a + p.stages_a * STAGE_BYTES;
    const int S_COL0 = TMEM_COLS - 128 * p.nsbuf;   // logits buffers of 128 columns behind the accumulators
    auto s_buf = [&](uint32_t gs) -> int { return p.nsbuf == 2 ? (int)(gs & 1u) : 0; };
    auto s_par = [&](uint32_t gs) -> uint32_t { return p.nsbuf == 2 ? ((gs >> 1) & 1u) : (gs & 1u); };

    if (warp == 0) {
      // ------------------------------------------------------------- TMA: resident X per item, then Y rows (K-major)
      if (ptx::elect_one()) {
        int stage = 0;
        uint32_t phase = 0;
        for (int r = 0; r < p.n_rounds; ++r) {
          const int item = r * p.P + pair_id;
          if (item >= p.n_items) break;
          const int i0 = (item % p.n_rb) * (2 * ROWS) + (int)rank * ROWS;
          const int t0 = (item / p.n_rb) * p.seg_steps;
          ptx::mbar_wait(bar(B_XEMPTY), (r & 1) ^ 1u);   // the previous item's logits MMAs have read X
          if (leader) ptx::mbar_arrive_expect_tx(bar(B_XFULL), 2 * p.nkc * X_CHUNK);
          for (int kc = 0; kc < p.nkc; ++kc)
            ptx::tma_load_2d_pair(x_smem + kc * X_CHUNK, &tmap_x, bar(B_XFULL), kc * 64, i0);
          for (int t = t0; t < t0 + p.seg_steps; ++t) {
            for (int g = 0; g < p.nkc; ++g) {
              ptx::mbar_wait(bar(B_EMPTY_A + stage), phase ^ 1u);
              if (leader) ptx::mbar_arrive_expect_tx(bar(B_FULL_A + stage), 2 * STAGE_BYTES);
              ptx::tma_load_2d_pair(ring_a + stage * STAGE_BYTES, &tmap_y, bar(B_FULL_A + stage), g * 64,
                                    t * STEP_J + (int)rank * 128);
              if (++stage == p.stages_a) { stage = 0; phase ^= 1u; }
            }
          }
        }
      }
      __syncwarp();
    } else if (warp == 2) {
      // ------------------------------------------------------------- TMA: Y[j, d slice] boxes (MN-major)
      if (ptx::elect_one()) {
        int stage = 0;
        uint32_t phase = 0;
        for (int r = 0; r < p.n_rounds; ++r) {
          const int item = r * p.P + pair_id;
          if (item >= p.n_items) break;
          const int t0 = (item / p.n_rb) * p.seg_steps;
          for (int t = t0; t < t0 + p.seg_steps; ++t) {
            for (int kc = 0; kc < 4; ++kc) {
              for (int q = 0; q < p.nq2; ++q) {
                const int wq = min(256, p.d - 256 * q);
                const int half = wq >> 1;
                const int ngr = half >> 6;
                ptx::mbar_wait(bar(B_EMPTY_B + stage), phase ^ 1u);
                if (leader) ptx::mbar_arrive_expect_tx(bar(B_FULL_B + stage), 2 * ngr * 8192);
                for (int gi = 0; gi < ngr; ++gi)
                  ptx::tma_load_2d_pair(ring_b + stage * STAGE_BYTES + gi * 8192, &tmap_yg, bar(B_FULL_B + stage),
                                        256 * q + half * (int)rank + 64 * gi, t * STEP_J + 64 * kc);
                if (++stage == p.stages_b) { stage = 0; phase ^= 1u; }
              }
            }
          }
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      // ------------------------------------------------------------- logits MMA issuer (leader)
      if (leader && ptx::elect_one()) {
        constexpr uint32_t idesc_s = ptx::idesc_bf16_f32_major(2 * ROWS, STEP_J, 0, 0);
        const uint32_t x_lo0 = desc_lo(x_smem, 1), a_lo0 = desc_lo(ring_a, 1);
        int stage = 0;
        uint32_t phase = 0, ready = 0, gs = 0;
        for (int r = 0; r < p.n_rounds; ++r) {
          if (r * p.P + pair_id >= p.n_items) break;
          ptx::mbar_wait(bar(B_XFULL), r & 1);
          for (int t = 0; t < p.seg_steps; ++t, ++gs) {
            const int sb = s_buf(gs);
            ptx::mbar_wait(bar(B_SEMPTY + sb), s_par(gs) ^ 1u);
            const uint32_t d_tmem = tmem_base + S_COL0 + sb * 128;
            for (int g = 0; g < p.nkc; ++g) {
              if (!ready) ptx::mbar_wait(bar(B_FULL_A + stage), phase);
              ptx::tc_fence_after();
              int ns = stage + 1;
              uint32_t np = phase;
              if (ns == p.stages_a) { ns = 0; np ^= 1u; }
              ready = ptx::mma_box_pair(d_tmem, mk(desc_hi_k, x_lo0 + g * (X_CHUNK >> 4)),
                                        mk(desc_hi_k, a_lo0 + stage * (STAGE_BYTES >> 4)), 2, 2, idesc_s, g != 0,
                                        bar(B_FULL_A + ns), np);
              ptx::mma_commit_pair(bar(B_EMPTY_A + stage));
              if (g == p.nkc - 1) ptx::mma_commit_pair(bar(B_SFULL + sb));
              stage = ns;
              phase = np;
            }
          }
          ptx::mma_commit_pair(bar(B_XEMPTY));   // every logits MMA of this item has read X
        }
      }
      __syncwarp();
    } else if (warp == 3) {
      // ------------------------------------------------------------- dX gradient MMA issuer (leader)
      if (leader && ptx::elect_one()) {
        const uint32_t g_lo0 = desc_lo(g_smem, 1), b_lo0 = desc_lo(ring_b, 8192 >> 4);
        int stage = 0;
        uint32_t phase = 0, ready = 0, gs = 0;
        for (int r = 0; r < p.n_rounds; ++r) {
          if (r * p.P + pair_id >= p.n_items) break;
          ptx::mbar_wait(bar(B_ACCEMPTY), (r & 1) ^ 1u);   // the previous item's accumulators have been drained
          ptx::tc_fence_after();
          for (int t = 0; t < p.seg_steps; ++t, ++gs) {
            for (int kc = 0; kc < 4; ++kc) {
              ptx::mbar_wait(bar(B_GFULL + kc), gs & 1u);
              for (int q = 0; q < p.nq2; ++q) {
                const int wq = min(256, p.d - 256 * q);
                const uint32_t idesc_g = ptx::idesc_bf16_f32_major(2 * ROWS, wq, 0, 1);
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
      }
      __syncwarp();
    } else if (warp == STORE_WARP) {
      // ------------------------------------------------------------- ring store: G boxes of this CTA -> global ring
      // A thread of its own, so that nothing on the epilogue's critical path touches global memory: the back-pressure
      // spin (done[g - depth]), the bulk-group waits and the release that publishes a step all live here.
      if (ptx::elect_one()) {
        uint32_t gs = 0;
        bool pending = false;
        uint32_t g_prev = 0;
        const uint64_t keep = ptx::l2_policy_evict_last();   // ring lines stay in L2 until their slot is overwritten
        for (int r = 0; r < p.n_rounds; ++r) {
          if (r * p.P + pair_id >= p.n_items) break;
          const bool more_rounds = (r + 1) * p.P + pair_id < p.n_items;
          for (int t = 0; t < p.seg_steps; ++t, ++gs) {
            const uint32_t g = (uint32_t)r * (uint32_t)p.seg_steps + (uint32_t)t;
            const int row0 = ((int)(g % (uint32_t)p.depth) * p.P + pair_id) * 128 + (int)rank * ROWS;
            // latency-critical part: the epilogue of the NEXT step waits for these boxes to be released
            for (int kc = 0; kc < 4; ++kc) {
              ptx::mbar_wait(bar(B_GSFULL + kc), gs & 1u);
              ptx::tma_store_2d_hint(&tmap_g, g_smem + kc * 8192, 64 * kc, row0, keep);
              ptx::bulk_commit_group();
            }
            ptx::bulk_wait_group_read0();               // shared memory of the four boxes has been read
            for (int kc = 0; kc < 4; ++kc) ptx::mbar_arrive(bar(B_GSTORED + kc));
            // off the critical path: publish the PREVIOUS step (its four groups are older than the four just committed,
            // so this does not wait for an L2 round trip), then the back-pressure check for the next step
            if (pending) {
              ptx::bulk_wait_group_le<4>();
              publish(p.ready + g_prev);
            }
            pending = true;
            g_prev = g;
            if (g + 1 >= (uint32_t)p.depth && (t + 1 < p.seg_steps || more_rounds)) {
              const uint32_t go = g + 1 - (uint32_t)p.depth;
              ptx::spin_until_ge(p.done + go, (uint32_t)(round_subs(p, (int)(go / (uint32_t)p.seg_steps)) * p.n_half));
            }
          }
        }
        if (pending) {
          ptx::bulk_wait_group0();
          publish(p.ready + g_prev);
        }
      }
      __syncwarp();
    } else {
      // ------------------------------------------------------------- epilogue: S tile -> bf16 G'' tile (MMA operand + ring)
      const int e = warp - 4;
      const int q = warp & 3;
      const int h = e >> 2;
      const int jh = q >> 1;
      const int i_local = 32 * (q & 1) + lane;
      const int te = threadIdx.x - 128;
      const int jl0 = 128 * jh + 64 * h;
      const int kc = 2 * jh + h;
      const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
      const uint32_t g_row = g_smem + kc * 8192 + (i_local >> 3) * 1024 + (i_local & 7) * 128;
      const uint32_t sw = i_local & 7;
      const uint32_t sempty_leader = ptx::mapa(bar(B_SEMPTY), 0);
      const uint32_t gfull_leader = ptx::mapa(bar(B_GFULL + kc), 0);
      const uint32_t accempty_leader = ptx::mapa(bar(B_ACCEMPTY), 0);
      uint32_t gs = 0;

      for (int r = 0; r < p.n_rounds; ++r) {
        const int item = r * p.P + pair_id;
        if (item >= p.n_items) break;
        const int seg = item / p.n_rb;
        const int t0 = seg * p.seg_steps;
        const int i_glob = (item % p.n_rb) * (2 * ROWS) + (int)rank * ROWS + i_local;
        const float rx = p.rinv_x[i_glob];
        const float u = TWO_EXP ? 0.f : p.row_w[i_glob] * pair::ex2((sc - p.row_m[i_glob]) * LOG2E);
        const float rm2 = TWO_EXP ? p.row_m[i_glob] * LOG2E : 0.f;
        const float rw = TWO_EXP ? p.row_w[i_glob] : 0.f;
        const long long dcol = (long long)i_glob + p.diag_offset;   // column of this row's positive
        float cw_n, cm_n, ry_n;
        {
          const long long jn = (long long)t0 * STEP_J + te;
          cw_n = p.col_w[jn]; cm_n = p.col_m[jn]; ry_n = p.rinv_y[jn];
        }

        for (int t = t0; t < t0 + p.seg_steps; ++t, ++gs) {
          const int sb = s_buf(gs);
          float* const cv = colv + (gs & 1) * 1024;
          cv[te] = ry_n * k2;                                                   // S_ij log2(e) = acc * rinv_x[i] * cj
          cv[256 + te] = (TWO_EXP ? cw_n : cw_n * pair::ex2((sc - cm_n) * LOG2E)) * ry_n;   // v_j / |y_j|  (TWO_EXP: w_j / |y_j|)
          cv[512 + te] = ry_n;
          if (TWO_EXP) cv[768 + te] = cw_n > 0.f ? cm_n * LOG2E : 0.f;          // weight 0: keep the exponent finite
          if (t + 1 < t0 + p.seg_steps) {
            const long long jn = (long long)(t + 1) * STEP_J + te;
            cw_n = p.col_w[jn]; cm_n = p.col_m[jn]; ry_n = p.rinv_y[jn];
          }
          pair::named_bar_sync(1, EPI_WARPS * 32);
          const long long dl = dcol - ((long long)t * STEP_J + jl0);   // step-local index of the positive, if in [0, 64)
          const bool has_diag = dl >= 0 && dl < 64;

          ptx::mbar_wait(bar(B_SFULL + sb), s_par(gs));
          ptx::tc_fence_after();
          uint32_t pk[32];
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            uint32_t rr[32];
            ptx::tmem_ld_32x32b_x32(t_lane + S_COL0 + sb * 128 + 64 * h + 32 * c, rr);
            ptx::tmem_ld_wait();
            if (c == 1) {
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
                  const float y = __uint_as_float(rr[4 * x4 + xx]) * rx;
                  const float er = pair::ex2(fmaf(y, cjv[xx], -rm2)) * rw;    // exp(S_ij - m_i) w_i
                  const float ec = pair::ex2(fmaf(y, cjv[xx], -cmv[xx]));     // exp(S_ij - m_j)
                  g[xx] = rx * fmaf(er, ryv[xx], ec * vrv[xx]);                 // (...) / (|x_i| |y_j|)
                }
              } else {
#pragma unroll
                for (int xx = 0; xx < 4; ++xx) {
                  const float y = __uint_as_float(rr[4 * x4 + xx]) * rx;
                  const float ev = pair::ex2(fmaf(y, cjv[xx], -k2)) * rx;     // exp(S_ij - s) / |x_i|
                  g[xx] = ev * fmaf(u, ryv[xx], vrv[xx]);                       // (u_i + v_j) / |y_j|
                }
              }
              if (has_diag) {
#pragma unroll
                for (int xx = 0; xx < 4; ++xx)
                  if (dl == 32 * c + 4 * x4 + xx) g[xx] -= p.diag_w * rx * ryv[xx];
              }
              const __nv_bfloat162 p0 = __floats2bfloat162_rn(g[0], g[1]);
              const __nv_bfloat162 p1 = __floats2bfloat162_rn(g[2], g[3]);
              pk[16 * c + 2 * x4] = *reinterpret_cast<const uint32_t*>(&p0);
              pk[16 * c + 2 * x4 + 1] = *reinterpret_cast<const uint32_t*>(&p1);
            }
          }
          ptx::mbar_wait(bar(B_GEMPTY + kc), (gs & 1u) ^ 1u);    // the gradient MMAs that last read this box are done
          ptx::mbar_wait(bar(B_GSTORED + kc), (gs & 1u) ^ 1u);   // ... and so is its ring store
#pragma unroll
          for (int ch = 0; ch < 8; ++ch)
            pair::st_shared_v4(g_row + ((static_cast<uint32_t>(ch) ^ sw) << 4), pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2],
                               pk[4 * ch + 3]);
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            ptx::mbar_arrive_cluster(gfull_leader);
            ptx::mbar_arrive(bar(B_GSFULL + kc));
          }
        }

        // the item's accumulators: slot q2 holds sum_j G''_ij y_j [i, 256 q2 + ...] in the 2x2 layout; dXhat = s |x_i| (...)
        ptx::mbar_wait(bar(B_ACCFULL), r & 1);
        ptx::tc_fence_after();
        const float osc = sc / rx;
        float* const slab = p.dx + (long long)seg * p.n_rows * p.d;
        for (int q2 = 0; q2 < p.nq2; ++q2) {
          const int halfw = min(256, p.d - 256 * q2) >> 1;
          if (64 * h < halfw) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
              uint32_t rr[32];
              ptx::tmem_ld_32x32b_x32(t_lane + 128 * q2 + 64 * h + 32 * c, rr);
              ptx::tmem_ld_wait();
              float* const dst = slab + (long long)i_glob * p.d + 256 * q2 + halfw * jh + 64 * h + 32 * c;
#pragma unroll
              for (int x4 = 0; x4 < 8; ++x4)
                *reinterpret_cast<float4*>(dst + 4 * x4) =
                    make_float4(__uint_as_float(rr[4 * x4]) * osc, __uint_as_float(rr[4 * x4 + 1]) * osc,
                                __uint_as_float(rr[4 * x4 + 2]) * osc, __uint_as_float(rr[4 * x4 + 3]) * osc);
            }
          }
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive_cluster(accempty_leader);
      }
    }
  } else {
    // =========================================================================================== CONSUMER PAIR
    // task = (round, sub, tau, d half); it belongs to the consumer with index (t n_half + hh) % Q, t = the column step
    const int cidx = pair_id - p.P;
    const uint32_t ring_c = base;

    if (warp == 0) {
      // ------------------------------------------------------------- TMA: G^T boxes from the ring + X boxes
      if (ptx::elect_one()) {
        int stage = 0;
        uint32_t phase = 0;
        const uint64_t keep = ptx::l2_policy_evict_last();
        for (int r = 0; r < p.n_rounds; ++r) {
          const int pw = round_items(p, r);
          const int nsub = round_subs(p, r);
          for (int tau = 0; tau < p.seg_steps; ++tau) {
            const uint32_t g = (uint32_t)r * (uint32_t)p.seg_steps + (uint32_t)tau;
            const int slot = (int)(g % (uint32_t)p.depth);
            bool step_ready = false;
            for (int k = 0; k < nsub; ++k) {
              const Sub sub = round_sub(p, r, k);
              const int t = sub.seg * p.seg_steps + tau;
              for (int hh = 0; hh < p.n_half; ++hh) {
                if ((t * p.n_half + hh) % p.Q != cidx) continue;
                if (!step_ready) {
                  ptx::spin_until_ge(p.ready + g, 2u * (uint32_t)pw);
                  ptx::fence_proxy_async_all();
                  step_ready = true;
                }
                const int wq = min(256, p.d - 256 * hh);
                const int ngr = wq >> 7;                   // 64-wide d groups this CTA supplies (N split over the pair)
                for (int pp = sub.p_lo; pp < sub.p_hi; ++pp) {
                  for (int kb = 0; kb < 2; ++kb) {
                    ptx::mbar_wait(bar(B_EMPTY_A + stage), phase ^ 1u);
                    if (leader) ptx::mbar_arrive_expect_tx(bar(B_FULL_A + stage), 2 * (2 + ngr) * 8192);
                    const uint32_t st = ring_c + stage * C_STAGE;
                    const int grow = (slot * p.P + pp) * 128 + 64 * kb;
                    const int xrow = (sub.rb_lo + pp - sub.p_lo) * 128 + 64 * kb;
                    for (int gi = 0; gi < 2; ++gi)
                      ptx::tma_load_2d_pair_hint(st + gi * 8192, &tmap_g, bar(B_FULL_A + stage), 128 * (int)rank + 64 * gi, grow, keep);
                    for (int gi = 0; gi < ngr; ++gi)
                      ptx::tma_load_2d_pair(st + 16384 + gi * 8192, &tmap_x, bar(B_FULL_A + stage),
                                            256 * hh + (wq >> 1) * (int)rank + 64 * gi, xrow);
                    if (++stage == p.stages_c) { stage = 0; phase ^= 1u; }
                  }
                }
              }
            }
          }
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      // ------------------------------------------------------------- dY gradient MMA issuer (leader)
      if (leader && ptx::elect_one()) {
        const uint32_t a_lo0 = desc_lo(ring_c, 8192 >> 4), b_lo0 = desc_lo(ring_c + 16384, 8192 >> 4);
        int stage = 0;
        uint32_t phase = 0, ready = 0, nt = 0;
        for (int r = 0; r < p.n_rounds; ++r) {
          const int nsub = round_subs(p, r);
          for (int tau = 0; tau < p.seg_steps; ++tau) {
            for (int k = 0; k < nsub; ++k) {
              const Sub sub = round_sub(p, r, k);
              const int t = sub.seg * p.seg_steps + tau;
              for (int hh = 0; hh < p.n_half; ++hh) {
                if ((t * p.n_half + hh) % p.Q != cidx) continue;
                const int buf = nt & 1;
                ptx::mbar_wait(bar(B_ACCEMPTY + buf), ((nt >> 1) & 1) ^ 1u);
                ptx::tc_fence_after();
                const int wq = min(256, p.d - 256 * hh);
                const uint32_t idesc = ptx::idesc_bf16_f32_major(256, wq, 1, 1);
                const uint32_t d_tmem = tmem_base + buf * 256;
                const int nk = 2 * (sub.p_hi - sub.p_lo);
                for (int kk = 0; kk < nk; ++kk) {
                  if (!ready) ptx::mbar_wait(bar(B_FULL_A + stage), phase);
                  ptx::tc_fence_after();
                  int ns = stage + 1;
                  uint32_t np = phase;
                  if (ns == p.stages_c) { ns = 0; np ^= 1u; }
                  ready = ptx::mma_box_pair(d_tmem, mk(desc_hi_mn, a_lo0 + stage * (C_STAGE >> 4)),
                                            mk(desc_hi_mn, b_lo0 + stage * (C_STAGE >> 4)), 2048 >> 4, 2048 >> 4, idesc,
                                            kk != 0, bar(B_FULL_A + ns), np);
                  ptx::mma_commit_pair(bar(B_EMPTY_A + stage));
                  stage = ns;
                  phase = np;
                }
                ptx::mma_commit_pair(bar(B_ACCFULL + buf));
                ++nt;
              }
            }
          }
        }
      }
      __syncwarp();
    } else if (warp >= 4 && warp < 4 + EPI_WARPS) {
      // ------------------------------------------------------------- epilogue: accumulator -> dY (store / read-modify-write / peer)
      const int q = warp & 3;
      const int hcol = (warp - 4) >> 2;
      const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
      const uint32_t accempty_leader = ptx::mapa(bar(B_ACCEMPTY), 0);
      const uint32_t scratch = ring_c + p.stages_c * C_STAGE + (warp - 4) * 4096;
      uint32_t nt = 0;
      for (int r = 0; r < p.n_rounds; ++r) {
        const int nsub = round_subs(p, r);
        for (int tau = 0; tau < p.seg_steps; ++tau) {
          for (int k = 0; k < nsub; ++k) {
            const Sub sub = round_sub(p, r, k);
            const int t = sub.seg * p.seg_steps + tau;
            for (int hh = 0; hh < p.n_half; ++hh) {
              if ((t * p.n_half + hh) % p.Q != cidx) continue;
              const int buf = nt & 1;
              const long long j = (long long)t * STEP_J + (int)rank * 128 + 32 * q + lane;
              const float osc = sc / p.rinv_y[j];              // dYhat_j = s |y_j| sum_i G''_ij x_i
              ptx::mbar_wait(bar(B_ACCFULL + buf), (nt >> 1) & 1);
              ptx::tc_fence_after();
              if (leader && warp == 4 && lane == 0)   // every MMA of the task is complete: its ring tiles have been read
                ptx::red_release_gpu_add(p.done + ((uint32_t)r * (uint32_t)p.seg_steps + (uint32_t)tau), 1u);
              const int wq = min(256, p.d - 256 * hh);
              const int wh = wq >> 1;                  // columns per epilogue-warp half
              const long long col0 = 256 * hh + hcol * wh;
              // Rows leave the warp as full 128-byte lines: the accumulator arrives with thread = row (32 consecutive
              // floats each), is staged through a swizzled [32][32] scratch and written with 8 lanes per row -- 16-byte
              // stores scattered over 32 rows reached 75 GB/s into NVLink peer memory, whole lines ride at link rate.
              // The segment's last contribution of a row-sharded step goes to the owner's slot in peer memory.
              const long long j0 = j - lane;           // first row of this warp
              const bool remote = sub.last && p.world > 0;
              float* const obase = remote ? p.dy_peer[sub.seg] + (j0 - (long long)sub.seg * p.seg_steps * STEP_J) * p.d + col0
                                          : p.dy + j0 * p.d + col0;
              const float* const lbase = p.dy + j0 * p.d + col0;
              const int rsub = lane >> 3, ch = lane & 7;
              for (int c = 0; c < (wh >> 5); ++c) {
                uint32_t rr[32];
                ptx::tmem_ld_32x32b_x32(t_lane + buf * 256 + hcol * wh + 32 * c, rr);
                ptx::tmem_ld_wait();
#pragma unroll
                for (int k4 = 0; k4 < 8; ++k4)
                  pair::st_shared_v4(scratch + lane * 128 + ((static_cast<uint32_t>(k4) ^ (lane & 7)) << 4),
                                     __float_as_uint(__uint_as_float(rr[4 * k4]) * osc), __float_as_uint(__uint_as_float(rr[4 * k4 + 1]) * osc),
                                     __float_as_uint(__uint_as_float(rr[4 * k4 + 2]) * osc), __float_as_uint(__uint_as_float(rr[4 * k4 + 3]) * osc));
                __syncwarp();
                float4 v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  const int row = 4 * i + rsub;
                  v[i] = ld_shared_v4(scratch + row * 128 + ((static_cast<uint32_t>(ch) ^ (row & 7)) << 4));
                }
                if (!sub.first) {
                  float4 old[8];
#pragma unroll
                  for (int i = 0; i < 8; ++i)
                    old[i] = *reinterpret_cast<const float4*>(lbase + (long long)(4 * i + rsub) * p.d + 32 * c + 4 * ch);
#pragma unroll
                  for (int i = 0; i < 8; ++i) { v[i].x += old[i].x; v[i].y += old[i].y; v[i].z += old[i].z; v[i].w += old[i].w; }
                }
#pragma unroll
                for (int i = 0; i < 8; ++i)
                  *reinterpret_cast<float4*>(obase + (long long)(4 * i + rsub) * p.d + 32 * c + 4 * ch) = v[i];
                __syncwarp();
              }
              ptx::tc_fence_before();
              __syncwarp();
              if (lane == 0) ptx::mbar_arrive_cluster(accempty_leader + 8u * buf);
              ++nt;
            }
          }
        }
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  ptx::cluster_sync();
  if (warp == 2) ptx::tmem_dealloc_pair(tmem_base, TMEM_COLS);
}

}  // namespace pair2
