// C-ABI entry points (include/clipnce.h): argument validation, workspace carving, TMA descriptor
// construction and kernel launches.  No torch types, no host synchronisation, no allocation.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <set>
#include <string>
#include <utility>

#include "../../include/clipnce.h"
#include "kernels_aux.cuh"
#include "kernels_head.cuh"
#include "kernels_link.cuh"
#include "kernels_pair.cuh"
#include "kernels_pair2.cuh"
#include "kernels_simt.cuh"
#include "kernels_tc.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                              \
  do {                                                                                              \
    cudaError_t e_ = (expr);                                                                        \
    if (e_ != cudaSuccess) return fail(CLIPNCE_ECUDA, "%s: %s", #expr, cudaGetErrorString(e_));     \
  } while (0)

// Integer value of the environment variable `name`, `dflt` where it is unset.  Every CLIPNCE_* variable the library reads
// goes through here (the list: INTEGRATION.md).  Test hooks are read on every call: tests switch them inside one process.
long long env_int(const char* name, long long dflt) {
  const char* e = getenv(name);
  return e ? atoll(e) : dflt;
}

// a peer that does not arrive within this time is fatal (barriers and per-block waits trap)
unsigned long long link_timeout_ns() {
  static const unsigned long long ns = [] {
    const long long ms = env_int("CLIPNCE_LINK_TIMEOUT_MS", 600000);   // 10 minutes, the order of NCCL's watchdog
    return (unsigned long long)(ms > 0 ? ms : 600000) * 1000000ull;
  }();
  return ns;
}
inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline size_t elem_size(int dtype) { return dtype == CLIPNCE_BF16 ? 2 : 4; }

// CTA-pair kernels (kernels_pair.cuh): the main tensor-core path.
bool pair_eligible(int64_t d) { return d % 128 == 0 && d >= 128 && d <= 768; }

// Kernel family.  0: exact CUDA-core kernels (fp32 check mode, shapes the tensor-core kernels do not take).
// 1: tensor cores with the FIXED shift -- |S_ij| <= s, so exp(S - s) needs no running maximum; valid while e^(-2s) is a
//    normal fp32.  The host's s may be a step or two stale (functional._ScaleHint), hence 2 s <= 80 instead of 86.
// 2: tensor cores with TRUE maxima (online soft-max forward, two-exponential backward): any s -- the clamp(max=100)
//    regime of old/clip_opt.py:100, run1/full.py:76 -- and logits not bounded by s (CLIPNCE_FLAG_UNBOUNDED: the
//    un-normalised queue rows of tong/utils/losses.py:10-14).  CTA-pair kernels only (d % 128 == 0).
int tc_family(int dtype, int64_t d, float scale, int flags) {
  if (dtype != CLIPNCE_BF16 || (flags & CLIPNCE_FLAG_FORCE_EXACT) || d < 8 || d % 8 != 0 || d > 768 || !(scale > 0.f)) return 0;
  if (!(flags & CLIPNCE_FLAG_UNBOUNDED) && 2.f * scale <= 80.f) return 1;
  return pair_eligible(d) ? 2 : 0;
}
bool tc_eligible(int dtype, int64_t d, float scale, int flags) { return tc_family(dtype, d, scale, flags) == 1; }

// ---- driver entry point for cuTensorMapEncodeTiled (no link-time dependency on libcuda) ----------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
std::mutex g_mu;
EncodeTiledFn g_encode = nullptr;
std::set<std::pair<const void*, int>> g_smem_allowed;   // (kernel, device) pairs whose shared-memory limit is raised

int get_encode(EncodeTiledFn* out) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (!g_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || fn == nullptr)
      return fail(CLIPNCE_ECUDA, "cuTensorMapEncodeTiled not available from this driver");
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  }
  *out = g_encode;
  return 0;
}

// bf16 row-major [outer, inner] (row stride ld elements), box {64, box_rows}, 128-byte swizzle.
int make_tmap(CUtensorMap* m, const void* base, int64_t inner, int64_t outer, int64_t ld, int box_rows) {
  EncodeTiledFn enc;
  int rc = get_encode(&enc);
  if (rc) return rc;
  cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(CLIPNCE_ECUDA, "cuTensorMapEncodeTiled failed (%d) for [%lld x %lld] ld %lld", (int)r, (long long)outer,
                (long long)inner, (long long)ld);
  return 0;
}

// Let `kern` take `bytes` of dynamic shared memory.  The attribute belongs to the kernel as loaded on one device, so it
// is set once per (kernel, current device).
template <typename Kernel>
int allow_smem(Kernel* kern, int bytes) {
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  const std::pair<const void*, int> key(reinterpret_cast<const void*>(kern), dev);
  std::lock_guard<std::mutex> lk(g_mu);
  if (g_smem_allowed.count(key)) return 0;
  CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  g_smem_allowed.insert(key);
  return 0;
}

int check_device_sm100() {
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  int major = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  if (major != 10) return fail(CLIPNCE_EUNSUPPORTED, "clipnce needs an sm_100 (B200) device, found sm_%d", major * 10);
  return 0;
}

template <int MODE, int BLOCK_I>
int launch_tc(const CUtensorMap& tx, const CUtensorMap& ty, const CUtensorMap& tyt, tc::Params p,
              int grid, cudaStream_t st) {
  auto kern = tc::clip_tc_kernel<MODE, BLOCK_I>;
  const int fixed = tc::smem_bytes(MODE, BLOCK_I, p.nkc, 0);
  const int total_boxes = (tc::SMEM_LIMIT - fixed) / tc::BOX_BYTES;   // 16 KiB ring stages that fit
  if (total_boxes < (MODE == 1 ? 2 : 1)) return fail(CLIPNCE_EUNSUPPORTED, "d=%d leaves no room for a TMA ring", p.d);
  auto cap = [](int v) { return v > tc::MAX_STAGES ? tc::MAX_STAGES : v; };
  if (MODE == 1) {
    p.stages_b = cap(total_boxes / 2);
    p.stages_a = cap(total_boxes - total_boxes / 2);
  } else {
    p.stages_a = cap(total_boxes);
    p.stages_b = 0;
  }
  const int smem = tc::smem_bytes(MODE, BLOCK_I, p.nkc, p.stages_a + p.stages_b);
  if (int rc = allow_smem(kern, tc::SMEM_LIMIT)) return rc;
  kern<<<grid, tc::num_threads(MODE, BLOCK_I), smem, st>>>(tx, ty, tyt, p);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int pair_slots() {   // CTA pairs that can be resident at once: one per two SMs
  static const int slots = [] {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms / 2 > 0 ? sms / 2 : 1;
  }();
  return slots;
}

// Cut a row block's column sweep into work items so that the grid fills whole waves of CTA pairs; every item pays a
// fixed prologue / drain (~0.75 step), so fewer, longer items win ties.  Returns steps per item.
int pick_split_steps(int n_pairs, int n_steps, int max_split) {
  {   // test hook: force the number of steps per work item
    const int v = (int)env_int("CLIPNCE_SPLIT_STEPS", 0);
    if (v >= 1) return (int)ceil_div(n_steps, v) <= max_split ? v : (int)ceil_div(n_steps, max_split);
  }
  const int slots = pair_slots();
  double best = -1.0;
  int best_sps = n_steps;
  for (int ns = 1; ns <= max_split; ++ns) {
    const int sps = (int)ceil_div(n_steps, ns);
    if (ns > 1 && sps < 8) break;
    const int items = n_pairs * (int)ceil_div(n_steps, sps);
    const double eff = (double)items / ((double)slots * (double)ceil_div(items, slots)) * (double)sps / ((double)sps + 0.75);
    if (eff > best + 1e-9) { best = eff; best_sps = sps; }
  }
  return best_sps;
}

template <int ROWS, int MODE = 0, int KT = 1>
int launch_pair_fwd(const void* x, const void* y, pair::FwdParams p, cudaStream_t st) {
  auto kern = pair::fwd_kernel<ROWS, MODE, KT>;
  int stages = (pair::SMEM_LIMIT - pair::fwd_smem_bytes(ROWS, p.nkc, 0)) / pair::STAGE_BYTES;
  if (stages > pair::MAX_STAGES) stages = pair::MAX_STAGES;
  if (stages < 2) return fail(CLIPNCE_EUNSUPPORTED, "d=%d leaves no room for a TMA ring", p.d);
  p.stages = stages;
  CUtensorMap tx, ty;
  int rc;
  // several problems in one launch: both operands are members of one stacked matrix, indexed by stack row
  if ((rc = make_tmap(&tx, x, p.d, p.grp.n_prob ? p.grp.stack_rows : p.n_rows, p.d, ROWS))) return rc;
  if ((rc = make_tmap(&ty, y, p.d, p.grp.n_prob ? p.grp.stack_rows : p.n_cols, p.d, 128))) return rc;
  if ((rc = allow_smem(kern, pair::SMEM_LIMIT))) return rc;
  const int grid = 2 * p.n_pairs * (int)ceil_div(p.n_steps, p.split_steps);
  kern<<<grid, pair::FWD_THREADS, pair::fwd_smem_bytes(ROWS, p.nkc, stages), st>>>(tx, ty, p);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

template <bool TWO_EXP>
int launch_pair_bwd(const void* x, const void* y, pair::BwdParams p, cudaStream_t st) {
  const int total = (pair::SMEM_LIMIT - pair::bwd_smem_bytes(p.nkc, 0)) / pair::STAGE_BYTES;
  if (total < 4) return fail(CLIPNCE_EUNSUPPORTED, "d=%d leaves no room for the TMA rings", p.d);
  auto cap = [](int v) { return v > pair::MAX_STAGES ? pair::MAX_STAGES : v; };
  p.stages_b = cap(total / 2);
  p.stages_a = cap(total - total / 2);
  p.nsbuf = p.nq2 <= 2 ? 2 : 1;   // 128 nq2 accumulator columns + 128 per logits buffer <= 512
  CUtensorMap tx, ty, tyg;
  int rc;
  const int64_t x_rows = p.grp.n_prob ? p.grp.stack_rows : p.n_rows, y_rows = p.grp.n_prob ? p.grp.stack_rows : p.n_cols;
  if ((rc = make_tmap(&tx, x, p.d, x_rows, p.d, pair::BWD_ROWS))) return rc;
  if ((rc = make_tmap(&ty, y, p.d, y_rows, p.d, 128))) return rc;
  if ((rc = make_tmap(&tyg, y, p.d, y_rows, p.d, 64))) return rc;
  const size_t smem = pair::bwd_smem_bytes(p.nkc, p.stages_a + p.stages_b);
  const int grid = 2 * p.n_pairs * (int)ceil_div(p.n_steps, p.split_steps);
  auto kern = pair::bwd_kernel<TWO_EXP>;
  if ((rc = allow_smem(kern, pair::SMEM_LIMIT))) return rc;
  kern<<<grid, pair::BWD_THREADS, smem, st>>>(tx, ty, tyg, p);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int fwd_block_i(int64_t n_rows, int64_t d) { return (d <= 512 && n_rows >= 128 * 148) ? 128 : 64; }

struct SimtFwdWs {
  float *row_pm, *row_pl, *col_pm, *col_pl;
  int64_t n_it, n_jt;
  size_t bytes;
};
SimtFwdWs simt_fwd_ws(void* ws, int64_t n_rows, int64_t n_cols) {
  SimtFwdWs w;
  w.n_it = ceil_div(n_rows, simt::TILE);
  w.n_jt = ceil_div(n_cols, simt::TILE);
  float* f = reinterpret_cast<float*>(ws);
  w.row_pm = f;
  w.row_pl = w.row_pm + w.n_jt * n_rows;
  w.col_pm = w.row_pl + w.n_jt * n_rows;
  w.col_pl = w.col_pm + w.n_it * n_cols;
  w.bytes = sizeof(float) * 2 * (size_t)(w.n_jt * n_rows + w.n_it * n_cols);
  return w;
}

}  // namespace

extern "C" {

int clipnce_version(void) { return CLIPNCE_VERSION; }
const char* clipnce_last_error(void) { return g_err.c_str(); }

int clipnce_uses_tensor_cores(int dtype, int64_t d, float scale, int flags) { return tc_family(dtype, d, scale, flags); }

int clipnce_needs_transposed(int dtype, int64_t d, float scale, int flags) {
  return (tc_eligible(dtype, d, scale, flags) && !pair_eligible(d)) ? 1 : 0;
}

int clipnce_workspace_bytes(int64_t n_rows, int64_t n_cols, int64_t d, int dtype, int flags, size_t* out) {
  if (!out || n_rows < 1 || n_cols < 1 || d < 1) return fail(CLIPNCE_EINVAL, "workspace_bytes: bad shape");
  if (dtype != CLIPNCE_BF16 && dtype != CLIPNCE_F32) return fail(CLIPNCE_EINVAL, "workspace_bytes: bad dtype %d", dtype);
  (void)flags;
  // tensor-core path (worst case over BLOCK_I choices) and exact path, forward and backward
  size_t tc_fwd = sizeof(float) * 2 * (size_t)ceil_div(n_rows, 64) * (size_t)round_up(n_cols, 32);
  size_t tc_bwd = round_up(sizeof(float) * (size_t)ceil_div(n_rows, 8), 256);
  {   // pair backward: per-split partial gradients when the row blocks alone cannot fill the GPU (capped at 256 MiB)
    const size_t slab = sizeof(float) * (size_t)n_rows * (size_t)d;
    const int n_pairs = (int)ceil_div(n_rows, 128);
    if (pair_eligible(d) && n_pairs < 4 * pair_slots()) {
      size_t ns = pair::MAX_SPLIT;
      while (ns > 1 && ns * slab > ((size_t)256 << 20)) --ns;
      if (ns > 1) tc_bwd += ns * slab;
    }
  }
  size_t pair_fwd = sizeof(float) * (2 * (size_t)ceil_div(n_rows, 128) * (size_t)round_up(n_cols, 256) +
                                     (size_t)pair::MAX_SPLIT * (size_t)n_rows);
  if (pair_fwd > tc_fwd) tc_fwd = pair_fwd;
  const size_t online_fwd = sizeof(float) * 2 * (size_t)pair::MAX_SPLIT * (size_t)(n_rows + n_cols);   // (max, sum) partials, both launches
  tc_fwd = (pair_fwd > tc_fwd ? pair_fwd : tc_fwd) + online_fwd + 512;   // the speculative large-scale forward uses both regions + a flag
  SimtFwdWs w = simt_fwd_ws(nullptr, n_rows, n_cols);
  size_t simt_bwd = sizeof(float) * (size_t)ceil_div(n_rows, simt::TILE);
  size_t m = tc_fwd;
  if (tc_bwd > m) m = tc_bwd;
  if (w.bytes > m) m = w.bytes;
  if (simt_bwd > m) m = simt_bwd;
  // clipnce_backward_dx keeps the fp32 gradient of the normalised rows in the workspace instead of a caller buffer
  *out = round_up(m + 256, 256) + round_up(sizeof(float) * (size_t)n_rows * (size_t)d, 256);
  return 0;
}

int clipnce_normalize(const void* x, int in_dtype, int64_t n, int64_t d, float* rinv, void* x_hat, int hat_dtype,
                      void* stream) {
  if (!x || !rinv || n < 1 || d < 1) return fail(CLIPNCE_EINVAL, "normalize: null pointer or empty shape");
  if ((in_dtype != CLIPNCE_BF16 && in_dtype != CLIPNCE_F32) ||
      (x_hat && hat_dtype != CLIPNCE_BF16 && hat_dtype != CLIPNCE_F32))
    return fail(CLIPNCE_EINVAL, "normalize: bad dtype");
  if (d > (1 << 20)) return fail(CLIPNCE_EINVAL, "normalize: d too large");
  cudaStream_t st = as_stream(stream);
  const int wpb = 8;
  dim3 grid((unsigned)ceil_div(n, wpb)), block(32 * wpb);
  const int di = (int)d;
  const bool hat_bf16 = x_hat && hat_dtype == CLIPNCE_BF16;
  if (in_dtype == CLIPNCE_BF16 && hat_bf16)
    aux::normalize_rows<<<grid, block, 0, st>>>((const __nv_bfloat16*)x, n, di, (__nv_bfloat16*)x_hat, rinv);
  else if (in_dtype == CLIPNCE_F32 && hat_bf16)
    aux::normalize_rows<<<grid, block, 0, st>>>((const float*)x, n, di, (__nv_bfloat16*)x_hat, rinv);
  else if (in_dtype == CLIPNCE_BF16)
    aux::normalize_rows<<<grid, block, 0, st>>>((const __nv_bfloat16*)x, n, di, (float*)x_hat, rinv);
  else
    aux::normalize_rows<<<grid, block, 0, st>>>((const float*)x, n, di, (float*)x_hat, rinv);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_stage_operand(const void* x, int in_dtype, int64_t n, int64_t d, void* x_c, void* x_c_t, int64_t ld_t,
                          int c_dtype, void* stream) {
  if (!x || n < 1 || d < 1) return fail(CLIPNCE_EINVAL, "stage_operand: bad argument");
  if (!x_c && !x_c_t) return 0;
  if (x_c_t && (ld_t < n || ld_t % 8 != 0)) return fail(CLIPNCE_EINVAL, "stage_operand: ld_t must be >= n and a multiple of 8");
  if ((in_dtype != CLIPNCE_BF16 && in_dtype != CLIPNCE_F32) || (c_dtype != CLIPNCE_BF16 && c_dtype != CLIPNCE_F32))
    return fail(CLIPNCE_EINVAL, "stage_operand: bad dtype");
  cudaStream_t st = as_stream(stream);
  dim3 grid((unsigned)ceil_div(n, 32), (unsigned)ceil_div(d, 32)), block(32, 8);
  const int di = (int)d;
  if (in_dtype == CLIPNCE_BF16 && c_dtype == CLIPNCE_BF16)
    aux::stage_operand<<<grid, block, 0, st>>>((const __nv_bfloat16*)x, n, di, (__nv_bfloat16*)x_c, (__nv_bfloat16*)x_c_t, ld_t);
  else if (in_dtype == CLIPNCE_F32 && c_dtype == CLIPNCE_BF16)
    aux::stage_operand<<<grid, block, 0, st>>>((const float*)x, n, di, (__nv_bfloat16*)x_c, (__nv_bfloat16*)x_c_t, ld_t);
  else if (in_dtype == CLIPNCE_BF16 && c_dtype == CLIPNCE_F32)
    aux::stage_operand<<<grid, block, 0, st>>>((const __nv_bfloat16*)x, n, di, (float*)x_c, (float*)x_c_t, ld_t);
  else
    aux::stage_operand<<<grid, block, 0, st>>>((const float*)x, n, di, (float*)x_c, (float*)x_c_t, ld_t);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // extern "C"

namespace {
// the gather of the columns runs beside the sweep (clipnce_forward_gathered): where the flags live and how the columns
// map to source ranks
struct Gathered {
  const uint32_t* flags = nullptr;
  const uint32_t* epoch = nullptr;
  int world = 0, rank = 0;
};
void set_gathered(pair::FwdParams& p, const Gathered* g) {
  if (!g || !g->flags) return;
  p.src_flags = g->flags;
  p.src_epoch = g->epoch;
  p.steps_per_src = p.n_steps / g->world;
  p.rot_steps = g->rank * p.steps_per_src;
  p.self_src = g->rank;
  p.wait_timeout_ns = link_timeout_ns();
}

int forward_impl(const void* x, const void* y, const float* rinv_x, const float* rinv_y, int64_t n_rows,
                 int64_t n_cols, int64_t d, int64_t diag_offset, float scale, const float* scale_dev, int dtype,
                 int flags, float* row_m,
                 float* row_l, float* col_m, float* col_l, float* diag, void* workspace, size_t workspace_bytes,
                 void* stream, const Gathered* gat) {
  if (!x || !y || !rinv_x || !rinv_y || !row_m || !row_l || !col_m || !col_l || !diag || !workspace)
    return fail(CLIPNCE_EINVAL, "forward: null pointer");
  if (n_rows < 1 || n_cols < 1 || d < 1 || n_rows > (1ll << 30) || n_cols > (1ll << 30))
    return fail(CLIPNCE_EINVAL, "forward: bad shape");
  if (dtype != CLIPNCE_BF16 && dtype != CLIPNCE_F32) return fail(CLIPNCE_EINVAL, "forward: bad dtype %d", dtype);
  if (!std::isfinite(scale)) return fail(CLIPNCE_EINVAL, "forward: scale is not finite");
  cudaStream_t st = as_stream(stream);
  int rc = check_device_sm100();
  if (rc) return rc;

  if (tc_family(dtype, d, scale, flags) == 2) {
    if (!aligned16(x) || !aligned16(y)) return fail(CLIPNCE_EINVAL, "forward: operands must be 16-byte aligned");
    const int rows = d <= 512 ? 128 : 64;
    float* wsf = reinterpret_cast<float*>(workspace);
    size_t used = 0;
    const int* gate = nullptr;
    // Bounded logits (|S| <= s: normalised rows; the clamp at 100 of old/clip_opt.py:100 is the case that matters).  The exact online
    // sweeps below cost two passes over the logits.  Speculate instead: ONE fixed-shift sweep (the family-1 kernel) with
    // the shift lowered to p = s - 72, so that e^(S - p) neither overflows (sums <= n e^72) nor -- for any row or column
    // whose largest logit is above p - 62 = s - 134 -- loses mass to the terms that flush to zero (< n e^-87 in all,
    // 1e-6 of a sum >= e^-62).  Rows / columns below that (a positive pair AND every negative with cosine < -0.34 at
    // s = 100) raise a device flag in the reduction, and the exact sweeps run after all, gated on it: same results in
    // every case, decided on the device (graph-capturable, no host read), one sweep in the common one.
    // (any scale: beyond ~105 more rows fall under the bound and the fallback runs more often, the results stay exact;
    // the decision must not depend on the scale -- ranks of a row-sharded step hold slightly different host copies of it)
    const bool speculate = !(flags & CLIPNCE_FLAG_UNBOUNDED) && n_cols <= (1ll << 22) && n_rows <= (1ll << 22) &&
                           env_int("CLIPNCE_NO_SPECULATE", 0) == 0;
    if (gat && !speculate) return fail(CLIPNCE_EUNSUPPORTED, "forward_gathered: no fixed-shift sweep for these arguments");
    if (speculate) {
      constexpr float kOff = 72.f;
      // a sum of n terms loses less than n e^-87.3 to flushed terms: demand 1e6 times that (n = 65536: 1.1e-27 = e^-62)
      const float thr_row = 1.2e-38f * 1e6f * (float)n_cols, thr_col = 1.2e-38f * 1e6f * (float)n_rows;
      pair::FwdParams p;
      memset(&p, 0, sizeof p);
      p.n_rows = (int)n_rows; p.n_cols = (int)n_cols; p.d = (int)d;
      p.nkc = (int)ceil_div(d, 64); p.n_steps = (int)ceil_div(n_cols, pair::STEP_J);
      p.diag_offset = diag_offset; p.scale = scale; p.scale_dev = scale_dev;
      p.rinv_x = rinv_x; p.rinv_y = rinv_y; p.diag = diag; p.shift_off = kOff;
      p.n_pairs = (int)ceil_div(n_rows, 2 * rows);
      p.split_steps = pick_split_steps(p.n_pairs, p.n_steps, pair::MAX_SPLIT);
      const int n_split = (int)ceil_div(p.n_steps, p.split_steps);
      p.col_ld = (long long)p.n_steps * pair::STEP_J;
      const int n_part = 2 * p.n_pairs;
      const size_t col_bytes = sizeof(float) * (size_t)n_part * (size_t)p.col_ld;
      const size_t need = round_up(col_bytes + sizeof(float) * (size_t)n_split * (size_t)n_rows, 256) + 256;
      if (workspace_bytes < need) return fail(CLIPNCE_EWORKSPACE, "forward: workspace %zu < %zu", workspace_bytes, need);
      p.col_part = wsf;
      p.row_part = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + col_bytes);
      int* flag = reinterpret_cast<int*>(reinterpret_cast<char*>(workspace) + need - 256);
      CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(int), st));
      set_gathered(p, gat);
      rc = rows == 128 ? launch_pair_fwd<128>(x, y, p, st) : launch_pair_fwd<64>(x, y, p, st);
      if (rc) return rc;
      aux::reduce_shifted_partials<<<(unsigned)ceil_div(n_cols, 256), 256, 0, st>>>(p.col_part, n_part, p.col_ld, n_cols, scale,
                                                                                      scale_dev, kOff, thr_col, col_m, col_l, flag);
      aux::reduce_shifted_partials<<<(unsigned)ceil_div(n_rows, 256), 256, 0, st>>>(p.row_part, n_split, n_rows, n_rows, scale,
                                                                                      scale_dev, kOff, thr_row, row_m, row_l, flag);
      CUDA_TRY(cudaGetLastError());
      gate = flag;
      used = need;
    }
    // online soft-max: row statistics of (x, y), then of (y, x) -- the column statistics -- with true running maxima
    for (int side = 0; side < 2; ++side) {
      const int64_t nr = side == 0 ? n_rows : n_cols, nc = side == 0 ? n_cols : n_rows;
      pair::FwdParams p;
      memset(&p, 0, sizeof p);
      p.n_rows = (int)nr; p.n_cols = (int)nc; p.d = (int)d;
      p.nkc = (int)ceil_div(d, 64); p.n_steps = (int)ceil_div(nc, pair::STEP_J);
      p.diag_offset = diag_offset; p.scale = scale; p.scale_dev = scale_dev;
      p.rinv_x = side == 0 ? rinv_x : rinv_y; p.rinv_y = side == 0 ? rinv_y : rinv_x;
      p.diag = side == 0 ? diag : nullptr;
      p.gate = gate;
      p.n_pairs = (int)ceil_div(nr, 2 * rows);
      p.split_steps = pick_split_steps(p.n_pairs, p.n_steps, pair::MAX_SPLIT);
      const int n_split = (int)ceil_div(p.n_steps, p.split_steps);
      const size_t need = used + sizeof(float) * 2 * (size_t)n_split * (size_t)nr;
      if (workspace_bytes < need) return fail(CLIPNCE_EWORKSPACE, "forward: workspace %zu < %zu", workspace_bytes, need);
      p.row_part_m = wsf + used / sizeof(float);
      p.row_part = p.row_part_m + (size_t)n_split * (size_t)nr;
      used = need;
      const void* xs = side == 0 ? x : y;
      const void* ys = side == 0 ? y : x;
      rc = rows == 128 ? launch_pair_fwd<128, 2>(xs, ys, p, st) : launch_pair_fwd<64, 2>(xs, ys, p, st);
      if (rc) return rc;
      aux::reduce_ml_partials<<<(unsigned)ceil_div(nr, 256), 256, 0, st>>>(p.row_part_m, p.row_part, n_split, nr, nr,
                                                                            side == 0 ? row_m : col_m, side == 0 ? row_l : col_l, gate);
      CUDA_TRY(cudaGetLastError());
    }
    return 0;
  }

  if (tc_eligible(dtype, d, scale, flags)) {
    if (!aligned16(x) || !aligned16(y)) return fail(CLIPNCE_EINVAL, "forward: operands must be 16-byte aligned");
    if (pair_eligible(d)) {
      const int rows = d <= 512 ? 128 : 64;
      pair::FwdParams p;
      memset(&p, 0, sizeof p);
      p.n_rows = (int)n_rows; p.n_cols = (int)n_cols; p.d = (int)d;
      p.nkc = (int)ceil_div(d, 64); p.n_steps = (int)ceil_div(n_cols, pair::STEP_J);
      p.diag_offset = diag_offset; p.scale = scale; p.scale_dev = scale_dev;
      p.rinv_x = rinv_x; p.rinv_y = rinv_y; p.diag = diag;
      p.n_pairs = (int)ceil_div(n_rows, 2 * rows);
      p.split_steps = pick_split_steps(p.n_pairs, p.n_steps, pair::MAX_SPLIT);
      const int n_split = (int)ceil_div(p.n_steps, p.split_steps);
      p.col_ld = (long long)p.n_steps * pair::STEP_J;
      const int n_part = 2 * p.n_pairs;
      const size_t col_bytes = sizeof(float) * (size_t)n_part * (size_t)p.col_ld;
      const size_t need = col_bytes + sizeof(float) * (size_t)n_split * (size_t)n_rows;
      if (workspace_bytes < need) return fail(CLIPNCE_EWORKSPACE, "forward: workspace %zu < %zu", workspace_bytes, need);
      p.col_part = reinterpret_cast<float*>(workspace);
      p.row_part = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + col_bytes);
      set_gathered(p, gat);
      rc = rows == 128 ? launch_pair_fwd<128>(x, y, p, st) : launch_pair_fwd<64>(x, y, p, st);
      if (rc) return rc;
      aux::reduce_col_partials<<<(unsigned)ceil_div(n_cols, 256), 256, 0, st>>>(p.col_part, n_part, p.col_ld, n_cols, scale,
                                                                                  scale_dev, col_m, col_l);
      aux::reduce_col_partials<<<(unsigned)ceil_div(n_rows, 256), 256, 0, st>>>(p.row_part, n_split, n_rows, n_rows, scale,
                                                                                  scale_dev, row_m, row_l);
      CUDA_TRY(cudaGetLastError());
      return 0;
    }
    const int bi = fwd_block_i(n_rows, d);
    const int64_t n_ib = ceil_div(n_rows, bi);
    const int64_t col_ld = round_up(n_cols, 32);
    const size_t need = sizeof(float) * (size_t)(bi / 32) * (size_t)n_ib * (size_t)col_ld;
    if (workspace_bytes < need) return fail(CLIPNCE_EWORKSPACE, "forward: workspace %zu < %zu", workspace_bytes, need);
    CUtensorMap tx, ty;
    if ((rc = make_tmap(&tx, x, d, n_rows, d, bi))) return rc;
    if ((rc = make_tmap(&ty, y, d, n_cols, d, tc::BLOCK_J))) return rc;
    tc::Params p;
    memset(&p, 0, sizeof p);
    p.n_rows = (int)n_rows; p.n_cols = (int)n_cols; p.d = (int)d;
    p.nkc = (int)ceil_div(d, 64); p.nq = (int)ceil_div(d, 128); p.n_jt = (int)ceil_div(n_cols, tc::BLOCK_J);
    p.diag_offset = diag_offset; p.scale = scale; p.k2 = scale * tc::LOG2E; p.scale_dev = scale_dev;
    p.rinv_x = rinv_x; p.rinv_y = rinv_y;
    p.row_m = row_m; p.row_l = row_l; p.col_part = reinterpret_cast<float*>(workspace); p.col_ld = col_ld; p.diag = diag;
    if (bi == 128) rc = launch_tc<0, 128>(tx, ty, ty, p, (int)n_ib, st);
    else           rc = launch_tc<0, 64>(tx, ty, ty, p, (int)n_ib, st);
    if (rc) return rc;
    aux::reduce_col_partials<<<(unsigned)ceil_div(n_cols, 256), 256, 0, st>>>(p.col_part, (int)((bi / 32) * n_ib), col_ld,
                                                                                n_cols, scale, scale_dev, col_m, col_l);
    CUDA_TRY(cudaGetLastError());
    return 0;
  }

  // exact CUDA-core path
  SimtFwdWs w = simt_fwd_ws(workspace, n_rows, n_cols);
  if (workspace_bytes < w.bytes) return fail(CLIPNCE_EWORKSPACE, "forward: workspace %zu < %zu", workspace_bytes, w.bytes);
  if (w.n_it > 65535) return fail(CLIPNCE_EUNSUPPORTED, "forward (exact path): n_rows too large");
  dim3 grid((unsigned)w.n_jt, (unsigned)w.n_it);
  if (dtype == CLIPNCE_BF16)
    simt::fwd_stats<<<grid, simt::THREADS, 0, st>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)y, rinv_x, rinv_y,
                                                     n_rows, n_cols, (int)d, diag_offset, scale, scale_dev, w.row_pm,
                                                     w.row_pl, w.col_pm, w.col_pl, diag);
  else
    simt::fwd_stats<<<grid, simt::THREADS, 0, st>>>((const float*)x, (const float*)y, rinv_x, rinv_y, n_rows, n_cols,
                                                     (int)d, diag_offset, scale, scale_dev, w.row_pm, w.row_pl, w.col_pm,
                                                     w.col_pl, diag);
  CUDA_TRY(cudaGetLastError());
  aux::reduce_ml_partials<<<(unsigned)ceil_div(n_rows, 256), 256, 0, st>>>(w.row_pm, w.row_pl, (int)w.n_jt, n_rows,
                                                                             n_rows, row_m, row_l);
  aux::reduce_ml_partials<<<(unsigned)ceil_div(n_cols, 256), 256, 0, st>>>(w.col_pm, w.col_pl, (int)w.n_it, n_cols,
                                                                             n_cols, col_m, col_l);
  CUDA_TRY(cudaGetLastError());
  return 0;
}
}  // namespace

extern "C" {

int clipnce_forward(const void* x, const void* y, const float* rinv_x, const float* rinv_y, int64_t n_rows,
                    int64_t n_cols, int64_t d, int64_t diag_offset, float scale, const float* scale_dev, int dtype,
                    int flags, float* row_m, float* row_l, float* col_m, float* col_l, float* diag, void* workspace,
                    size_t workspace_bytes, void* stream) {
  return forward_impl(x, y, rinv_x, rinv_y, n_rows, n_cols, d, diag_offset, scale, scale_dev, dtype, flags, row_m, row_l, col_m,
                      col_l, diag, workspace, workspace_bytes, stream, nullptr);
}

int clipnce_forward_gathered_ok(int dtype, int64_t d, float scale, int flags) {
  const int fam = tc_family(dtype, d, scale, flags);
  if (fam == 1) return pair_eligible(d) ? 1 : 0;
  return (fam == 2 && !(flags & CLIPNCE_FLAG_UNBOUNDED) && env_int("CLIPNCE_NO_SPECULATE", 0) == 0) ? 1 : 0;
}

int clipnce_forward_gathered(const void* x, const void* y, const float* rinv_x, const float* rinv_y, int64_t n_rows,
                             int64_t n_cols, int64_t d, float scale, const float* scale_dev, int dtype, int flags,
                             float* row_m, float* row_l, float* col_m, float* col_l, float* diag, void* const* peer_base,
                             int world, int rank, int phase, void* workspace, size_t workspace_bytes, void* stream) {
  if (!peer_base || world < 2 || world > link::MAX_WORLD || rank < 0 || rank >= world || phase < 0 || phase >= link::MAX_PHASE)
    return fail(CLIPNCE_EINVAL, "forward_gathered: bad peers / phase");
  if (n_cols != n_rows * world || n_rows % pair::STEP_J != 0 || n_cols > (1ll << 22))
    return fail(CLIPNCE_EUNSUPPORTED, "forward_gathered: n_cols must be world * n_rows <= 2^22, n_rows a multiple of 256");
  if (!clipnce_forward_gathered_ok(dtype, d, scale, flags))
    return fail(CLIPNCE_EUNSUPPORTED, "forward_gathered: kernel family without a fixed-shift sweep (use clipnce_link_barrier + clipnce_forward)");
  if (!peer_base[rank]) return fail(CLIPNCE_EINVAL, "forward_gathered: null peer buffer");
  Gathered g;
  const char* mine = reinterpret_cast<const char*>(peer_base[rank]);
  g.flags = reinterpret_cast<const uint32_t*>(mine + link::OFF_FLAGS) + phase * link::MAX_WORLD;
  g.epoch = reinterpret_cast<const uint32_t*>(mine + link::OFF_EPOCH) + phase;
  g.world = world;
  g.rank = rank;
  return forward_impl(x, y, rinv_x, rinv_y, n_rows, n_cols, d, (int64_t)rank * n_rows, scale, scale_dev, dtype, flags, row_m,
                      row_l, col_m, col_l, diag, workspace, workspace_bytes, stream, &g);
}

}  // extern "C"

namespace {
// What clipnce_backward_dx asks the contraction to leave undone: the pair kernels' split partials stay unsummed and the
// row dots untaken -- finish_rows does all of it in one pass together with the normalise backward.
struct Deferred {
  const float* parts = nullptr;
  int n_split = 1;
  bool ds_pending = false;
};

// A side of the finishing pass with one contribution of n_split slabs of [n, d].
aux::FinishSide finish_side(const float* parts, int n_split, int64_t n, int64_t d, const void* xc, const void* xo,
                            const float* rinv, void* dx, float* ds_part) {
  aux::FinishSide s;
  memset(&s, 0, sizeof s);
  s.parts[0] = parts; s.n_contrib = 1; s.n_split = n_split; s.slab = n * d; s.n = n;
  s.xc = xc; s.xo = xo; s.rinv = rinv; s.dx = dx; s.ds_part = ds_part;
  return s;
}

template <typename TC, typename TI, typename TO>
void finish_kernel(const aux::FinishSides& fs, dim3 grid, size_t smem, bool v4, const float* grad_scale, int d, cudaStream_t st) {
  if (v4) aux::finish_rows<TC, TI, TO, 4><<<grid, 256, smem, st>>>(fs, grad_scale, d);
  else aux::finish_rows<TC, TI, TO, 1><<<grid, 256, smem, st>>>(fs, grad_scale, d);
}

// ONE launch of the finishing pass over sides[0, n_sides), each of at most n rows, all of the same types: the compute
// type `dtype` (xc), the caller's rows `in_dtype` (xo), the gradient `out_dtype` (dx).  v4: 16-byte accesses (d % 4 == 0,
// every row base 4-element aligned).  8 d floats of shared memory per block: d <= 1536.
int launch_finish(const aux::FinishSide* sides, int n_sides, int64_t n, int64_t d, int dtype, int in_dtype, int out_dtype,
                  const float* grad_scale, bool v4, cudaStream_t st) {
  aux::FinishSides fs;
  memset(&fs, 0, sizeof fs);
  for (int i = 0; i < n_sides; ++i) fs.s[i] = sides[i];
  const dim3 grid((unsigned)ceil_div(n, 8), (unsigned)n_sides);
  const size_t smem = sizeof(float) * 8 * (size_t)d;
  const int di = (int)d;
  using bf = __nv_bfloat16;
  const bool ib = in_dtype == CLIPNCE_BF16, ob = out_dtype == CLIPNCE_BF16;
  if (dtype == CLIPNCE_BF16 && ib && ob) finish_kernel<bf, bf, bf>(fs, grid, smem, v4, grad_scale, di, st);
  else if (dtype == CLIPNCE_BF16 && ib) finish_kernel<bf, bf, float>(fs, grid, smem, v4, grad_scale, di, st);
  else if (dtype == CLIPNCE_BF16 && ob) finish_kernel<bf, float, bf>(fs, grid, smem, v4, grad_scale, di, st);
  else if (dtype == CLIPNCE_BF16) finish_kernel<bf, float, float>(fs, grid, smem, v4, grad_scale, di, st);
  else if (ob) finish_kernel<float, float, bf>(fs, grid, smem, v4, grad_scale, di, st);
  else finish_kernel<float, float, float>(fs, grid, smem, v4, grad_scale, di, st);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int backward_impl(const void* x, const void* y, const void* y_t, int64_t ld_t, const float* rinv_x,
                  const float* rinv_y, int64_t n_rows, int64_t n_cols, int64_t d, int64_t diag_offset, float scale,
                  const float* scale_dev, const float* row_m, const float* row_w, const float* col_m, const float* col_w, float diag_w,
                  float grad_out, int dtype, int flags, float* dx_hat, float* d_scale_sum, void* workspace,
                  size_t workspace_bytes, void* stream, Deferred* defer) {
  if (!x || !y || !rinv_x || !rinv_y || !row_m || !row_w || !dx_hat || !workspace)
    return fail(CLIPNCE_EINVAL, "backward: null pointer");
  if ((col_m == nullptr) != (col_w == nullptr)) return fail(CLIPNCE_EINVAL, "backward: col_m and col_w go together");
  if (n_rows < 1 || n_cols < 1 || d < 1 || n_rows > (1ll << 30) || n_cols > (1ll << 30))
    return fail(CLIPNCE_EINVAL, "backward: bad shape");
  if (dtype != CLIPNCE_BF16 && dtype != CLIPNCE_F32) return fail(CLIPNCE_EINVAL, "backward: bad dtype %d", dtype);
  if (!std::isfinite(scale)) return fail(CLIPNCE_EINVAL, "backward: scale is not finite");
  cudaStream_t st = as_stream(stream);
  int rc = check_device_sm100();
  if (rc) return rc;

  const int fam = tc_family(dtype, d, scale, flags);
  if ((fam == 1 && pair_eligible(d)) || fam == 2) {
    if (!aligned16(x) || !aligned16(y)) return fail(CLIPNCE_EINVAL, "backward: operands must be 16-byte aligned");
    const int64_t n_blk = ceil_div(n_rows, 8);
    const size_t part_bytes = round_up(sizeof(float) * (size_t)n_blk, 256);
    pair::BwdParams p;
    memset(&p, 0, sizeof p);
    p.n_rows = (int)n_rows; p.n_cols = (int)n_cols; p.d = (int)d;
    p.nkc = (int)ceil_div(d, 64); p.nq2 = (int)ceil_div(d, 256); p.n_steps = (int)ceil_div(n_cols, pair::STEP_J);
    p.diag_offset = diag_offset; p.scale = scale; p.scale_dev = scale_dev; p.diag_w = diag_w; p.grad_out = grad_out;
    p.rinv_x = rinv_x; p.rinv_y = rinv_y; p.row_m_in = row_m; p.row_w = row_w; p.col_m_in = col_m; p.col_w = col_w;
    p.n_pairs = (int)ceil_div(n_rows, 2 * pair::BWD_ROWS);
    // split the column sweep only where the row blocks alone leave SMs idle (few local rows: the row-sharded step),
    // and only as far as the scratch for the per-split partial gradients reaches
    int max_split = (int)((workspace_bytes > part_bytes ? workspace_bytes - part_bytes : 0) / (sizeof(float) * (size_t)n_rows * (size_t)d));
    if (max_split > pair::MAX_SPLIT) max_split = pair::MAX_SPLIT;
    p.split_steps = max_split >= 2 ? pick_split_steps(p.n_pairs, p.n_steps, max_split) : p.n_steps;
    const int n_split = (int)ceil_div(p.n_steps, p.split_steps);
    if (workspace_bytes < part_bytes) return fail(CLIPNCE_EWORKSPACE, "backward: workspace %zu < %zu", workspace_bytes, part_bytes);
    float* dx_part = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + part_bytes);
    p.dx = n_split > 1 ? dx_part : dx_hat;
    if ((rc = fam == 2 ? launch_pair_bwd<true>(x, y, p, st) : launch_pair_bwd<false>(x, y, p, st))) return rc;
    if (defer) {
      defer->parts = p.dx;
      defer->n_split = n_split;
      defer->ds_pending = d_scale_sum != nullptr;
      return 0;
    }
    if (n_split > 1) {
      const int64_t n4 = n_rows * d / 4;
      aux::sum_splits<<<(unsigned)ceil_div(n4, 256), 256, 0, st>>>(reinterpret_cast<const float4*>(dx_part), n_split, n4,
                                                                     reinterpret_cast<float4*>(dx_hat));
      CUDA_TRY(cudaGetLastError());
    }
    if (d_scale_sum) {
      // sum_ij G_ij S_ij = sum_i <xhat_i, dxhat_i> / grad_out: read it off the finished gradient instead of
      // carrying an extra FMA per logit through the epilogue
      float* part = reinterpret_cast<float*>(workspace);
      aux::rowdot_partials<<<(unsigned)n_blk, 256, 0, st>>>((const __nv_bfloat16*)x, rinv_x, dx_hat, n_rows, (int)d, part);
      aux::reduce_scalar_partials_par<<<1, 256, 0, st>>>(part, (int)n_blk, 1.f, d_scale_sum);
      CUDA_TRY(cudaGetLastError());
    }
    return 0;
  }

  if (tc_eligible(dtype, d, scale, flags)) {
    if (!y_t) return fail(CLIPNCE_EINVAL, "backward: the tensor-core path needs y_t");
    if (ld_t < n_cols || ld_t % 8 != 0) return fail(CLIPNCE_EINVAL, "backward: ld_t must be >= n_cols and a multiple of 8");
    if (!aligned16(x) || !aligned16(y) || !aligned16(y_t))
      return fail(CLIPNCE_EINVAL, "backward: operands must be 16-byte aligned");
    // rows per CTA: the gradient accumulators (ceil(d/128) * BLOCK_I TMEM columns) plus two logits buffers share the
    // 512 TMEM columns (measured on a B200 at N = 65536, d = 512: 9.6 ms per side, against 11.4 with 96 rows and one buffer)
    const int bi = 64;
    const int64_t n_ib = ceil_div(n_rows, bi);
    const size_t need = sizeof(float) * (size_t)n_ib;
    if (workspace_bytes < need) return fail(CLIPNCE_EWORKSPACE, "backward: workspace %zu < %zu", workspace_bytes, need);
    CUtensorMap tx, ty, tyt;
    if ((rc = make_tmap(&tx, x, d, n_rows, d, bi))) return rc;
    if ((rc = make_tmap(&ty, y, d, n_cols, d, tc::BLOCK_J))) return rc;
    if ((rc = make_tmap(&tyt, y_t, n_cols, d, ld_t, 128))) return rc;
    tc::Params p;
    memset(&p, 0, sizeof p);
    p.n_rows = (int)n_rows; p.n_cols = (int)n_cols; p.d = (int)d;
    p.nkc = (int)ceil_div(d, 64); p.nq = (int)ceil_div(d, 128); p.n_jt = (int)ceil_div(n_cols, tc::BLOCK_J);
    p.diag_offset = diag_offset; p.scale = scale; p.k2 = scale * tc::LOG2E; p.scale_dev = scale_dev; p.grad_out = grad_out;
    p.rinv_x = rinv_x; p.rinv_y = rinv_y;
    p.row_m_in = row_m; p.row_w = row_w; p.col_m_in = col_m; p.col_w = col_w; p.diag_w = diag_w; p.out_scale = grad_out * scale;
    p.dx = dx_hat; p.ds_part = d_scale_sum ? reinterpret_cast<float*>(workspace) : nullptr;
    if ((rc = launch_tc<1, 64>(tx, ty, tyt, p, (int)n_ib, st))) return rc;
    if (d_scale_sum) {
      aux::reduce_scalar_partials<<<1, 32, 0, st>>>(p.ds_part, (int)n_ib, grad_out, d_scale_sum);
      CUDA_TRY(cudaGetLastError());
    }
    return 0;
  }

  const int64_t n_it = ceil_div(n_rows, simt::TILE);
  const size_t need = sizeof(float) * (size_t)n_it;
  if (workspace_bytes < need) return fail(CLIPNCE_EWORKSPACE, "backward: workspace %zu < %zu", workspace_bytes, need);
  if (n_it > 65535) return fail(CLIPNCE_EUNSUPPORTED, "backward (exact path): n_rows too large");
  float* ds_part = d_scale_sum ? reinterpret_cast<float*>(workspace) : nullptr;
  dim3 grid((unsigned)ceil_div(d, simt::TILE), (unsigned)n_it);
  if (dtype == CLIPNCE_BF16)
    simt::bwd_side<<<grid, simt::THREADS, 0, st>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)y, rinv_x, rinv_y,
                                                    n_rows, n_cols, (int)d, diag_offset, scale, scale_dev, row_m, row_w, col_m,
                                                    col_w, diag_w, grad_out * scale, dx_hat, ds_part);
  else
    simt::bwd_side<<<grid, simt::THREADS, 0, st>>>((const float*)x, (const float*)y, rinv_x, rinv_y, n_rows, n_cols,
                                                    (int)d, diag_offset, scale, scale_dev, row_m, row_w, col_m, col_w, diag_w,
                                                    grad_out * scale, dx_hat, ds_part);
  CUDA_TRY(cudaGetLastError());
  if (d_scale_sum) {
    aux::reduce_scalar_partials<<<1, 32, 0, st>>>(ds_part, (int)n_it, grad_out, d_scale_sum);
    CUDA_TRY(cudaGetLastError());
  }
  return 0;
}

}  // namespace

extern "C" {

int clipnce_backward(const void* x, const void* y, const void* y_t, int64_t ld_t, const float* rinv_x,
                     const float* rinv_y, int64_t n_rows, int64_t n_cols, int64_t d, int64_t diag_offset, float scale,
                     const float* scale_dev, const float* row_m, const float* row_w, const float* col_m, const float* col_w, float diag_w,
                     float grad_out, int dtype, int flags, float* dx_hat, float* d_scale_sum, void* workspace,
                     size_t workspace_bytes, void* stream) {
  return backward_impl(x, y, y_t, ld_t, rinv_x, rinv_y, n_rows, n_cols, d, diag_offset, scale, scale_dev, row_m, row_w, col_m,
                       col_w, diag_w, grad_out, dtype, flags, dx_hat, d_scale_sum, workspace, workspace_bytes, stream, nullptr);
}

int clipnce_backward_dx(const void* x, const void* y, const void* y_t, int64_t ld_t, const float* rinv_x,
                        const float* rinv_y, int64_t n_rows, int64_t n_cols, int64_t d, int64_t diag_offset, float scale,
                        const float* scale_dev, const float* row_m, const float* row_w, const float* col_m,
                        const float* col_w, float diag_w, int dtype, int flags, const void* x_orig, int in_dtype,
                        const float* grad_scale, void* dx, int out_dtype, float* d_scale_sum, void* workspace,
                        size_t workspace_bytes, void* stream) {
  if (!x_orig || !dx) return fail(CLIPNCE_EINVAL, "backward_dx: null pointer");
  if ((in_dtype != CLIPNCE_BF16 && in_dtype != CLIPNCE_F32) || (out_dtype != CLIPNCE_BF16 && out_dtype != CLIPNCE_F32))
    return fail(CLIPNCE_EINVAL, "backward_dx: bad dtype");
  if (n_rows < 1 || d < 1) return fail(CLIPNCE_EINVAL, "backward_dx: bad shape");
  if (in_dtype == dtype && x_orig != x) return fail(CLIPNCE_EINVAL, "backward_dx: x_orig of the compute type must be x itself");
  if (dtype == CLIPNCE_F32 && in_dtype != CLIPNCE_F32) return fail(CLIPNCE_EINVAL, "backward_dx: fp32 compute needs fp32 rows");
  const size_t slab = round_up(sizeof(float) * (size_t)n_rows * (size_t)d, 256);
  if (!workspace || workspace_bytes < slab + 256) return fail(CLIPNCE_EWORKSPACE, "backward_dx: workspace %zu too small", workspace_bytes);
  const size_t core_bytes = (workspace_bytes - slab) & ~(size_t)255;
  float* dx_hat = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + core_bytes);
  Deferred df;
  df.parts = dx_hat;
  int rc = backward_impl(x, y, y_t, ld_t, rinv_x, rinv_y, n_rows, n_cols, d, diag_offset, scale, scale_dev, row_m, row_w, col_m,
                         col_w, diag_w, 1.0f, dtype, flags, dx_hat, d_scale_sum, workspace, core_bytes, stream, &df);
  if (rc) return rc;
  cudaStream_t st = as_stream(stream);
  const int64_t n_blk = ceil_div(n_rows, 8);
  const int di = (int)d;
  const size_t smem = sizeof(float) * 8 * (size_t)d;
  if (smem > 48 * 1024) {   // rows too long to stage: the three separate passes
    if (df.n_split > 1) {
      const int64_t n4 = n_rows * d / 4;
      aux::sum_splits<<<(unsigned)ceil_div(n4, 256), 256, 0, st>>>(reinterpret_cast<const float4*>(df.parts), df.n_split, n4,
                                                                     reinterpret_cast<float4*>(dx_hat));
    }
    if (df.ds_pending) {
      float* part = reinterpret_cast<float*>(workspace);
      aux::rowdot_partials<<<(unsigned)n_blk, 256, 0, st>>>((const __nv_bfloat16*)x, rinv_x, dx_hat, n_rows, di, part);
      aux::reduce_scalar_partials_par<<<1, 256, 0, st>>>(part, (int)n_blk, 1.f, d_scale_sum);
    }
    CUDA_TRY(cudaGetLastError());
    return clipnce_normalize_backward(x_orig, in_dtype, rinv_x, dx_hat, grad_scale, n_rows, d, dx, out_dtype, stream);
  }
  float* ds_part = df.ds_pending ? reinterpret_cast<float*>(workspace) : nullptr;   // [n_blk] at the workspace start
  // 16-byte accesses when every row base is 4-element aligned (always so for the tensor-core path: d % 8 == 0)
  const bool v4 = d % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15u) == 0 && (reinterpret_cast<uintptr_t>(x_orig) & 15u) == 0 &&
                  (reinterpret_cast<uintptr_t>(dx) & 15u) == 0 && (reinterpret_cast<uintptr_t>(df.parts) & 15u) == 0;
  const aux::FinishSide side = finish_side(df.parts, df.n_split, n_rows, d, x, x_orig, rinv_x, dx, ds_part);
  if ((rc = launch_finish(&side, 1, n_rows, d, dtype, in_dtype, out_dtype, grad_scale, v4, st))) return rc;
  if (df.ds_pending) {
    aux::reduce_scalar_partials_par<<<1, 256, 0, st>>>(ds_part, (int)n_blk, 1.f, d_scale_sum);
    CUDA_TRY(cudaGetLastError());
  }
  return 0;
}

}  // extern "C"

// ---- several pair problems in one launch (pair::Group) ------------------------------------------------------------------
namespace {
struct GroupPlan {
  int fam, rows;            // kernel family (1 / 2); resident rows per CTA of the forward (128 / 64)
  int64_t n_pad, V;         // rows per member (n rounded up to 256); virtual rows of the forward: n_prob * n_pad
  int fwd_pairs, bwd_pairs; // row blocks per problem
  int steps;                // 256-column steps per problem
  int bwd_split_steps, bwd_n_split;
  size_t off_w, off_ds, off_sq, off_slab, bytes;   // backward layout of the workspace
  size_t fwd_bytes;
  int n_blk;
};

int group_plan(int n_members, int n_prob, int64_t n, int64_t d, int dtype, float scale, int flags, GroupPlan* pl) {
  memset(pl, 0, sizeof *pl);
  if (n_members < 1 || n_members > aux::FINISH_SIDES || n_prob < 1 || 2 * n_prob > pair::MAX_GROUP || n < 1 || d < 1)
    return fail(CLIPNCE_EINVAL, "group: 1..%d members, 1..%d problems", aux::FINISH_SIDES, pair::MAX_GROUP / 2);
  pl->fam = tc_family(dtype, d, scale, flags);
  if (!((pl->fam == 1 && pair_eligible(d)) || pl->fam == 2) || (flags & CLIPNCE_FLAG_UNBOUNDED)) { pl->fam = 0; return 0; }
  pl->rows = d <= 512 ? 128 : 64;
  pl->n_pad = round_up(n, 256);
  pl->V = (int64_t)n_prob * pl->n_pad;
  if ((int64_t)n_members * pl->n_pad > (1ll << 30) || 2 * pl->V > (1ll << 30)) { pl->fam = 0; return 0; }
  pl->fwd_pairs = (int)(pl->n_pad / (2 * pl->rows));
  pl->bwd_pairs = (int)(pl->n_pad / (2 * pair::BWD_ROWS));
  pl->steps = (int)(pl->n_pad / pair::STEP_J);
  // forward scratch: fixed shift -- column partials [2 fwd_pairs][V] + row partials [MAX_SPLIT][V];
  // true maxima -- (max, sum) row partials of both launches
  const size_t f1 = sizeof(float) * ((size_t)2 * pl->fwd_pairs + pair::MAX_SPLIT) * (size_t)pl->V;
  const size_t f2 = sizeof(float) * 4 * (size_t)pair::MAX_SPLIT * (size_t)pl->V;
  pl->fwd_bytes = round_up(pl->fam == 2 ? f1 + f2 + 1024 : f1, 256);   // family 2: the speculative sweep's partials + the exact sweeps'
  // backward: soft-max weights [2 V] | row-dot and |dx|^2 block partials | split slabs [n_split][2 V, d] f32 (<= 512 MiB)
  pl->n_blk = (int)ceil_div(pl->n_pad, 8);
  const size_t slab = sizeof(float) * 2 * (size_t)pl->V * (size_t)d;
  int max_split = (int)(((size_t)512 << 20) / slab);
  if (max_split < 1) max_split = 1;
  if (max_split > pair::MAX_SPLIT) max_split = pair::MAX_SPLIT;
  pl->bwd_split_steps = max_split >= 2 ? pick_split_steps(2 * n_prob * pl->bwd_pairs, pl->steps, max_split) : pl->steps;
  pl->bwd_n_split = (int)ceil_div(pl->steps, pl->bwd_split_steps);
  pl->off_w = 0;
  pl->off_ds = round_up(sizeof(float) * 2 * (size_t)pl->V, 256);
  pl->off_sq = pl->off_ds + round_up(sizeof(float) * (size_t)n_members * pl->n_blk, 256);
  pl->off_slab = pl->off_sq + round_up(sizeof(float) * (size_t)n_members * pl->n_blk, 256);
  pl->bytes = pl->off_slab + (size_t)pl->bwd_n_split * slab;
  if (pl->fwd_bytes > pl->bytes) pl->bytes = pl->fwd_bytes;
  return 0;
}

int group_members_ok(int n_members, int n_prob, const int* xm, const int* ym) {
  if (!xm || !ym) return fail(CLIPNCE_EINVAL, "group: null member list");
  for (int k = 0; k < n_prob; ++k)
    if (xm[k] < 0 || xm[k] >= n_members || ym[k] < 0 || ym[k] >= n_members)
      return fail(CLIPNCE_EINVAL, "group: problem %d names a member outside 0..%d", k, n_members - 1);
  return 0;
}
}  // namespace

extern "C" {

int clipnce_group_workspace_bytes(int n_members, int n_prob, int64_t n, int64_t d, int dtype, float scale, int flags,
                                  size_t* out) {
  if (!out) return fail(CLIPNCE_EINVAL, "group_workspace_bytes: null pointer");
  GroupPlan pl;
  int rc = group_plan(n_members, n_prob, n, d, dtype, scale, flags, &pl);
  if (rc) return rc;
  *out = pl.fam ? pl.bytes : 0;
  return 0;
}

int clipnce_group_forward(const void* stack, const float* rinv, int n_members, int n_prob, const int* x_member,
                          const int* y_member, int64_t n, int64_t d, float scale, const float* scale_dev, int dtype,
                          int flags, float* stat_m, float* stat_l, float* diag, float* loss, void* workspace,
                          size_t workspace_bytes, void* stream) {
  if (!stack || !rinv || !stat_m || !stat_l || !diag || !loss || !workspace)
    return fail(CLIPNCE_EINVAL, "group_forward: null pointer");
  if (!std::isfinite(scale)) return fail(CLIPNCE_EINVAL, "group_forward: scale is not finite");
  GroupPlan pl;
  int rc = group_plan(n_members, n_prob, n, d, dtype, scale, flags, &pl);
  if (rc) return rc;
  if (!pl.fam) return fail(CLIPNCE_EUNSUPPORTED, "group_forward: shape / type not served (bf16, d %% 128 == 0, d <= 768)");
  if ((rc = group_members_ok(n_members, n_prob, x_member, y_member))) return rc;
  if (workspace_bytes < pl.fwd_bytes) return fail(CLIPNCE_EWORKSPACE, "group_forward: workspace %zu < %zu", workspace_bytes, pl.fwd_bytes);
  if (!aligned16(stack)) return fail(CLIPNCE_EINVAL, "group_forward: the stack must be 16-byte aligned");
  if ((rc = check_device_sm100())) return rc;
  cudaStream_t st = as_stream(stream);
  const int64_t V = pl.V;

  pair::FwdParams p;
  memset(&p, 0, sizeof p);
  p.n_rows = (int)V; p.n_cols = (int)V; p.d = (int)d;
  p.nkc = (int)ceil_div(d, 64); p.n_steps = pl.steps;
  p.diag_offset = 0; p.scale = scale; p.scale_dev = scale_dev;
  p.rinv_x = rinv; p.rinv_y = rinv;
  p.n_pairs = n_prob * pl.fwd_pairs;
  p.split_steps = pick_split_steps(p.n_pairs, p.n_steps, pair::MAX_SPLIT);
  const int n_split = (int)ceil_div(p.n_steps, p.split_steps);
  p.grp.n_prob = n_prob; p.grp.pairs_per_prob = pl.fwd_pairs; p.grp.steps_per_prob = pl.steps; p.grp.n_valid = (int)n;
  p.grp.stack_rows = (int)(n_members * pl.n_pad);
  float* wsf = reinterpret_cast<float*>(workspace);

  const int* gate = nullptr;
  size_t exact_off = 0;   // floats: where the exact sweeps' partials start
  if (pl.fam == 2 && env_int("CLIPNCE_NO_SPECULATE", 0) == 0) {
    // bounded logits: one fixed-shift sweep with the shift lowered to s - 72, the exact sweeps gated on a device flag
    // (see clipnce_forward)
    constexpr float kOff = 72.f;
    const float thr = 1.2e-38f * 1e6f * (float)n;
    for (int k = 0; k < n_prob; ++k) {
      p.grp.xshift[k] = (int)((x_member[k] - k) * pl.n_pad);
      p.grp.yshift[k] = (int)((y_member[k] - k) * pl.n_pad);
    }
    p.diag = diag;
    p.col_ld = V;
    p.shift_off = kOff;
    const int n_part = 2 * pl.fwd_pairs;
    p.col_part = wsf;
    p.row_part = wsf + (size_t)n_part * (size_t)V;
    exact_off = (size_t)round_up((int64_t)(((size_t)n_part + (size_t)n_split) * (size_t)V), 64) + 64;
    int* flag = reinterpret_cast<int*>(wsf + exact_off - 64);
    CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(int), st));
    rc = pl.rows == 128 ? launch_pair_fwd<128>(stack, stack, p, st) : launch_pair_fwd<64>(stack, stack, p, st);
    if (rc) return rc;
    aux::reduce_shifted_partials<<<(unsigned)ceil_div(V, 256), 256, 0, st>>>(p.col_part, n_part, V, V, scale, scale_dev, kOff, thr,
                                                                              stat_m + V, stat_l + V, flag, pl.n_pad, n);
    aux::reduce_shifted_partials<<<(unsigned)ceil_div(V, 256), 256, 0, st>>>(p.row_part, n_split, V, V, scale, scale_dev, kOff, thr,
                                                                              stat_m, stat_l, flag, pl.n_pad, n);
    CUDA_TRY(cudaGetLastError());
    p.shift_off = 0.f; p.col_part = nullptr; p.col_ld = 0;
    gate = flag;
  }
  if (pl.fam == 2) {   // true maxima: row statistics of (x, y), then of (y, x) = the column statistics
    p.gate = gate;
    for (int side = 0; side < 2; ++side) {
      for (int k = 0; k < n_prob; ++k) {
        const int res = side == 0 ? x_member[k] : y_member[k], str = side == 0 ? y_member[k] : x_member[k];
        p.grp.xshift[k] = (int)((res - k) * pl.n_pad);
        p.grp.yshift[k] = (int)((str - k) * pl.n_pad);
      }
      p.diag = side == 0 ? diag : nullptr;
      p.row_part_m = wsf + exact_off + (size_t)side * 2 * (size_t)n_split * (size_t)V;
      p.row_part = p.row_part_m + (size_t)n_split * (size_t)V;
      rc = pl.rows == 128 ? launch_pair_fwd<128, 2>(stack, stack, p, st) : launch_pair_fwd<64, 2>(stack, stack, p, st);
      if (rc) return rc;
      aux::reduce_ml_partials<<<(unsigned)ceil_div(V, 256), 256, 0, st>>>(p.row_part_m, p.row_part, n_split, V, V,
                                                                           stat_m + side * V, stat_l + side * V, gate);
      CUDA_TRY(cudaGetLastError());
    }
  } else {
    for (int k = 0; k < n_prob; ++k) {
      p.grp.xshift[k] = (int)((x_member[k] - k) * pl.n_pad);
      p.grp.yshift[k] = (int)((y_member[k] - k) * pl.n_pad);
    }
    p.diag = diag;
    p.col_ld = V;
    const int n_part = 2 * pl.fwd_pairs;
    p.col_part = wsf;
    p.row_part = wsf + (size_t)n_part * (size_t)V;
    rc = pl.rows == 128 ? launch_pair_fwd<128>(stack, stack, p, st) : launch_pair_fwd<64>(stack, stack, p, st);
    if (rc) return rc;
    aux::reduce_col_partials<<<(unsigned)ceil_div(V, 256), 256, 0, st>>>(p.col_part, n_part, V, V, scale, scale_dev,
                                                                          stat_m + V, stat_l + V);
    aux::reduce_col_partials<<<(unsigned)ceil_div(V, 256), 256, 0, st>>>(p.row_part, n_split, V, V, scale, scale_dev,
                                                                          stat_m, stat_l);
    CUDA_TRY(cudaGetLastError());
  }
  aux::loss_reduce_group<<<1, 1024, 0, st>>>(stat_m, stat_l, diag, n_prob, n, pl.n_pad, loss);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_group_backward(const void* stack, const float* rinv, int n_members, int n_prob, const int* x_member,
                           const int* y_member, int64_t n, int64_t d, float scale, const float* scale_dev,
                           const float* stat_m, const float* stat_l, int dtype, int flags, const void* stack_orig,
                           int in_dtype, const float* grad_scale, void* d_stack, int out_dtype, float* d_scale_sum,
                           float* grad_sumsq, void* workspace, size_t workspace_bytes, void* stream) {
  if (!stack || !rinv || !stat_m || !stat_l || !stack_orig || !d_stack || !workspace)
    return fail(CLIPNCE_EINVAL, "group_backward: null pointer");
  if ((in_dtype != CLIPNCE_BF16 && in_dtype != CLIPNCE_F32) || (out_dtype != CLIPNCE_BF16 && out_dtype != CLIPNCE_F32))
    return fail(CLIPNCE_EINVAL, "group_backward: bad dtype");
  if (in_dtype == dtype && stack_orig != stack) return fail(CLIPNCE_EINVAL, "group_backward: stack_orig of the compute type must be the stack itself");
  if (!std::isfinite(scale)) return fail(CLIPNCE_EINVAL, "group_backward: scale is not finite");
  GroupPlan pl;
  int rc = group_plan(n_members, n_prob, n, d, dtype, scale, flags, &pl);
  if (rc) return rc;
  if (!pl.fam) return fail(CLIPNCE_EUNSUPPORTED, "group_backward: shape / type not served (bf16, d %% 128 == 0, d <= 768)");
  if ((rc = group_members_ok(n_members, n_prob, x_member, y_member))) return rc;
  if (workspace_bytes < pl.bytes) return fail(CLIPNCE_EWORKSPACE, "group_backward: workspace %zu < %zu", workspace_bytes, pl.bytes);
  if (!aligned16(stack) || !aligned16(stack_orig) || !aligned16(d_stack))
    return fail(CLIPNCE_EINVAL, "group_backward: buffers must be 16-byte aligned");
  if (sizeof(float) * 8 * (size_t)d > 48 * 1024) return fail(CLIPNCE_EUNSUPPORTED, "group_backward: d too large");
  if ((rc = check_device_sm100())) return rc;
  cudaStream_t st = as_stream(stream);
  const int64_t V = pl.V;
  char* ws = reinterpret_cast<char*>(workspace);
  float* w = reinterpret_cast<float*>(ws + pl.off_w);
  float* ds_part = reinterpret_cast<float*>(ws + pl.off_ds);
  float* sq_part = reinterpret_cast<float*>(ws + pl.off_sq);
  float* slabs = reinterpret_cast<float*>(ws + pl.off_slab);

  // w = 1 / (2 n l) for row and column sums alike (entries of the padding are never read)
  aux::softmax_weights<<<(unsigned)ceil_div(2 * V, 256), 256, 0, st>>>(stat_l, 2 * V, 1.0f / (2.0f * (float)n), w);
  CUDA_TRY(cudaGetLastError());

  // ONE sweep launch over 2 n_prob virtual problems: k < n_prob the X side of problem k (rows of x_member[k] resident),
  // k >= n_prob the Y side of problem k - n_prob (rows of y_member resident; the column statistics play the row role)
  pair::BwdParams p;
  memset(&p, 0, sizeof p);
  p.n_rows = (int)(2 * V); p.n_cols = (int)(2 * V); p.d = (int)d;
  p.nkc = (int)ceil_div(d, 64); p.nq2 = (int)ceil_div(d, 256); p.n_steps = pl.steps;
  p.diag_offset = 0; p.scale = scale; p.scale_dev = scale_dev; p.diag_w = 1.0f / (float)n; p.grad_out = 1.0f;
  p.rinv_x = rinv; p.rinv_y = rinv; p.row_m_in = stat_m; p.row_w = w; p.col_m_in = stat_m; p.col_w = w;
  p.n_pairs = 2 * n_prob * pl.bwd_pairs;
  p.split_steps = pl.bwd_split_steps;
  p.dx = slabs;
  p.grp.n_prob = 2 * n_prob; p.grp.pairs_per_prob = pl.bwd_pairs; p.grp.steps_per_prob = pl.steps; p.grp.n_valid = (int)n;
  p.grp.stack_rows = (int)(n_members * pl.n_pad);
  p.grp.gscale = grad_scale; p.grp.gmod = n_prob;
  // the finishing pass, one side per member: the gradient of member m's normalised rows is the sum of the slabs of every
  // virtual problem in which m was the resident operand (its X sides and its Y sides).  Every pair's sum G.S appears once
  // per side in the row dots: reduce_group_scalars halves it.
  aux::FinishSide sides[aux::FINISH_SIDES];
  memset(sides, 0, sizeof sides);
  for (int m = 0; m < n_members; ++m) {
    aux::FinishSide& s = sides[m];
    s.n_split = pl.bwd_n_split; s.slab = 2 * V * d; s.row0 = m * pl.n_pad; s.n = n;
    s.xc = stack; s.xo = stack_orig; s.rinv = rinv; s.dx = d_stack;
    s.ds_part = ds_part + (size_t)m * pl.n_blk; s.sq_part = sq_part + (size_t)m * pl.n_blk;
  }
  for (int k = 0; k < 2 * n_prob; ++k) {
    const int q = k % n_prob;
    const int res = k < n_prob ? x_member[q] : y_member[q], str = k < n_prob ? y_member[q] : x_member[q];
    p.grp.xshift[k] = (int)((res - k) * pl.n_pad);
    p.grp.yshift[k] = (int)((str - k) * pl.n_pad);
    p.grp.cshift[k] = (int)(k < n_prob ? V : -V);
    aux::FinishSide& s = sides[res];
    if (s.n_contrib >= aux::FINISH_CONTRIB) return fail(CLIPNCE_EINVAL, "group_backward: too many problems share member %d", res);
    s.parts[s.n_contrib++] = slabs + (size_t)k * pl.n_pad * d;
  }
  if ((rc = pl.fam == 2 ? launch_pair_bwd<true>(stack, stack, p, st) : launch_pair_bwd<false>(stack, stack, p, st))) return rc;

  if ((rc = launch_finish(sides, n_members, pl.n_pad, d, CLIPNCE_BF16, in_dtype, out_dtype, nullptr, true, st))) return rc;
  if (d_scale_sum || grad_sumsq) {
    aux::reduce_group_scalars<<<1 + n_members, 256, 0, st>>>(ds_part, sq_part, n_members, pl.n_blk, d_scale_sum, grad_sumsq);
    CUDA_TRY(cudaGetLastError());
  }
  return 0;
}

}  // extern "C"

// ---- two-sided backward (kernels_pair2.cuh) ----------------------------------------------------------------------------
namespace {
struct Bwd2Plan {
  int P, Q, n_rb, n_seg, seg_steps, n_items, n_rounds, n_steps, n_half, depth, stages_a, stages_b, stages_c, smem;
  size_t off_flags, off_ring, off_dxh, off_dyh, off_part, bytes;
};

bool bwd2_device_ok() {   // every CTA pair of the persistent grid must be resident at once
  if (env_int("CLIPNCE_NO_BWD2", 0) != 0) return false;   // test hook: the two-sweep path instead
  // the occupancy query below counts on the raised shared-memory limit
  if (allow_smem(pair2::bwd2_kernel<false>, pair::SMEM_LIMIT) || allow_smem(pair2::bwd2_kernel<true>, pair::SMEM_LIMIT)) {
    cudaGetLastError();
    return false;
  }
  static const bool ok = [] {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.gridDim = dim3(2 * pair_slots());
    cfg.blockDim = dim3(pair2::THREADS);
    cfg.dynamicSmemBytes = pair::SMEM_LIMIT;
    int n = 0, n2 = 0;
    if (cudaOccupancyMaxActiveClusters(&n, pair2::bwd2_kernel<false>, &cfg) != cudaSuccess ||
        cudaOccupancyMaxActiveClusters(&n2, pair2::bwd2_kernel<true>, &cfg) != cudaSuccess) {
      cudaGetLastError();
      return false;
    }
    return n >= pair_slots() && n2 >= pair_slots();
  }();
  return ok;
}

// world == 0: one GPU (n_rows == n_cols, every column segment stays local); world >= 2: row-sharded step, the rank's
// n_rows = n_cols / world rows against all columns, one segment per owner rank.
bool bwd2_plan(int64_t n_rows, int64_t n_cols, int64_t d, int dtype, float scale, int flags, int world, Bwd2Plan* pl) {
  // family 1 (fixed shift) or family 2 with bounded logits (scales up to the clamp at 100); not the un-normalised queue
  // columns (extra columns are not served at all: positives on the diagonal of a square / row-sharded batch only)
  const int fam = tc_family(dtype, d, scale, flags);
  if (!((fam == 1 || fam == 2) && pair_eligible(d)) || (flags & CLIPNCE_FLAG_UNBOUNDED)) return false;
  if (world == 1 || world < 0 || world > pair2::MAX_WORLD) return false;
  if (world == 0 ? n_rows != n_cols : n_rows * world != n_cols) return false;
  // below this the items do not fill the producer pairs; measured on one GPU, d = 512 (tools/run_bwd2_threshold.sh): 12288 rows
  // 0.571 ms per step against 0.692 with two sweeps, 8192 rows 0.329 against 0.307 (CLIPNCE_BWD2_MIN_N: test hook)
  const int64_t min_n = env_int("CLIPNCE_BWD2_MIN_N", 12288);
  if (n_rows % 128 != 0 || n_cols % 256 != 0 || n_rows * n_cols < min_n * min_n || n_cols > (1ll << 22)) return false;
  if (world >= 2 && (n_cols / world) % 256 != 0) return false;
  const int slots = pair_slots();
  if (slots < 8) return false;
  pl->n_rb = (int)(n_rows / 128);
  pl->n_steps = (int)(n_cols / 256);
  pl->n_half = (int)ceil_div(d, 256);
  // Split of the CTA pairs into producers and consumers, and (one GPU) the number of column segments.  Model, in units of
  // one producer step: a producer item costs seg_steps + 1 (accumulator drain, reload of the resident rows, pipeline
  // refill), the consumers work through one tile unit per producer tile at `r` times a producer's rate (measured on B200,
  // N = 65536, d = 512: P = 48..52 within 1 %), every segment beyond the first costs a pass over an [n_rows, d] fp32 slab.
  // CLIPNCE_BWD2_P / CLIPNCE_BWD2_SEG (test hooks) force the split and the number of segments.
  const int forced_p = (int)env_int("CLIPNCE_BWD2_P", 0);
  const int forced_seg = (int)env_int("CLIPNCE_BWD2_SEG", 0);
  constexpr double r = 1.0;
  double best_t = 1e300;
  int best_p = 0, best_seg = 0;
  for (int n_seg = 1; n_seg <= 8; n_seg *= 2) {
    int ns = world >= 2 ? world : n_seg;
    if (world == 0 && forced_seg >= 1) ns = forced_seg;
    if (pl->n_steps % ns != 0) continue;
    const int seg_steps = pl->n_steps / ns;
    if (seg_steps < 8 && ns > 1 && world == 0 && forced_seg < 1) continue;
    const int64_t n_items = (int64_t)pl->n_rb * ns;
    const double slab_steps = (double)(ns - 1) * (double)n_rows * (double)d * 8.0 / 3e12 / 3.9e-6;
    const bool force = forced_p >= 1 && forced_p <= slots - 1;
    for (int Pe = force ? forced_p : slots / 2; Pe <= (force ? forced_p : slots - 2); ++Pe) {
      const int Q = slots - Pe;
      const double tp = (double)ceil_div(n_items, Pe) * ((double)seg_steps + 1.0);
      const double tc_ = (double)n_items * (double)seg_steps / ((double)Q * 2.0 * r);
      // measured (one GPU, N = 65536, d = 512): 1 segment 11.9 ms, 2 (auto) 12.1, 4 12.5 -- the extra slabs and item
      // prologues cost more than the fuller rounds return, so more segments must win by a clear margin
      const double t = ((tp > tc_ ? tp : tc_) + slab_steps) * (world == 0 && ns > 1 ? 1.08 : 1.0);
      if (t < best_t - 1e-9) { best_t = t; best_p = Pe; best_seg = ns; }
    }
    if (world >= 2 || forced_seg >= 1) break;
  }
  if (best_p == 0) return false;
  pl->P = best_p;
  pl->Q = slots - best_p;
  pl->n_seg = best_seg;
  pl->seg_steps = pl->n_steps / best_seg;
  pl->n_items = pl->n_rb * best_seg;
  pl->n_rounds = (int)ceil_div(pl->n_items, pl->P);
  pl->depth = pair2::RING_DEPTH;
  const int nkc = (int)(d / 64);
  const int total = (pair::SMEM_LIMIT - pair2::producer_smem(nkc, 0)) / pair::STAGE_BYTES;
  if (total < 4) return false;
  auto cap = [](int v) { return v > pair2::MAXS ? pair2::MAXS : v; };
  pl->stages_b = cap(total / 2);
  pl->stages_a = cap(total - total / 2);
  pl->stages_c = cap((pair::SMEM_LIMIT - pair2::consumer_smem(0)) / pair2::C_STAGE);
  const int ps = pair2::producer_smem(nkc, pl->stages_a + pl->stages_b), cs = pair2::consumer_smem(pl->stages_c);
  pl->smem = ps > cs ? ps : cs;
  size_t off = 0;
  auto region = [&](size_t bytes) { const size_t o = off; off = (size_t)round_up((int64_t)(off + bytes), 256); return o; };
  pl->off_flags = region(sizeof(uint32_t) * 2 * (size_t)pl->n_rounds * (size_t)pl->seg_steps);
  pl->off_ring = region((size_t)pl->depth * (size_t)pl->P * 128 * 256 * 2);
  pl->off_dxh = region(sizeof(float) * (size_t)pl->n_seg * (size_t)n_rows * (size_t)d);
  pl->off_dyh = region(sizeof(float) * (size_t)n_cols * (size_t)d);
  pl->off_part = region(sizeof(float) * (size_t)ceil_div(n_rows > n_cols ? n_rows : n_cols, 8));
  pl->bytes = off;
  return true;
}

int bwd2_launch(const Bwd2Plan& pl, const void* x, const void* y, const float* rinv_x, const float* rinv_y, int64_t n_rows,
                int64_t n_cols, int64_t d, int64_t diag_offset, float scale, const float* scale_dev, const float* row_m,
                const float* row_w, const float* col_m, const float* col_w, float diag_w, char* ws, float* const* dy_peer,
                int world, cudaStream_t st) {
  uint32_t* flags_dev = reinterpret_cast<uint32_t*>(ws + pl.off_flags);
  const size_t n_flags = (size_t)pl.n_rounds * (size_t)pl.seg_steps;
  CUDA_TRY(cudaMemsetAsync(flags_dev, 0, sizeof(uint32_t) * 2 * n_flags, st));
  pair2::Params p;
  memset(&p, 0, sizeof p);
  p.n_rows = (int)n_rows; p.n_cols = (int)n_cols; p.d = (int)d;
  p.nkc = (int)(d / 64); p.nq2 = (int)ceil_div(d, 256); p.n_half = pl.n_half;
  p.nsbuf = p.nq2 <= 2 ? 2 : 1;   // 128 nq2 accumulator columns + 128 per logits buffer <= 512
  p.n_rb = pl.n_rb; p.n_seg = pl.n_seg; p.seg_steps = pl.seg_steps; p.n_items = pl.n_items; p.n_rounds = pl.n_rounds;
  p.P = pl.P; p.Q = pl.Q; p.depth = pl.depth;
  p.stages_a = pl.stages_a; p.stages_b = pl.stages_b; p.stages_c = pl.stages_c;
  p.diag_offset = diag_offset; p.scale = scale; p.scale_dev = scale_dev; p.diag_w = diag_w;
  p.rinv_x = rinv_x; p.rinv_y = rinv_y; p.row_m = row_m; p.row_w = row_w; p.col_m = col_m; p.col_w = col_w;
  p.dx = reinterpret_cast<float*>(ws + pl.off_dxh);
  p.dy = reinterpret_cast<float*>(ws + pl.off_dyh);
  p.world = world;
  for (int s = 0; s < world; ++s) p.dy_peer[s] = dy_peer[s];
  p.ready = flags_dev; p.done = flags_dev + n_flags;
  CUtensorMap tx, ty, tyg, tg;
  int rc;
  if ((rc = make_tmap(&tx, x, d, n_rows, d, pair2::ROWS))) return rc;
  if ((rc = make_tmap(&ty, y, d, n_cols, d, 128))) return rc;
  if ((rc = make_tmap(&tyg, y, d, n_cols, d, 64))) return rc;
  if ((rc = make_tmap(&tg, ws + pl.off_ring, 256, (int64_t)pl.depth * pl.P * 128, 256, 64))) return rc;
  auto kern = tc_family(CLIPNCE_BF16, d, scale, 0) == 2 ? pair2::bwd2_kernel<true> : pair2::bwd2_kernel<false>;
  if ((rc = allow_smem(kern, pair::SMEM_LIMIT))) return rc;
  kern<<<2 * (pl.P + pl.Q), pair2::THREADS, pl.smem, st>>>(tx, ty, tyg, tg, p);
  CUDA_TRY(cudaGetLastError());
  return 0;
}
}  // namespace

extern "C" {

int clipnce_backward_both_workspace_bytes(int64_t n_rows, int64_t n_cols, int64_t d, int dtype, float scale, int flags,
                                          int world, size_t* out) {
  if (!out) return fail(CLIPNCE_EINVAL, "backward_both_workspace_bytes: null pointer");
  Bwd2Plan pl;
  *out = (n_rows >= 1 && n_cols >= 1 && d >= 1 && bwd2_plan(n_rows, n_cols, d, dtype, scale, flags, world, &pl) &&
          check_device_sm100() == 0 && bwd2_device_ok()) ? pl.bytes : 0;
  return 0;
}

int clipnce_backward_both_dx(const void* x, const void* y, const float* rinv_x, const float* rinv_y, int64_t n,
                             int64_t d, float scale, const float* scale_dev, const float* row_m, const float* row_w,
                             const float* col_m, const float* col_w, float diag_w, int dtype, int flags,
                             const void* x_orig, const void* y_orig, int in_dtype, const float* grad_scale, void* dx,
                             void* dy, int out_dtype, float* d_scale_sum, void* workspace, size_t workspace_bytes,
                             void* stream) {
  if (!x || !y || !rinv_x || !rinv_y || !row_m || !row_w || !col_m || !col_w || !x_orig || !y_orig || !dx || !dy || !workspace)
    return fail(CLIPNCE_EINVAL, "backward_both_dx: null pointer");
  if ((in_dtype != CLIPNCE_BF16 && in_dtype != CLIPNCE_F32) || (out_dtype != CLIPNCE_BF16 && out_dtype != CLIPNCE_F32))
    return fail(CLIPNCE_EINVAL, "backward_both_dx: bad dtype");
  if (in_dtype == dtype && (x_orig != x || y_orig != y))
    return fail(CLIPNCE_EINVAL, "backward_both_dx: x_orig / y_orig of the compute type must be x / y themselves");
  if (!aligned16(x) || !aligned16(y) || !aligned16(workspace)) return fail(CLIPNCE_EINVAL, "backward_both_dx: operands must be 16-byte aligned");
  int rc = check_device_sm100();
  if (rc) return rc;
  Bwd2Plan pl;
  if (!bwd2_plan(n, n, d, dtype, scale, flags, 0, &pl) || !bwd2_device_ok())
    return fail(CLIPNCE_EUNSUPPORTED, "backward_both_dx: shape not served (see clipnce_backward_both_workspace_bytes)");
  if (workspace_bytes < pl.bytes) return fail(CLIPNCE_EWORKSPACE, "backward_both_dx: workspace %zu < %zu", workspace_bytes, pl.bytes);
  cudaStream_t st = as_stream(stream);
  char* ws = reinterpret_cast<char*>(workspace);
  if ((rc = bwd2_launch(pl, x, y, rinv_x, rinv_y, n, n, d, 0, scale, scale_dev, row_m, row_w, col_m, col_w, diag_w, ws, nullptr,
                        0, st)))
    return rc;
  // tails: segment sum + row dots (sum G.S, side A only) + normalise backward, one pass per side
  float* ds_part = reinterpret_cast<float*>(ws + pl.off_part);
  const aux::FinishSide sx = finish_side(reinterpret_cast<float*>(ws + pl.off_dxh), pl.n_seg, n, d, x, x_orig, rinv_x, dx,
                                         d_scale_sum ? ds_part : nullptr);
  const aux::FinishSide sy = finish_side(reinterpret_cast<float*>(ws + pl.off_dyh), 1, n, d, y, y_orig, rinv_y, dy, nullptr);
  if ((rc = launch_finish(&sx, 1, n, d, CLIPNCE_BF16, in_dtype, out_dtype, grad_scale, true, st))) return rc;
  if ((rc = launch_finish(&sy, 1, n, d, CLIPNCE_BF16, in_dtype, out_dtype, grad_scale, true, st))) return rc;
  if (d_scale_sum) {
    aux::reduce_scalar_partials_par<<<1, 256, 0, st>>>(ds_part, (int)ceil_div(n, 8), 1.f, d_scale_sum);
    CUDA_TRY(cudaGetLastError());
  }
  return 0;
}

int clipnce_backward_both_sharded(const void* x, const void* y, const float* rinv_x, const float* rinv_y, int64_t n_rows,
                                  int64_t n_cols, int64_t d, int64_t diag_offset, float scale, const float* scale_dev,
                                  const float* row_m, const float* row_w, const float* col_m, const float* col_w,
                                  float diag_w, int dtype, int flags, void* const* peer_base, int world, int rank,
                                  int64_t slots_offset, void* workspace, size_t workspace_bytes, void* stream) {
  if (!x || !y || !rinv_x || !rinv_y || !row_m || !row_w || !col_m || !col_w || !workspace || !peer_base)
    return fail(CLIPNCE_EINVAL, "backward_both_sharded: null pointer");
  if (!aligned16(x) || !aligned16(y) || !aligned16(workspace)) return fail(CLIPNCE_EINVAL, "backward_both_sharded: operands must be 16-byte aligned");
  if (world < 2 || world > pair2::MAX_WORLD || rank < 0 || rank >= world || slots_offset < 0 || slots_offset % 16 != 0)
    return fail(CLIPNCE_EINVAL, "backward_both_sharded: bad world / rank / slots_offset");
  if (diag_offset != (int64_t)rank * n_rows) return fail(CLIPNCE_EINVAL, "backward_both_sharded: diag_offset must be rank * n_rows");
  int rc = check_device_sm100();
  if (rc) return rc;
  Bwd2Plan pl;
  if (!bwd2_plan(n_rows, n_cols, d, dtype, scale, flags, world, &pl) || !bwd2_device_ok())
    return fail(CLIPNCE_EUNSUPPORTED, "backward_both_sharded: shape not served (see clipnce_backward_both_workspace_bytes)");
  if (workspace_bytes < pl.bytes) return fail(CLIPNCE_EWORKSPACE, "backward_both_sharded: workspace %zu < %zu", workspace_bytes, pl.bytes);
  char* ws = reinterpret_cast<char*>(workspace);
  float* dy_peer[pair2::MAX_WORLD];
  for (int s = 0; s < world; ++s) {   // this rank's slot in rank s's buffer: [n_rows, d] f32 (n_rows == columns per owner)
    if (!peer_base[s] || !aligned16(peer_base[s])) return fail(CLIPNCE_EINVAL, "backward_both_sharded: peer buffer %d is null or unaligned", s);
    dy_peer[s] = reinterpret_cast<float*>(reinterpret_cast<char*>(peer_base[s]) + slots_offset) + (size_t)rank * (size_t)n_rows * (size_t)d;
  }
  return bwd2_launch(pl, x, y, rinv_x, rinv_y, n_rows, n_cols, d, diag_offset, scale, scale_dev, row_m, row_w, col_m, col_w,
                     diag_w, ws, dy_peer, world, as_stream(stream));
}

int clipnce_finish_sharded(const void* x, const void* x_orig, const float* rinv_x, void* dx, const void* y_local,
                           const void* y_orig, const float* rinv_y_local, void* dy, const float* slots, int64_t n_rows,
                           int64_t n_cols, int64_t d, int dtype, float scale, int flags, int world, int x_in_dtype,
                           int x_out_dtype, int y_in_dtype, int y_out_dtype, const float* grad_scale, float* d_scale_sum,
                           void* workspace, size_t workspace_bytes, void* stream) {
  if (!x || !x_orig || !rinv_x || !dx || !y_local || !y_orig || !rinv_y_local || !dy || !slots || !workspace)
    return fail(CLIPNCE_EINVAL, "finish_sharded: null pointer");
  for (int t : {x_in_dtype, x_out_dtype, y_in_dtype, y_out_dtype})
    if (t != CLIPNCE_BF16 && t != CLIPNCE_F32) return fail(CLIPNCE_EINVAL, "finish_sharded: bad dtype");
  if ((x_in_dtype == dtype && x_orig != x) || (y_in_dtype == dtype && y_orig != y_local))
    return fail(CLIPNCE_EINVAL, "finish_sharded: x_orig / y_orig of the compute type must be x / y_local themselves");
  Bwd2Plan pl;
  if (!bwd2_plan(n_rows, n_cols, d, dtype, scale, flags, world, &pl))
    return fail(CLIPNCE_EUNSUPPORTED, "finish_sharded: shape not served by the two-sided backward");
  if (workspace_bytes < pl.bytes) return fail(CLIPNCE_EWORKSPACE, "finish_sharded: workspace %zu < %zu", workspace_bytes, pl.bytes);
  cudaStream_t st = as_stream(stream);
  char* ws = reinterpret_cast<char*>(workspace);
  float* ds_part = reinterpret_cast<float*>(ws + pl.off_part);
  // side 0 sums the segment slabs of dA_hat, side 1 the ranks' slots of dB_hat; sides of the same types share ONE launch
  // instead of queueing behind each other
  const aux::FinishSide sides[2] = {
      finish_side(reinterpret_cast<float*>(ws + pl.off_dxh), pl.n_seg, n_rows, d, x, x_orig, rinv_x, dx, d_scale_sum ? ds_part : nullptr),
      finish_side(slots, world, n_rows, d, y_local, y_orig, rinv_y_local, dy, nullptr)};
  int rc;
  if (x_in_dtype == y_in_dtype && x_out_dtype == y_out_dtype) {
    if ((rc = launch_finish(sides, 2, n_rows, d, CLIPNCE_BF16, x_in_dtype, x_out_dtype, grad_scale, true, st))) return rc;
  } else {
    if ((rc = launch_finish(&sides[0], 1, n_rows, d, CLIPNCE_BF16, x_in_dtype, x_out_dtype, grad_scale, true, st))) return rc;
    if ((rc = launch_finish(&sides[1], 1, n_rows, d, CLIPNCE_BF16, y_in_dtype, y_out_dtype, grad_scale, true, st))) return rc;
  }
  if (d_scale_sum) {
    aux::reduce_scalar_partials_par<<<1, 256, 0, st>>>(ds_part, (int)ceil_div(n_rows, 8), 1.f, d_scale_sum);
    CUDA_TRY(cudaGetLastError());
  }
  return 0;
}

}  // extern "C"

namespace {
int topk_kt(int k) { return k <= 1 ? 1 : (k <= 10 ? 10 : 16); }
struct TopkPlan {
  int n_pairs, n_steps, split_steps, n_split, kt;
  size_t cand_elems;
};
int topk_plan(int64_t n_q, int64_t n_lib, int64_t d, int k, int dtype, TopkPlan* pl) {
  if (n_q < 1 || n_lib < 1 || n_lib >= (1ll << 31) || n_q >= (1ll << 31)) return fail(CLIPNCE_EINVAL, "topk: bad shape");
  if (dtype != CLIPNCE_BF16 || d % 128 != 0 || d < 128 || d > 512 || k < 1 || k > 16)
    return fail(CLIPNCE_EUNSUPPORTED, "topk: served for bf16, d in {128,256,384,512}, 1 <= k <= 16 (got dtype %d, d %lld, k %d)",
                dtype, (long long)d, k);
  pl->kt = topk_kt(k);
  pl->n_pairs = (int)ceil_div(n_q, 256);
  pl->n_steps = (int)ceil_div(n_lib, pair::STEP_J);
  pl->split_steps = pick_split_steps(pl->n_pairs, pl->n_steps, pair::MAX_SPLIT);
  pl->n_split = (int)ceil_div(pl->n_steps, pl->split_steps);
  pl->cand_elems = (size_t)pl->n_split * 4 * (size_t)n_q * (size_t)pl->kt;
  return 0;
}
}  // namespace

extern "C" {

int clipnce_topk_workspace_bytes(int64_t n_q, int64_t n_lib, int64_t d, int k, int dtype, size_t* out) {
  if (!out) return fail(CLIPNCE_EINVAL, "topk_workspace_bytes: null pointer");
  TopkPlan pl;
  int rc = topk_plan(n_q, n_lib, d, k, dtype, &pl);
  if (rc) return rc;
  *out = pl.cand_elems * 8 + sizeof(int) * (size_t)n_q + 256;
  return 0;
}

int clipnce_topk(const void* q, const void* lib, const float* rinv_q, const float* rinv_lib, int64_t n_q, int64_t n_lib,
                 int64_t d, int64_t col_offset, int k, int dtype, float* out_score, int64_t* out_idx, void* workspace,
                 size_t workspace_bytes, void* stream) {
  if (!q || !lib || !rinv_q || !rinv_lib || !out_score || !out_idx || !workspace) return fail(CLIPNCE_EINVAL, "topk: null pointer");
  if (!aligned16(q) || !aligned16(lib)) return fail(CLIPNCE_EINVAL, "topk: operands must be 16-byte aligned");
  if (col_offset < 0 || col_offset + n_lib >= (1ll << 31)) return fail(CLIPNCE_EINVAL, "topk: library index range must fit int32");
  TopkPlan pl;
  int rc = topk_plan(n_q, n_lib, d, k, dtype, &pl);
  if (rc) return rc;
  if ((rc = check_device_sm100())) return rc;
  const size_t need = pl.cand_elems * 8 + sizeof(int) * (size_t)n_q;
  if (workspace_bytes < need) return fail(CLIPNCE_EWORKSPACE, "topk: workspace %zu < %zu", workspace_bytes, need);
  cudaStream_t st = as_stream(stream);
  pair::FwdParams p;
  memset(&p, 0, sizeof p);
  p.n_rows = (int)n_q; p.n_cols = (int)n_lib; p.d = (int)d;
  p.nkc = (int)ceil_div(d, 64); p.n_steps = pl.n_steps; p.n_pairs = pl.n_pairs; p.split_steps = pl.split_steps;
  p.rinv_x = rinv_q; p.rinv_y = rinv_lib; p.col_offset = col_offset;
  p.cand_score = reinterpret_cast<float*>(workspace);
  p.cand_idx = reinterpret_cast<int*>(p.cand_score + pl.cand_elems);
  p.row_thr = p.cand_idx + pl.cand_elems;
  CUDA_TRY(cudaMemsetAsync(p.row_thr, 0x80, sizeof(int) * (size_t)n_q, st));   // key 0x80808080: below every real score
  if (pl.kt == 1) rc = launch_pair_fwd<128, 1, 1>(q, lib, p, st);
  else if (pl.kt == 10) rc = launch_pair_fwd<128, 1, 10>(q, lib, p, st);
  else rc = launch_pair_fwd<128, 1, 16>(q, lib, p, st);
  if (rc) return rc;
  aux::topk_merge<<<(unsigned)ceil_div(n_q, 8), 256, 0, st>>>(p.cand_score, p.cand_idx, pl.n_split * 4, n_q, pl.kt, k, out_score,
                                                               out_idx);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_softmax_weights(const float* l, int64_t n, float coef, float* w, void* stream) {
  if (!l || !w || n < 1) return fail(CLIPNCE_EINVAL, "softmax_weights: bad argument");
  aux::softmax_weights<<<(unsigned)ceil_div(n, 256), 256, 0, as_stream(stream)>>>(l, n, coef, w);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_combine_lse(const float* m, const float* l, int64_t n, float* lse, void* stream) {
  if (!m || !l || !lse || n < 1) return fail(CLIPNCE_EINVAL, "combine_lse: bad argument");
  aux::combine_lse<<<(unsigned)ceil_div(n, 256), 256, 0, as_stream(stream)>>>(m, l, n, lse);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_normalize_backward(const void* x, int in_dtype, const float* rinv, const float* dx_hat,
                               const float* grad_scale, int64_t n, int64_t d, void* dx, int out_dtype, void* stream) {
  if (!x || !rinv || !dx_hat || !dx || n < 1 || d < 1) return fail(CLIPNCE_EINVAL, "normalize_backward: bad argument");
  if ((in_dtype != CLIPNCE_BF16 && in_dtype != CLIPNCE_F32) || (out_dtype != CLIPNCE_BF16 && out_dtype != CLIPNCE_F32))
    return fail(CLIPNCE_EINVAL, "normalize_backward: bad dtype");
  cudaStream_t st = as_stream(stream);
  const int wpb = 8;
  dim3 grid((unsigned)ceil_div(n, wpb)), block(32 * wpb);
  const int di = (int)d;
  if (in_dtype == CLIPNCE_BF16 && out_dtype == CLIPNCE_BF16)
    aux::normalize_rows_bwd<<<grid, block, 0, st>>>((const __nv_bfloat16*)x, rinv, dx_hat, grad_scale, n, di, (__nv_bfloat16*)dx);
  else if (in_dtype == CLIPNCE_F32 && out_dtype == CLIPNCE_BF16)
    aux::normalize_rows_bwd<<<grid, block, 0, st>>>((const float*)x, rinv, dx_hat, grad_scale, n, di, (__nv_bfloat16*)dx);
  else if (in_dtype == CLIPNCE_BF16 && out_dtype == CLIPNCE_F32)
    aux::normalize_rows_bwd<<<grid, block, 0, st>>>((const __nv_bfloat16*)x, rinv, dx_hat, grad_scale, n, di, (float*)dx);
  else
    aux::normalize_rows_bwd<<<grid, block, 0, st>>>((const float*)x, rinv, dx_hat, grad_scale, n, di, (float*)dx);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_loss(const float* row_m, const float* row_l, const float* col_m, const float* col_l, const float* diag,
                 int64_t n_rows, int64_t diag_offset, int64_t n_global, int symmetric, float* loss, void* stream) {
  if (!row_m || !row_l || !diag || !loss || n_rows < 1 || n_global < 1) return fail(CLIPNCE_EINVAL, "loss: bad argument");
  if (symmetric && (!col_m || !col_l)) return fail(CLIPNCE_EINVAL, "loss: symmetric loss needs column statistics");
  const double inv = 1.0 / ((symmetric ? 2.0 : 1.0) * (double)n_global);
  aux::loss_reduce<<<1, 1024, 0, as_stream(stream)>>>(row_m, row_l, col_m, col_l, diag, n_rows, diag_offset, inv,
                                                       symmetric, loss);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ---- projection-head tail (kernels_head.cuh) -----------------------------------------------------------------------------
int clipnce_head_tail(const void* h, const void* w, const float* bias, const float* gamma, const float* beta, int64_t n,
                      int64_t k, int64_t p, float ln_eps, void* e, void* zhat, float* rstd, float* rinv, void* stream) {
  if (!h || !w || !gamma || !beta || !e || !rinv) return fail(CLIPNCE_EINVAL, "head_tail: null pointer");
  if (n < 1 || n >= (1ll << 31) || k < 64 || k % 64 != 0 || k > (1 << 16) || p < 128 || p > 512 || p % 128 != 0)
    return fail(CLIPNCE_EUNSUPPORTED, "head_tail: served for hidden %% 64 == 0 and output width in {128, 256, 384, 512} "
                                      "(got hidden %lld, width %lld)", (long long)k, (long long)p);
  if (!aligned16(h) || !aligned16(w) || !aligned16(e) || (zhat && !aligned16(zhat)))
    return fail(CLIPNCE_EINVAL, "head_tail: operands must be 16-byte aligned");
  int rc = check_device_sm100();
  if (rc) return rc;
  head::Params hp;
  memset(&hp, 0, sizeof hp);
  hp.n = (int)n; hp.k = (int)k; hp.p = (int)p; hp.nkb = (int)(k / 64);
  int stages = (pair::SMEM_LIMIT - head::SMALL) / head::stage_bytes((int)p);
  if (stages > head::MAX_STAGES) stages = head::MAX_STAGES;
  if (stages < 2) return fail(CLIPNCE_EUNSUPPORTED, "head_tail: no room for a TMA ring");
  hp.stages = stages;
  hp.ln_eps = ln_eps; hp.norm_eps = aux::kNormEps;
  hp.bias = bias; hp.gamma = gamma; hp.beta = beta;
  hp.e = reinterpret_cast<__nv_bfloat16*>(e); hp.zhat = reinterpret_cast<__nv_bfloat16*>(zhat); hp.rstd = rstd; hp.rinv = rinv;
  CUtensorMap th, tw;
  if ((rc = make_tmap(&th, h, k, n, k, head::ROWS))) return rc;
  if ((rc = make_tmap(&tw, w, k, p, k, 128))) return rc;
  if ((rc = allow_smem(head::linear_ln_kernel, pair::SMEM_LIMIT))) return rc;
  head::linear_ln_kernel<<<(unsigned)ceil_div(n, head::ROWS), head::THREADS, head::smem_bytes((int)p, stages), as_stream(stream)>>>(th, tw, hp);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_head_tail_backward(const void* de, int de_dtype, const void* zhat, const float* rstd, const float* gamma, int64_t n,
                               int64_t p, void* dz, void* stream) {
  if (!de || !zhat || !rstd || !gamma || !dz || n < 1 || p < 1) return fail(CLIPNCE_EINVAL, "head_tail_backward: bad argument");
  if (de_dtype != CLIPNCE_BF16 && de_dtype != CLIPNCE_F32) return fail(CLIPNCE_EINVAL, "head_tail_backward: bad dtype");
  const int wpb = 8;
  dim3 grid((unsigned)ceil_div(n, wpb)), block(32 * wpb);
  if (de_dtype == CLIPNCE_BF16)
    head::ln_backward_rows<<<grid, block, 0, as_stream(stream)>>>((const __nv_bfloat16*)de, (const __nv_bfloat16*)zhat, rstd, gamma, n,
                                                                  (int)p, (__nv_bfloat16*)dz);
  else
    head::ln_backward_rows<<<grid, block, 0, as_stream(stream)>>>((const float*)de, (const __nv_bfloat16*)zhat, rstd, gamma, n, (int)p,
                                                                  (__nv_bfloat16*)dz);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

// ---- exchange over NVLink peer memory (kernels_link.cuh) ------------------------------------------------------------
namespace {
int make_peers(void* const* peer_base, int world, int rank, link::Peers* out) {
  if (!peer_base || world < 1 || world > link::MAX_WORLD || rank < 0 || rank >= world)
    return fail(CLIPNCE_EINVAL, "link: need 1 <= world <= %d peer buffers and 0 <= rank < world", link::MAX_WORLD);
  memset(out, 0, sizeof *out);
  for (int r = 0; r < world; ++r) {
    if (!peer_base[r] || !aligned16(peer_base[r])) return fail(CLIPNCE_EINVAL, "link: peer buffer %d is null or unaligned", r);
    out->base[r] = peer_base[r];
  }
  return 0;
}
}  // namespace

int clipnce_link_control_bytes(int64_t* control_bytes, int64_t* status_offset) {
  if (!control_bytes) return fail(CLIPNCE_EINVAL, "link_control_bytes: null pointer");
  *control_bytes = link::CONTROL_BYTES;
  if (status_offset) *status_offset = link::OFF_STATUS;
  return 0;
}

int clipnce_link_barrier(void* const* peer_base, int world, int rank, int phase, void* stream) {
  link::Peers peers;
  int rc = make_peers(peer_base, world, rank, &peers);
  if (rc) return rc;
  if (phase < 0 || phase >= link::MAX_PHASE) return fail(CLIPNCE_EINVAL, "link_barrier: bad phase %d", phase);
  link::barrier<<<1, 32, 0, as_stream(stream)>>>(peers, world, rank, phase, link_timeout_ns());
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_link_push_rows(const void* x, int in_dtype, int64_t n, int64_t d, int c_dtype, void* const* peer_base,
                           int world, int rank, int64_t rows_offset, int64_t rinv_offset, int64_t row0, void* stream) {
  link::Peers peers;
  int rc = make_peers(peer_base, world, rank, &peers);
  if (rc) return rc;
  if (!x || n < 1 || d < 1 || row0 < 0) return fail(CLIPNCE_EINVAL, "link_push_rows: bad argument");
  if ((in_dtype != CLIPNCE_BF16 && in_dtype != CLIPNCE_F32) || (c_dtype != CLIPNCE_BF16 && c_dtype != CLIPNCE_F32))
    return fail(CLIPNCE_EINVAL, "link_push_rows: bad dtype");
  if (rows_offset < link::CONTROL_BYTES || rows_offset % 16 != 0 || rinv_offset < link::CONTROL_BYTES || rinv_offset % 4 != 0)
    return fail(CLIPNCE_EINVAL, "link_push_rows: offsets must lie behind the control block and be aligned");
  if (in_dtype == CLIPNCE_BF16 && c_dtype == CLIPNCE_BF16 && (d % 8 != 0 || !aligned16(x)))
    return fail(CLIPNCE_EINVAL, "link_push_rows: bf16 rows need d %% 8 == 0 and 16-byte alignment");
  cudaStream_t st = as_stream(stream);
  const int wpb = 8;   // one warp per row over the whole GPU
  dim3 grid((unsigned)ceil_div(n, wpb)), block(32 * wpb);
  const int di = (int)d;
  if (in_dtype == CLIPNCE_BF16 && c_dtype == CLIPNCE_BF16)
    link::push_rows<__nv_bfloat16, __nv_bfloat16><<<grid, block, 0, st>>>((const __nv_bfloat16*)x, n, di, peers, world, rank, rows_offset, rinv_offset, row0);
  else if (in_dtype == CLIPNCE_F32 && c_dtype == CLIPNCE_BF16)
    link::push_rows<float, __nv_bfloat16><<<grid, block, 0, st>>>((const float*)x, n, di, peers, world, rank, rows_offset, rinv_offset, row0);
  else if (in_dtype == CLIPNCE_BF16 && c_dtype == CLIPNCE_F32)
    link::push_rows<__nv_bfloat16, float><<<grid, block, 0, st>>>((const __nv_bfloat16*)x, n, di, peers, world, rank, rows_offset, rinv_offset, row0);
  else
    link::push_rows<float, float><<<grid, block, 0, st>>>((const float*)x, n, di, peers, world, rank, rows_offset, rinv_offset, row0);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_link_copy(const void* src, size_t bytes, void* const* peer_base, int world, int rank, int64_t dst_offset,
                      void* stream) {
  link::Peers peers;
  int rc = make_peers(peer_base, world, rank, &peers);
  if (rc) return rc;
  if (!src || bytes < 1 || dst_offset < link::CONTROL_BYTES) return fail(CLIPNCE_EINVAL, "link_copy: bad argument");
  cudaStream_t st = as_stream(stream);
  for (int k = 1; k <= world; ++k) {   // start behind the own rank: the ranks' copies fan out over different peers
    const int r = (rank + k) % world;
    CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(peers.base[r]) + dst_offset, src, bytes, cudaMemcpyDeviceToDevice, st));
  }
  return 0;
}

int clipnce_link_epoch_advance(void* const* peer_base, int world, int rank, int phase, void* stream) {
  link::Peers peers;
  int rc = make_peers(peer_base, world, rank, &peers);
  if (rc) return rc;
  if (phase < 0 || phase >= link::MAX_PHASE) return fail(CLIPNCE_EINVAL, "link_epoch_advance: bad phase %d", phase);
  link::epoch_advance<<<1, 32, 0, as_stream(stream)>>>(peers, rank, phase);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_link_send_blocks(const void* rows, size_t row_bytes, const float* rinv, size_t rinv_bytes, void* const* peer_base,
                             int world, int rank, int64_t rows_offset, int64_t rinv_offset, int phase, void* stream) {
  link::Peers peers;
  int rc = make_peers(peer_base, world, rank, &peers);
  if (rc) return rc;
  if (!rows || !rinv || row_bytes < 1 || rinv_bytes < 1 || rows_offset < link::CONTROL_BYTES || rinv_offset < link::CONTROL_BYTES)
    return fail(CLIPNCE_EINVAL, "link_send_blocks: bad argument");
  if (phase < 0 || phase >= link::MAX_PHASE) return fail(CLIPNCE_EINVAL, "link_send_blocks: bad phase %d", phase);
  cudaStream_t st = as_stream(stream);
  // rank r sweeps the blocks in the order r, r + 1, r + 2, ...: send first to the rank that needs this block first
  for (int k = 1; k < world; ++k) {
    const int dst = (rank - k + world) % world;
    char* base = reinterpret_cast<char*>(peers.base[dst]);
    CUDA_TRY(cudaMemcpyAsync(base + rows_offset, rows, row_bytes, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(base + rinv_offset, rinv, rinv_bytes, cudaMemcpyDeviceToDevice, st));
    link::signal<<<1, 32, 0, st>>>(peers, rank, dst, phase);
    CUDA_TRY(cudaGetLastError());
  }
  return 0;
}

int clipnce_link_push_f32(const float* const* src, const int64_t* n, const int64_t* dst_offset, int n_seg,
                          void* const* peer_base, int world, int rank, void* stream) {
  link::Peers peers;
  int rc = make_peers(peer_base, world, rank, &peers);
  if (rc) return rc;
  if (!src || !n || !dst_offset || n_seg < 1 || n_seg > 4) return fail(CLIPNCE_EINVAL, "link_push_f32: 1..4 segments");
  link::PushSegs s;
  memset(&s, 0, sizeof s);
  int64_t n_max = 0;
  for (int i = 0; i < n_seg; ++i) {
    if (!src[i] || n[i] < 1 || dst_offset[i] < link::CONTROL_BYTES || dst_offset[i] % 4 != 0)
      return fail(CLIPNCE_EINVAL, "link_push_f32: bad segment %d", i);
    s.src[i] = src[i]; s.n[i] = n[i]; s.dst_off[i] = dst_offset[i];
    if (n[i] > n_max) n_max = n[i];
  }
  s.n_seg = n_seg;
  int64_t gx = ceil_div(n_max, 256);
  if (gx > 1024) gx = 1024;
  link::push_f32<<<dim3((unsigned)gx, (unsigned)n_seg), 256, 0, as_stream(stream)>>>(s, peers, world, rank);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_link_sum_scalars(const float* vals, int cnt, void* const* peer_base, int world, int rank, int phase,
                             float* out, void* stream) {
  link::Peers peers;
  int rc = make_peers(peer_base, world, rank, &peers);
  if (rc) return rc;
  if (!vals || !out || cnt < 1 || cnt > link::MAX_SCALARS) return fail(CLIPNCE_EINVAL, "link_sum_scalars: 1..%d values", link::MAX_SCALARS);
  if (phase < 0 || phase >= link::MAX_PHASE) return fail(CLIPNCE_EINVAL, "link_sum_scalars: bad phase %d", phase);
  link::sum_scalars<<<1, 128, 0, as_stream(stream)>>>(vals, cnt, peers, world, rank, phase, link_timeout_ns(), out);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

int clipnce_combine_partials(const float* part_m, const float* part_l, int n_part, int64_t ld, int64_t n, float* out_m,
                             float* out_l, void* stream) {
  if (!part_m || !part_l || !out_m || !out_l || n_part < 1 || n < 1 || ld < n)
    return fail(CLIPNCE_EINVAL, "combine_partials: bad argument");
  aux::reduce_ml_partials<<<(unsigned)ceil_div(n, 256), 256, 0, as_stream(stream)>>>(part_m, part_l, n_part, ld, n, out_m, out_l);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // extern "C"
