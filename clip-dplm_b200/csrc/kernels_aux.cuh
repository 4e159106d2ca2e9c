// HBM-bound helper kernels around the two contraction kernels: normalise (+ its backward),
// transpose, LSE plumbing on [N] vectors, deterministic reductions of per-CTA partials.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <cstdint>

namespace aux {

template <typename T> __device__ __forceinline__ float ld_f(const T* p);
template <> __device__ __forceinline__ float ld_f<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ld_f<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <typename T> __device__ __forceinline__ void st_f(T* p, float v);
template <> __device__ __forceinline__ void st_f<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void st_f<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

constexpr float kNormEps = 1e-12f;  // F.normalize default eps

// One lane's share of a row's sum of squares (the caller adds the lanes with warp_sum).  bf16 rows with d % 8 == 0 are read
// as 16-byte chunks.  Every kernel that needs 1/|x| goes through this function, so that a row's norm has the same bits
// wherever it is computed (normalize_rows on the owner, link::push_rows for the gathered copies).
template <typename TI>
__device__ __forceinline__ float row_sumsq_lane(const TI* __restrict__ xr, int d, int lane) {
  float ss = 0.f;
  if constexpr (sizeof(TI) == 2) {
    if ((d & 7) == 0 && (reinterpret_cast<uintptr_t>(xr) & 15u) == 0) {
      const uint4* xv = reinterpret_cast<const uint4*>(xr);
      for (int c = lane; c < (d >> 3); c += 32) {
        const uint4 v = xv[c];
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 f = __bfloat1622float2(h[k]);
          ss = fmaf(f.x, f.x, ss);
          ss = fmaf(f.y, f.y, ss);
        }
      }
      return ss;
    }
  }
  for (int k = lane; k < d; k += 32) {
    const float v = ld_f(xr + k);
    ss = fmaf(v, v, ss);
  }
  return ss;
}

// One warp per row: rinv = 1 / max(|x|, eps), optionally x_hat = x / max(|x|, eps)   (old/clip.py:63-64).
template <typename TI, typename TO>
__global__ void normalize_rows(const TI* __restrict__ x, int64_t n, int d, TO* __restrict__ xh, float* __restrict__ rinv) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const TI* xr = x + row * d;
  const float ss = warp_sum(row_sumsq_lane(xr, d, lane));
  const float denom = fmaxf(sqrtf(ss), kNormEps);
  if (xh != nullptr) {
    TO* o = xh + row * d;
    for (int k = lane; k < d; k += 32) st_f(o + k, ld_f(xr + k) / denom);
  }
  if (lane == 0) rinv[row] = 1.f / denom;
}

// Operand staging: out_c = convert(in) [n,d] (optional) and out_t = convert(in)^T [d,ld_t] (optional).
// Padding columns n..ld_t of out_t are left untouched (TMA never reads them: the map's extent is n).
template <typename TI, typename TO>
__global__ void stage_operand(const TI* __restrict__ in, int64_t n, int d, TO* __restrict__ out_c, TO* __restrict__ out_t,
                              int64_t ld_t) {
  __shared__ TO tile[32][33];
  const int64_t r0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    int64_t rr = r0 + r;
    int cc = c0 + threadIdx.x;
    if (rr < n && cc < d) {
      TO v;
      st_f(&v, ld_f(in + rr * d + cc));
      tile[r][threadIdx.x] = v;
      if (out_c != nullptr) out_c[rr * d + cc] = v;
    }
  }
  if (out_t == nullptr) return;
  __syncthreads();
  for (int c = threadIdx.y; c < 32; c += blockDim.y) {
    int cc = c0 + c;
    int64_t rr = r0 + threadIdx.x;
    if (rr < n && cc < d) out_t[(int64_t)cc * ld_t + rr] = tile[threadIdx.x][c];
  }
}

// dx_i = rinv_i (g_i - xhat_i (xhat_i . g_i));  clamped rows (|x| < eps): dx_i = g_i * rinv_i.
template <typename TI, typename TO>
__global__ void normalize_rows_bwd(const TI* __restrict__ x, const float* __restrict__ rinv,
                                   const float* __restrict__ g, const float* __restrict__ grad_scale, int64_t n, int d,
                                   TO* __restrict__ dx) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n) return;
  const float ri = rinv[row];
  const float gs = grad_scale ? grad_scale[0] : 1.f;
  const TI* xr = x + row * d;
  const float* gr = g + row * d;
  TO* o = dx + row * d;
  const bool clamped = ri >= 0.5f / kNormEps;
  float dot = 0.f;
  if (!clamped) {
    for (int k = lane; k < d; k += 32) dot = fmaf(ld_f(xr + k) * ri, gr[k], dot);
    dot = warp_sum(dot);
  }
  for (int k = lane; k < d; k += 32) {
    float xh = ld_f(xr + k) * ri;
    st_f(o + k, (gr[k] - xh * dot) * (ri * gs));
  }
}

__global__ void softmax_weights(const float* __restrict__ l, int64_t n, float coef, float* __restrict__ w) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) w[i] = coef / l[i];   // l = +inf (column without positives) -> 0
}

__global__ void combine_lse(const float* __restrict__ m, const float* __restrict__ l, int64_t n, float* __restrict__ lse) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) lse[i] = m[i] + logf(l[i]);
}

// Deterministic single-block loss reduction (fp64 accumulators, fixed order).
__global__ void loss_reduce(const float* __restrict__ row_m, const float* __restrict__ row_l,
                            const float* __restrict__ col_m, const float* __restrict__ col_l,
                            const float* __restrict__ diag, int64_t n_rows, int64_t diag_offset, double inv_denom,
                            int symmetric, float* __restrict__ loss) {
  __shared__ double sh[1024];
  double acc = 0.0;
  for (int64_t i = threadIdx.x; i < n_rows; i += blockDim.x) {
    // fp32 logf (1 ulp) + fp64 accumulation: the fp64 log cost 100 us on one SM at N = 65536 and buys nothing --
    // the sums l are fp32 quantities and ATen's log_softmax takes this log in fp32 as well
    const double dg = diag[i];
    acc += ((double)row_m[i] - dg) + (double)logf(row_l[i]);
    if (symmetric) acc += ((double)col_m[i + diag_offset] - dg) + (double)logf(col_l[i + diag_offset]);
  }
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) loss[0] = (float)(sh[0] * inv_denom);
}

// col_l[j] = sum_p part[p][j] (fixed order), col_m[j] = shift.   Used by the tensor-core forward
// whose partials all share the fixed shift s.
__global__ void reduce_col_partials(const float* __restrict__ part, int n_part, int64_t ld, int64_t n_cols, float shift,
                                    const float* __restrict__ shift_dev, float* __restrict__ col_m,
                                    float* __restrict__ col_l) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_cols) return;
  if (shift_dev != nullptr) shift = __ldg(shift_dev);
  float acc = 0.f;
  for (int p = 0; p < n_part; ++p) acc += part[(int64_t)p * ld + j];
  col_m[j] = shift;
  col_l[j] = acc;
}

// Sums taken relative to the offset shift p = s - off (the speculative large-scale forward): l = sum_p part[p][j] in fixed
// order, returned as an exactly rescaled pair (m = p + k ln 2, l 2^-k in [1, 2)) so that the soft-max weights coef / l of
// the backward stay normal numbers whatever the magnitude of the sum (up to n e^off).  A sum below `thr` means the
// entry's largest logit lies so far under the shift that terms were flushed to zero: *flag is raised and the exact
// sweeps that follow (gated on it) replace the statistics.
// n_pad > 0 (grouped launch): entry j belongs to a problem's padding when j % n_pad >= n_valid -- written, never flagged.
__global__ void reduce_shifted_partials(const float* __restrict__ part, int n_part, int64_t ld, int64_t n, float scale,
                                        const float* __restrict__ scale_dev, float off, float thr, float* __restrict__ out_m,
                                        float* __restrict__ out_l, int* __restrict__ flag, int64_t n_pad = 0,
                                        int64_t n_valid = 0) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  if (scale_dev != nullptr) scale = __ldg(scale_dev);
  float acc = 0.f;
  for (int p = 0; p < n_part; ++p) acc += part[(int64_t)p * ld + j];
  if (!(acc >= thr) || !(acc < INFINITY)) {
    if (n_pad == 0 || j % n_pad < n_valid) *flag = 1;   // every writer stores the same value
    out_m[j] = scale - off;
    out_l[j] = acc;
    return;
  }
  const int k = ilogbf(acc);
  out_m[j] = fmaf((float)k, 0.6931471805599453f, scale - off);
  out_l[j] = ldexpf(acc, -k);
}

// Combine (m,l) partial pairs: out over `n` entries, `n_part` partials with leading dimension ld.  gate: optional DEVICE
// flag, the kernel does nothing while it is 0.
__global__ void reduce_ml_partials(const float* __restrict__ pm, const float* __restrict__ pl, int n_part, int64_t ld,
                                   int64_t n, float* __restrict__ out_m, float* __restrict__ out_l,
                                   const int* __restrict__ gate = nullptr) {
  if (gate != nullptr && __ldg(gate) == 0) return;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float M = -INFINITY;
  for (int p = 0; p < n_part; ++p) M = fmaxf(M, pm[(int64_t)p * ld + i]);
  float L = 0.f;
  for (int p = 0; p < n_part; ++p) {
    float m = pm[(int64_t)p * ld + i];
    if (m > -INFINITY) L += pl[(int64_t)p * ld + i] * expf(m - M);
  }
  out_m[i] = M;
  out_l[i] = L;
}

// *dst += coef * sum_p part[p]   (single thread, fixed order -> deterministic).
__global__ void reduce_scalar_partials(const float* __restrict__ part, int n_part, float coef, float* __restrict__ dst) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double acc = 0.0;
    for (int p = 0; p < n_part; ++p) acc += (double)part[p];
    dst[0] += (float)(acc * (double)coef);
  }
}

// out = sum_s part[s] over n_split slabs of `n4` float4 each (fixed order).
__global__ void sum_splits(const float4* __restrict__ part, int n_split, int64_t n4, float4* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  float4 acc = part[i];
  for (int s = 1; s < n_split; ++s) {
    const float4 v = part[(int64_t)s * n4 + i];
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  out[i] = acc;
}

// Retrieval: merge `n_slot` candidate lists of KT entries per row into the row's k best (one warp per row; ties -> lower
// column index).  cand_* are [n_slot][n_rows][KT]; out_* are [n_rows][k].
__global__ void topk_merge(const float* __restrict__ cand_score, const int* __restrict__ cand_idx, int n_slot, int64_t n_rows,
                           int kt, int k, float* __restrict__ out_score, int64_t* __restrict__ out_idx) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int n_cand = n_slot * kt;                 // <= 32 * 64
  unsigned long long used = 0ull;                 // this lane's candidates c = lane + 32 u, u < 64
  for (int r = 0; r < k; ++r) {
    float best = -INFINITY;
    int best_i = 0x7fffffff, best_u = -1;
    for (int u = 0, c = lane; c < n_cand; ++u, c += 32) {
      if ((used >> u) & 1ull) continue;
      const int64_t o = ((int64_t)(c / kt) * n_rows + row) * kt + (c % kt);
      const float v = cand_score[o];
      const int ix = cand_idx[o];
      if (ix >= 0 && (v > best || (v == best && ix < best_i))) { best = v; best_i = ix; best_u = u; }
    }
    float wv = best;
    int wi = best_i;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, wv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, wi, o);
      if (ov > wv || (ov == wv && oi < wi)) { wv = ov; wi = oi; }
    }
    if (best_u >= 0 && best == wv && best_i == wi) used |= 1ull << best_u;   // (score, index) pairs are unique per row
    if (lane == 0) {
      out_score[row * k + r] = wi == 0x7fffffff ? -INFINITY : wv;
      out_idx[row * k + r] = wi == 0x7fffffff ? -1 : (int64_t)wi;
    }
  }
}

// part[block] = sum over the block's 8 rows of rinv_i <x_i, g_i>   (= <xhat_i, dxhat_i>; one warp per row)
template <typename TI>
__global__ void rowdot_partials(const TI* __restrict__ x, const float* __restrict__ rinv, const float* __restrict__ g,
                                int64_t n, int d, float* __restrict__ part) {
  __shared__ float sh[8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * 8 + w;
  float dot = 0.f;
  if (row < n) {
    const TI* xr = x + row * d;
    const float* gr = g + row * d;
    for (int k = lane; k < d; k += 32) dot = fmaf(ld_f(xr + k), gr[k], dot);
    dot = warp_sum(dot) * rinv[row];
  }
  if (lane == 0) sh[w] = dot;
  __syncthreads();
  if (threadIdx.x == 0) part[blockIdx.x] = ((sh[0] + sh[1]) + (sh[2] + sh[3])) + ((sh[4] + sh[5]) + (sh[6] + sh[7]));
}

// Loads and stores of VEC consecutive elements as floats: 16-byte accesses for VEC = 4 (fp32) and 8-byte ones for bf16.
template <int VEC, typename T>
__device__ __forceinline__ void ldv(const T* p, float (&v)[VEC]) {
  if constexpr (VEC == 1) {
    v[0] = ld_f(p);
  } else if constexpr (sizeof(T) == 4) {
    const float4 f = *reinterpret_cast<const float4*>(p);
    v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
  } else {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
    const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
  }
}
template <int VEC, typename T>
__device__ __forceinline__ void stv(T* p, const float (&v)[VEC]) {
  if constexpr (VEC == 1) {
    st_f(p, v[0]);
  } else if constexpr (sizeof(T) == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  } else {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
    uint2 u;
    u.x = *reinterpret_cast<const uint32_t*>(&a);
    u.y = *reinterpret_cast<const uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p) = u;
  }
}

// One output side of the finishing pass.  Its gradient g_i is the sum of the slabs of every contribution, each split into
// n_split slabs `slab` elements apart: one contribution for a plain side (the split partials of a column sweep, the
// segments of the two-sided sweep, the ranks' slots), one per virtual problem in which a group member was the resident
// operand.  parts[] are indexed by the side's row, xc / xo / rinv / dx by row0 + that row.
constexpr int FINISH_SIDES = 4, FINISH_CONTRIB = 8;
struct FinishSide {
  const float* parts[FINISH_CONTRIB];
  int n_contrib, n_split;
  int64_t slab;
  int64_t row0, n;     // first row in xc / xo / rinv / dx, valid rows
  const void* xc;      // the rows the contraction saw (compute type)
  const void* xo;      // the caller's rows (their own type): the same pointer for rows of the compute type
  const float* rinv;
  void* dx;
  float* ds_part;      // [gridDim.x] block sums of the row dots, or null
  float* sq_part;      // [gridDim.x] block sums of |dx_i|^2, or null
};
struct FinishSides {
  FinishSide s[FINISH_SIDES];
};

// The tail of a backward side in ONE pass over the fp32 gradient of the normalised rows (one warp per row, the row staged
// in shared memory; blockIdx.y = side):
//   g_i     = sum of the side's slabs (contribution-major, then split-major; fixed order)
//   ds_part = sum over the block's 8 rows of rinv_i <xc_i, g_i>      (= <xhat_i, dxhat_i>: sum G.S, d logit_scale)
//   dx_i    = rinv_i (g_i - xhat_i (xhat_i . g_i)) * grad_scale      (normalise backward; clamped rows: g_i rinv_i)
//   sq_part = sum over the block's 8 rows of |dx_i|^2                 (the embeddings' share of a gradient norm)
// Replaces sum_splits + rowdot_partials + normalize_rows_bwd (three passes over [n,d] fp32).  VEC = 4 (d % 4 == 0, every
// row base 4-element aligned): every lane owns four consecutive features per 128-feature stripe, with 16-byte accesses;
// VEC = 1: one feature per 32.  The slabs are added into the row's shared-memory copy one slab at a time, so that a lane's
// loads of a slab are independent of each other -- memory-level parallelism is what this pass lives on.  Every lane
// re-reads only what it wrote: no barrier needed.  grad_scale may be null (1).
template <typename TC, typename TI, typename TO, int VEC>
__global__ void finish_rows(const __grid_constant__ FinishSides sides, const float* __restrict__ grad_scale, int d) {
  const FinishSide& s = sides.s[blockIdx.y];
  extern __shared__ __align__(16) float g_sh[];   // [8][d]
  __shared__ float dot_sh[8], sq_sh[8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t r = (int64_t)blockIdx.x * 8 + w;   // row within the side
  float* g = g_sh + (size_t)w * d;
  float dot_c = 0.f, sq = 0.f;
  if (r < s.n) {
    const int64_t row = s.row0 + r;
    const float ri = s.rinv[row];
    const float gs = grad_scale ? grad_scale[0] : 1.f;
    const TC* xcr = static_cast<const TC*>(s.xc) + row * d;
    const TI* xor_ = static_cast<const TI*>(s.xo) + row * d;
    const bool same = s.xc == s.xo;
    float dot_o = 0.f;
    // g = the side's slabs summed contribution-major, then split-major (fixed order), accumulated in shared memory
    const int n_slabs = s.n_contrib * s.n_split;
    for (int t = 0; t < n_slabs; ++t) {
      const float* pr = s.parts[t / s.n_split] + (int64_t)(t % s.n_split) * s.slab + r * d;
      for (int k = lane * VEC; k < d; k += 32 * VEC) {
        float v[VEC];
        ldv(pr + k, v);
        if (t > 0) {
          float acc[VEC];
          ldv(g + k, acc);
#pragma unroll
          for (int j = 0; j < VEC; ++j) v[j] = acc[j] + v[j];
        }
        stv(g + k, v);
      }
    }
    for (int k = lane * VEC; k < d; k += 32 * VEC) {
      float acc[VEC] = {};   // a group member that is resident in no problem has no slabs: g = 0
      if (n_slabs > 0) ldv(g + k, acc);
      else stv(g + k, acc);
      float vc[VEC];
      ldv(xcr + k, vc);
#pragma unroll
      for (int j = 0; j < VEC; ++j) dot_c = fmaf(vc[j], acc[j], dot_c);
      if (!same) {
        float vo[VEC];
        ldv(xor_ + k, vo);
#pragma unroll
        for (int j = 0; j < VEC; ++j) dot_o = fmaf(vo[j], acc[j], dot_o);
      }
    }
    dot_c = warp_sum(dot_c) * ri;
    dot_o = same ? dot_c : warp_sum(dot_o) * ri;
    if (ri >= 0.5f / kNormEps) dot_o = 0.f;   // clamped row: dx = g * rinv
    const float k2 = ri * gs;
    TO* out = static_cast<TO*>(s.dx) + row * d;
    for (int k = lane * VEC; k < d; k += 32 * VEC) {
      float gv[VEC], xv[VEC], o[VEC];
      ldv(g + k, gv);
      ldv(xor_ + k, xv);
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        o[j] = (gv[j] - xv[j] * ri * dot_o) * k2;
        sq = fmaf(o[j], o[j], sq);
      }
      stv(out + k, o);
    }
    sq = warp_sum(sq);
  }
  if (s.ds_part != nullptr || s.sq_part != nullptr) {
    if (lane == 0) { dot_sh[w] = dot_c; sq_sh[w] = sq; }
    __syncthreads();
    if (threadIdx.x == 0 && s.ds_part != nullptr)
      s.ds_part[blockIdx.x] = ((dot_sh[0] + dot_sh[1]) + (dot_sh[2] + dot_sh[3])) + ((dot_sh[4] + dot_sh[5]) + (dot_sh[6] + dot_sh[7]));
    if (threadIdx.x == 0 && s.sq_part != nullptr)
      s.sq_part[blockIdx.x] = ((sq_sh[0] + sq_sh[1]) + (sq_sh[2] + sq_sh[3])) + ((sq_sh[4] + sq_sh[5]) + (sq_sh[6] + sq_sh[7]));
  }
}

// *dst += coef * sum_p part[p]: 256 threads, strided fp64 partial sums + a fixed-order tree (deterministic).
__global__ void reduce_scalar_partials_par(const float* __restrict__ part, int n_part, float coef, float* __restrict__ dst) {
  __shared__ double sh[256];
  double acc = 0.0;
  for (int p = threadIdx.x; p < n_part; p += 256) acc += (double)part[p];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) dst[0] += (float)(sh[0] * (double)coef);
}

// ---- several pair problems in one launch (kernels_pair.cuh `Group`; the tri-modal model of tf_clip_codes (1).ipynb:13152-13165)
// Per-problem mean loss of the symmetric InfoNCE, problem k over the virtual rows / columns [k n_pad, k n_pad + n):
// loss[k] = [ sum_i (r_i - diag_i) + (c_i - diag_i) ] / (2 n), loss[n_prob] = their sum.  stat_* = [row statistics | column
// statistics], each [n_prob n_pad].  One block, fp64 accumulators, fixed order.
__global__ void loss_reduce_group(const float* __restrict__ stat_m, const float* __restrict__ stat_l,
                                  const float* __restrict__ diag, int n_prob, int64_t n, int64_t n_pad,
                                  float* __restrict__ loss) {
  __shared__ double sh[1024];
  const int64_t V = (int64_t)n_prob * n_pad;
  double total = 0.0;
  for (int k = 0; k < n_prob; ++k) {
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
      const int64_t r = (int64_t)k * n_pad + i;
      const double dg = diag[r];
      acc += ((double)stat_m[r] - dg) + (double)logf(stat_l[r]);
      acc += ((double)stat_m[V + r] - dg) + (double)logf(stat_l[V + r]);
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = blockDim.x >> 1; s > 0; s >>= 1) {
      if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
      __syncthreads();
    }
    const double lk = sh[0] / (2.0 * (double)n);
    if (threadIdx.x == 0) loss[k] = (float)lk;
    total += lk;
    __syncthreads();
  }
  if (threadIdx.x == 0) loss[n_prob] = (float)total;
}

// block 0: *d_scale_sum += 0.5 sum ds_part[all];  block 1 + m: sumsq[m] = sum sq_part[m][:]   (fp64, fixed-order tree)
__global__ void reduce_group_scalars(const float* __restrict__ ds_part, const float* __restrict__ sq_part, int n_members,
                                     int n_blk, float* __restrict__ d_scale_sum, float* __restrict__ sumsq) {
  __shared__ double sh[256];
  const int b = blockIdx.x;
  const float* src = b == 0 ? ds_part : sq_part + (int64_t)(b - 1) * n_blk;
  const int cnt = b == 0 ? n_members * n_blk : n_blk;
  if ((b == 0 && d_scale_sum == nullptr) || (b > 0 && sumsq == nullptr)) return;
  double acc = 0.0;
  for (int p = threadIdx.x; p < cnt; p += 256) acc += (double)src[p];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (b == 0) d_scale_sum[0] += (float)(0.5 * sh[0]);
    else sumsq[b - 1] = (float)sh[0];
  }
}

}  // namespace aux
