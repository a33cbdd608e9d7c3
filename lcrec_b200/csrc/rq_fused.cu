// Fused all-levels residual quantisation (argmin branch).
//
// Replaces the per-level torch ops of VectorQuantizer.forward (reference index/models/vq.py:63-75,
// 87-99) chained by ResidualVectorQuantizer.forward (index/models/rq.py:39-56): for every level
//   d_k = (|r|^2 + |c_k|^2) - 2 r.c_k        fp32, same evaluation order as vq.py:71-73
//   idx = first argmin_k d_k                  torch.argmin tie rule
//   x_res = r + (c_idx - r)                   straight-through forward value, vq.py:95
//   r <- r - x_res ; x_q <- x_q + x_res       rq.py:47-48
// One thread owns one item and keeps the residual in registers for all levels; the codebooks of
// all levels (4 x 256 x 32 fp32 = 128 KB at the run.sh shape) and their squared norms are staged
// once per CTA in shared memory and read as warp-wide broadcasts.  The kernel is FP32-FMA bound
// (65 536 FLOP per 128 B read), not HBM bound.
#include <cuda_fp16.h>

#include "common.cuh"
#include "linear.cuh"

namespace lcrec {

constexpr int kRqThreads = 256;

struct RqArgs {
  const float* z; int64_t n; int n_levels; int n_levels_run; int resid_level;
  const float* cb[LCREC_MAX_LEVELS]; int k[LCREC_MAX_LEVELS];
  int64_t* codes; float* xq; float* resid_last; double* sq_err;
};

__device__ __forceinline__ double block_sum_double(double v, double* scratch) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  double t = 0.0;
  if (warp == 0) {
    t = lane < (blockDim.x >> 5) ? scratch[lane] : 0.0;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
  }
  __syncthreads();
  return t;  // valid in warp 0
}

// smem layout: for each staged level: codebook (k*D floats) then norms (k floats).
// IPT items per thread share every broadcast codebook load (one LDS.128 feeds 4 * IPT FMAs: with one item per
// thread the kernel is bound by shared-memory instruction issue, not by the FMA pipe); TRAIN adds the
// straight-through x_q and the per-level squared errors of the training forward.
template <int D, int IPT, bool TRAIN, int THREADS>
__global__ void __launch_bounds__(THREADS, 1) rq_quantize_smem_kernel(const RqArgs a) {
  extern __shared__ __align__(16) float smem_f[];
  __shared__ double red[THREADS / 32];
  float* cbs[LCREC_MAX_LEVELS];
  float* nrm[LCREC_MAX_LEVELS];
  {
    float* p = smem_f;
    for (int l = 0; l < a.n_levels_run; ++l) { cbs[l] = p; p += (size_t)a.k[l] * D; nrm[l] = p; p += (a.k[l] + 3) & ~3; }
  }
  for (int l = 0; l < a.n_levels_run; ++l) {
    const float4* src = reinterpret_cast<const float4*>(a.cb[l]);
    float4* dst = reinterpret_cast<float4*>(cbs[l]);
    for (int i = threadIdx.x; i < a.k[l] * D / 4; i += blockDim.x) dst[i] = __ldg(src + i);
  }
  __syncthreads();
  for (int l = 0; l < a.n_levels_run; ++l)
    for (int c = threadIdx.x; c < a.k[l]; c += blockDim.x) {
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < D; ++d) s = fmaf(cbs[l][c * D + d], cbs[l][c * D + d], s);
      nrm[l][c] = s;
    }
  __syncthreads();

  double err[TRAIN ? LCREC_MAX_LEVELS : 1];
#pragma unroll
  for (int l = 0; l < (TRAIN ? LCREC_MAX_LEVELS : 1); ++l) err[l] = 0.0;

  for (int64_t base = blockIdx.x * (int64_t)blockDim.x * IPT; base < a.n; base += (int64_t)gridDim.x * blockDim.x * IPT) {
    int64_t item[IPT]; bool ok[IPT];
    float r[IPT][D];
    float xq[TRAIN ? IPT : 1][TRAIN ? D : 1];
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
      item[j] = base + (int64_t)j * blockDim.x + threadIdx.x;
      ok[j] = item[j] < a.n;
      const float4* zp = reinterpret_cast<const float4*>(a.z + (ok[j] ? item[j] : 0) * D);
#pragma unroll
      for (int d = 0; d < D / 4; ++d) {
        const float4 t = __ldg(zp + d);
        r[j][4 * d] = t.x; r[j][4 * d + 1] = t.y; r[j][4 * d + 2] = t.z; r[j][4 * d + 3] = t.w;
      }
      if constexpr (TRAIN) {
#pragma unroll
        for (int d = 0; d < D; ++d) xq[j][d] = 0.f;
      }
    }
#pragma unroll 1
    for (int l = 0; l < a.n_levels_run; ++l) {
      float xx[IPT], best[IPT]; int best_k[IPT];
#pragma unroll
      for (int j = 0; j < IPT; ++j) {
        if (a.resid_last != nullptr && l == a.resid_level && ok[j]) {
          float4* rp = reinterpret_cast<float4*>(a.resid_last + item[j] * D);
#pragma unroll
          for (int d = 0; d < D / 4; ++d) rp[d] = make_float4(r[j][4 * d], r[j][4 * d + 1], r[j][4 * d + 2], r[j][4 * d + 3]);
        }
        xx[j] = 0.f;
#pragma unroll
        for (int d = 0; d < D; ++d) xx[j] = fmaf(r[j][d], r[j][d], xx[j]);
        best[j] = INFINITY; best_k[j] = 0;
      }
      const float* cb = cbs[l];
      const float* nr = nrm[l];
      const int kl = a.k[l];
#pragma unroll 2
      for (int c = 0; c < kl; ++c) {
        const float4* cp = reinterpret_cast<const float4*>(cb + c * D);
        float dot0[IPT], dot1[IPT];
#pragma unroll
        for (int j = 0; j < IPT; ++j) { dot0[j] = 0.f; dot1[j] = 0.f; }
#pragma unroll
        for (int d = 0; d < D / 4; d += 2) {
          const float4 u = cp[d];
#pragma unroll
          for (int j = 0; j < IPT; ++j) {
            dot0[j] = fmaf(r[j][4 * d], u.x, dot0[j]); dot0[j] = fmaf(r[j][4 * d + 1], u.y, dot0[j]);
            dot0[j] = fmaf(r[j][4 * d + 2], u.z, dot0[j]); dot0[j] = fmaf(r[j][4 * d + 3], u.w, dot0[j]);
          }
          if (d + 1 < D / 4) {
            const float4 w = cp[d + 1];
#pragma unroll
            for (int j = 0; j < IPT; ++j) {
              dot1[j] = fmaf(r[j][4 * d + 4], w.x, dot1[j]); dot1[j] = fmaf(r[j][4 * d + 5], w.y, dot1[j]);
              dot1[j] = fmaf(r[j][4 * d + 6], w.z, dot1[j]); dot1[j] = fmaf(r[j][4 * d + 7], w.w, dot1[j]);
            }
          }
        }
        const float nc = nr[c];
#pragma unroll
        for (int j = 0; j < IPT; ++j) {
          const float dist = (xx[j] + nc) - 2.f * (dot0[j] + dot1[j]);
          if (dist < best[j]) { best[j] = dist; best_k[j] = c; }
        }
      }
#pragma unroll
      for (int j = 0; j < IPT; ++j) {
        if (a.codes && ok[j]) a.codes[item[j] * a.n_levels + l] = best_k[j];
        const float* q = cb + best_k[j] * D;
        double e = 0.0;
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const float t = q[d] - r[j][d];
          if constexpr (TRAIN) e += (double)(t * t);
          const float xres = r[j][d] + t;
          r[j][d] = r[j][d] - xres;
          if constexpr (TRAIN) xq[j][d] += xres;
        }
        if constexpr (TRAIN) { if (ok[j]) err[l] += e; }
      }
    }
#pragma unroll
    for (int j = 0; j < IPT; ++j) {
      if (!ok[j]) continue;
      if (a.resid_last != nullptr && a.resid_level >= a.n_levels_run) {
        float4* rp = reinterpret_cast<float4*>(a.resid_last + item[j] * D);
#pragma unroll
        for (int d = 0; d < D / 4; ++d) rp[d] = make_float4(r[j][4 * d], r[j][4 * d + 1], r[j][4 * d + 2], r[j][4 * d + 3]);
      }
      if constexpr (TRAIN) {
        if (a.xq) {
          float4* xp = reinterpret_cast<float4*>(a.xq + item[j] * D);
#pragma unroll
          for (int d = 0; d < D / 4; ++d) xp[d] = make_float4(xq[j][4 * d], xq[j][4 * d + 1], xq[j][4 * d + 2], xq[j][4 * d + 3]);
        }
      }
    }
  }
  if constexpr (TRAIN) {
    if (a.sq_err) {
      for (int l = 0; l < a.n_levels_run; ++l) {
        const double t = block_sum_double(err[l], red);
        if (threadIdx.x == 0) atomicAdd(a.sq_err + l, t);
      }
    }
  }
}

// Generic path: any e_dim / codebook size, codebooks read from global memory (L2).  One warp per
// item; lanes stride over the codes; residual kept in shared memory.  Correct for every shape the
// reference accepts; the large-codebook configuration (8192 x 256) is served by this kernel until
// the tensor-core distance path lands.
__global__ void __launch_bounds__(256) rq_quantize_generic_kernel(const RqArgs a, const int D,
                                                                 const float* __restrict__ norms_all) {
  extern __shared__ float sm[];
  const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* r = sm + (size_t)warp * 2 * D;
  float* xq = r + D;
  double err[LCREC_MAX_LEVELS];
  for (int l = 0; l < LCREC_MAX_LEVELS; ++l) err[l] = 0.0;
  for (int64_t item = blockIdx.x * (int64_t)warps + warp; item < a.n; item += (int64_t)gridDim.x * warps) {
    for (int d = lane; d < D; d += 32) { r[d] = a.z[item * D + d]; xq[d] = 0.f; }
    __syncwarp();
    int norm_off = 0;
    for (int l = 0; l < a.n_levels_run; ++l) {
      if (a.resid_last != nullptr && l == a.resid_level)
        for (int d = lane; d < D; d += 32) a.resid_last[item * D + d] = r[d];
      float xx = 0.f;
      for (int d = 0; d < D; ++d) xx = fmaf(r[d], r[d], xx);
      float best = INFINITY; int best_k = 0x7fffffff;
      const float* cb = a.cb[l];
      for (int c = lane; c < a.k[l]; c += 32) {
        const float* cp = cb + (size_t)c * D;
        float dot = 0.f;
        for (int d = 0; d < D; ++d) dot = fmaf(r[d], __ldg(cp + d), dot);
        const float dist = (xx + norms_all[norm_off + c]) - 2.f * dot;
        if (dist < best) { best = dist; best_k = c; }
      }
      for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int ok = __shfl_xor_sync(0xffffffffu, best_k, o);
        if (ob < best || (ob == best && ok < best_k)) { best = ob; best_k = ok; }
      }
      if (best_k == 0x7fffffff) best_k = 0;   // all-NaN row
      if (lane == 0 && a.codes) a.codes[item * a.n_levels + l] = best_k;
      const float* q = cb + (size_t)best_k * D;
      double e = 0.0;
      for (int d = lane; d < D; d += 32) {
        const float t = __ldg(q + d) - r[d];
        e += (double)(t * t);
        const float xres = r[d] + t;
        r[d] = r[d] - xres;
        xq[d] += xres;
      }
      err[l] += e;
      norm_off += a.k[l];
      __syncwarp();
    }
    if (a.resid_last != nullptr && a.resid_level >= a.n_levels_run)
      for (int d = lane; d < D; d += 32) a.resid_last[item * D + d] = r[d];
    if (a.xq) for (int d = lane; d < D; d += 32) a.xq[item * D + d] = xq[d];
    __syncwarp();
  }
  if (a.sq_err) {
    __shared__ double red[8];
    for (int l = 0; l < a.n_levels_run; ++l) {
      const double t = block_sum_double(err[l], red);
      if (threadIdx.x == 0) atomicAdd(a.sq_err + l, t);
    }
  }
}

__global__ void code_norms_kernel(const float* __restrict__ cb, int k, int D, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= k) return;
  float s = 0.f;
  for (int d = 0; d < D; ++d) s = fmaf(cb[(size_t)c * D + d], cb[(size_t)c * D + d], s);
  out[c] = s;
}

// d[i][k] = (|r_i|^2 + |c_k|^2) - 2 r_i.c_k   (vq.py:71-73); block = 256 threads over codes, rows by blockIdx
__global__ void vq_distances_kernel(const float* __restrict__ r, int64_t n, int D, const float* __restrict__ cb,
                                    int k, float* __restrict__ out) {
  extern __shared__ float row[];
  for (int64_t i = blockIdx.x; i < n; i += gridDim.x) {
    for (int d = threadIdx.x; d < D; d += blockDim.x) row[d] = r[i * D + d];
    __syncthreads();
    float xx = 0.f;
    for (int d = 0; d < D; ++d) xx = fmaf(row[d], row[d], xx);
    for (int c = threadIdx.x; c < k; c += blockDim.x) {
      const float* cp = cb + (size_t)c * D;
      float cc = 0.f, dot = 0.f;
      for (int d = 0; d < D; ++d) { const float v = __ldg(cp + d); cc = fmaf(v, v, cc); dot = fmaf(row[d], v, dot); }
      out[i * k + c] = (xx + cc) - 2.f * dot;
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------- tensor-core path (large codebooks)
// Level step of the tensor-core residual quantiser: apply the codes of the previous level (x_res = r + (q - r),
// r -= x_res, x_q += x_res, squared error; vq.py:87-95 / rq.py:47-48), then prepare the operand of the next distance
// GEMM: |r|^2 (sequential fma chain, the order of the other kernels), fp16 hi/lo with one power-of-two scale per
// (row, 256 columns).  One warp per row, the row lives in shared memory.
struct RqTcPrep {
  const float* src; float* r; int64_t n; int D;
  const int64_t* codes; int64_t codes_stride; const float* cb_prev;     // null on the first level
  float* xq; int xq_first; double* sq_err; float* resid_out;
  __half* hi; __half* lo; int64_t ld_out; float* inv_scale; int64_t ld_scale; float* xx;    // hi == null: apply only
};
__global__ void __launch_bounds__(256) rq_tc_prepare_kernel(const RqTcPrep a) {
  extern __shared__ float sm[];
  __shared__ double red[8];
  const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* row = sm + (size_t)warp * a.D;
  double err = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)warps + warp; i < a.n; i += (int64_t)gridDim.x * warps) {
    const int64_t code = a.cb_prev ? a.codes[i * a.codes_stride] : 0;
    for (int d = lane; d < a.D; d += 32) {
      float v = a.src[i * a.D + d];
      if (a.cb_prev) {
        const float t = __ldg(a.cb_prev + code * a.D + d) - v;
        err += (double)(t * t);
        const float xres = v + t;
        v = v - xres;
        if (a.xq) a.xq[i * a.D + d] = a.xq_first ? xres : a.xq[i * a.D + d] + xres;
      }
      row[d] = v;
      if (a.r) a.r[i * a.D + d] = v;
      if (a.resid_out) a.resid_out[i * a.D + d] = v;
    }
    __syncwarp();
    if (a.hi != nullptr) {
      float xx = 0.f;
      for (int d = 0; d < a.D; ++d) xx = fmaf(row[d], row[d], xx);      // every lane runs the same chain
      if (lane == 0) a.xx[i] = xx;
      for (int g0 = 0; g0 < a.ld_out; g0 += 256) {
        float m = 0.f;
        for (int d = g0 + lane; d < min(g0 + 256, a.D); d += 32) m = fmaxf(m, fabsf(row[d]));
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float s = 1.f, is = 1.f;
        if (m > 0.f && m < INFINITY) {
          int e;
          frexpf(m, &e);
          const int sh = min(max(15 - e, -126), 126);
          s = ldexpf(1.f, sh); is = ldexpf(1.f, -sh);
        }
        if (lane == 0) a.inv_scale[(int64_t)(g0 >> 8) * a.ld_scale + i] = is;
        for (int d = g0 + lane; d < min((int64_t)g0 + 256, a.ld_out); d += 32) {
          const float xs = (d < a.D ? row[d] : 0.f) * s;
          const __half h = __float2half_rn(xs);
          a.hi[i * a.ld_out + d] = h;
          a.lo[i * a.ld_out + d] = __float2half_rn(xs - __half2float(h));
        }
      }
    }
    __syncwarp();
  }
  if (a.sq_err) {
    const double t = block_sum_double(err, red);
    if (threadIdx.x == 0) atomicAdd(a.sq_err, t);
  }
}

// Same step for small e_dim (<= 64): one THREAD per row, the row in registers (a 128-byte row is one cache line per thread;
// no shuffles, no shared memory), same arithmetic and the same sequential |r|^2 chain.
template <int D>
__global__ void __launch_bounds__(256) rq_tc_prepare_small_kernel(const RqTcPrep a) {
  __shared__ double red[8];
  double err = 0.0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < a.n; i += (int64_t)gridDim.x * blockDim.x) {
    float v[D];
    const float4* sp = reinterpret_cast<const float4*>(a.src + i * D);
#pragma unroll
    for (int d = 0; d < D / 4; ++d) { const float4 t = __ldg(sp + d); v[4 * d] = t.x; v[4 * d + 1] = t.y; v[4 * d + 2] = t.z; v[4 * d + 3] = t.w; }
    if (a.cb_prev) {
      const float4* qp = reinterpret_cast<const float4*>(a.cb_prev + a.codes[i * a.codes_stride] * D);
      float xr[D];
#pragma unroll
      for (int d = 0; d < D / 4; ++d) {
        const float4 q = __ldg(qp + d);
        const float qq[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float t = qq[e] - v[4 * d + e];
          err += (double)(t * t);
          const float xres = v[4 * d + e] + t;
          v[4 * d + e] = v[4 * d + e] - xres;
          xr[4 * d + e] = xres;
        }
      }
      if (a.xq) {
        float4* xp = reinterpret_cast<float4*>(a.xq + i * D);
#pragma unroll
        for (int d = 0; d < D / 4; ++d) {
          float4 o = make_float4(xr[4 * d], xr[4 * d + 1], xr[4 * d + 2], xr[4 * d + 3]);
          if (!a.xq_first) { const float4 p = xp[d]; o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w; }
          xp[d] = o;
        }
      }
    }
    if (a.r) {
      float4* rp = reinterpret_cast<float4*>(a.r + i * D);
#pragma unroll
      for (int d = 0; d < D / 4; ++d) rp[d] = make_float4(v[4 * d], v[4 * d + 1], v[4 * d + 2], v[4 * d + 3]);
    }
    if (a.resid_out) {
      float4* rp = reinterpret_cast<float4*>(a.resid_out + i * D);
#pragma unroll
      for (int d = 0; d < D / 4; ++d) rp[d] = make_float4(v[4 * d], v[4 * d + 1], v[4 * d + 2], v[4 * d + 3]);
    }
    if (a.hi != nullptr) {
      float xx = 0.f, m = 0.f;
#pragma unroll
      for (int d = 0; d < D; ++d) { xx = fmaf(v[d], v[d], xx); m = fmaxf(m, fabsf(v[d])); }
      a.xx[i] = xx;
      float s = 1.f, is = 1.f;
      if (m > 0.f && m < INFINITY) {
        int e;
        frexpf(m, &e);
        const int sh = min(max(15 - e, -126), 126);
        s = ldexpf(1.f, sh); is = ldexpf(1.f, -sh);
      }
      a.inv_scale[i] = is;                         // D <= 64: a single scale group
      __align__(16) __half h[D];
      __align__(16) __half l[D];
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const float xs = v[d] * s;
        h[d] = __float2half_rn(xs);
        l[d] = __float2half_rn(xs - __half2float(h[d]));
      }
      uint4* hp = reinterpret_cast<uint4*>(a.hi + i * a.ld_out);
      uint4* lp = reinterpret_cast<uint4*>(a.lo + i * a.ld_out);
#pragma unroll
      for (int d = 0; d < D / 8; ++d) { hp[d] = reinterpret_cast<const uint4*>(h)[d]; lp[d] = reinterpret_cast<const uint4*>(l)[d]; }
    }
  }
  if (a.sq_err) {
    const double t = block_sum_double(err, red);
    if (threadIdx.x == 0) atomicAdd(a.sq_err, t);
  }
}

int launch_split_f16(const float* x, int64_t rows, int k, int64_t ldx, __half* hi, __half* lo, int64_t ld_out,
                     float* inv_scale, cudaStream_t st);                      // linear_tf32x3.cu
__global__ void code_norms_kernel(const float* __restrict__ cb, int k, int D, float* __restrict__ out);

// All levels on the tensor cores: per level {prepare, distance GEMM + argmin on CTA pairs (launch_argmin_pair)}.
// Used for codebooks that do not fit the shared-memory kernel (>= 4096 codes or e_dim >= 128, e.g. 4 x 8192 x 256).
static int rq_quantize_tc(const RqArgs& a, int D, cudaStream_t st) {
  const int64_t n = a.n;
  const int64_t ldh = round_up(D, 8);
  const int64_t groups = ceil_div(ldh, 256);
  int kmax = 0;
  for (int l = 0; l < a.n_levels_run; ++l) kmax = std::max(kmax, a.k[l]);
  const size_t bytes_r = sizeof(float) * n * D, bytes_h = sizeof(__half) * n * ldh, bytes_s = sizeof(float) * n * groups,
               bytes_x = sizeof(float) * n, bytes_wh = sizeof(__half) * (size_t)kmax * ldh, bytes_ws = sizeof(float) * kmax;
  auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t total = al(bytes_r) + 2 * al(bytes_h) + al(bytes_s) + al(bytes_x) + 2 * al(bytes_wh) + 2 * al(bytes_ws) + 256;
  static bool pool_set = false;
  if (!pool_set) {      // keep the stream-ordered pool's memory between calls (the default threshold returns it at every sync)
    int dev = 0; cudaMemPool_t pool;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
      uint64_t keep = ~0ull;
      (void)cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    (void)cudaGetLastError();
    pool_set = true;
  }
  char* ws = nullptr;
  LC_CUDA(cudaMallocAsync((void**)&ws, total, st));
  char* p = ws;
  auto take = [&](size_t b) { char* q = p; p += al(b); return q; };
  float* r = (float*)take(bytes_r);
  __half* hi = (__half*)take(bytes_h); __half* lo = (__half*)take(bytes_h);
  float* sc = (float*)take(bytes_s); float* xx = (float*)take(bytes_x);
  __half* w_hi = (__half*)take(bytes_wh); __half* w_lo = (__half*)take(bytes_wh);
  float* w_sc = (float*)take(bytes_ws); float* cc = (float*)take(bytes_ws);
  const int warps = 8;
  const int64_t blocks = std::min<int64_t>(ceil_div(n, warps), (int64_t)num_sms() * 8);
  const size_t smem = sizeof(float) * warps * D;
  int rc = LCREC_OK;
  auto run = [&]() -> int {
    for (int l = 0; l <= a.n_levels_run; ++l) {
      const bool last = l == a.n_levels_run;
      if (last && !(a.xq || a.sq_err || (a.resid_last && a.resid_level >= a.n_levels_run))) break;
      RqTcPrep q{};
      q.src = l == 0 ? a.z : r; q.r = r; q.n = n; q.D = D;
      if (l > 0) { q.codes = a.codes + (l - 1); q.codes_stride = a.n_levels; q.cb_prev = a.cb[l - 1]; q.xq = a.xq; q.xq_first = l == 1; q.sq_err = a.sq_err ? a.sq_err + (l - 1) : nullptr; }
      q.resid_out = (a.resid_last && (l == a.resid_level || (last && a.resid_level >= a.n_levels_run))) ? a.resid_last : nullptr;
      if (!last) { q.hi = hi; q.lo = lo; q.ld_out = ldh; q.inv_scale = sc; q.ld_scale = n; q.xx = xx; }
      const bool vec_ok = ((reinterpret_cast<uintptr_t>(q.src) | reinterpret_cast<uintptr_t>(a.xq) | reinterpret_cast<uintptr_t>(a.resid_last) |
                            (l > 0 ? reinterpret_cast<uintptr_t>(a.cb[l - 1]) : 0)) & 15) == 0;
      const int64_t tblocks = std::min<int64_t>(ceil_div(n, 256), (int64_t)num_sms() * 16);
      if (D == 32 && vec_ok) rq_tc_prepare_small_kernel<32><<<(unsigned)tblocks, 256, 0, st>>>(q);
      else if (D == 64 && vec_ok) rq_tc_prepare_small_kernel<64><<<(unsigned)tblocks, 256, 0, st>>>(q);
      else if (D == 16 && vec_ok) rq_tc_prepare_small_kernel<16><<<(unsigned)tblocks, 256, 0, st>>>(q);
      else rq_tc_prepare_kernel<<<(unsigned)blocks, warps * 32, smem, st>>>(q);
      LC_LAUNCH_CHECK("rq_tc_prepare_kernel");
      if (last) break;
      LC_TRY(launch_split_f16(a.cb[l], a.k[l], D, D, w_hi, w_lo, ldh, w_sc, st));
      code_norms_kernel<<<(unsigned)ceil_div(a.k[l], 256), 256, 0, st>>>(a.cb[l], a.k[l], D, cc);
      LC_LAUNCH_CHECK("code_norms_kernel");
      PairProblem pp{};
      pp.a.hi = hi; pp.a.lo = lo; pp.a.ld = ldh; pp.a.inv_scale = sc; pp.a.ld_scale = n; pp.a.group = kPairGroup;
      pp.n_rows = n; pp.k = D; pp.w_hi = w_hi; pp.w_lo = w_lo; pp.ldw = ldh; pp.w_inv_scale = w_sc; pp.n_out = a.k[l];
      pp.xx = xx; pp.cc = cc; pp.codes = a.codes + l; pp.codes_stride = a.n_levels;
      LC_TRY(launch_argmin_pair(pp, st));
    }
    return LCREC_OK;
  };
  rc = run();
  (void)cudaFreeAsync(ws, st);
  return rc;
}

static int g_rq_ipt = 4;      // items per thread of the generation-path kernel (2 or 4; lcrec_rq_set_tc_mode(10 + ipt) for experiments)

template <int D, int IPT, bool TRAIN, int THREADS>
static int launch_rq_smem_impl(const RqArgs& a, size_t smem, cudaStream_t st) {
  static bool attr = false;
  auto kern = rq_quantize_smem_kernel<D, IPT, TRAIN, THREADS>;
  if (!attr) { LC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024)); attr = true; }
  const int threads = THREADS;
  const int64_t blocks = std::min<int64_t>(ceil_div(a.n, threads * IPT), (int64_t)num_sms());
  kern<<<(unsigned)blocks, threads, smem, st>>>(a);
  LC_LAUNCH_CHECK("rq_quantize_smem_kernel");
  return LCREC_OK;
}
template <int D>
static int launch_rq_smem(const RqArgs& a, int64_t n_select, size_t smem, cudaStream_t st) {
  if (a.xq != nullptr || a.sq_err != nullptr) return launch_rq_smem_impl<D, 1, true, 256>(a, smem, st);
  if constexpr (D <= 32) {
    if (n_select >= 4096) {
      if (g_rq_ipt == 4 && n_select >= 65536) return launch_rq_smem_impl<D, 4, false, 256>(a, smem, st);
      return launch_rq_smem_impl<D, 2, false, 512>(a, smem, st);
    }
  }
  return launch_rq_smem_impl<D, 1, false, 256>(a, smem, st);
}

}  // namespace lcrec

using namespace lcrec;

static int g_rq_tc_mode = 1;
// 0 = never use the tensor-core distance path, 1 (default) = for large codebooks (>= 4096 codes or e_dim >= 128),
// 2 = whenever the shape allows it (cross-checks)
extern "C" int lcrec_rq_set_tc_mode(int mode) {
  if (mode == 12 || mode == 14) { g_rq_ipt = mode - 10; return LCREC_OK; }      // experiment switch: items per thread
  LC_ARG(mode >= 0 && mode <= 2);
  g_rq_tc_mode = mode;
  return LCREC_OK;
}

namespace lcrec {
// lcrec_rq_quantize with the kernel path chosen as if the call had n_select rows (n_select >= n).  The tensor-core and SIMT
// paths agree only up to near-ties, so a caller that quantises part of a larger batch passes the batch's row count to get
// the codes the whole batch would get (lcrec_indexer_pass0_host_ex).  lcrec_rq_quantize is n_select = n.
int rq_quantize_select(const float* z, int64_t n, int64_t n_select, int e_dim, int n_levels, const float* const* codebooks,
                       const int32_t* n_codes, int n_levels_run, int resid_level, int64_t* codes, float* xq, float* resid_last,
                       double* sq_err, void* stream) {
  LC_ARG(n >= 0 && n_select >= n && e_dim > 0 && n_levels >= 1 && n_levels <= LCREC_MAX_LEVELS && codebooks && n_codes);
  LC_ARG(n_levels_run >= 0 && n_levels_run <= n_levels);
  LC_TRY(lcrec_device_check());
  if (n == 0) return LCREC_OK;
  LC_ARG(z != nullptr);
  cudaStream_t st = (cudaStream_t)stream;
  RqArgs a{};
  a.z = z; a.n = n; a.n_levels = n_levels; a.n_levels_run = n_levels_run; a.resid_level = resid_level;
  a.codes = codes; a.xq = xq; a.resid_last = resid_last; a.sq_err = sq_err;
  size_t smem = 0; int64_t total_codes = 0;
  for (int l = 0; l < n_levels; ++l) {
    LC_ARG(codebooks[l] != nullptr && n_codes[l] > 0);
    a.cb[l] = codebooks[l]; a.k[l] = n_codes[l];
    if (l < n_levels_run) { smem += sizeof(float) * ((size_t)n_codes[l] * e_dim + ((n_codes[l] + 3) & ~3)); total_codes += n_codes[l]; }
  }
  const bool aligned = (reinterpret_cast<uintptr_t>(z) & 15) == 0 && (!xq || (reinterpret_cast<uintptr_t>(xq) & 15) == 0) &&
                       (!resid_last || (reinterpret_cast<uintptr_t>(resid_last) & 15) == 0);
  bool cb_aligned = true;
  for (int l = 0; l < n_levels_run; ++l) cb_aligned = cb_aligned && (reinterpret_cast<uintptr_t>(codebooks[l]) & 15) == 0;
  // tensor-core distance path (CTA-pair GEMM + argmin epilogue) for the shapes it serves
  bool tc_ok = codes != nullptr && n_levels_run > 0 && g_rq_tc_mode != 0 && n_select >= 1024, tc_big = false;
  for (int l = 0; l < n_levels_run; ++l) { tc_ok = tc_ok && argmin_pair_supported(e_dim, n_codes[l]); tc_big = tc_big || n_codes[l] >= 4096; }
  if (tc_ok && g_rq_tc_mode == 2) return rq_quantize_tc(a, e_dim, st);
  // small e_dim with 256-multiple codebooks: the tensor-core path (thread-per-row prepare + CTA-pair distance GEMM) is
  // 1.7x the SIMT kernel from a few thousand rows on (1 M items, 4 x 256 x 32: 1.43 vs 2.38 ms)
  if (tc_ok && n_select >= 4096 && (e_dim == 16 || e_dim == 32 || e_dim == 64) && aligned && cb_aligned) return rq_quantize_tc(a, e_dim, st);
  if (smem <= 200 * 1024 && aligned && cb_aligned && n_levels_run > 0) {
    if (e_dim == 32) return launch_rq_smem<32>(a, n_select, smem, st);
    if (e_dim == 16) return launch_rq_smem<16>(a, n_select, smem, st);
    if (e_dim == 64) return launch_rq_smem<64>(a, n_select, smem, st);
  }
  if (tc_ok && (tc_big || e_dim >= 128)) return rq_quantize_tc(a, e_dim, st);
  // generic path
  float* norms = nullptr;
  LC_CUDA(cudaMallocAsync(&norms, sizeof(float) * std::max<int64_t>(total_codes, 1), st));
  int off = 0;
  for (int l = 0; l < n_levels_run; ++l) {
    code_norms_kernel<<<(unsigned)ceil_div(n_codes[l], 256), 256, 0, st>>>(codebooks[l], n_codes[l], e_dim, norms + off);
    LC_LAUNCH_CHECK("code_norms_kernel");
    off += n_codes[l];
  }
  const int warps = 8;
  const int64_t blocks = std::min<int64_t>(ceil_div(n, warps), (int64_t)num_sms() * 8);
  rq_quantize_generic_kernel<<<(unsigned)blocks, warps * 32, sizeof(float) * warps * 2 * e_dim, st>>>(a, e_dim, norms);
  LC_LAUNCH_CHECK("rq_quantize_generic_kernel");
  LC_CUDA(cudaFreeAsync(norms, st));
  return LCREC_OK;
}
}  // namespace lcrec

extern "C" int lcrec_rq_quantize(const float* z, int64_t n, int e_dim, int n_levels, const float* const* codebooks,
                                 const int32_t* n_codes, int n_levels_run, int resid_level, int64_t* codes,
                                 float* xq, float* resid_last, double* sq_err, void* stream) {
  return rq_quantize_select(z, n, n, e_dim, n_levels, codebooks, n_codes, n_levels_run, resid_level, codes, xq, resid_last,
                            sq_err, stream);
}

extern "C" int lcrec_vq_distances(const float* r, int64_t n, int e_dim, const float* codebook, int n_codes,
                                  float* d, void* stream) {
  LC_ARG(n >= 0 && e_dim > 0 && n_codes > 0 && codebook);
  LC_TRY(lcrec_device_check());
  if (n == 0) return LCREC_OK;
  LC_ARG(r && d);
  const int64_t blocks = std::min<int64_t>(n, (int64_t)num_sms() * 8);
  vq_distances_kernel<<<(unsigned)blocks, 256, sizeof(float) * e_dim, (cudaStream_t)stream>>>(r, n, e_dim, codebook, n_codes, d);
  LC_LAUNCH_CHECK("vq_distances_kernel");
  return LCREC_OK;
}
