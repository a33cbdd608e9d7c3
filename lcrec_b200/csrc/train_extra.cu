// Training-step pieces that ran on torch in round 1 (reference index/trainer.py:98-125 with index/run.sh's configuration):
//
//   * BatchNorm1d in TRAINING mode, fused with the ReLU that follows it (index/models/layers.py:25-29: Linear ->
//     BatchNorm1d -> ReLU; `run.sh --bn False` parses to bn=True, index/main.py:31): batch statistics, normalisation +
//     affine + ReLU, running-statistics update, and the analytic backward.  Split into a REDUCE launch and an APPLY launch
//     with the per-channel sums in between, so that a data-parallel job can all-reduce the sums (synchronised BatchNorm =
//     the single-device global-batch semantics of the reference) between the two.
//   * the reconstruction loss of RQVAE.compute_loss (index/models/rqvae.py:74-85): F.mse_loss / F.l1_loss with
//     reduction="mean" and its backward.
//
// All of it is HBM / L2-bound byte work: the activations of one batch (n x C fp32, 8 MB at 1024 x 2048) are read once per
// launch with coalesced rows; sums accumulate in fp64 in a fixed order (deterministic, no atomics).
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace lcrec {

constexpr int kBnThreads = 256;            // 8 row lanes x 32 channels
constexpr int kBnChan = 32;
constexpr int kBnMaxSplits = 16;

// sums[s][0][c] = sum over the rows of split s of v, sums[s][1][c] = sum of v * w   (fp64)
//   forward : v = y,                      w = y                      (sum, sum of squares)
//   backward: v = g = gy * (out > 0),     w = xhat = (y - mean) * invstd   (g_beta, g_gamma)
template <bool BACKWARD>
__global__ void __launch_bounds__(kBnThreads)
bn_reduce_kernel(const float* __restrict__ y, const float* __restrict__ gy, const float* __restrict__ out, int relu,
                 const float* __restrict__ mean, const float* __restrict__ invstd, int64_t n, int C, int splits,
                 double* __restrict__ sums) {
  __shared__ double red[2][kBnThreads / kBnChan][kBnChan];
  const int c = blockIdx.x * kBnChan + (threadIdx.x & (kBnChan - 1));
  const int rl = threadIdx.x / kBnChan, nrl = kBnThreads / kBnChan;
  const int s = blockIdx.y;
  const int64_t r0 = n * s / splits, r1 = n * (s + 1) / splits;
  double a = 0.0, b = 0.0;
  if (c < C) {
    float mu = 0.f, is = 0.f;
    if (BACKWARD) { mu = mean[c]; is = invstd[c]; }
    for (int64_t r = r0 + rl; r < r1; r += nrl) {
      const int64_t o = r * C + c;
      if (BACKWARD) {
        float g = gy[o];
        if (relu && !(out[o] > 0.f)) g = 0.f;
        const float xh = (y[o] - mu) * is;
        a += (double)g;
        b += (double)g * (double)xh;
      } else {
        const float v = y[o];
        a += (double)v;
        b += (double)v * (double)v;
      }
    }
  }
  red[0][rl][threadIdx.x & (kBnChan - 1)] = a;
  red[1][rl][threadIdx.x & (kBnChan - 1)] = b;
  __syncthreads();
  if (rl == 0 && c < C) {
    double ta = 0.0, tb = 0.0;
    for (int k = 0; k < nrl; ++k) { ta += red[0][k][threadIdx.x]; tb += red[1][k][threadIdx.x]; }
    sums[((size_t)s * 2 + 0) * C + c] = ta;
    sums[((size_t)s * 2 + 1) * C + c] = tb;
  }
}

// forward apply: statistics from the sums of `splits` partial blocks over n_total rows (n_total >= n when the sums were
// all-reduced over ranks), then out = relu?((y - mean) * invstd * gamma + beta) for this rank's n rows.
__global__ void __launch_bounds__(kBnThreads)
bn_apply_kernel(const float* __restrict__ y, const double* __restrict__ sums, int splits, int64_t n, int64_t n_total, int C,
                const float* __restrict__ gamma, const float* __restrict__ beta, float eps, float momentum, int relu,
                float* __restrict__ out, float* __restrict__ save_mean, float* __restrict__ save_invstd,
                float* __restrict__ running_mean, float* __restrict__ running_var) {
  const int c = blockIdx.x * kBnChan + (threadIdx.x & (kBnChan - 1));
  const int rl = threadIdx.x / kBnChan, nrl = kBnThreads / kBnChan;
  if (c >= C) return;
  double sa = 0.0, sb = 0.0;
  for (int s = 0; s < splits; ++s) { sa += sums[((size_t)s * 2 + 0) * C + c]; sb += sums[((size_t)s * 2 + 1) * C + c]; }
  const double m = sa / (double)n_total;
  double var = sb / (double)n_total - m * m;                 // biased variance (what normalises the batch)
  var = var < 0.0 ? 0.0 : var;                               // NaN passes (inf in a channel: inf - inf), like torch
  const float mu = (float)m;
  const float is = (float)(1.0 / sqrt(var + (double)eps));
  if (blockIdx.y == 0 && rl == 0) {
    save_mean[c] = mu;
    save_invstd[c] = is;
    if (running_mean) {                                      // torch: running = (1 - momentum) * running + momentum * stat,
      const double unb = n_total > 1 ? var * (double)n_total / (double)(n_total - 1) : var;      // unbiased variance here
      running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mu;
      running_var[c] = (1.f - momentum) * running_var[c] + momentum * (float)unb;
    }
  }
  const float ga = gamma ? gamma[c] : 1.f, be = beta ? beta[c] : 0.f;
  const int64_t r0 = n * blockIdx.y / gridDim.y, r1 = n * (blockIdx.y + 1) / gridDim.y;
  for (int64_t r = r0 + rl; r < r1; r += nrl) {
    const int64_t o = r * C + c;
    float v = (y[o] - mu) * is * ga + be;
    if (relu) v = v < 0.f ? 0.f : v;                      // NaN passes, like torch.relu
    out[o] = v;
  }
}

// backward apply: gx = gamma * invstd * (g - g_beta / N - xhat * g_gamma / N), N = n_total
__global__ void __launch_bounds__(kBnThreads)
bn_backward_apply_kernel(const float* __restrict__ y, const float* __restrict__ gy, const float* __restrict__ out, int relu,
                         const double* __restrict__ sums, int splits, int64_t n, int64_t n_total, int C,
                         const float* __restrict__ gamma, const float* __restrict__ mean, const float* __restrict__ invstd,
                         float* __restrict__ gx, float* __restrict__ g_gamma, float* __restrict__ g_beta) {
  const int c = blockIdx.x * kBnChan + (threadIdx.x & (kBnChan - 1));
  const int rl = threadIdx.x / kBnChan, nrl = kBnThreads / kBnChan;
  if (c >= C) return;
  double sa = 0.0, sb = 0.0;
  for (int s = 0; s < splits; ++s) { sa += sums[((size_t)s * 2 + 0) * C + c]; sb += sums[((size_t)s * 2 + 1) * C + c]; }
  if (blockIdx.y == 0 && rl == 0) {
    if (g_beta) g_beta[c] = (float)sa;
    if (g_gamma) g_gamma[c] = (float)sb;
  }
  if (!gx) return;
  const float mu = mean[c], is = invstd[c], ga = gamma ? gamma[c] : 1.f;
  const float mb = (float)(sa / (double)n_total), mg = (float)(sb / (double)n_total);
  const float k = ga * is;
  const int64_t r0 = n * blockIdx.y / gridDim.y, r1 = n * (blockIdx.y + 1) / gridDim.y;
  for (int64_t r = r0 + rl; r < r1; r += nrl) {
    const int64_t o = r * C + c;
    float g = gy[o];
    if (relu && !(out[o] > 0.f)) g = 0.f;
    const float xh = (y[o] - mu) * is;
    gx[o] = k * (g - mb - xh * mg);
  }
}

// ---- reconstruction loss
// VEC: every pointer is 16-byte aligned and groups of 4 elements move as float4; otherwise the same groups are loaded and
// stored one float at a time.  The arithmetic is the same either way, so an offset view gives the aligned copy's values.
constexpr int kLossThreads = 256;
constexpr int kLossPerCta = kLossThreads * 16;

template <bool VEC>
__device__ __forceinline__ float4 ld4(const float* p) {
  if (VEC) return *reinterpret_cast<const float4*>(p);
  return make_float4(p[0], p[1], p[2], p[3]);
}

template <bool VEC>
__device__ __forceinline__ void st4(float* p, float4 v) {
  if (VEC) { *reinterpret_cast<float4*>(p) = v; return; }
  p[0] = v.x; p[1] = v.y; p[2] = v.z; p[3] = v.w;
}

static bool aligned16(const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <bool VEC>
__global__ void __launch_bounds__(kLossThreads)
recon_partial_kernel(const float* __restrict__ out, const float* __restrict__ x, int64_t total, int l1, double* __restrict__ partial) {
  __shared__ double red[kLossThreads / 32];
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * kLossPerCta + threadIdx.x * 4; i < total; i += (int64_t)gridDim.x * kLossPerCta) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t j = i + (int64_t)u * kLossThreads * 4;
      if (j + 3 < total) {
        const float4 a = ld4<VEC>(out + j), b = ld4<VEC>(x + j);
        const float d0 = a.x - b.x, d1 = a.y - b.y, d2 = a.z - b.z, d3 = a.w - b.w;
        const float t = l1 ? (fabsf(d0) + fabsf(d1)) + (fabsf(d2) + fabsf(d3)) : fmaf(d0, d0, d1 * d1) + fmaf(d2, d2, d3 * d3);
        s += (double)t;
      } else {
        for (int64_t q = j; q < total && q < j + 4; ++q) { const float d = out[q] - x[q]; s += l1 ? (double)fabsf(d) : (double)d * (double)d; }
      }
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < kLossThreads / 32; ++w) t += red[w];
    partial[blockIdx.x] = t;
  }
}

__global__ void recon_final_kernel(const double* __restrict__ partial, int n_partial, double inv_total, float* __restrict__ loss) {
  __shared__ double red[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < n_partial; i += blockDim.x) s += partial[i];
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x / 32); ++w) t += red[w];
    *loss = (float)(t * inv_total);
  }
}

// grad = upstream * d mean(loss) / d out:  mse: 2 (out - x) / total;  l1: sign(out - x) / total
template <bool VEC>
__global__ void __launch_bounds__(kLossThreads)
recon_backward_kernel(const float* __restrict__ out, const float* __restrict__ x, int64_t total, int l1,
                      const float* __restrict__ upstream, float inv_total, float* __restrict__ grad) {
  const float up = upstream ? *upstream : 1.f;
  const float k = (l1 ? 1.f : 2.f) * inv_total * up;
  for (int64_t i = ((int64_t)blockIdx.x * kLossThreads + threadIdx.x) * 4; i < total; i += (int64_t)gridDim.x * kLossThreads * 4) {
    if (i + 3 < total) {
      const float4 a = ld4<VEC>(out + i), b = ld4<VEC>(x + i);
      float4 g;
      if (l1) {
        g.x = k * (float)((a.x > b.x) - (a.x < b.x)); g.y = k * (float)((a.y > b.y) - (a.y < b.y));
        g.z = k * (float)((a.z > b.z) - (a.z < b.z)); g.w = k * (float)((a.w > b.w) - (a.w < b.w));
      } else {
        g.x = k * (a.x - b.x); g.y = k * (a.y - b.y); g.z = k * (a.z - b.z); g.w = k * (a.w - b.w);
      }
      st4<VEC>(grad + i, g);
    } else {
      for (int64_t q = i; q < total; ++q) {
        const float d = out[q] - x[q];
        grad[q] = l1 ? k * (float)((d > 0.f) - (d < 0.f)) : k * d;
      }
    }
  }
}

static int bn_splits(int64_t n, int C) {
  // enough CTAs to cover the chip: C / 32 channel blocks x row splits, at least 64 rows per split
  const int64_t cb = ceil_div(C, kBnChan);
  int64_t s = std::max<int64_t>(1, std::min<int64_t>(kBnMaxSplits, (2 * num_sms()) / std::max<int64_t>(cb, 1)));
  s = std::min<int64_t>(s, std::max<int64_t>(1, n / 64));
  return (int)s;
}

}  // namespace lcrec

using namespace lcrec;

extern "C" int64_t lcrec_bn_sums_elems(int n_channels) { return (int64_t)kBnMaxSplits * 2 * n_channels; }
extern "C" int lcrec_bn_splits(int64_t n_rows, int n_channels) { return bn_splits(std::max<int64_t>(n_rows, 1), std::max(n_channels, 1)); }

extern "C" int lcrec_bn_forward_reduce(const float* y, int64_t n_rows, int n_channels, double* sums, void* stream) {
  LC_ARG(n_rows >= 0 && n_channels > 0 && sums);
  LC_TRY(lcrec_device_check());
  LC_ARG(n_rows == 0 || y);
  const int splits = bn_splits(std::max<int64_t>(n_rows, 1), n_channels);
  dim3 grid((unsigned)ceil_div(n_channels, kBnChan), (unsigned)splits);
  bn_reduce_kernel<false><<<grid, kBnThreads, 0, (cudaStream_t)stream>>>(y, nullptr, nullptr, 0, nullptr, nullptr, n_rows, n_channels,
                                                                      splits, sums);
  LC_LAUNCH_CHECK("bn_reduce_kernel<fwd>");
  return LCREC_OK;
}

extern "C" int lcrec_bn_forward_apply(const float* y, const double* sums, int n_splits, int64_t n_rows, int64_t n_rows_total,
                                      int n_channels, const float* gamma, const float* beta, double eps, double momentum, int relu,
                                      float* out, float* save_mean, float* save_invstd, float* running_mean, float* running_var,
                                      void* stream) {
  LC_ARG(n_rows >= 0 && n_rows_total >= n_rows && n_rows_total >= 1 && n_channels > 0 && sums && n_splits >= 1 && n_splits <= kBnMaxSplits);
  LC_ARG(save_mean && save_invstd && (n_rows == 0 || (y && out)) && ((running_mean == nullptr) == (running_var == nullptr)));
  LC_TRY(lcrec_device_check());
  dim3 grid((unsigned)ceil_div(n_channels, kBnChan), (unsigned)bn_splits(std::max<int64_t>(n_rows, 1), n_channels));
  bn_apply_kernel<<<grid, kBnThreads, 0, (cudaStream_t)stream>>>(y, sums, n_splits, n_rows, n_rows_total, n_channels, gamma, beta, (float)eps,
                                                               (float)momentum, relu, out, save_mean, save_invstd, running_mean, running_var);
  LC_LAUNCH_CHECK("bn_apply_kernel");
  return LCREC_OK;
}

extern "C" int lcrec_bn_backward_reduce(const float* y, const float* gy, const float* out, int relu, const float* save_mean,
                                        const float* save_invstd, int64_t n_rows, int n_channels, double* sums, void* stream) {
  LC_ARG(n_rows >= 0 && n_channels > 0 && sums && save_mean && save_invstd && (!relu || out || n_rows == 0));
  LC_ARG(n_rows == 0 || (y && gy));
  LC_TRY(lcrec_device_check());
  const int splits = bn_splits(std::max<int64_t>(n_rows, 1), n_channels);
  dim3 grid((unsigned)ceil_div(n_channels, kBnChan), (unsigned)splits);
  bn_reduce_kernel<true><<<grid, kBnThreads, 0, (cudaStream_t)stream>>>(y, gy, out, relu, save_mean, save_invstd, n_rows, n_channels, splits,
                                                                     sums);
  LC_LAUNCH_CHECK("bn_reduce_kernel<bwd>");
  return LCREC_OK;
}

extern "C" int lcrec_bn_backward_apply(const float* y, const float* gy, const float* out, int relu, const double* sums, int n_splits,
                                       int64_t n_rows, int64_t n_rows_total, int n_channels, const float* gamma, const float* save_mean,
                                       const float* save_invstd, float* gx, float* g_gamma, float* g_beta, void* stream) {
  LC_ARG(n_rows >= 0 && n_rows_total >= n_rows && n_rows_total >= 1 && n_channels > 0 && sums && n_splits >= 1 && n_splits <= kBnMaxSplits);
  LC_ARG(save_mean && save_invstd && (n_rows == 0 || (y && gy)) && (!relu || out || n_rows == 0));
  LC_TRY(lcrec_device_check());
  dim3 grid((unsigned)ceil_div(n_channels, kBnChan), (unsigned)bn_splits(std::max<int64_t>(n_rows, 1), n_channels));
  bn_backward_apply_kernel<<<grid, kBnThreads, 0, (cudaStream_t)stream>>>(y, gy, out, relu, sums, n_splits, n_rows, n_rows_total, n_channels,
                                                                        gamma, save_mean, save_invstd, gx, g_gamma, g_beta);
  LC_LAUNCH_CHECK("bn_backward_apply_kernel");
  return LCREC_OK;
}

extern "C" int64_t lcrec_recon_loss_workspace_bytes(int64_t total) {
  const int64_t ctas = std::max<int64_t>(1, std::min<int64_t>(ceil_div(std::max<int64_t>(total, 1), kLossPerCta), 4096));
  return arena_need(ctas * 8);
}

// loss (1 fp32, device) = mean over `total` elements of (out - x)^2 (loss_type 0, F.mse_loss) or |out - x| (1, F.l1_loss).
// Any 4-byte-aligned out / x (an offset view included); 16-byte-aligned pointers take the float4 loads.
extern "C" int lcrec_recon_loss(const float* out, const float* x, int64_t total, int loss_type, float* loss, void* ws,
                                int64_t ws_bytes, void* stream) {
  LC_ARG(total >= 1 && out && x && loss && (loss_type == 0 || loss_type == 1));
  LC_TRY(lcrec_device_check());
  const int ctas = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(total, kLossPerCta), 4096));
  Arena ar(ws, ws_bytes);
  double* partial = ar.take<double>(ctas);
  if (!ar.ok()) { set_error("recon_loss: workspace too small"); return LCREC_ERR_NOMEM; }
  if (aligned16(out) && aligned16(x))
    recon_partial_kernel<true><<<ctas, kLossThreads, 0, (cudaStream_t)stream>>>(out, x, total, loss_type, partial);
  else
    recon_partial_kernel<false><<<ctas, kLossThreads, 0, (cudaStream_t)stream>>>(out, x, total, loss_type, partial);
  LC_LAUNCH_CHECK("recon_partial_kernel");
  recon_final_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(partial, ctas, 1.0 / (double)total, loss);
  LC_LAUNCH_CHECK("recon_final_kernel");
  return LCREC_OK;
}

// grad = (*upstream, or 1 when NULL) * d loss / d out; any 4-byte-aligned out / x / grad, float4 accesses when all three are 16-byte aligned
extern "C" int lcrec_recon_loss_backward(const float* out, const float* x, int64_t total, int loss_type, const float* upstream,
                                         float* grad, void* stream) {
  LC_ARG(total >= 1 && out && x && grad && (loss_type == 0 || loss_type == 1));
  LC_TRY(lcrec_device_check());
  const int ctas = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div(total, kLossThreads * 4 * 4), (int64_t)num_sms() * 16));
  const float inv_total = (float)(1.0 / (double)total);
  if (aligned16(out) && aligned16(x) && aligned16(grad))
    recon_backward_kernel<true><<<ctas, kLossThreads, 0, (cudaStream_t)stream>>>(out, x, total, loss_type, upstream, inv_total, grad);
  else
    recon_backward_kernel<false><<<ctas, kLossThreads, 0, (cudaStream_t)stream>>>(out, x, total, loss_type, upstream, inv_total, grad);
  LC_LAUNCH_CHECK("recon_backward_kernel");
  return LCREC_OK;
}
