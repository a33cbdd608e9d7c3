// EMA codebook update, usage statistics (SURVEY 8(f) rank 3; reference index_improve/models/vq.py:146-187, 205-217).
//
// One CTA owns one code k: ordered_code_sum (segsum.cuh) adds the rows assigned to k in ascending item order - the
// summation order of torch's CPU index_add_ (vq.py:166-167), so the sums are bit-identical to the reference and
// independent of the grid (deterministic, no floating-point atomics).  The same CTA
// then applies the smoothing and the convex codebook update with the reference's roundings: `x.mul_(decay)` is one
// rounding, `.add_(t, alpha=a)` is a fused multiply-add, `c * (1 - r) + n * r` is three roundings.
#include "common.cuh"
#include "segsum.cuh"

namespace lcrec {

constexpr int kEmaThreads = kSegThreads;

__global__ void __launch_bounds__(kEmaThreads)
ema_update_kernel(const float* __restrict__ latent, const int64_t* __restrict__ indices, int64_t n, int e_dim,
                  float decay, float alpha, float eps, float keep, float rate,
                  float* __restrict__ cluster_size, float* __restrict__ ema_w, float* __restrict__ codebook) {
  extern __shared__ float acc[];                 // e_dim running sums
  __shared__ SegSumSmem sm;
  const int k = blockIdx.x;
  const int tid = threadIdx.x;
  const int64_t count = ordered_code_sum(latent, indices, n, e_dim, k, acc, sm);

  // smoothing + codebook step (vq.py:155-184)
  const float cs = fmaf((float)count, alpha, __fmul_rn(cluster_size[k], decay));
  const bool used = cs > eps;
  const float denom = __fadd_rn(cs, eps);
  for (int d = tid; d < e_dim; d += kEmaThreads) {
    const int64_t o = (int64_t)k * e_dim + d;
    const float w = fmaf(acc[d], alpha, __fmul_rn(ema_w[o], decay));
    ema_w[o] = w;
    if (used) codebook[o] = __fadd_rn(__fmul_rn(codebook[o], keep), __fmul_rn(__fdiv_rn(w, denom), rate));
  }
  __syncthreads();                               // every thread has read cluster_size[k]
  if (tid == 0) cluster_size[k] = cs;
}

// usage = cs / (sum(cs) + eps); used = usage > threshold, unused = usage < threshold (vq.py:83-87, 208-211).
// The sum is taken in fp64 and rounded once (torch's fp32 tree sums differ between its own back ends by an ulp, which
// only matters for a code sitting exactly on the threshold).
__global__ void __launch_bounds__(256)
codebook_usage_kernel(const float* __restrict__ cluster_size, int n_codes, float eps, float threshold,
                      int64_t* __restrict__ used_codes, uint8_t* __restrict__ unused_mask) {
  __shared__ double part[8];
  __shared__ int used_part[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double s = 0.0;
  for (int i = tid; i < n_codes; i += 256) s += (double)cluster_size[i];
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) part[warp] = s;
  __syncthreads();
  double tot = 0.0;
#pragma unroll
  for (int w = 0; w < 8; ++w) tot += part[w];
  const float total = __fadd_rn((float)tot, eps);
  int used = 0;
  for (int i = tid; i < n_codes; i += 256) {
    const float u = __fdiv_rn(cluster_size[i], total);
    used += u > threshold;
    if (unused_mask) unused_mask[i] = u < threshold;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) used += __shfl_xor_sync(0xffffffffu, used, o);
  if (lane == 0) used_part[warp] = used;
  __syncthreads();
  if (tid == 0) {
    int t = 0;
    for (int w = 0; w < 8; ++w) t += used_part[w];
    *used_codes = t;
  }
}

// ---------------------------------------------------------------------------- EMA step, rows split over GPUs
// Data-parallel form: every rank holds a contiguous row block of the global batch (ShardPlan: rank r has n / world rows,
// plus one if r < n % world).  The step must equal the single-device step on the concatenated batch bit for bit, and
// floating-point sums of per-rank partials would not, so each rank GATHERS the global batch through peer memory and runs
// the unchanged ema_update_kernel on it: the same member order, the same sums, the same buffers on every rank.
//
// Symmetric buffer of each rank (zeroed once, peer-mapped): [0] u64 publish counter, [64] u32 CTA ticket of the publish
// launch (local use only), then from byte 256 two slots of ema_dist_slot_bytes(rows_per_rank, e_dim), each
// [i64 n_rows | rows_per_rank i64 indices | pad to 16 B | rows_per_rank x e_dim fp32 latent | pad to 16 B].
// Call c (epoch = c, counting every call on these buffers) publishes into slot c & 1 and sets the counter to c + 1.
//
// Two slots suffice.  Rank A overwrites slot p in call c + 2 only after its gather of call c + 1 has seen every peer B's
// counter at c + 2, i.e. B's publish of call c + 1.  B's stream issued that publish after B's gather of call c - the last
// read of slot p of call c, on any rank's buffer by B - had completed.  So no rank writes a slot a peer may still read.
// The slot stride depends on (rows_per_rank, e_dim) only, which stay fixed for a buffer: calls differ in n and K.
constexpr int kEmaDistThreads = 256;

__host__ __device__ inline int64_t ema_dist_align16(int64_t b) { return (b + 15) & ~(int64_t)15; }
__host__ __device__ inline int64_t ema_dist_latent_offset(int64_t rows_per_rank) { return ema_dist_align16(8 + 8 * rows_per_rank); }
__host__ __device__ inline int64_t ema_dist_slot_bytes(int64_t rows_per_rank, int e_dim) {
  return ema_dist_align16(ema_dist_latent_offset(rows_per_rank) + 4 * rows_per_rank * (int64_t)e_dim);
}

struct EmaDistArgs {
  const float* latent; const int64_t* indices; int64_t n_local; int64_t n_global; int e_dim;
  float* gathered_latent; int64_t* gathered_indices; int32_t* flags;
  unsigned char* const* peers; int world; int rank; int64_t rows_per_rank; unsigned long long epoch;
};

__device__ __forceinline__ void ema_st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ema_ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float ema_ld_relaxed_sys(const float* p) {
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ long long ema_ld_relaxed_sys(const int64_t* p) {
  long long v;
  asm volatile("ld.relaxed.sys.global.s64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// Launch 1: zero flags, this rank's rows into its own slot, then (last CTA of the launch, after every CTA's writes are fenced
// system-wide) the release-store of counter = epoch + 1.
__global__ void __launch_bounds__(kEmaDistThreads) ema_dist_publish_kernel(const EmaDistArgs a) {
  __shared__ bool last;
  unsigned char* base = a.peers[a.rank];
  unsigned char* slot = base + 256 + (a.epoch & 1ull) * ema_dist_slot_bytes(a.rows_per_rank, a.e_dim);
  int64_t* s_idx = reinterpret_cast<int64_t*>(slot + 8);
  float* s_lat = reinterpret_cast<float*>(slot + ema_dist_latent_offset(a.rows_per_rank));
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t0 == 0) {
    *reinterpret_cast<int64_t*>(slot) = a.n_local;
    *a.flags = 0;                                                // the gather launch, stream-ordered after this one, ORs in
  }
  for (int64_t i = t0; i < a.n_local; i += stride) s_idx[i] = a.indices[i];
  const int64_t total = a.n_local * a.e_dim;
  for (int64_t i = t0; i < total; i += stride) s_lat[i] = a.latent[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int* ticket = reinterpret_cast<unsigned int*>(base + 64);
    last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (last && threadIdx.x == 0) {
    *reinterpret_cast<unsigned int*>(base + 64) = 0u;            // the next publish is stream-ordered after this launch
    __threadfence_system();
    ema_st_release_sys(reinterpret_cast<unsigned long long*>(base), a.epoch + 1ull);
  }
}

// Launch 2: every CTA waits for every rank's publish of this call (bounded: flags bit 0 when a peer never arrives), then
// copies its share of the global rows, in rank order, into the local gathered buffers.  No CTA waits on another CTA.
// CTA 0 checks each published n_rows against the ShardPlan count (flags bit 1); the copy reads the ShardPlan counts, which
// never exceed rows_per_rank, so a bad peer cannot make it read past a slot.
__global__ void __launch_bounds__(kEmaDistThreads) ema_dist_gather_kernel(const EmaDistArgs a) {
  __shared__ int s_missing;
  const int tid = threadIdx.x;
  if (tid == 0) s_missing = 0;
  __syncthreads();
  const int64_t slot_off = 256 + (int64_t)(a.epoch & 1ull) * ema_dist_slot_bytes(a.rows_per_rank, a.e_dim);
  const int64_t base = a.n_global / a.world, rem = a.n_global % a.world;
  if (tid < a.world) {
    const unsigned long long* f = reinterpret_cast<const unsigned long long*>(a.peers[tid]);
    long long spins = 0;
    bool arrived = true;
    while (ema_ld_acquire_sys(f) < a.epoch + 1ull) {
      if (++spins > (1ll << 28)) { arrived = false; s_missing = 1; break; }      // a peer never arrived: flag, do not hang
    }
    if (arrived && blockIdx.x == 0) {
      const int64_t want = base + (tid < rem ? 1 : 0);
      if (ema_ld_relaxed_sys(reinterpret_cast<const int64_t*>(a.peers[tid] + slot_off)) != want) atomicOr(a.flags, 2);
    }
  }
  __syncthreads();
  if (s_missing) {
    if (tid == 0) atomicOr(a.flags, 1);
    return;
  }
  const int64_t big = rem * (base + 1);                          // rows held by the ranks with one extra row
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t g = t0; g < a.n_global; g += stride) {
    const int64_t r = g < big ? g / (base + 1) : rem + (g - big) / base;
    const int64_t j = g < big ? g % (base + 1) : (g - big) % base;
    a.gathered_indices[g] = ema_ld_relaxed_sys(reinterpret_cast<const int64_t*>(a.peers[r] + slot_off + 8) + j);
  }
  const int64_t total = a.n_global * a.e_dim;
  const int64_t lat_off = slot_off + ema_dist_latent_offset(a.rows_per_rank);
  for (int64_t e = t0; e < total; e += stride) {
    const int64_t g = e / a.e_dim, d = e - g * a.e_dim;
    const int64_t r = g < big ? g / (base + 1) : rem + (g - big) / base;
    const int64_t j = g < big ? g % (base + 1) : (g - big) % base;
    a.gathered_latent[e] = ema_ld_relaxed_sys(reinterpret_cast<const float*>(a.peers[r] + lat_off) + j * a.e_dim + d);
  }
}

}  // namespace lcrec

using namespace lcrec;

static int launch_ema_update(const float* latent, const int64_t* indices, int64_t n, int n_codes, int e_dim,
                             double ema_decay, double epsilon, float* cluster_size, float* ema_w, float* codebook,
                             cudaStream_t st) {
  // Python doubles meet fp32 tensors as fp32 scalars: decay, 1 - decay, and for the convex step 1 - (1 - decay)
  const double update_rate = 1.0 - ema_decay;
  ema_update_kernel<<<n_codes, kEmaThreads, (size_t)e_dim * sizeof(float), st>>>(
      latent, indices, n, e_dim, (float)ema_decay, (float)(1.0 - ema_decay), (float)epsilon,
      (float)(1.0 - update_rate), (float)update_rate, cluster_size, ema_w, codebook);
  LC_LAUNCH_CHECK("ema_update_kernel");
  return LCREC_OK;
}

extern "C" int lcrec_ema_update(const float* latent, const int64_t* indices, int64_t n, int n_codes, int e_dim,
                                double ema_decay, double epsilon, float* cluster_size, float* ema_w, float* codebook,
                                void* stream) {
  LC_ARG(n >= 0 && n < (int64_t)1 << 31);
  LC_ARG(n_codes > 0 && e_dim > 0 && e_dim <= 8192);
  LC_ARG(cluster_size && ema_w && codebook);
  LC_ARG(n == 0 || (latent && indices));
  LC_TRY(lcrec_device_check());
  return launch_ema_update(latent, indices, n, n_codes, e_dim, ema_decay, epsilon, cluster_size, ema_w, codebook,
                           (cudaStream_t)stream);
}

extern "C" int64_t lcrec_ema_dist_symmetric_bytes(int64_t rows_per_rank, int e_dim) {
  if (rows_per_rank < 1 || e_dim < 1) return -1;
  return 256 + 2 * ema_dist_slot_bytes(rows_per_rank, e_dim);
}

extern "C" int lcrec_ema_update_dist(const float* latent, const int64_t* indices, int64_t n_local, int64_t n_global,
                                     int n_codes, int e_dim, double ema_decay, double epsilon, float* cluster_size,
                                     float* ema_w, float* codebook, float* gathered_latent, int64_t* gathered_indices,
                                     int32_t* flags, void* const* peers_dev, int world, int rank, int64_t rows_per_rank,
                                     uint64_t epoch, void* stream) {
  LC_ARG(world >= 1 && world <= 64 && rank >= 0 && rank < world);
  LC_ARG(rows_per_rank >= 1 && n_local >= 0 && n_local <= rows_per_rank);
  LC_ARG(n_global >= 0 && n_global <= (int64_t)world * rows_per_rank && n_global < (int64_t)1 << 31);
  LC_ARG(n_codes > 0 && e_dim > 0 && e_dim <= 8192);
  LC_ARG(peers_dev && cluster_size && ema_w && codebook && gathered_latent && gathered_indices && flags);
  LC_ARG(n_local == 0 || (latent && indices));
  LC_TRY(lcrec_device_check());
  cudaStream_t st = (cudaStream_t)stream;
  EmaDistArgs a{};
  a.latent = latent; a.indices = indices; a.n_local = n_local; a.n_global = n_global; a.e_dim = e_dim;
  a.gathered_latent = gathered_latent; a.gathered_indices = gathered_indices; a.flags = flags;
  a.peers = (unsigned char* const*)peers_dev; a.world = world; a.rank = rank; a.rows_per_rank = rows_per_rank;
  a.epoch = epoch;
  const auto blocks = [](int64_t elems) {
    return (unsigned)std::min<int64_t>(std::max<int64_t>(1, (elems + kEmaDistThreads - 1) / kEmaDistThreads), 1184);
  };
  ema_dist_publish_kernel<<<blocks(n_local * e_dim), kEmaDistThreads, 0, st>>>(a);
  LC_LAUNCH_CHECK("ema_dist_publish_kernel");
  ema_dist_gather_kernel<<<blocks(n_global * e_dim), kEmaDistThreads, 0, st>>>(a);
  LC_LAUNCH_CHECK("ema_dist_gather_kernel");
  return launch_ema_update(gathered_latent, gathered_indices, n_global, n_codes, e_dim, ema_decay, epsilon,
                           cluster_size, ema_w, codebook, st);
}

extern "C" int lcrec_codebook_usage(const float* cluster_size, int n_codes, double epsilon, double reset_threshold,
                                    int64_t* used_codes, uint8_t* unused_mask, void* stream) {
  LC_ARG(cluster_size && used_codes && n_codes > 0);
  LC_TRY(lcrec_device_check());
  codebook_usage_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(cluster_size, n_codes, (float)epsilon,
                                                            (float)reset_threshold, used_codes, unused_mask);
  LC_LAUNCH_CHECK("codebook_usage_kernel");
  return LCREC_OK;
}
