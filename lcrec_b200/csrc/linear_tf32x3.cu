// fp32-accurate Linear(+bias, +ReLU) on the 5th-gen tensor cores (tcgen05 / TMEM / TMA).
//
// Replaces nn.Linear + ReLU inside MLPLayers.forward (reference index/models/layers.py:22-43).
// The reference computes in IEEE fp32; bf16 or single-pass TF32 change 11 % / 1.2 % of the
// emitted codes (SURVEY.md F2), so every product is evaluated with the 3xTF32 split
//     x*w ~= x_hi*w_hi + x_lo*w_hi + x_hi*w_lo,   x_hi = tf32(x), x_lo = tf32(x - x_hi)
// which carries ~22 mantissa bits per operand.  Operands arrive pre-split (A_hi/A_lo from
// split_tf32_kernel or from the previous layer's epilogue, W_hi/W_lo prepared once per
// checkpoint), are staged by TMA into 128B/64B-swizzled shared memory, and one elected thread
// issues tcgen05.mma.kind::tf32 into a TMEM accumulator.
//
// Accumulation accuracy: the tensor core adds into an fp32 TMEM accumulator; to keep the
// rounding error of a K=4096 reduction at fp32-SIMT level the K loop can be cut into chunks
// (`chunk_kblocks`): each chunk accumulates in one of two TMEM buffers and the epilogue warps
// fold finished chunks into fp32 registers with round-to-nearest adds while the next chunk is
// being multiplied (two TMEM buffers = the chunks ping-pong).
//
// Two operand encodings share the kernel (template F16):
//   tf32 x3  operands fp32 in memory, each value a tf32 number; MMA kind::tf32 (K = 8 per instruction);
//   f16  x3  operands fp16 with a per-row power-of-two scale s: h = fp16(x s), l = fp16(x s - h); MMA kind::f16
//            (K = 16 per instruction, twice the tensor rate).  h + l carries 22 significant bits for every
//            element within 2^-18 of its row maximum and an absolute error <= 2^-40 of the row maximum below
//            that; hi*hi products are exact in fp32.  The epilogue multiplies by 1/(s_row s_col).
//
// CTA = 10 warps: warps 0-7 fold/epilogue (TMEM -> registers -> bias/ReLU/split -> global),
// warp 8 = TMA producer (one lane), warp 9 = TMEM allocator + MMA issuer (one lane).
// Tile: 128 rows x BN columns, K block = BK fp32 (BK*4 bytes = swizzle span).
#include <cuda.h>
#include <cuda_fp16.h>

#include <mutex>
#include <vector>

#include "common.cuh"
#include "linear.cuh"
#include "sm100_ptx.cuh"

namespace lcrec {

using namespace ptx;

struct LinearArgs {
  int64_t n_rows;     // M
  int n_out;          // N
  int num_kblocks;    // ceil(K / BK)
  int chunk_kblocks;  // K blocks per TMEM accumulation chunk (>= 1)
  int relu;
  const float* bias;  // (n_out) or null
  float* y;           // (n_rows, ldy) fp32 or null
  int64_t ldy;
  float* y_hi;        // split output for the next layer, or null (tf32 engine only)
  float* y_lo;
  int64_t ld_split;
  const float* row_scale;   // f16 engine: 1 / s_row (n_rows) and 1 / s_col (n_out); null = 1
  const float* col_scale;
  int debug;          // measurement only: bit 0 = no TMA loads after the first ring fill, bit 1 = no MMAs (results are garbage)
};

constexpr int kTileM = 128;
constexpr int kThreads = 320;

template <int BN, int BK, int STAGES, bool F16 = false>
struct LinearCfg {
  static constexpr int ELEM = F16 ? 2 : 4;
  static constexpr int KSTEP = 32 / ELEM;              // elements per MMA instruction (32 bytes of K)
  static constexpr int A_BYTES = kTileM * BK * ELEM;
  static constexpr int B_BYTES = BN * BK * ELEM;
  static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + BAR_BYTES + 1024;  // + alignment slack
  static constexpr int TMEM_COLS = 2 * BN < 32 ? 32 : 2 * BN;
  static constexpr uint32_t ROW_BYTES = BK * ELEM;     // 128 or 64
  static constexpr uint32_t SBO = 8 * ROW_BYTES;
  static constexpr uint32_t LAYOUT = ROW_BYTES == 128 ? 2u : (ROW_BYTES == 64 ? 4u : 6u);
  static_assert(ROW_BYTES == 128 || ROW_BYTES == 64, "a K block must span a 128B or 64B swizzle row");
  static_assert(BN % 16 == 0 && BN >= 32 && BN <= 256, "UMMA N");
  static_assert(SMEM_BYTES <= 232448, "shared memory");
};

template <int BN, int BK, int STAGES, bool F16>
__global__ void __launch_bounds__(kThreads, 1)
linear_split3_kernel(const __grid_constant__ CUtensorMap map_ahi, const __grid_constant__ CUtensorMap map_alo,
                     const __grid_constant__ CUtensorMap map_bhi, const __grid_constant__ CUtensorMap map_blo,
                     const LinearArgs args, const int tiles_n) {
  using C = LinearCfg<BN, BK, STAGES, F16>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);

  const uint32_t bar0 = base + STAGES * C::STAGE_BYTES;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (STAGES + s); };
  auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * STAGES + b); };
  auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * STAGES + 2 + b); };
  const uint32_t tmem_slot = bar0 + 8u * (2 * STAGES + 4);
  volatile uint32_t* tmem_slot_ptr = (volatile uint32_t*)(smem + STAGES * C::STAGE_BYTES + 8 * (2 * STAGES + 4));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tile_n = blockIdx.x % tiles_n;
  const int64_t tile_m = blockIdx.x / tiles_n;
  const int nkb = args.num_kblocks;
  const int ckb = args.chunk_kblocks;
  const int nchunks = (nkb + ckb - 1) / ckb;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 8); }
    fence_barrier_init();
  }
  if (warp == 8 && lane == 0) {
    prefetch_tensormap(&map_ahi); prefetch_tensormap(&map_alo);
    prefetch_tensormap(&map_bhi); prefetch_tensormap(&map_blo);
  }
  if (warp == 9) tmem_alloc(tmem_slot, C::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 8) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      const int row0 = (int)(tile_m * kTileM);
      const int col0 = tile_n * BN;
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % STAGES;
        const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
        mbar_wait(empty_bar(s), ph ^ 1u);
        if ((args.debug & 1) && kb >= STAGES) { mbar_arrive(full_bar(s)); continue; }
        mbar_expect_tx(full_bar(s), C::STAGE_BYTES);
        const uint32_t dst = base + s * C::STAGE_BYTES;
        tma_load_2d(dst, &map_ahi, full_bar(s), kb * BK, row0);
        tma_load_2d(dst + C::A_BYTES, &map_alo, full_bar(s), kb * BK, row0);
        tma_load_2d(dst + 2 * C::A_BYTES, &map_bhi, full_bar(s), kb * BK, col0);
        tma_load_2d(dst + 2 * C::A_BYTES + C::B_BYTES, &map_blo, full_bar(s), kb * BK, col0);
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = umma_idesc(kTileM, BN, F16 ? 0 : 2);
      int kb = 0;
      for (int c = 0; c < nchunks; ++c) {
        const int b = c & 1;
        mbar_wait(tempty_bar(b), (((uint32_t)c >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(b * BN);
        const int kb_end = min(nkb, kb + ckb);
        bool first = true;
        for (; kb < kb_end; ++kb) {
          const int s = kb % STAGES;
          const uint32_t ph = (uint32_t)(kb / STAGES) & 1u;
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t a_hi = base + s * C::STAGE_BYTES;
          const uint64_t d_ahi = umma_smem_desc(a_hi, C::SBO, C::LAYOUT);
          const uint64_t d_alo = umma_smem_desc(a_hi + C::A_BYTES, C::SBO, C::LAYOUT);
          const uint64_t d_bhi = umma_smem_desc(a_hi + 2 * C::A_BYTES, C::SBO, C::LAYOUT);
          const uint64_t d_blo = umma_smem_desc(a_hi + 2 * C::A_BYTES + C::B_BYTES, C::SBO, C::LAYOUT);
          if (!(args.debug & 2))
#pragma unroll
          for (int k = 0; k < BK / C::KSTEP; ++k) {
            const uint64_t adv = (uint64_t)(k * 32 >> 4);   // one MMA consumes 32 bytes along K
            // small cross terms first, then the dominant hi*hi product
            if constexpr (F16) {
              umma_f16(d_tmem, d_alo + adv, d_bhi + adv, idesc, first ? 0u : 1u);
              umma_f16(d_tmem, d_ahi + adv, d_blo + adv, idesc, 1u);
              umma_f16(d_tmem, d_ahi + adv, d_bhi + adv, idesc, 1u);
            } else {
              umma_tf32(d_tmem, d_alo + adv, d_bhi + adv, idesc, first ? 0u : 1u);
              umma_tf32(d_tmem, d_ahi + adv, d_blo + adv, idesc, 1u);
              umma_tf32(d_tmem, d_ahi + adv, d_bhi + adv, idesc, 1u);
            }
            first = false;
          }
          umma_commit(empty_bar(s));   // smem slot reusable once these MMAs have read it
        }
        umma_commit(tfull_bar(b));     // chunk complete in TMEM
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------ fold + epilogue warps
    constexpr int NCOL = BN / 2;
    constexpr int LDW = NCOL >= 32 ? 32 : 16;
    const int q = warp & 3;        // TMEM lane quarter this warp may access
    const int half = warp >> 2;    // column half
    float acc[NCOL];
#pragma unroll
    for (int i = 0; i < NCOL; ++i) acc[i] = 0.f;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * NCOL);
    for (int c = 0; c < nchunks; ++c) {
      const int b = c & 1;
      mbar_wait(tfull_bar(b), ((uint32_t)c >> 1) & 1u);
      tc_fence_after();
#pragma unroll
      for (int j = 0; j < NCOL; j += LDW) {
        uint32_t v[LDW];
        if constexpr (LDW == 32) tmem_ld32(t_lane + (uint32_t)(b * BN + j), v);
        else tmem_ld16(t_lane + (uint32_t)(b * BN + j), v);
        tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < LDW; ++i) acc[j + i] += __uint_as_float(v[i]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(b));
    }
    // epilogue: bias, ReLU, optional 3xTF32 split for the next layer
    const int64_t row = tile_m * kTileM + q * 32 + lane;
    const int col_base = tile_n * BN + half * NCOL;
    if (row < args.n_rows) {
      const float rscale = args.row_scale ? __ldg(args.row_scale + row) : 1.f;
#pragma unroll
      for (int j = 0; j < NCOL; j += 4) {
        const int col = col_base + j;
        if (col >= args.n_out) break;
        float v[4], hi[4], lo[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float t = acc[j + i];
          if constexpr (F16) { if (col + i < args.n_out) t = (t * rscale) * (args.col_scale ? __ldg(args.col_scale + col + i) : 1.f); }
          if (args.bias != nullptr && col + i < args.n_out) t += __ldg(args.bias + col + i);
          if (args.relu) t = t < 0.f ? 0.f : t;            // NaN passes, like torch.relu
          v[i] = t;
          hi[i] = to_tf32(t);
          lo[i] = to_tf32(t - hi[i]);
        }
        if (col + 3 < args.n_out) {
          if (args.y) *reinterpret_cast<float4*>(args.y + row * args.ldy + col) = make_float4(v[0], v[1], v[2], v[3]);
          if (args.y_hi) {
            *reinterpret_cast<float4*>(args.y_hi + row * args.ld_split + col) = make_float4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<float4*>(args.y_lo + row * args.ld_split + col) = make_float4(lo[0], lo[1], lo[2], lo[3]);
          }
        } else {
          for (int i = 0; i < 4 && col + i < args.n_out; ++i) {
            if (args.y) args.y[row * args.ldy + col + i] = v[i];
            if (args.y_hi) { args.y_hi[row * args.ld_split + col + i] = hi[i]; args.y_lo[row * args.ld_split + col + i] = lo[i]; }
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, C::TMEM_COLS);
  }
}

// x -> (hi, lo) with hi = tf32(x), lo = tf32(x - hi); pads columns [k, ld_out) with zeros.
__global__ void split_tf32_kernel(const float* __restrict__ x, int64_t rows, int k, int64_t ldx,
                                  float* __restrict__ hi, float* __restrict__ lo, int64_t ld_out) {
  const int64_t groups_per_row = ld_out >> 2;
  const int64_t total = rows * groups_per_row;
  const bool vec_ok = ((ldx & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < total;
       g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = g / groups_per_row;
    const int c = (int)(g - r * groups_per_row) << 2;
    float v[4];
    if (vec_ok && c + 3 < k) {
      const float4 t = __ldcs(reinterpret_cast<const float4*>(x + r * ldx + c));
      v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) v[i] = (c + i < k) ? x[r * ldx + c + i] : 0.f;
    }
    float h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { h[i] = to_tf32(v[i]); l[i] = to_tf32(v[i] - h[i]); }
    *reinterpret_cast<float4*>(hi + r * ld_out + c) = make_float4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<float4*>(lo + r * ld_out + c) = make_float4(l[0], l[1], l[2], l[3]);
  }
}

// x (rows, k) fp32 / fp16 / bf16 -> per-row power-of-two scale s with max|x s| in [2^14, 2^15), hi = fp16(x s),
// lo = fp16(x s - hi) (both padded with zeros to ld_out), inv_scale[row] = 1 / s.  One warp per row, two
// passes over the row (the second one hits L1/L2).  Half inputs are converted to fp32 on load (exact).
template <typename T>
__global__ void __launch_bounds__(256) split_f16_rows_kernel(const T* __restrict__ x, int64_t rows, int k, int64_t ldx,
                                                             __half* __restrict__ hi, __half* __restrict__ lo, int64_t ld_out,
                                                             float* __restrict__ inv_scale) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const bool vec_ok = ((ldx & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & (4 * sizeof(T) - 1)) == 0);
  for (int64_t r = warp0; r < rows; r += nwarps) {
    const T* xr = x + r * ldx;
    float m = 0.f;
    if (vec_ok) {
      for (int c = lane * 4; c + 3 < k; c += 128) {
        float t[4];
        load4_f32<false>(xr + c, t);
        m = fmaxf(fmaxf(m, fmaxf(fabsf(t[0]), fabsf(t[1]))), fmaxf(fabsf(t[2]), fabsf(t[3])));
      }
      for (int c = (k & ~3) + lane; c < k; c += 32) m = fmaxf(m, fabsf(to_f32(xr[c])));
    } else {
      for (int c = lane; c < k; c += 32) m = fmaxf(m, fabsf(to_f32(xr[c])));
    }
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    // exponent-only scale: s = 2^(14 - floor(log2 m)); m == 0, inf or nan -> s = 1
    float s = 1.f, is = 1.f;
    if (m > 0.f && m < INFINITY) {
      int e;
      frexpf(m, &e);                 // m = f * 2^e, f in [0.5, 1)  ->  floor(log2 m) = e - 1
      const int sh = min(max(15 - e, -100), 100);
      s = ldexpf(1.f, sh); is = ldexpf(1.f, -sh);
    }
    if (lane == 0) inv_scale[r] = is;
    __half* hr = hi + r * ld_out;
    __half* lr = lo + r * ld_out;
    for (int c = lane * 4; c < ld_out; c += 128) {
      float v[4];
      if (vec_ok && c + 3 < k) {
        load4_f32<false>(xr + c, v);
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = (c + i < k) ? to_f32(xr[c + i]) : 0.f;
      }
      __half h[4], l[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float xs = v[i] * s;                       // exact (power of two)
        h[i] = __float2half_rn(xs);
        l[i] = __float2half_rn(xs - __half2float(h[i]));  // the difference is exact in fp32
      }
      *reinterpret_cast<uint2*>(hr + c) = *reinterpret_cast<const uint2*>(h);
      *reinterpret_cast<uint2*>(lr + c) = *reinterpret_cast<const uint2*>(l);
    }
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  });
  return fn;
}

// fp32 row-major (rows, k) matrix with row stride ld; box = (bk, box_rows); OOB reads give zeros.
int make_map(CUtensorMap* m, const void* ptr, int64_t rows, int k, int64_t ld, int bk, int box_rows, int elem) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled not available from the driver"); return LCREC_ERR_CUDA; }
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) || ((ld * elem) & 15)) {
    set_error("TMA operand must be 16-byte aligned with a row stride multiple of 16 bytes");
    return LCREC_ERR_ARG;
  }
  cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * elem};
  cuuint32_t box[2] = {(cuuint32_t)bk, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMapSwizzle sw = bk * elem == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = fn(m, elem == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)ptr, dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows %lld k %d ld %lld)", (int)r, (long long)rows, k, (long long)ld); return LCREC_ERR_CUDA; }
  return LCREC_OK;
}

struct LinearProblem {
  const void *a_hi, *a_lo; int64_t n_rows; int k; int64_t lda;     // fp32 (tf32 engine) or __half (f16 engine)
  const void *w_hi, *w_lo; int n_out; int64_t ldw;
  bool f16 = false; const float* row_scale = nullptr; const float* col_scale = nullptr;
  const float* bias; int relu;
  float* y; int64_t ldy; float *y_hi, *y_lo; int64_t ld_split;
  int acc_chunk;   // K elements per TMEM chunk, 0 = all
  int variant;     // 0 = default tile choice; 1 = force BK=32 two-stage for BN=256
};

template <int BN, int BK, int STAGES, bool F16 = false>
static int launch_cfg(const LinearProblem& p, cudaStream_t st) {
  using C = LinearCfg<BN, BK, STAGES, F16>;
  static bool attr_set = false;
  auto kern = linear_split3_kernel<BN, BK, STAGES, F16>;
  if (!attr_set) {
    LC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set = true;
  }
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  LC_TRY(make_map(&ma_hi, p.a_hi, p.n_rows, p.k, p.lda, BK, kTileM, C::ELEM));
  LC_TRY(make_map(&ma_lo, p.a_lo, p.n_rows, p.k, p.lda, BK, kTileM, C::ELEM));
  LC_TRY(make_map(&mb_hi, p.w_hi, p.n_out, p.k, p.ldw, BK, BN, C::ELEM));
  LC_TRY(make_map(&mb_lo, p.w_lo, p.n_out, p.k, p.ldw, BK, BN, C::ELEM));
  LinearArgs a;
  a.n_rows = p.n_rows; a.n_out = p.n_out;
  a.num_kblocks = (int)ceil_div(p.k, BK);
  a.chunk_kblocks = p.acc_chunk <= 0 ? a.num_kblocks : (int)std::max<int64_t>(1, p.acc_chunk / BK);
  a.relu = p.relu; a.bias = p.bias; a.y = p.y; a.ldy = p.ldy; a.y_hi = p.y_hi; a.y_lo = p.y_lo; a.ld_split = p.ld_split;
  a.row_scale = p.row_scale; a.col_scale = p.col_scale; a.debug = (p.variant >> 2) & 3;   // variant bits 2, 3
  const int tiles_n = (int)ceil_div(p.n_out, BN);
  const int64_t tiles_m = ceil_div(p.n_rows, kTileM);
  const int64_t grid = tiles_m * tiles_n;
  if (grid <= 0 || grid > 0x7fffffffLL) { set_error("linear: grid %lld out of range", (long long)grid); return LCREC_ERR_ARG; }
  kern<<<(unsigned)grid, kThreads, C::SMEM_BYTES, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, a, tiles_n);
  LC_LAUNCH_CHECK("linear_split3_kernel");
  return LCREC_OK;
}

int launch_linear(const LinearProblem& p, cudaStream_t st) {
  if (p.n_rows == 0) return LCREC_OK;
  if (p.k <= 0 || p.n_out <= 0) { set_error("linear: empty K or N"); return LCREC_ERR_ARG; }
  if (p.f16) {   // same stage bytes as the tf32 configurations, twice the K per block
    if (p.n_out > 128) return (p.variant & 1) ? launch_cfg<256, 64, 2, true>(p, st) : launch_cfg<256, 32, 4, true>(p, st);
    if (p.n_out > 64) return launch_cfg<128, 64, 3, true>(p, st);
    if (p.n_out > 32) return launch_cfg<64, 64, 4, true>(p, st);
    return launch_cfg<32, 64, 4, true>(p, st);
  }
  if (p.n_out > 128) return (p.variant & 1) ? launch_cfg<256, 32, 2>(p, st) : launch_cfg<256, 16, 4>(p, st);
  if (p.n_out > 64) return launch_cfg<128, 32, 3>(p, st);
  if (p.n_out > 32) return launch_cfg<64, 32, 4>(p, st);
  return launch_cfg<32, 32, 4>(p, st);
}

template <typename T>
static int launch_split_f16_t(const T* x, int64_t rows, int k, int64_t ldx, __half* hi, __half* lo, int64_t ld_out,
                              float* inv_scale, cudaStream_t st) {
  if (rows == 0) return LCREC_OK;
  const int64_t blocks = std::min<int64_t>(ceil_div(rows, 8), (int64_t)num_sms() * 16);
  split_f16_rows_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(x, rows, k, ldx, hi, lo, ld_out, inv_scale);
  LC_LAUNCH_CHECK("split_f16_rows_kernel");
  return LCREC_OK;
}

int launch_split_f16(const float* x, int64_t rows, int k, int64_t ldx, __half* hi, __half* lo, int64_t ld_out,
                     float* inv_scale, cudaStream_t st) {
  return launch_split_f16_t(x, rows, k, ldx, hi, lo, ld_out, inv_scale, st);
}

// the same for x of element type `dtype` (kDtypeF32 / kDtypeF16 / kDtypeBF16)
static int launch_split_f16_ex(const void* x, int dtype, int64_t rows, int k, int64_t ldx, __half* hi, __half* lo, int64_t ld_out,
                               float* inv_scale, cudaStream_t st) {
  switch (dtype) {
    case kDtypeF32: return launch_split_f16_t(static_cast<const float*>(x), rows, k, ldx, hi, lo, ld_out, inv_scale, st);
    case kDtypeF16: return launch_split_f16_t(static_cast<const __half*>(x), rows, k, ldx, hi, lo, ld_out, inv_scale, st);
    case kDtypeBF16: return launch_split_f16_t(static_cast<const __nv_bfloat16*>(x), rows, k, ldx, hi, lo, ld_out, inv_scale, st);
    default: set_error("split_f16_rows: bad argument: dtype %d (0 = fp32, 1 = fp16, 2 = bf16)", dtype); return LCREC_ERR_ARG;
  }
}

int launch_split(const float* x, int64_t rows, int k, int64_t ldx, float* hi, float* lo, int64_t ld_out,
                 cudaStream_t st) {
  if (rows == 0) return LCREC_OK;
  const int64_t total = rows * (ld_out / 4);
  const int threads = 256;
  const int64_t blocks = std::min<int64_t>(ceil_div(total, threads), (int64_t)num_sms() * 16);
  split_tf32_kernel<<<(unsigned)blocks, threads, 0, st>>>(x, rows, k, ldx, hi, lo, ld_out);
  LC_LAUNCH_CHECK("split_tf32_kernel");
  return LCREC_OK;
}

}  // namespace lcrec

// ====================================================================== C ABI: MLP
using namespace lcrec;

struct lcrec_mlp {
  int n_layers = 0;
  std::vector<int> dims;
  std::vector<float*> w_hi, w_lo, bias;   // tf32 engine: device, owned
  std::vector<int64_t> ldw;
  std::vector<__half*> h_hi, h_lo;        // f16 engine: split weights + 1/s per output channel
  std::vector<float*> h_scale;
  std::vector<int64_t> ldh;
  int relu_last = 0;
  int acc_chunk = 64;   // fp32-SIMT-level accumulation error (measured: 4.8e-7 vs cuBLAS sgemm 1.0e-6 at K=4096)
  int variant = 0;
  int engine = 0;       // 0 = tf32 x3, 1 = f16 x3
  int max_hidden = 0;
  void* trace = nullptr;
};

static inline int64_t ld4(int64_t k) { return round_up(k, 4); }
static inline int64_t ld8(int64_t k) { return round_up(k, 8); }

extern "C" int lcrec_mlp_update(lcrec_mlp_t* m, const float* const* weights, const float* const* biases,
                                void* stream) {
  LC_ARG(m != nullptr && weights != nullptr);
  cudaStream_t st = (cudaStream_t)stream;
  for (int l = 0; l < m->n_layers; ++l) {
    LC_ARG(weights[l] != nullptr);
    LC_TRY(launch_split(weights[l], m->dims[l + 1], m->dims[l], m->dims[l], m->w_hi[l], m->w_lo[l], m->ldw[l], st));
    LC_TRY(launch_split_f16(weights[l], m->dims[l + 1], m->dims[l], m->dims[l], m->h_hi[l], m->h_lo[l], m->ldh[l],
                            m->h_scale[l], st));
    if (biases && biases[l]) {
      LC_CUDA(cudaMemcpyAsync(m->bias[l], biases[l], sizeof(float) * m->dims[l + 1], cudaMemcpyDeviceToDevice, st));
    } else {
      LC_CUDA(cudaMemsetAsync(m->bias[l], 0, sizeof(float) * m->dims[l + 1], st));
    }
  }
  return LCREC_OK;
}

extern "C" int lcrec_mlp_create(int n_layers, const int32_t* dims, const float* const* weights,
                                const float* const* biases, int relu_last, void* stream, lcrec_mlp_t** out) {
  LC_ARG(n_layers >= 1 && n_layers <= 64 && dims && weights && out);
  LC_TRY(lcrec_device_check());
  lcrec_mlp* m = new lcrec_mlp();
  m->n_layers = n_layers;
  m->dims.assign(dims, dims + n_layers + 1);
  m->relu_last = relu_last;
  for (int l = 0; l <= n_layers; ++l) {
    if (dims[l] <= 0) { delete m; set_error("mlp: non-positive dimension"); return LCREC_ERR_ARG; }
    if (l > 0 && l < n_layers) m->max_hidden = std::max<int>(m->max_hidden, dims[l]);
  }
  m->w_hi.assign(n_layers, nullptr); m->w_lo.assign(n_layers, nullptr); m->bias.assign(n_layers, nullptr);
  m->h_hi.assign(n_layers, nullptr); m->h_lo.assign(n_layers, nullptr); m->h_scale.assign(n_layers, nullptr);
  m->ldw.assign(n_layers, 0); m->ldh.assign(n_layers, 0);
  for (int l = 0; l < n_layers; ++l) {
    m->ldw[l] = ld4(dims[l]); m->ldh[l] = ld8(dims[l]);
    const size_t wbytes = sizeof(float) * (size_t)dims[l + 1] * m->ldw[l];
    const size_t hbytes = sizeof(__half) * (size_t)dims[l + 1] * m->ldh[l];
    if (cudaMalloc(&m->w_hi[l], wbytes) != cudaSuccess || cudaMalloc(&m->w_lo[l], wbytes) != cudaSuccess ||
        cudaMalloc(&m->h_hi[l], hbytes) != cudaSuccess || cudaMalloc(&m->h_lo[l], hbytes) != cudaSuccess ||
        cudaMalloc(&m->h_scale[l], sizeof(float) * dims[l + 1]) != cudaSuccess ||
        cudaMalloc(&m->bias[l], sizeof(float) * dims[l + 1]) != cudaSuccess) {
      set_error("mlp: cudaMalloc of split weights failed: %s", cudaGetErrorString(cudaGetLastError()));
      lcrec_mlp_destroy(m);
      return LCREC_ERR_NOMEM;
    }
  }
  int r = lcrec_mlp_update(m, weights, biases, stream);
  if (r != LCREC_OK) { lcrec_mlp_destroy(m); return r; }
  *out = m;
  return LCREC_OK;
}

extern "C" int lcrec_mlp_destroy(lcrec_mlp_t* m) {
  if (!m) return LCREC_OK;
  for (auto p : m->w_hi) if (p) cudaFree(p);
  for (auto p : m->w_lo) if (p) cudaFree(p);
  for (auto p : m->bias) if (p) cudaFree(p);
  for (auto p : m->h_hi) if (p) cudaFree(p);
  for (auto p : m->h_lo) if (p) cudaFree(p);
  for (auto p : m->h_scale) if (p) cudaFree(p);
  delete m;
  return LCREC_OK;
}

extern "C" int lcrec_mlp_set_acc_chunk(lcrec_mlp_t* m, int k_elems) {
  LC_ARG(m != nullptr && k_elems >= 0);
  m->acc_chunk = k_elems;
  return LCREC_OK;
}

extern "C" int lcrec_mlp_set_variant(lcrec_mlp_t* m, int variant) {
  LC_ARG(m != nullptr);
  m->variant = variant;
  return LCREC_OK;
}

extern "C" int lcrec_pair_set_cluster_cap(int cap) {
  LC_ARG(cap >= 0);
  set_pair_cluster_cap(cap);
  return LCREC_OK;
}

extern "C" int lcrec_mlp_set_trace(lcrec_mlp_t* m, void* trace) {
  LC_ARG(m != nullptr);
  m->trace = trace;
  return LCREC_OK;
}

extern "C" int lcrec_mlp_set_engine(lcrec_mlp_t* m, int engine) {
  LC_ARG(m != nullptr && (engine == 0 || engine == 1));
  m->engine = engine;
  return LCREC_OK;
}

extern "C" int lcrec_mlp_in_dim(const lcrec_mlp_t* m) { return m ? m->dims.front() : -1; }
extern "C" int lcrec_mlp_out_dim(const lcrec_mlp_t* m) { return m ? m->dims.back() : -1; }

static inline int64_t n_scale_groups(int64_t k) { return ceil_div(ld8(k), kPairGroup); }

extern "C" int64_t lcrec_mlp_workspace_bytes(const lcrec_mlp_t* m, int64_t n_rows) {
  if (!m || n_rows < 0) return -1;
  const int64_t hid = std::max(m->max_hidden, 8);
  // tf32 engine: split input (2 fp32) + hi/lo ping-pong (4 fp32 hidden); f16 engine: split input (2 fp16) + two
  // sets of split hidden activations (4 fp16) + one fp32 hidden + scales.  Sized for the larger of the two.
  const int64_t tf = 2 * arena_need(sizeof(float) * n_rows * ld4(m->dims[0])) + 4 * arena_need(sizeof(float) * n_rows * ld4(hid));
  const int64_t hf = 2 * arena_need(sizeof(__half) * n_rows * ld8(m->dims[0])) + 4 * arena_need(sizeof(__half) * n_rows * ld8(hid)) +
                     arena_need(sizeof(float) * n_rows * ld4(hid)) + arena_need(sizeof(float) * n_rows) +
                     arena_need(sizeof(float) * n_rows * n_scale_groups(m->dims[0])) + 2 * arena_need(sizeof(float) * n_rows * n_scale_groups(hid));
  return std::max(tf, hf) + 1024;
}

// f16 x3 engine.  Wide layers (n_out a multiple of 256) run on the CTA-pair kernel with group-scaled operands and
// hand the next wide layer its fp16 hi/lo operand straight from the epilogue; the narrow tail layers use the
// single-CTA kernel with per-row scales (fp32 activation + split_f16_rows pass in between).
static int mlp_forward_f16(lcrec_mlp_t* m, const void* x, int dtype, int64_t n_rows, float* y, float* const* acts, void* workspace,
                           int64_t workspace_bytes, cudaStream_t st) {
  Arena ar(workspace, workspace_bytes);
  const int64_t ld0 = ld8(m->dims[0]);
  const int64_t hid = std::max(m->max_hidden, 8);
  __half* in_hi = ar.take<__half>(n_rows * ld0);
  __half* in_lo = ar.take<__half>(n_rows * ld0);
  __half* set_hi[2]; __half* set_lo[2]; float* set_scale[2];
  for (int i = 0; i < 2; ++i) { set_hi[i] = ar.take<__half>(n_rows * ld8(hid)); set_lo[i] = ar.take<__half>(n_rows * ld8(hid)); }
  float* ybuf = ar.take<float>(n_rows * ld4(hid));
  float* rscale = ar.take<float>(n_rows);
  float* in_scale = ar.take<float>(n_rows * n_scale_groups(m->dims[0]));
  for (int i = 0; i < 2; ++i) set_scale[i] = ar.take<float>(n_rows * n_scale_groups(hid));
  if (!ar.ok()) { set_error("mlp_forward: workspace too small (%lld bytes given, %lld needed)", (long long)workspace_bytes, (long long)lcrec_mlp_workspace_bytes(m, n_rows)); return LCREC_ERR_NOMEM; }
  const bool allow_pair = !(m->variant & 16);
  auto pair_ok = [&](int l) { return allow_pair && l < m->n_layers && linear_pair_supported(m->dims[l], m->dims[l + 1], kPairGroup); };
  // current activation: (cur, ldc) of element type cur_dtype (the input's for layer 0, fp32 after it) or group-scaled fp16 (grp)
  const void* cur = x; int cur_dtype = dtype; int64_t ldc = m->dims[0];
  SplitOperand grp{}; bool grouped = false; int next_set = 0;
  for (int l = 0; l < m->n_layers; ++l) {
    const bool last = (l == m->n_layers - 1);
    const int k = m->dims[l], n_out = m->dims[l + 1];
    float* act_out = (acts && acts[l]) ? acts[l] : nullptr;
    if (pair_ok(l)) {
      if (!grouped) {
        ProfScope prof(l == 0 ? 0 : 17, st);
        __half* hi = l == 0 ? in_hi : set_hi[next_set];
        __half* lo = l == 0 ? in_lo : set_lo[next_set];
        float* sc = l == 0 ? in_scale : set_scale[next_set];
        if (l != 0) next_set ^= 1;
        LC_TRY(launch_split_groups(cur, cur_dtype, n_rows, k, ldc, hi, lo, ld8(k), sc, n_rows, st));
        grp.hi = hi; grp.lo = lo; grp.ld = ld8(k); grp.inv_scale = sc; grp.ld_scale = n_rows; grp.group = kPairGroup;
        grouped = true;
      }
      PairProblem p{};
      p.a = grp; p.n_rows = n_rows; p.k = k;
      p.w_hi = m->h_hi[l]; p.w_lo = m->h_lo[l]; p.ldw = m->ldh[l]; p.w_inv_scale = m->h_scale[l];
      p.n_out = n_out; p.bias = m->bias[l]; p.relu = last ? m->relu_last : 1;
      p.debug = ((m->variant >> 2) & 3) | ((m->variant & 32) ? 4 : 0) | ((m->variant & 64) ? 8 : 0);
      if (l == 0) p.trace = m->trace;
      const bool next_pair = !last && pair_ok(l + 1);
      if (next_pair) {
        p.o_hi = set_hi[next_set]; p.o_lo = set_lo[next_set]; p.ldo = ld8(n_out);
        p.o_inv_scale = set_scale[next_set]; p.ld_oscale = n_rows;
      }
      if (last) { p.y = y; p.ldy = n_out; }
      else if (act_out) { p.y = act_out; p.ldy = n_out; }
      else if (!next_pair) { p.y = ybuf; p.ldy = ld4(n_out); }
      { ProfScope prof(1 + std::min(l, 15), st); LC_TRY(launch_linear_pair(p, st)); }
      if (next_pair) {
        grp.hi = p.o_hi; grp.lo = p.o_lo; grp.ld = p.ldo; grp.inv_scale = p.o_inv_scale; grp.ld_scale = n_rows; grp.group = kPairGroup;
        next_set ^= 1;
      } else {
        grouped = false; cur = p.y; cur_dtype = kDtypeF32; ldc = p.ldy;
      }
      continue;
    }
    // single-CTA kernel, per-row scales
    {
      ProfScope prof(l == 0 ? 0 : 17, st);
      LC_TRY(launch_split_f16_ex(cur, cur_dtype, n_rows, k, ldc, l == 0 ? in_hi : set_hi[0], l == 0 ? in_lo : set_lo[0], ld8(k), rscale, st));
    }
    LinearProblem p{};
    p.f16 = true; p.row_scale = rscale; p.col_scale = m->h_scale[l];
    p.a_hi = l == 0 ? in_hi : set_hi[0]; p.a_lo = l == 0 ? in_lo : set_lo[0]; p.n_rows = n_rows; p.k = k; p.lda = ld8(k);
    p.w_hi = m->h_hi[l]; p.w_lo = m->h_lo[l]; p.n_out = n_out; p.ldw = m->ldh[l];
    p.bias = m->bias[l]; p.relu = last ? m->relu_last : 1;
    p.acc_chunk = m->acc_chunk; p.variant = m->variant & 15;
    float* out = last ? y : (act_out ? act_out : ybuf);
    const int64_t ldo = last ? n_out : (act_out ? n_out : ld4(n_out));
    p.y = out; p.ldy = ldo;
    if ((p.ldy & 3) || (reinterpret_cast<uintptr_t>(p.y) & 15)) {
      set_error("mlp_forward: output width %lld must be a multiple of 4 floats and 16-byte aligned", (long long)p.ldy);
      return LCREC_ERR_UNSUPPORTED;
    }
    { ProfScope prof(1 + std::min(l, 15), st); LC_TRY(launch_linear(p, st)); }
    cur = out; cur_dtype = kDtypeF32; ldc = ldo;
  }
  if (acts && acts[m->n_layers - 1] && acts[m->n_layers - 1] != y)
    LC_CUDA(cudaMemcpyAsync(acts[m->n_layers - 1], y, sizeof(float) * n_rows * m->dims[m->n_layers], cudaMemcpyDeviceToDevice, st));
  return LCREC_OK;
}

extern "C" int lcrec_mlp_forward(lcrec_mlp_t* m, const float* x, int64_t n_rows, float* y, float* const* acts,
                                 void* workspace, int64_t workspace_bytes, void* stream) {
  return lcrec_mlp_forward_ex(m, x, kDtypeF32, n_rows, y, acts, workspace, workspace_bytes, stream);
}

extern "C" int lcrec_mlp_forward_ex(lcrec_mlp_t* m, const void* x_in, int dtype, int64_t n_rows, float* y, float* const* acts,
                                    void* workspace, int64_t workspace_bytes, void* stream) {
  LC_ARG(dtype_ok(dtype));
  LC_ARG(m != nullptr && n_rows >= 0);
  if (n_rows == 0) return LCREC_OK;
  LC_ARG(x_in != nullptr && y != nullptr);
  cudaStream_t st = (cudaStream_t)stream;
  if (m->engine == 1) return mlp_forward_f16(m, x_in, dtype, n_rows, y, acts, workspace, workspace_bytes, st);
  if (dtype != kDtypeF32) {
    set_error("mlp_forward: engine 0 (tf32 x3) takes fp32 input only (dtype %d); half-precision input needs engine 1 (f16 x3)", dtype);
    return LCREC_ERR_UNSUPPORTED;
  }
  const float* x = static_cast<const float*>(x_in);
  Arena ar(workspace, workspace_bytes);
  const int64_t ld0 = ld4(m->dims[0]);
  float* in_hi = ar.take<float>(n_rows * ld0);
  float* in_lo = ar.take<float>(n_rows * ld0);
  const int64_t hld = ld4(std::max(m->max_hidden, 8));
  float* buf[2][2];
  for (int i = 0; i < 2; ++i) for (int j = 0; j < 2; ++j) buf[i][j] = ar.take<float>(n_rows * hld);
  if (!ar.ok()) { set_error("mlp_forward: workspace too small (%lld bytes given, %lld needed)", (long long)workspace_bytes, (long long)lcrec_mlp_workspace_bytes(m, n_rows)); return LCREC_ERR_NOMEM; }
  { ProfScope prof(0, st); LC_TRY(launch_split(x, n_rows, m->dims[0], m->dims[0], in_hi, in_lo, ld0, st)); }
  const float *a_hi = in_hi, *a_lo = in_lo;
  int64_t lda = ld0;
  for (int l = 0; l < m->n_layers; ++l) {
    const bool last = (l == m->n_layers - 1);
    LinearProblem p{};
    p.a_hi = a_hi; p.a_lo = a_lo; p.n_rows = n_rows; p.k = m->dims[l]; p.lda = lda;
    p.w_hi = m->w_hi[l]; p.w_lo = m->w_lo[l]; p.n_out = m->dims[l + 1]; p.ldw = m->ldw[l];
    p.bias = m->bias[l]; p.relu = last ? m->relu_last : 1;
    p.acc_chunk = m->acc_chunk; p.variant = m->variant;
    if (last) { p.y = y; p.ldy = m->dims[l + 1]; }
    else {
      p.y_hi = buf[l & 1][0]; p.y_lo = buf[l & 1][1]; p.ld_split = ld4(m->dims[l + 1]);
      if (acts && acts[l]) { p.y = acts[l]; p.ldy = m->dims[l + 1]; }
    }
    if (p.ldy && ((p.ldy & 3) || (reinterpret_cast<uintptr_t>(p.y) & 15))) {
      set_error("mlp_forward: output width %lld must be a multiple of 4 floats and 16-byte aligned", (long long)p.ldy);
      return LCREC_ERR_UNSUPPORTED;
    }
    { ProfScope prof(1 + std::min(l, 15), st); LC_TRY(launch_linear(p, st)); }
    a_hi = p.y_hi; a_lo = p.y_lo; lda = p.ld_split;
  }
  if (acts && acts[m->n_layers - 1] && acts[m->n_layers - 1] != y)
    LC_CUDA(cudaMemcpyAsync(acts[m->n_layers - 1], y, sizeof(float) * n_rows * m->dims[m->n_layers], cudaMemcpyDeviceToDevice, st));
  return LCREC_OK;
}

// Single fused Linear(+bias)(+ReLU) on raw fp32 operands (splits both on the fly into `ws`).
// variant: bit 0 = alternative tile for wide N, bit 1 = f16 x3 engine instead of tf32 x3.
extern "C" int64_t lcrec_linear_workspace_bytes(int64_t n_rows, int k_in, int n_out) {
  return 2 * arena_need(sizeof(float) * n_rows * ld4(k_in)) + 2 * arena_need(sizeof(float) * (int64_t)n_out * ld4(k_in)) +
         arena_need(sizeof(float) * n_rows * std::max<int64_t>(1, ceil_div(ld8(k_in), 128))) + arena_need(sizeof(float) * n_out) + 1024;
}
extern "C" int lcrec_linear_forward(const float* x, int64_t n_rows, int k_in, const float* w, const float* b,
                                    int n_out, int relu, float* y, int acc_chunk, int variant, void* ws,
                                    int64_t ws_bytes, void* stream) {
  LC_ARG(n_rows >= 0 && k_in > 0 && n_out > 0);
  LC_TRY(lcrec_device_check());
  if (n_rows == 0) return LCREC_OK;
  LC_ARG(x && w && y);
  LC_ARG((n_out & 3) == 0);
  cudaStream_t st = (cudaStream_t)stream;
  Arena ar(ws, ws_bytes);
  LinearProblem p{};
  p.n_rows = n_rows; p.k = k_in; p.n_out = n_out; p.bias = b; p.relu = relu;
  p.y = y; p.ldy = n_out; p.acc_chunk = acc_chunk; p.variant = variant & 1;
  if ((variant & 6) == 6) {      // CTA-pair kernel, group-scaled activations (n_out must be a multiple of 256)
    const int64_t ldk = ld8(k_in);
    __half* a_hi = ar.take<__half>(n_rows * ldk); __half* a_lo = ar.take<__half>(n_rows * ldk);
    __half* w_hi = ar.take<__half>((int64_t)n_out * ldk); __half* w_lo = ar.take<__half>((int64_t)n_out * ldk);
    float* cs = ar.take<float>(n_out);
    float* as = ar.take<float>(n_rows * ceil_div(ldk, kPairGroup));
    if (!ar.ok()) { set_error("linear_forward: workspace too small"); return LCREC_ERR_NOMEM; }
    LC_TRY(launch_split_groups(x, kDtypeF32, n_rows, k_in, k_in, a_hi, a_lo, ldk, as, n_rows, st));
    LC_TRY(launch_split_f16(w, n_out, k_in, k_in, w_hi, w_lo, ldk, cs, st));
    PairProblem q{};
    q.a.hi = a_hi; q.a.lo = a_lo; q.a.ld = ldk; q.a.inv_scale = as; q.a.ld_scale = n_rows; q.a.group = kPairGroup;
    q.n_rows = n_rows; q.k = k_in; q.w_hi = w_hi; q.w_lo = w_lo; q.ldw = ldk; q.w_inv_scale = cs; q.n_out = n_out;
    q.bias = b; q.relu = relu; q.y = y; q.ldy = n_out; q.debug = (variant & 1) ? 4 : 0;
    return launch_linear_pair(q, st);
  }
  if (variant & 2) {
    const int64_t ldk = ld8(k_in);
    __half* a_hi = ar.take<__half>(n_rows * ldk); __half* a_lo = ar.take<__half>(n_rows * ldk);
    __half* w_hi = ar.take<__half>((int64_t)n_out * ldk); __half* w_lo = ar.take<__half>((int64_t)n_out * ldk);
    float* rs = ar.take<float>(n_rows); float* cs = ar.take<float>(n_out);
    if (!ar.ok()) { set_error("linear_forward: workspace too small"); return LCREC_ERR_NOMEM; }
    LC_TRY(launch_split_f16(x, n_rows, k_in, k_in, a_hi, a_lo, ldk, rs, st));
    LC_TRY(launch_split_f16(w, n_out, k_in, k_in, w_hi, w_lo, ldk, cs, st));
    p.f16 = true; p.row_scale = rs; p.col_scale = cs;
    p.a_hi = a_hi; p.a_lo = a_lo; p.lda = ldk; p.w_hi = w_hi; p.w_lo = w_lo; p.ldw = ldk;
    return launch_linear(p, st);
  }
  const int64_t ldk = ld4(k_in);
  float* a_hi = ar.take<float>(n_rows * ldk); float* a_lo = ar.take<float>(n_rows * ldk);
  float* w_hi = ar.take<float>((int64_t)n_out * ldk); float* w_lo = ar.take<float>((int64_t)n_out * ldk);
  if (!ar.ok()) { set_error("linear_forward: workspace too small"); return LCREC_ERR_NOMEM; }
  LC_TRY(launch_split(x, n_rows, k_in, k_in, a_hi, a_lo, ldk, st));
  LC_TRY(launch_split(w, n_out, k_in, k_in, w_hi, w_lo, ldk, st));
  p.a_hi = a_hi; p.a_lo = a_lo; p.lda = ldk; p.w_hi = w_hi; p.w_lo = w_lo; p.ldw = ldk;
  return launch_linear(p, st);
}

// ====================================================================== backward of one Linear(+ReLU)
// Training path (trainer.py:114-118: loss.backward()): for y = relu?(x W^T + b)
//   g  = gy * (y > 0)            (ReLU mask, only when the forward fused the ReLU)
//   gb = sum_rows g              gx = g W              gw = g^T x
// Both GEMMs run on the same fp32-accurate split-operand tensor-core kernels as the forward (the contraction
// dimension has to be the fastest one of both operands, so W, g and x are transposed by a tiled copy first).
namespace lcrec {

// out (cols x ldo) = in (rows x cols)^T, ldo >= rows
__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ in, int64_t rows, int64_t cols,
                                                        float* __restrict__ out, int64_t ldo) {
  __shared__ float tile[32][33];
  const int64_t tiles_c = (cols + 31) / 32, tiles_r = (rows + 31) / 32;
  for (int64_t t = blockIdx.x; t < tiles_c * tiles_r; t += gridDim.x) {
    const int64_t r0 = (t / tiles_c) * 32, c0 = (t % tiles_c) * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int j = ty; j < 32; j += 8)
      if (r0 + j < rows && c0 + tx < cols) tile[j][tx] = in[(r0 + j) * cols + c0 + tx];
    __syncthreads();
    for (int j = ty; j < 32; j += 8)
      if (c0 + j < cols && r0 + tx < rows) out[(c0 + j) * ldo + r0 + tx] = tile[tx][j];
    __syncthreads();
  }
}

// g = gy * (y > 0) (y null: g = gy) and the bias gradient gb[c] = sum over rows of g[:, c].
// Grid = (column blocks of 32) x (row splits): one CTA per 32 columns only filled 2..128 CTAs and walked the whole batch
// serially per thread (35 us per launch on average at batch 1024, 0.5 ms per training step over the 14 layers).  Each CTA
// now sums its row block in a fixed order into part[split][c]; the second kernel adds the <= 16 partials in split order
// (deterministic, no atomics).
constexpr int kMaskSplits = 16;
__global__ void __launch_bounds__(256) relu_mask_bias_partial_kernel(const float* __restrict__ gy, const float* __restrict__ y,
                                                                     int64_t rows, int cols, int splits, float* __restrict__ g,
                                                                     float* __restrict__ part) {
  __shared__ float red[8][32];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + tx;
  const int64_t r0 = rows * blockIdx.y / splits, r1 = rows * (blockIdx.y + 1) / splits;
  float s = 0.f;
  if (c < cols)
    for (int64_t r = r0 + ty; r < r1; r += 8) {
      float v = gy[r * cols + c];
      if (y != nullptr && !(y[r * cols + c] > 0.f)) v = 0.f;
      if (g != nullptr) g[r * cols + c] = v;
      s += v;
    }
  red[ty][tx] = s;
  __syncthreads();
  if (ty == 0 && c < cols && part != nullptr) {
    float t = 0.f;
    for (int j = 0; j < 8; ++j) t += red[j][tx];
    part[(size_t)blockIdx.y * cols + c] = t;
  }
}

__global__ void bias_grad_final_kernel(const float* __restrict__ part, int cols, int splits, float* __restrict__ gb) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= cols) return;
  float t = 0.f;
  for (int s = 0; s < splits; ++s) t += part[(size_t)s * cols + c];
  gb[c] = t;
}

static int mask_splits(int64_t rows, int cols) {
  const int64_t cb = ceil_div(cols, 32);
  int64_t s = std::max<int64_t>(1, std::min<int64_t>(kMaskSplits, (4 * (int64_t)num_sms()) / std::max<int64_t>(cb, 1)));
  return (int)std::min<int64_t>(s, std::max<int64_t>(1, rows / 32));
}

static int launch_transpose(const float* in, int64_t rows, int64_t cols, float* out, int64_t ldo, cudaStream_t st) {
  if (rows == 0 || cols == 0) return LCREC_OK;
  const int64_t tiles = ceil_div(rows, 32) * ceil_div(cols, 32);
  transpose_kernel<<<(unsigned)std::min<int64_t>(tiles, (int64_t)num_sms() * 16), 256, 0, st>>>(in, rows, cols, out, ldo);
  LC_LAUNCH_CHECK("transpose_kernel");
  return LCREC_OK;
}

static inline int64_t pad8(int64_t v) { return round_up(std::max<int64_t>(v, 1), 8); }

}  // namespace lcrec

extern "C" int64_t lcrec_linear_backward_workspace_bytes(int64_t n_rows, int k_in, int n_out) {
  const int64_t nr = pad8(n_rows);
  // g, g^T (padded batch), x^T (padded batch), W^T + the workspaces of the two GEMM calls
  return arena_need(sizeof(float) * kMaskSplits * n_out) + arena_need(sizeof(float) * n_rows * n_out) + arena_need(sizeof(float) * (int64_t)n_out * nr) +
         arena_need(sizeof(float) * (int64_t)k_in * nr) + arena_need(sizeof(float) * (int64_t)k_in * n_out) +
         std::max(lcrec_linear_workspace_bytes(n_rows, n_out, k_in), lcrec_linear_workspace_bytes(n_out, (int)nr, k_in)) + 1024;
}

extern "C" int lcrec_linear_backward(const float* x, const float* w, const float* y_relu, const float* gy, int64_t n_rows,
                                     int k_in, int n_out, float* gx, float* gw, float* gb, void* ws, int64_t ws_bytes,
                                     void* stream) {
  LC_ARG(n_rows >= 0 && k_in > 0 && n_out > 0 && (k_in & 3) == 0 && (n_out & 3) == 0);
  LC_TRY(lcrec_device_check());
  cudaStream_t st = (cudaStream_t)stream;
  if (n_rows == 0) {
    if (gw) LC_CUDA(cudaMemsetAsync(gw, 0, sizeof(float) * (size_t)n_out * k_in, st));
    if (gb) LC_CUDA(cudaMemsetAsync(gb, 0, sizeof(float) * n_out, st));
    return LCREC_OK;
  }
  LC_ARG(gy != nullptr && (gx == nullptr || w != nullptr) && (gw == nullptr || x != nullptr));
  const int64_t nr = pad8(n_rows);
  Arena ar(ws, ws_bytes);
  float* g = ar.take<float>(n_rows * n_out);
  float* gt = ar.take<float>((int64_t)n_out * nr);
  float* xt = ar.take<float>((int64_t)k_in * nr);
  float* wt = ar.take<float>((int64_t)k_in * n_out);
  const int64_t sub_bytes = std::max(lcrec_linear_workspace_bytes(n_rows, n_out, k_in), lcrec_linear_workspace_bytes(n_out, (int)nr, k_in));
  char* sub = ar.take<char>(sub_bytes);
  float* gb_part = ar.take<float>((int64_t)kMaskSplits * n_out);
  if (!ar.ok()) { set_error("linear_backward: workspace too small (%lld given, %lld needed)", (long long)ws_bytes, (long long)lcrec_linear_backward_workspace_bytes(n_rows, k_in, n_out)); return LCREC_ERR_NOMEM; }
  const float* gsrc = gy;
  if (y_relu != nullptr || gb != nullptr) {
    const int splits = mask_splits(n_rows, n_out);
    relu_mask_bias_partial_kernel<<<dim3((unsigned)ceil_div(n_out, 32), (unsigned)splits), 256, 0, st>>>(
        gy, y_relu, n_rows, n_out, splits, y_relu ? g : nullptr, gb ? gb_part : nullptr);
    LC_LAUNCH_CHECK("relu_mask_bias_partial_kernel");
    if (gb) {
      bias_grad_final_kernel<<<(unsigned)ceil_div(n_out, 256), 256, 0, st>>>(gb_part, n_out, splits, gb);
      LC_LAUNCH_CHECK("bias_grad_final_kernel");
    }
    if (y_relu) gsrc = g;
  }
  auto variant_for = [](int k, int n) { return linear_pair_supported(k, n, kPairGroup) ? 6 : 2; };
  if (gx != nullptr) {      // gx (n x K) = g (n x N) . W (N x K): "weights" = W^T (K x N), contraction over N
    LC_TRY(launch_transpose(w, n_out, k_in, wt, n_out, st));
    LC_TRY(lcrec_linear_forward(gsrc, n_rows, n_out, wt, nullptr, k_in, 0, gx, 64, variant_for(n_out, k_in), sub, sub_bytes, stream));
  }
  if (gw != nullptr) {      // gw (N x K) = g^T (N x n) . x (n x K): "weights" = x^T (K x n), contraction over the batch
    if (nr != n_rows) {     // zero the padded batch columns (the split kernels read whole rows)
      LC_CUDA(cudaMemsetAsync(gt, 0, sizeof(float) * (size_t)n_out * nr, st));
      LC_CUDA(cudaMemsetAsync(xt, 0, sizeof(float) * (size_t)k_in * nr, st));
    }
    LC_TRY(launch_transpose(gsrc, n_rows, n_out, gt, nr, st));
    LC_TRY(launch_transpose(x, n_rows, k_in, xt, nr, st));
    LC_TRY(lcrec_linear_forward(gt, n_out, (int)nr, xt, nullptr, k_in, 0, gw, 64, variant_for((int)nr, k_in), sub, sub_bytes, stream));
  }
  return LCREC_OK;
}

// ====================================================================== backward of a whole MLP stack
// acts[l] = output of layer l (fp32, ReLU applied for l < n_layers - 1, exactly what lcrec_mlp_forward returns through
// `acts`); gy = gradient w.r.t. the last layer's output.  gw[l] / gb[l] receive the parameter gradients, gx (nullable)
// the gradient w.r.t. the input.  One native loop over lcrec_linear_backward (no per-layer host round trip).
extern "C" int64_t lcrec_mlp_backward_workspace_bytes(const lcrec_mlp_t* m, int64_t n_rows) {
  if (!m || n_rows < 0) return -1;
  int64_t sub = 0; int widest = 0;
  for (int l = 0; l < m->n_layers; ++l) {
    sub = std::max(sub, lcrec_linear_backward_workspace_bytes(n_rows, m->dims[l], m->dims[l + 1]));
    widest = std::max(widest, m->dims[l]);
  }
  return sub + 2 * arena_need(sizeof(float) * n_rows * widest) + 1024;
}

extern "C" int lcrec_mlp_backward(lcrec_mlp_t* m, const float* const* weights, const float* x, const float* const* acts,
                                  const float* gy, int64_t n_rows, float* gx, float* const* gw, float* const* gb, void* ws,
                                  int64_t ws_bytes, void* stream) {
  LC_ARG(m && weights && acts && gy && gw && n_rows >= 0);
  LC_ARG(x != nullptr || n_rows == 0);
  int widest = 0;
  for (int l = 0; l < m->n_layers; ++l) widest = std::max(widest, m->dims[l]);
  Arena ar(ws, ws_bytes);
  float* gbuf[2] = {ar.take<float>(n_rows * widest), ar.take<float>(n_rows * widest)};
  int64_t sub_bytes = 0;
  for (int l = 0; l < m->n_layers; ++l) sub_bytes = std::max(sub_bytes, lcrec_linear_backward_workspace_bytes(n_rows, m->dims[l], m->dims[l + 1]));
  char* sub = ar.take<char>(sub_bytes);
  if (!ar.ok()) { set_error("mlp_backward: workspace too small"); return LCREC_ERR_NOMEM; }
  const float* g = gy;
  for (int l = m->n_layers - 1; l >= 0; --l) {
    const bool relu = (l != m->n_layers - 1) || m->relu_last;
    const float* in = l == 0 ? x : acts[l - 1];
    float* g_prev = l == 0 ? gx : gbuf[l & 1];
    LC_ARG(weights[l] != nullptr && acts[l] != nullptr && gw[l] != nullptr);
    LC_TRY(lcrec_linear_backward(in, weights[l], relu ? acts[l] : nullptr, g, n_rows, m->dims[l], m->dims[l + 1], g_prev, gw[l],
                                 gb ? gb[l] : nullptr, sub, sub_bytes, stream));
    g = g_prev;
  }
  return LCREC_OK;
}
