// Internal interface between the GEMM translation units (linear_tf32x3.cu, linear_pair.cu).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace lcrec {

// 2-D tiled tensor map over a row-major (rows, k) matrix of `elem`-byte elements with row stride ld (elements);
// box = (bk, box_rows); swizzle span = bk * elem bytes (64 or 128); out-of-bounds reads give zeros.
int make_map(CUtensorMap* m, const void* ptr, int64_t rows, int k, int64_t ld, int bk, int box_rows, int elem);

// Group-scaled fp16 split operand: value(row, c) = (hi + lo)(row, c) * inv_scale[(c / group) * ld_scale + row]
struct SplitOperand {
  const __half* hi = nullptr;
  const __half* lo = nullptr;
  int64_t ld = 0;               // row stride in elements (multiple of 8)
  const float* inv_scale = nullptr;
  int64_t ld_scale = 0;         // stride between scale groups (>= n_rows)
  int group = 0;                // K elements per scale group
};

struct PairProblem {
  SplitOperand a; int64_t n_rows; int k;
  const __half *w_hi, *w_lo; int64_t ldw; const float* w_inv_scale;   // per output channel (n_out)
  int n_out;                    // multiple of 256
  const float* bias; int relu;
  float* y; int64_t ldy;        // fp32 output or null
  __half *o_hi, *o_lo; int64_t ldo; float* o_inv_scale; int64_t ld_oscale;   // group-scaled output (group 256) or null
  int debug;
  void* trace = nullptr;        // measurement only (see linear_pair.cu)
  // distance + argmin mode (launch_argmin_pair): squared norms of the rows / codes, output codes (stride in elements)
  const float* xx = nullptr; const float* cc = nullptr; int64_t* codes = nullptr; int64_t codes_stride = 0;
};

// Linear(+bias)(+ReLU) on CTA pairs (tcgen05 cta_group::2, 256 x 256 tiles, persistent).  n_out % 256 == 0.
int launch_linear_pair(const PairProblem& p, cudaStream_t st);
bool linear_pair_supported(int k, int n_out, int group);
int launch_argmin_pair(const PairProblem& p, cudaStream_t st);
bool argmin_pair_supported(int k, int n_out);
void set_pair_cluster_cap(int cap);   // 0 = all CTA pairs the device holds
constexpr int kPairGroup = 256;

// x (rows, k) of element type `dtype` (kDtypeF32 / kDtypeF16 / kDtypeBF16; ldx in elements) -> group-scaled fp16 hi/lo
// (one pass; scale groups of 256 elements)
int launch_split_groups(const void* x, int dtype, int64_t rows, int k, int64_t ldx, __half* hi, __half* lo, int64_t ld_out,
                        float* inv_scale, int64_t ld_scale, cudaStream_t st);

// ReLU of the GEMM epilogues: 0 for finite negative values only.  NaN passes like torch.relu; -inf passes too, because
// with finite operands it only comes from an overflow of the fp32 accumulator (which on the f16 x3 engine carries the
// channel scale 2^15 / max|w_c|), and a ReLU of it would turn an out-of-range result into a finite 0.  Unlike torch.relu
// it also keeps a truly -inf pre-activation (an input row holding inf); that row is non-finite either way.
__device__ __forceinline__ float relu_keep_nonfinite(float t) { return (t < 0.f && t > -INFINITY) ? 0.f : t; }

// Input loads of the operand splits.  Both half formats convert to fp32 exactly, so everything after the load is the
// arithmetic of the fp32 input.
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }

// four consecutive elements at p -> v[0..3]; p 16-byte aligned (fp32) or 8-byte aligned (halves).  STREAM: __ldcs, for
// an input that is read once.
template <bool STREAM>
__device__ __forceinline__ void load4_f32(const float* p, float* v) {
  float4 t;
  if constexpr (STREAM) t = __ldcs(reinterpret_cast<const float4*>(p));
  else t = *reinterpret_cast<const float4*>(p);
  v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <bool STREAM>
__device__ __forceinline__ void load4_f32(const __half* p, float* v) {
  uint2 t;
  if constexpr (STREAM) t = __ldcs(reinterpret_cast<const uint2*>(p));
  else t = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&t.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&t.y));
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
template <bool STREAM>
__device__ __forceinline__ void load4_f32(const __nv_bfloat16* p, float* v) {
  uint2 t;
  if constexpr (STREAM) t = __ldcs(reinterpret_cast<const uint2*>(p));
  else t = *reinterpret_cast<const uint2*>(p);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.y));
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}

}  // namespace lcrec
