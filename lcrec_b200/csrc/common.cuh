// Shared helpers for the lcrec_b200 C-ABI library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

#include "../../include/lcrec_b200.h"

namespace lcrec {

void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launches;

inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

#define LC_CUDA(expr)                                                                        \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess) {                                                                 \
      lcrec::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      (void)cudaGetLastError();                                                              \
      return LCREC_ERR_CUDA;                                                                 \
    }                                                                                        \
  } while (0)

#define LC_LAUNCH_CHECK(name)                                                                \
  do {                                                                                       \
    cudaError_t _e = cudaGetLastError();                                                     \
    if (_e != cudaSuccess) {                                                                 \
      lcrec::set_error("launch of %s failed: %s (%s:%d)", name, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return LCREC_ERR_CUDA;                                                                 \
    }                                                                                        \
    lcrec::count_launch();                                                                   \
  } while (0)

#define LC_ARG(cond)                                                                         \
  do {                                                                                       \
    if (!(cond)) {                                                                           \
      lcrec::set_error("bad argument: %s (%s:%d)", #cond, __FILE__, __LINE__);               \
      return LCREC_ERR_ARG;                                                                  \
    }                                                                                        \
  } while (0)

#define LC_TRY(expr)                                                                         \
  do {                                                                                       \
    int _r = (expr);                                                                         \
    if (_r != LCREC_OK) return _r;                                                           \
  } while (0)

// element type codes of inputs that may be half precision (the `dtype` arguments of the C ABI)
constexpr int kDtypeF32 = 0, kDtypeF16 = 1, kDtypeBF16 = 2;
inline bool dtype_ok(int dtype) { return dtype == kDtypeF32 || dtype == kDtypeF16 || dtype == kDtypeBF16; }
inline int64_t dtype_bytes(int dtype) { return dtype == kDtypeF32 ? 4 : 2; }

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }
inline int64_t ceil_div(int64_t x, int64_t m) { return (x + m - 1) / m; }

int num_sms();

// Optional per-stage device timing (CUDA events on the launching stream), used by bench.py for the
// live roofline figure.  Tags: 0 = split, 1..16 = MLP layer l, 17 = tail splits, 20 = rq, 21 = collide, 22 = sinkhorn of the
// first round, 23 = sinkhorn of the later rounds, 24 = warp-class kernels / 26 = literal re-run inside a sinkhorn call.
constexpr int kProfTags = 32;
void prof_begin(int tag, cudaStream_t st);
void prof_end(int tag, cudaStream_t st);
struct ProfScope {
  int tag; cudaStream_t st;
  ProfScope(int t, cudaStream_t s) : tag(t), st(s) { prof_begin(tag, st); }
  ~ProfScope() { prof_end(tag, st); }
};

// bump allocator over a caller-provided workspace
struct Arena {
  char* base; int64_t size; int64_t off;
  Arena(void* p, int64_t n) : base((char*)p), size(n), off(0) {}
  template <typename T> T* take(int64_t count) {
    int64_t start = round_up(off, 256);
    int64_t end = start + (int64_t)sizeof(T) * count;
    if (end > size || base == nullptr) { off = size + 1; return nullptr; }
    off = end;
    return (T*)(base + start);
  }
  bool ok() const { return off <= size; }
};
inline int64_t arena_need(int64_t bytes) { return round_up(bytes, 256) + 256; }

}  // namespace lcrec
