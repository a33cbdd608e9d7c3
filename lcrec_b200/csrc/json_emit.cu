// `.index.json` emission on the device (SURVEY 8(f) rank 2; reference index/generate_indices.py:83,138-145):
// json.dump({item: ["<a_%d>", "<b_%d>", ...]}) with int keys, default separators - byte for byte:
//     {"0": ["<a_12>", "<b_3>", "<c_4>", "<d_5>"], "1": [...], ...}
// The reference builds the dict and the string in Python (seconds at 1 M items against a 75 ms GPU step).  Here it is byte
// work over the code table already resident in HBM: row lengths -> block sums -> one-CTA scan -> every CTA formats its 1024
// rows at their final offsets (~50 B/row written once); the caller copies the bytes to the host and writes the file.
#include <algorithm>

#include "common.cuh"

namespace lcrec {

constexpr int kJsThreads = 256;
constexpr int kJsRowsPerThread = 4;
constexpr int kJsRowsPerCta = kJsThreads * kJsRowsPerThread;

__device__ __forceinline__ int dec_digits(unsigned long long v) {
  int d = 1;
  while (v >= 10ull) { v /= 10ull; ++d; }
  return d;
}

// bytes of row i (key item_base + i) including the ", " in front of every row whose key is not 0
__device__ __forceinline__ int row_bytes(const int64_t* __restrict__ codes, int64_t i, int64_t item_base, int L) {
  const int64_t key = item_base + i;
  int len = (key ? 2 : 0) + 1 + dec_digits((unsigned long long)key) + 1 + 2 + 1 + 1 + 2 * (L - 1);     // [, ]"key": [ ... ]
  for (int l = 0; l < L; ++l) len += 6 + dec_digits((unsigned long long)codes[i * L + l]);           // "<a_ digits >"
  return len;
}

__device__ __forceinline__ char* put_dec(char* p, unsigned long long v) {
  char tmp[20];
  int n = 0;
  do { tmp[n++] = (char)('0' + (int)(v % 10ull)); v /= 10ull; } while (v);
  while (n) *p++ = tmp[--n];
  return p;
}

__global__ void __launch_bounds__(kJsThreads) json_block_sums_kernel(const int64_t* __restrict__ codes, int64_t n, int64_t item_base,
                                                                     int L, long long* __restrict__ block_sums) {
  __shared__ long long red[kJsThreads / 32];
  const int64_t base = (int64_t)blockIdx.x * kJsRowsPerCta + (int64_t)threadIdx.x * kJsRowsPerThread;
  long long s = 0;
  for (int r = 0; r < kJsRowsPerThread; ++r)
    if (base + r < n) s += row_bytes(codes, base + r, item_base, L);
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long t = 0;
    for (int w = 0; w < kJsThreads / 32; ++w) t += red[w];
    block_sums[blockIdx.x] = t;
  }
}

// exclusive scan of n_blocks sums in place (+1 for the leading '{' if braces); total bytes (with the closing '}' if braces)
// -> sums[n_blocks]
__global__ void json_scan_kernel(long long* __restrict__ sums, int n_blocks, int braces) {
  __shared__ long long carry;
  __shared__ long long wsum[32];
  if (threadIdx.x == 0) carry = braces;
  __syncthreads();
  for (int base = 0; base < n_blocks; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const long long v = i < n_blocks ? sums[i] : 0;
    long long x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, x, o); if ((threadIdx.x & 31) >= o) x += y; }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = x;
    __syncthreads();
    if (threadIdx.x < 32) {
      long long w = threadIdx.x < (blockDim.x >> 5) ? wsum[threadIdx.x] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, w, o); if (threadIdx.x >= o) w += y; }
      wsum[threadIdx.x] = w;
    }
    __syncthreads();
    const long long before = carry + (threadIdx.x >= 32 ? wsum[(threadIdx.x >> 5) - 1] : 0) + x - v;
    if (i < n_blocks) sums[i] = before;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = before + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) sums[n_blocks] = carry + braces;
}

__global__ void __launch_bounds__(kJsThreads) json_write_kernel(const int64_t* __restrict__ codes, int64_t n, int64_t item_base,
                                                                int L, int braces, const long long* __restrict__ block_off,
                                                                char* __restrict__ out, long long cap) {
  __shared__ long long wsum[kJsThreads / 32];
  const int64_t base = (int64_t)blockIdx.x * kJsRowsPerCta + (int64_t)threadIdx.x * kJsRowsPerThread;
  int len[kJsRowsPerThread];
  long long mine = 0;
  for (int r = 0; r < kJsRowsPerThread; ++r) { len[r] = base + r < n ? row_bytes(codes, base + r, item_base, L) : 0; mine += len[r]; }
  long long x = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const long long y = __shfl_up_sync(0xffffffffu, x, o); if ((threadIdx.x & 31) >= o) x += y; }
  if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = x;
  __syncthreads();
  long long off = block_off[blockIdx.x] + x - mine;
  for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) off += wsum[w];
  if (braces && blockIdx.x == 0 && threadIdx.x == 0) {
    out[0] = '{';
    const long long total = block_off[gridDim.x];
    if (total <= cap) out[total - 1] = '}';
  }
  for (int r = 0; r < kJsRowsPerThread; ++r) {
    const int64_t i = base + r;
    if (i >= n) break;
    if (off + len[r] > cap) return;                  // caller's buffer too small: total is reported, nothing overruns
    char* p = out + off;
    const int64_t key = item_base + i;
    if (key) { *p++ = ','; *p++ = ' '; }
    *p++ = '"';
    p = put_dec(p, (unsigned long long)key);
    *p++ = '"'; *p++ = ':'; *p++ = ' '; *p++ = '[';
    for (int l = 0; l < L; ++l) {
      if (l) { *p++ = ','; *p++ = ' '; }
      *p++ = '"'; *p++ = '<'; *p++ = (char)('a' + l); *p++ = '_';
      p = put_dec(p, (unsigned long long)codes[i * L + l]);
      *p++ = '>'; *p++ = '"';
    }
    *p++ = ']';
    off += len[r];
  }
}

}  // namespace lcrec

using namespace lcrec;

extern "C" int64_t lcrec_index_json_workspace_bytes(int64_t n) {
  return arena_need((ceil_div(std::max<int64_t>(n, 1), kJsRowsPerCta) + 2) * 8);
}

// out (device, capacity out_cap bytes, nullable for a sizing call) <- the JSON text of codes (n x n_levels, int64, values >= 0),
// row i under the key item_base + i, with the enclosing braces if `braces`; total_bytes_dev (1 int64, device) <- its exact
// length.  n_levels <= 5 (the reference has five prefixes, :83).  The ", " goes in front of every row whose key is not 0, so the
// fragments of consecutive row blocks (braces 0), concatenated inside "{" and "}", are the text of the whole table.
extern "C" int lcrec_index_json_ex(const int64_t* codes, int64_t n, int n_levels, int64_t item_base, int braces, char* out,
                                   int64_t out_cap, int64_t* total_bytes_dev, void* ws, int64_t ws_bytes, void* stream) {
  LC_ARG(n >= 0 && n_levels >= 1 && n_levels <= 5 && total_bytes_dev && (n == 0 || codes) && out_cap >= 0);
  LC_ARG(item_base >= 0 && item_base <= INT64_MAX - n && (braces == 0 || braces == 1));
  LC_TRY(lcrec_device_check());
  cudaStream_t st = (cudaStream_t)stream;
  const int n_blocks = (int)ceil_div(std::max<int64_t>(n, 1), kJsRowsPerCta);
  Arena ar(ws, ws_bytes);
  long long* sums = ar.take<long long>(n_blocks + 2);
  if (!ar.ok()) { set_error("index_json: workspace too small"); return LCREC_ERR_NOMEM; }
  json_block_sums_kernel<<<n_blocks, kJsThreads, 0, st>>>(codes, n, item_base, n_levels, sums);
  LC_LAUNCH_CHECK("json_block_sums_kernel");
  json_scan_kernel<<<1, 1024, 0, st>>>(sums, n_blocks, braces);
  LC_LAUNCH_CHECK("json_scan_kernel");
  LC_CUDA(cudaMemcpyAsync(total_bytes_dev, sums + n_blocks, sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
  if (out && (braces ? out_cap >= 2 : n > 0)) {
    json_write_kernel<<<n_blocks, kJsThreads, 0, st>>>(codes, n, item_base, n_levels, braces, sums, out, out_cap);
    LC_LAUNCH_CHECK("json_write_kernel");
  }
  return LCREC_OK;
}

extern "C" int lcrec_index_json(const int64_t* codes, int64_t n, int n_levels, char* out, int64_t out_cap, int64_t* total_bytes_dev,
                                void* ws, int64_t ws_bytes, void* stream) {
  return lcrec_index_json_ex(codes, n, n_levels, 0, 1, out, out_cap, total_bytes_dev, ws, ws_bytes, stream);
}
