// fp32-accurate Linear(+bias, +ReLU) on CTA PAIRS: tcgen05.mma.cta_group::2, 256 x 256 output tiles, persistent.
//
// Same arithmetic as linear_split3_kernel<.., F16 = true> (reference: nn.Linear + ReLU inside MLPLayers.forward,
// index/models/layers.py:22-43): every fp32 product is evaluated as x_hi*w_hi + x_lo*w_hi + x_hi*w_lo on fp16
// operand pairs, accumulated in fp32 TMEM in chunks that fold warps add into fp32 registers.
//
// Why pairs.  The single-CTA 128 x 256 tile needs 48 KB of operands per 768 tensor-pipe cycles = 62.5 B/clk/SM from
// L2; the chip delivers ~45 B/clk/SM (measured: the kernel with its MMAs switched off runs at 12.3 TB/s and is only
// 1.4x faster than with them on).  With cta_group::2 the two SMs of a TPC share one 256-wide B tile, each CTA
// stages its own 128 A rows and HALF of the B rows: 32 KB per 768 cycles = 41.7 B/clk/SM.
//
// Operands carry per-(row, 128-column group) power-of-two scales instead of per-row scales: a scale group is
// exactly one TMEM accumulation chunk, so the fold is acc += chunk * inv_scale[row][chunk] (one FMA, exact scaling),
// and the epilogue of a layer can emit the NEXT layer's fp16 hi/lo operand directly (each epilogue thread owns one
// row x 128 columns = one scale group): no separate split pass and no fp32 round trip between the wide layers.
//
// CTA = 10 warps: warps 0-7 fold + epilogue, warp 8 = TMA producer (one lane), warp 9 = TMEM allocator + (leader
// CTA only) MMA issuer.  Persistent: cluster c walks tiles c, c + n_clusters, ...; the producer and the MMA thread
// run ahead into the next tile while the fold warps finish the epilogue of the previous one from registers.
#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>

#include "linear.cuh"
#include "sm100_ptx.cuh"

namespace lcrec {

using namespace ptx;

namespace {

constexpr int kPairThreads = 384;      // 12 warps = 3 warpgroups (setmaxnreg works on whole warpgroups); warps 10, 11 idle
constexpr int kStageWords = 32 * 32;   // per-warp epilogue transpose buffer (32 rows x 32 words, XOR-swizzled columns)
constexpr int kGroup = 256;            // K elements per scale group = TMEM accumulation chunk (see header comment)
constexpr int kTileN = 256;
constexpr int kHalfM = 128;            // rows per CTA

struct PairArgs {
  int64_t n_rows; int n_out; int k;
  int tiles_n; int64_t n_tiles;        // tiles of 256 x 256
  const float* a_inv_scale; int64_t ld_ascale;
  const float* w_inv_scale; const float* bias; int relu;
  float* y; int64_t ldy;
  __half* o_hi; __half* o_lo; int64_t ldo; float* o_inv_scale; int64_t ld_oscale;
  // ARGMIN mode (distance GEMM of the residual quantiser): d = (xx[row] + cc[col]) - 2 dot, first argmin over all n_out columns
  const float* xx; const float* cc; int64_t* codes; int64_t codes_stride;
  int debug;
  long long* trace;   // measurement only: clock64 stamps of cluster 0's leader CTA (6 roles x 512 events x 4)
};

template <int BK, int STAGES, int TILE_N = 256>
struct PairCfg {
  static constexpr int ROW_BYTES = BK * 2;
  static constexpr int A_BYTES = kHalfM * ROW_BYTES;             // this CTA's 128 A rows (one of hi / lo)
  static constexpr int B_BYTES = (TILE_N / 2) * ROW_BYTES;       // this CTA's half of the B rows (one of hi / lo)
  static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;  // A_hi, A_lo, B_hi, B_lo
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 256 + 8 * kStageWords * 4 + 1024 /* xch */ + 1024 /* alignment */;
  static constexpr uint32_t SBO = 8 * ROW_BYTES;
  static constexpr uint32_t LAYOUT = ROW_BYTES == 128 ? 2u : 4u;
  static constexpr int KB_PER_CHUNK = kGroup / BK;
  static_assert(ROW_BYTES == 128 || ROW_BYTES == 64, "a K block spans one 128 B or 64 B swizzle row");
  static_assert(kGroup % BK == 0, "a chunk is a whole number of K blocks");
  static_assert(TILE_N == 256 || TILE_N == 128 || TILE_N == 64, "tile widths");
  static_assert(B_BYTES % 1024 == 0, "operand slabs start on swizzle-atom boundaries");
  static_assert(SMEM_BYTES <= 232448, "shared memory");
};

__device__ __forceinline__ uint32_t leader_addr(uint32_t a) { return a & kPeerBitMask; }
__device__ __forceinline__ void stamp(long long* trace, int role, uint32_t idx, int slot) {
  if (trace != nullptr && idx < 512u) trace[((size_t)role * 512 + idx) * 4 + slot] = clock64();
}

template <int BK, int STAGES, bool ARGMIN, int TILE_N>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPairThreads, 1)
linear_pair_kernel(const __grid_constant__ CUtensorMap map_ahi, const __grid_constant__ CUtensorMap map_alo,
                   const __grid_constant__ CUtensorMap map_bhi, const __grid_constant__ CUtensorMap map_blo,
                   const PairArgs args) {
  using C = PairCfg<BK, STAGES, TILE_N>;
  static_assert(!ARGMIN || TILE_N == 256, "the argmin epilogue walks 256-wide code tiles");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;      // same offset in both CTAs of the pair
  uint8_t* smem = smem_raw + (base - raw);

  const uint32_t bar0 = base + STAGES * C::STAGE_BYTES;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };                      // leader's copy is the live one
  auto empty_bar = [&](int s) { return bar0 + 8u * (STAGES + s); };          // per CTA (multicast commit)
  auto tfull_bar = [&](int b) { return bar0 + 8u * (2 * STAGES + b); };      // per CTA (multicast commit)
  auto tempty_bar = [&](int b) { return bar0 + 8u * (2 * STAGES + 2 + b); }; // leader's copy is the live one
  const uint32_t tmem_slot = bar0 + 8u * (2 * STAGES + 4);
  volatile uint32_t* tmem_slot_ptr = (volatile uint32_t*)(smem + STAGES * C::STAGE_BYTES + 8 * (2 * STAGES + 4));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();           // 0 = leader
  const int64_t cluster_id = blockIdx.x >> 1;
  const int64_t n_clusters = gridDim.x >> 1;
  const int nkb = (args.k + BK - 1) / BK;
  const int nchunks = (nkb + C::KB_PER_CHUNK - 1) / C::KB_PER_CHUNK;
  long long* const trace = (blockIdx.x == 0) ? args.trace : nullptr;
  // work units: one 256 x 256 tile (linear mode, n fastest) or one 256-row block with ALL its column tiles (ARGMIN mode:
  // the running minimum of a row stays in the registers of the thread that owns it)
  const int inner = ARGMIN ? args.tiles_n : 1;
  const int64_t n_units = ARGMIN ? args.n_tiles / args.tiles_n : args.n_tiles;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(tfull_bar(b), 1); mbar_init(tempty_bar(b), 16); }
    fence_barrier_init();
  }
  if (warp == 8 && lane == 0) {
    prefetch_tensormap(&map_ahi); prefetch_tensormap(&map_alo);
    prefetch_tensormap(&map_bhi); prefetch_tensormap(&map_blo);
  }
  if (warp == 9) tmem_alloc_2sm(tmem_slot, 512);
  tc_fence_before();
  cluster_sync_all();                                 // barriers of both CTAs initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // register budget: the fold warps hold a 128-column fp32 accumulator + 64 TMEM words in flight
  // (setmaxnreg at the head of each role branch: warps 0-7 -> 224 registers, warps 8-11 -> 56)

  if (warp == 8) {
    // ------------------------------------------------------------ TMA producer (both CTAs)
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (lane == 0) {
      uint32_t it = 0;
      for (int64_t unit = cluster_id; unit < n_units; unit += n_clusters)
      for (int nn = 0; nn < inner; ++nn) {
        const int tile_n = ARGMIN ? nn : (int)(unit % args.tiles_n);
        const int64_t tile_m = ARGMIN ? unit : unit / args.tiles_n;
        const int row0 = (int)(tile_m * 256 + rank * kHalfM);
        const int col0 = tile_n * TILE_N + (int)rank * (TILE_N / 2);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1u;
          stamp(trace, 0, it, 0);
          mbar_wait(empty_bar(s), ph ^ 1u);
          stamp(trace, 0, it, 1);
          if (rank == 0) mbar_expect_tx(full_bar(s), 2 * C::STAGE_BYTES);    // bytes of both CTAs
          if ((args.debug & 1) && it >= (uint32_t)STAGES) {                  // measurement: no loads after the fill
            if (rank == 0) { asm volatile("mbarrier.complete_tx.shared::cta.b64 [%0], %1;" ::"r"(full_bar(s)), "r"(2 * C::STAGE_BYTES) : "memory"); }
            continue;
          }
          const uint32_t dst = base + s * C::STAGE_BYTES;
          const uint32_t bar = leader_addr(full_bar(s));
          tma_load_2d_2sm(dst, &map_ahi, bar, kb * BK, row0);
          tma_load_2d_2sm(dst + C::A_BYTES, &map_alo, bar, kb * BK, row0);
          tma_load_2d_2sm(dst + 2 * C::A_BYTES, &map_bhi, bar, kb * BK, col0);
          tma_load_2d_2sm(dst + 2 * C::A_BYTES + C::B_BYTES, &map_blo, bar, kb * BK, col0);
        }
      }
    }
    __syncwarp();
  } else if (warp == 9) {
    // ------------------------------------------------------------ MMA issuer (leader CTA, one thread)
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (rank == 0 && lane == 0) {
      constexpr uint32_t idesc = umma_idesc(256, TILE_N, 0);
      uint32_t it = 0, cc = 0;
      for (int64_t unit = cluster_id; unit < n_units; unit += n_clusters)
      for (int nn = 0; nn < inner; ++nn) {
        int kb = 0;
        for (int c = 0; c < nchunks; ++c, ++cc) {
          const uint32_t b = cc & 1u;
          stamp(trace, 2, cc, 0);
          mbar_wait(tempty_bar(b), ((cc >> 1) & 1u) ^ 1u);
          stamp(trace, 2, cc, 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + b * TILE_N;
          const int kb_end = min(nkb, kb + C::KB_PER_CHUNK);
          bool first = true;
          for (; kb < kb_end; ++kb, ++it) {
            const int s = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1u;
            stamp(trace, 1, it, 0);
            mbar_wait(full_bar(s), ph);
            stamp(trace, 1, it, 1);
            tc_fence_after();
            const uint32_t a_hi = base + s * C::STAGE_BYTES;
            const uint64_t d_ahi = umma_smem_desc(a_hi, C::SBO, C::LAYOUT);
            const uint64_t d_alo = umma_smem_desc(a_hi + C::A_BYTES, C::SBO, C::LAYOUT);
            const uint64_t d_bhi = umma_smem_desc(a_hi + 2 * C::A_BYTES, C::SBO, C::LAYOUT);
            const uint64_t d_blo = umma_smem_desc(a_hi + 2 * C::A_BYTES + C::B_BYTES, C::SBO, C::LAYOUT);
            if (!(args.debug & 2)) {
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) {
                const uint64_t adv = (uint64_t)(k * 32 >> 4);     // one MMA consumes 32 bytes along K
                umma_f16_2sm(d_tmem, d_alo + adv, d_bhi + adv, idesc, first ? 0u : 1u);   // small cross terms first
                umma_f16_2sm(d_tmem, d_ahi + adv, d_blo + adv, idesc, 1u);
                umma_f16_2sm(d_tmem, d_ahi + adv, d_bhi + adv, idesc, 1u);
                first = false;
              }
            }
            umma_commit_2sm(empty_bar(s), 3);         // both CTAs may refill this slot
            stamp(trace, 1, it, 2);
          }
          umma_commit_2sm(tfull_bar(b), 3);           // chunk complete in both CTAs' TMEM
        }
      }
    }
    __syncwarp();
  } else if (warp < 8) {
    // ------------------------------------------------------------ fold + epilogue warps (both CTAs)
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;");
    constexpr int NCOL = TILE_N / 2;                  // columns per thread (128 at full width) = half an output scale group
    const int q = warp & 3;                           // TMEM lane quarter this warp may access
    const int half = warp >> 2;                       // column half
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * NCOL);
    const uint32_t tempty_leader[2] = {leader_addr(tempty_bar(0)), leader_addr(tempty_bar(1))};
    uint32_t* stg = reinterpret_cast<uint32_t*>(smem + STAGES * C::STAGE_BYTES + 256) + warp * kStageWords;
    float* xch = reinterpret_cast<float*>(smem + STAGES * C::STAGE_BYTES + 256 + 8 * kStageWords * 4);   // 2 x 128 maxima
    uint32_t cc = 0, tcount = 0;
    float run_best = INFINITY; int run_idx = 0;            // ARGMIN: running minimum of this thread's row and column half
    for (int64_t unit = cluster_id; unit < n_units; unit += n_clusters)
    for (int nn = 0; nn < inner; ++nn, ++tcount) {
      const int tile_n = ARGMIN ? nn : (int)(unit % args.tiles_n);
      const int64_t tile_m = ARGMIN ? unit : unit / args.tiles_n;
      const int64_t row = tile_m * 256 + rank * kHalfM + q * 32 + lane;
      const bool row_ok = row < args.n_rows;
      const float* sc_ptr = args.a_inv_scale + (row_ok ? row : 0);
      float acc[NCOL];
#pragma unroll
      for (int i = 0; i < NCOL; ++i) acc[i] = 0.f;
      for (int c = 0; c < nchunks; ++c, ++cc) {
        const uint32_t b = cc & 1u;
        const float sc = __ldg(sc_ptr + (int64_t)c * args.ld_ascale);
        if (warp == 0 && lane == 0) stamp(trace, 3, cc, 0);
        mbar_wait(tfull_bar(b), (cc >> 1) & 1u);
        if (warp == 0 && lane == 0) stamp(trace, 3, cc, 1);
        tc_fence_after();
        if constexpr (NCOL >= 64) {
#pragma unroll
          for (int j = 0; j < NCOL; j += 64) {      // two TMEM loads in flight per wait
            uint32_t v0[32], v1[32];
            tmem_ld32(t_lane + b * TILE_N + (uint32_t)j, v0);
            tmem_ld32(t_lane + b * TILE_N + (uint32_t)(j + 32), v1);
            tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[j + i] = fmaf(__uint_as_float(v0[i]), sc, acc[j + i]);
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[j + 32 + i] = fmaf(__uint_as_float(v1[i]), sc, acc[j + 32 + i]);
          }
        } else {
          uint32_t v0[32];
          tmem_ld32(t_lane + b * TILE_N, v0);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[i] = fmaf(__uint_as_float(v0[i]), sc, acc[i]);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(tempty_leader[b]);
        if (warp == 0 && lane == 0) stamp(trace, 3, cc, 2);
      }
      const int col_base = tile_n * TILE_N + half * NCOL;
      if constexpr (ARGMIN) {
        // ---- distance + first-argmin epilogue (vq.py:71-75): d = (|r|^2 + |c|^2) - 2 r.c in fp32, strict < keeps the lowest
        // index inside the thread's ascending column scan; the two column halves of a row are merged at the end
        if (nn == 0) { run_best = INFINITY; run_idx = 0; }
        const float xr = __ldg(args.xx + (row_ok ? row : 0));
#pragma unroll
        for (int j = 0; j < NCOL; j += 4) {
          const float4 cs = __ldg(reinterpret_cast<const float4*>(args.w_inv_scale + col_base + j));
          const float4 cn = __ldg(reinterpret_cast<const float4*>(args.cc + col_base + j));
          const float d0 = (xr + cn.x) - 2.f * (acc[j] * cs.x), d1 = (xr + cn.y) - 2.f * (acc[j + 1] * cs.y);
          const float d2 = (xr + cn.z) - 2.f * (acc[j + 2] * cs.z), d3 = (xr + cn.w) - 2.f * (acc[j + 3] * cs.w);
          if (d0 < run_best) { run_best = d0; run_idx = col_base + j; }
          if (d1 < run_best) { run_best = d1; run_idx = col_base + j + 1; }
          if (d2 < run_best) { run_best = d2; run_idx = col_base + j + 2; }
          if (d3 < run_best) { run_best = d3; run_idx = col_base + j + 3; }
        }
        if (nn == inner - 1) {
          float* xb = xch;                                           // 2 x 128 best values
          int* xi = reinterpret_cast<int*>(stg);                     // this warp's staging words: 32 indices
          if (half == 1) { xb[kHalfM + q * 32 + lane] = run_best; xi[lane] = run_idx; }
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (half == 0) {
            const float ob = xb[kHalfM + q * 32 + lane];
            const int oi = reinterpret_cast<const int*>(stg + 4 * kStageWords)[lane];     // warp + 4 owns the other half
            if (ob < run_best || (ob == run_best && oi < run_idx)) { run_best = ob; run_idx = oi; }
            if (row_ok) args.codes[row * args.codes_stride] = (int64_t)run_idx;
          }
          asm volatile("bar.sync 1, 256;" ::: "memory");
        }
        continue;
      }
      // ---- epilogue from registers: 1/s_col, bias, ReLU; fp32 and / or the next layer's group-scaled fp16 pair
      if (warp == 0 && lane == 0) stamp(trace, 4, tcount, 0);
      float amax = 0.f;
#pragma unroll
      for (int j = 0; j < NCOL; j += 4) {
        const float4 cs = __ldg(reinterpret_cast<const float4*>(args.w_inv_scale + col_base + j));
        float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (args.bias) bv = __ldg(reinterpret_cast<const float4*>(args.bias + col_base + j));
        float t0 = acc[j] * cs.x + bv.x, t1 = acc[j + 1] * cs.y + bv.y, t2 = acc[j + 2] * cs.z + bv.z, t3 = acc[j + 3] * cs.w + bv.w;
        // ReLU that lets NaN through like torch.relu (fmaxf(NaN, 0) would be 0 and hide a diverged run from trainer.py:93-95),
        // and an accumulator overflow to -inf (linear.cuh)
        if (args.relu) { t0 = relu_keep_nonfinite(t0); t1 = relu_keep_nonfinite(t1); t2 = relu_keep_nonfinite(t2); t3 = relu_keep_nonfinite(t3); }
        acc[j] = t0; acc[j + 1] = t1; acc[j + 2] = t2; acc[j + 3] = t3;
        amax = fmaxf(fmaxf(amax, fmaxf(fabsf(t0), fabsf(t1))), fmaxf(fabsf(t2), fabsf(t3)));
      }
      if (warp == 0 && lane == 0) stamp(trace, 4, tcount, 1);
      // stores go through a per-warp shared-memory transpose so that every store instruction writes whole row
      // segments (a thread owns a ROW of the tile; written directly, each instruction would touch 32 rows)
      const int64_t row_base = tile_m * 256 + rank * kHalfM + q * 32;
      // staging layout: row r, 16-byte chunk c (4 columns) at word r * 32 + ((c ^ (r & 7)) << 2): conflict-free for the
      // row-per-lane 16-byte writes and for the 8-lanes-per-row 16-byte reads
      const int rsub = lane >> 3, csub = lane & 7;
      if (args.y && !(args.debug & 8)) {
#pragma unroll
        for (int jb = 0; jb < NCOL; jb += 32) {
#pragma unroll
          for (int c = 0; c < 8; ++c)
            *reinterpret_cast<float4*>(stg + lane * 32 + ((c ^ (lane & 7)) << 2)) =
                make_float4(acc[jb + 4 * c], acc[jb + 4 * c + 1], acc[jb + 4 * c + 2], acc[jb + 4 * c + 3]);
          __syncwarp();
          if (warp == 0 && lane == 0) stamp(trace, 5, tcount * 8 + jb / 16, 0);
          float* yb = args.y + row_base * args.ldy + col_base + jb + 4 * csub;
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int r = 4 * it + rsub;
            const float4 v = *reinterpret_cast<const float4*>(stg + r * 32 + ((csub ^ (r & 7)) << 2));
            if (row_base + r < args.n_rows) *reinterpret_cast<float4*>(yb + (int64_t)r * args.ldy) = v;
          }
          __syncwarp();
          if (warp == 0 && lane == 0) stamp(trace, 5, tcount * 8 + jb / 16 + 1, 0);
        }
      }
      if (args.o_hi) {
        // one scale per row and 256-column group = both column halves of the tile: exchange the maxima between the
        // two warps that own the halves of a row (named barrier over the 8 fold warps)
        xch[half * kHalfM + q * 32 + lane] = amax;
        asm volatile("bar.sync 1, 256;" ::: "memory");
        amax = fmaxf(amax, xch[(half ^ 1) * kHalfM + q * 32 + lane]);
        asm volatile("bar.sync 1, 256;" ::: "memory");     // xch is rewritten by the next tile
        // exponent-only scale: max|v s| in [2^14, 2^15); zero / inf / nan group -> s = 1
        float s = 1.f, is = 1.f;
        if (amax > 0.f && amax < INFINITY) {
          const int e = (int)((__float_as_uint(amax) >> 23) & 0xffu) - 127;      // floor(log2 amax) (normal numbers)
          const int sh = min(max(14 - e, -126), 126);
          s = __uint_as_float((uint32_t)(sh + 127) << 23); is = __uint_as_float((uint32_t)(127 - sh) << 23);
        }
        if (row_ok && half == 0) args.o_inv_scale[(int64_t)tile_n * args.ld_oscale + row] = is;
#pragma unroll
        for (int jb = 0; jb < NCOL; jb += 32) {
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            uint32_t w[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float xs = acc[jb + 4 * c + i] * s;                          // exact (power of two)
              const __half h = __float2half_rn(xs);
              const __half l = __float2half_rn(xs - __half2float(h));            // the difference is exact in fp32
              w[i] = (uint32_t)__half_as_ushort(h) | ((uint32_t)__half_as_ushort(l) << 16);
            }
            *reinterpret_cast<uint4*>(stg + lane * 32 + ((c ^ (lane & 7)) << 2)) = make_uint4(w[0], w[1], w[2], w[3]);
          }
          __syncwarp();
          __half* hb = args.o_hi + row_base * args.ldo + col_base + jb + 4 * csub;
          __half* lb = args.o_lo + row_base * args.ldo + col_base + jb + 4 * csub;
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            const int r = 4 * it + rsub;
            const uint4 w = *reinterpret_cast<const uint4*>(stg + r * 32 + ((csub ^ (r & 7)) << 2));
            if (row_base + r < args.n_rows) {
              *reinterpret_cast<uint2*>(hb + (int64_t)r * args.ldo) = make_uint2(__byte_perm(w.x, w.y, 0x5410), __byte_perm(w.z, w.w, 0x5410));
              *reinterpret_cast<uint2*>(lb + (int64_t)r * args.ldo) = make_uint2(__byte_perm(w.x, w.y, 0x7632), __byte_perm(w.z, w.w, 0x7632));
            }
          }
          __syncwarp();
        }
      }
      if (warp == 0 && lane == 0) stamp(trace, 4, tcount, 2);
    }
  }
  else {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");      // idle warps 10, 11 of the third warpgroup
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, 512);
  }
}

// x (rows, k) fp32 / fp16 / bf16 -> group-scaled fp16 pair, one pass: a warp owns a row, each iteration covers one
// 256-element group (two 4-element vectors per lane: float4, or 8 bytes of halves), group maximum by warp shuffles.
// Every element is converted to fp32 on load (exact for both half formats), so a half input gives the bits the fp32
// input x.float() gives.  Scales are staged in shared memory and written group-major ([group][row], coalesced over
// rows) - the layout the fold warps read.
constexpr int kSplitRowsPerCta = 32;
template <typename T>
__global__ void __launch_bounds__(256) split_groups_kernel(const T* __restrict__ x, int64_t rows, int k, int64_t ldx,
                                                           __half* __restrict__ hi, __half* __restrict__ lo, int64_t ld_out,
                                                           float* __restrict__ inv_scale, int64_t ld_scale, int n_groups) {
  extern __shared__ float s_scale[];                 // n_groups x 32 rows
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool vec_ok = ((ldx & 3) == 0) && ((reinterpret_cast<uintptr_t>(x) & (4 * sizeof(T) - 1)) == 0);
  for (int64_t blk = blockIdx.x; blk * kSplitRowsPerCta < rows; blk += gridDim.x) {
    const int64_t r0 = blk * kSplitRowsPerCta;
    for (int rr = warp; rr < kSplitRowsPerCta; rr += 8) {
      const int64_t r = r0 + rr;
      if (r >= rows) { for (int g = lane; g < n_groups; g += 32) s_scale[g * 32 + rr] = 1.f; continue; }
      const T* xr = x + r * ldx;
      __half* hr = hi + r * ld_out;
      __half* lr = lo + r * ld_out;
#pragma unroll 2
      for (int g = 0; g < n_groups; ++g) {
        float v[8];
#pragma unroll
        for (int hseg = 0; hseg < 2; ++hseg) {
          const int c = g * kGroup + hseg * 128 + lane * 4;
          if (vec_ok && c + 3 < k) {
            load4_f32<true>(xr + c, v + 4 * hseg);
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) v[4 * hseg + i] = (c + i < k) ? to_f32(xr[c + i]) : 0.f;
          }
        }
        float m = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) m = fmaxf(m, fabsf(v[i]));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float s = 1.f, is = 1.f;
        if (m > 0.f && m < INFINITY) {
          int e;
          frexpf(m, &e);                               // floor(log2 m) = e - 1 (also for subnormal m)
          const int sh = min(max(15 - e, -126), 126);
          s = ldexpf(1.f, sh); is = ldexpf(1.f, -sh);
        }
        if (lane == 0) s_scale[g * 32 + rr] = is;
#pragma unroll
        for (int hseg = 0; hseg < 2; ++hseg) {
          const int c = g * kGroup + hseg * 128 + lane * 4;
          if (c < ld_out) {
            __align__(8) __half h[4];
            __align__(8) __half l[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float xs = v[4 * hseg + i] * s;
              h[i] = __float2half_rn(xs);
              l[i] = __float2half_rn(xs - __half2float(h[i]));
            }
            *reinterpret_cast<uint2*>(hr + c) = *reinterpret_cast<const uint2*>(h);
            *reinterpret_cast<uint2*>(lr + c) = *reinterpret_cast<const uint2*>(l);
          }
        }
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_groups * 32; i += 256) {
      const int g = i >> 5, rr = i & 31;
      if (r0 + rr < rows) inv_scale[(int64_t)g * ld_scale + r0 + rr] = s_scale[i];
    }
    __syncthreads();
  }
}

int g_pair_cluster_cap = 0;     // > 0: persistent grid limited to this many CTA pairs (leaves SMs to concurrent kernels)

template <int BK, int STAGES, bool ARGMIN, int TILE_N = 256>
int launch_pair_cfg(const PairProblem& p, cudaStream_t st) {
  using C = PairCfg<BK, STAGES, TILE_N>;
  auto kern = linear_pair_kernel<BK, STAGES, ARGMIN, TILE_N>;
  static bool attr_set = false;
  static int max_clusters = 0;
  if (!attr_set) {
    LC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2 * (unsigned)num_sms()); cfg.blockDim = dim3(kPairThreads); cfg.dynamicSmemBytes = C::SMEM_BYTES;
    cudaLaunchAttribute at{};
    at.id = cudaLaunchAttributeClusterDimension; at.val.clusterDim.x = 2; at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
    cfg.attrs = &at; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n < 1) { (void)cudaGetLastError(); n = num_sms() / 2; }
    max_clusters = n;
    attr_set = true;
  }
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  LC_TRY(make_map(&ma_hi, p.a.hi, p.n_rows, p.k, p.a.ld, BK, kHalfM, 2));
  LC_TRY(make_map(&ma_lo, p.a.lo, p.n_rows, p.k, p.a.ld, BK, kHalfM, 2));
  LC_TRY(make_map(&mb_hi, p.w_hi, p.n_out, p.k, p.ldw, BK, TILE_N / 2, 2));
  LC_TRY(make_map(&mb_lo, p.w_lo, p.n_out, p.k, p.ldw, BK, TILE_N / 2, 2));
  PairArgs a{};
  a.n_rows = p.n_rows; a.n_out = p.n_out; a.k = p.k;
  a.tiles_n = p.n_out / TILE_N;
  a.n_tiles = ceil_div(p.n_rows, 256) * a.tiles_n;
  a.a_inv_scale = p.a.inv_scale; a.ld_ascale = p.a.ld_scale;
  a.w_inv_scale = p.w_inv_scale; a.bias = p.bias; a.relu = p.relu;
  a.y = p.y; a.ldy = p.ldy;
  a.o_hi = p.o_hi; a.o_lo = p.o_lo; a.ldo = p.ldo; a.o_inv_scale = p.o_inv_scale; a.ld_oscale = p.ld_oscale;
  a.debug = p.debug; a.trace = (long long*)p.trace;
  a.xx = p.xx; a.cc = p.cc; a.codes = p.codes; a.codes_stride = p.codes_stride;
  int cap = max_clusters;
  if (g_pair_cluster_cap > 0) cap = std::min(cap, g_pair_cluster_cap);
  const int64_t clusters = std::min<int64_t>(ARGMIN ? a.n_tiles / a.tiles_n : a.n_tiles, cap);
  kern<<<(unsigned)(2 * clusters), kPairThreads, C::SMEM_BYTES, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, a);
  LC_LAUNCH_CHECK("linear_pair_kernel");
  return LCREC_OK;
}

}  // namespace

void set_pair_cluster_cap(int cap) { g_pair_cluster_cap = cap; }

// full-width tiles for n_out a multiple of 256; one narrower tile for the 128- and 64-wide tail layers
bool linear_pair_supported(int k, int n_out, int group) {
  return group == kGroup && ((n_out >= kTileN && n_out % kTileN == 0) || n_out == 128 || n_out == 64) && k >= 64 && k % 8 == 0;
}
bool argmin_pair_supported(int k, int n_out) { return n_out >= kTileN && n_out % kTileN == 0 && k >= 8 && k % 8 == 0; }

int launch_linear_pair(const PairProblem& p, cudaStream_t st) {
  if (p.n_rows == 0) return LCREC_OK;
  if (!linear_pair_supported(p.k, p.n_out, p.a.group)) { set_error("linear_pair: unsupported shape k=%d n_out=%d group=%d", p.k, p.n_out, p.a.group); return LCREC_ERR_UNSUPPORTED; }
  if ((p.y && ((p.ldy & 3) || (reinterpret_cast<uintptr_t>(p.y) & 15))) || (p.o_hi && ((p.ldo & 7) || (reinterpret_cast<uintptr_t>(p.o_hi) & 15) || (reinterpret_cast<uintptr_t>(p.o_lo) & 15)))) {
    set_error("linear_pair: outputs must be 16-byte aligned with 16-byte row strides");
    return LCREC_ERR_ARG;
  }
  if ((reinterpret_cast<uintptr_t>(p.w_inv_scale) & 15) || (p.bias && (reinterpret_cast<uintptr_t>(p.bias) & 15))) {
    set_error("linear_pair: bias / channel scales must be 16-byte aligned");
    return LCREC_ERR_ARG;
  }
  if (p.n_out == 128) return launch_pair_cfg<64, 4, false, 128>(p, st);
  if (p.n_out == 64) return launch_pair_cfg<64, 4, false, 64>(p, st);
  if (p.debug & 4) return launch_pair_cfg<32, 6, false>(p, st);
  return launch_pair_cfg<64, 3, false>(p, st);
}

// codes[row * codes_stride] = first argmin over the n_out codes of (xx[row] + cc[code]) - 2 <a_row, w_code>
int launch_argmin_pair(const PairProblem& p, cudaStream_t st) {
  if (p.n_rows == 0) return LCREC_OK;
  if (!argmin_pair_supported(p.k, p.n_out) || p.a.group != kGroup || !p.xx || !p.cc || !p.codes) {
    set_error("argmin_pair: unsupported problem k=%d n_out=%d", p.k, p.n_out);
    return LCREC_ERR_UNSUPPORTED;
  }
  if ((reinterpret_cast<uintptr_t>(p.w_inv_scale) & 15) || (reinterpret_cast<uintptr_t>(p.cc) & 15)) {
    set_error("argmin_pair: code norms / scales must be 16-byte aligned");
    return LCREC_ERR_ARG;
  }
  if (p.k <= 32) return launch_pair_cfg<32, 6, true>(p, st);      // e_dim <= 32: one 64-byte K block, no zero-padded half
  return launch_pair_cfg<64, 3, true>(p, st);
}

template <typename T>
static int launch_split_groups_t(const T* x, int64_t rows, int k, int64_t ldx, __half* hi, __half* lo, int64_t ld_out,
                                 float* inv_scale, int64_t ld_scale, cudaStream_t st) {
  if (rows == 0) return LCREC_OK;
  const int n_groups = (int)ceil_div(ld_out, kGroup);
  const size_t smem = sizeof(float) * 32 * n_groups;
  if (smem > 48 * 1024) { set_error("split_groups: k = %d too wide", k); return LCREC_ERR_UNSUPPORTED; }
  const int64_t blocks = std::min<int64_t>(ceil_div(rows, kSplitRowsPerCta), (int64_t)num_sms() * 8);
  split_groups_kernel<T><<<(unsigned)blocks, 256, smem, st>>>(x, rows, k, ldx, hi, lo, ld_out, inv_scale, ld_scale, n_groups);
  LC_LAUNCH_CHECK("split_groups_kernel");
  return LCREC_OK;
}

int launch_split_groups(const void* x, int dtype, int64_t rows, int k, int64_t ldx, __half* hi, __half* lo, int64_t ld_out,
                        float* inv_scale, int64_t ld_scale, cudaStream_t st) {
  switch (dtype) {
    case kDtypeF32: return launch_split_groups_t(static_cast<const float*>(x), rows, k, ldx, hi, lo, ld_out, inv_scale, ld_scale, st);
    case kDtypeF16: return launch_split_groups_t(static_cast<const __half*>(x), rows, k, ldx, hi, lo, ld_out, inv_scale, ld_scale, st);
    case kDtypeBF16: return launch_split_groups_t(static_cast<const __nv_bfloat16*>(x), rows, k, ldx, hi, lo, ld_out, inv_scale, ld_scale, st);
    default: set_error("split_groups: bad argument: dtype %d (0 = fp32, 1 = fp16, 2 = bf16)", dtype); return LCREC_ERR_ARG;
  }
}

}  // namespace lcrec
