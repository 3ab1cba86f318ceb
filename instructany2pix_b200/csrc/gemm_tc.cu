// tcgen05 / TMEM / TMA "tap-table" implicit GEMM for sm_100a.
//
//   out[pixel, n] = epilogue( sum over taps e, channel chunks c of  A_e[pixel shifted by (dx,dy), c*64..] . W[n, wk0_e + c*64..] )
//
// One kernel covers: plain Linear (1 tap), K-concat of two sources (2 taps), 3x3 conv pad 1 (9 taps over one 4-D
// NHWC tensor map; TMA zero-fills the halo), stride-2 conv (9 taps over 4 parity-decimated maps) and a fused 1x1
// shortcut conv (extra taps over the raw block input).  Reference ops replaced: see include/ia2p.h.
//
// CTA = 6 warps: w0 TMA producer, w1 tcgen05.mma issuer (also owns TMEM alloc), w2..w5 epilogue (TMEM -> regs ->
// bias/rowbias/residual/GEGLU -> bf16 -> global).  Persistent over (m_tile, n_tile); STAGES-deep smem ring
// (full/empty mbarriers), two TMEM accumulator buffers (tmem_full/tmem_empty) so the epilogue of tile i overlaps the
// main loop of tile i+1.  Tile 128 x BLOCK_N x 64, operands K-major SWIZZLE_128B.
#include <cuda.h>

#include <cstdlib>
#include <mutex>

#ifdef IA2P_TC_TRACE
#define IA2P_TRACE_ROW ((size_t)p.trace_id * (size_t)g_tc_trace_stride + (size_t)blockIdx.x)
#endif
#include "common.cuh"
#include "tensormap.cuh"

// Two few-row experiments live behind compile-time switches and are NOT part of the shipped library (make variant
// DEFS="-DIA2P_WITH_SPLITK -DIA2P_WITH_MC"): split-K through an L2 workspace and A-operand TMA multicast in clusters.  Both
// were measured slower than / equal to one narrow tile per CTA (profiles/README.md section 9), and merely compiling their
// run-time branches into the kernel cost the batch-1 512^2 step 7 % (14.0 vs 13.0 ms, same box): hence compiled out.
// ia2p_tc_features() reports what a build contains (bit 0 split-K, bit 1 multicast).
#ifndef IA2P_EPI3_SLOTS
#define IA2P_EPI3_SLOTS 2   // staging slots per epilogue half-group of the bf16 TMA-store epilogue (1: one more main-loop stage)
#endif
#ifndef IA2P_MAX_STAGES
#define IA2P_MAX_STAGES 6   // smem ring depth cap (experiments: make variant NAME=.. DEFS=-DIA2P_MAX_STAGES=..)
#endif

namespace ia2p {

struct TapEntry {
  int16_t map_id, dx, dy, nchunks;
  int32_t wk0;
};
constexpr int kMaxTaps = 24;

struct alignas(64) TcMaps {
  CUtensorMap a[4];
  CUtensorMap w;
  CUtensorMap w2;                  // same matrix, box of HALF the rows: the B operand of a tail-split half tile
  CUtensorMap o, o2;               // EPI >= 1: fp32 output / bf16 copy, boxes of 16 columns x the 128 tile pixels
  CUtensorMap r;                   // EPI == 2: fp32 residual, same boxes
};

struct TcParams {
  TapEntry taps[kMaxTaps];
  int ntaps, num_kb;
  int tw_log2, th_log2;            // M tile = TB x TH x TW output pixels, TB*TH*TW == 128
  int tiles_x, tiles_y, m_tiles, n_tiles;
  // Tail split (wave quantisation): work items [0, full_items) are whole 128 x BLOCK_N tiles; the remaining tiles -- the
  // ones that would form a last, mostly idle wave -- are cut into `split` column slices each, so that every SM gets a slice.
  int full_items, total_items, split;
  // Split-K (few-row problems: fewer tiles than half the SMs).  Every tile is computed by `ksplit` CTAs, each over kb_per
  // consecutive k-blocks; splits 1.. dump their fp32 accumulators to `ws` and bump flags[tile]; split 0 waits for them, adds
  // the partials in split order (bit-reproducible), writes the sums back to TMEM and runs the normal epilogue.
  int ksplit, kb_per;
  float* ws;
  unsigned* flags;
  // A-operand multicast (single-wave problems on the single-CTA kernel): `mc` CTAs of a cluster own consecutive n-tiles of the
  // SAME row tile; each loads 1/mc of the 128 A rows per k-block (the a[] maps then carry the slice box) and multicasts it to
  // all of them, so the L2 -> SM traffic of A drops by mc (host side: pick_mc / slice_box).
  int mc;
  int trace_id;                    // debug build: launch id for the in-graph timeline
  // Weight prefetch hint (ia2p_tc_prefetch_hint): the NEXT tcgen05 launch's weight matrix.  Every CTA pulls its slice into L2
  // once its first tile's loads are under way, so the next kernel's first wave does not start on cold DRAM misses.
  const char* pf_ptr;
  long long pf_bytes;
  int early_b;           // programmatic dependent launch: issue the first weight loads ahead of griddepcontrol.wait
  int Wo, Ho, B;                   // output pixel grid (plain GEMM: Wo = M, Ho = B = 1)
  int N;                           // GEMM N (pre-GEGLU)
  int rows_per_batch;              // rowbias row = pixel / rows_per_batch
  const float* bias;
  const float* rowbias;
  const void* residual;            // bf16 or fp32 (res_f32)
  void* out;                       // bf16 or fp32 (out_f32)
  long long ldo, ldr;
  long long ost_x, ost_y, ost_b;   // EPI >= 1 output map: element strides of the pixel grid (0 -> dense: ldo, ldo*Wo, ldo*Wo*Ho)
  int geglu, out_f32, res_f32;
  int act;                         // EPI 3 only: IA2P_EPI_GELU | IA2P_EPI_QUICK_GELU on (LN-corrected acc + bias), else 0
  // LayerNorm folding (DESIGN.md): a PRODUCER of the fp32 residual stream also emits a bf16 copy of its output rows and
  // per-row partial (sum, sum of squares) over each column half of every N tile; a CONSUMER multiplies the raw bf16 rows
  // by gamma-scaled weights and finishes LN in its epilogue: rstd[m] * (acc - mean[m] * c1[n]) + c2[n].
  __nv_bfloat16* out2;             // producer: bf16 copy of out (row pitch ldo2) | NULL
  long long ldo2;
  float* stats_out;                // producer: [rows][2 * n_tiles][2] partial sums | NULL
  float* colstats;                 // EPI >= 1: [m_tiles][N][2] per-tile column (sum, sum of squares) for a following GroupNorm | NULL
  const float* ln_stats;           // consumer: [rows][ln_parts][2] | NULL
  const float* ln_c1;              // consumer: [N]  (row sums of the gamma-scaled weight)
  int ln_parts;
  float ln_inv_n, ln_eps;          // 1 / (normalised width), epsilon
};

#ifdef IA2P_TC_TRACE
#define IA2P_TRACE_BUF g_tc_trace
__device__ unsigned long long* g_tc_trace = nullptr;
__device__ int g_tc_trace_stride = 0;                          // 0: one row per CTA (last launch); > 0: rows per launch (whole-step traces)
__device__ unsigned long long* g_tc_timeline = nullptr;
static int g_tc_launch_id = 0;                                 // host: id handed to the next launch (fixed per graph node)
#endif

struct TcItem { int m_unit, n_tile, n_off, w; };
__device__ __forceinline__ TcItem tc_decode_item(const TcParams& p, int item, int block_n) {
  TcItem it;
  int tile = item;
  it.n_off = 0;
  it.w = block_n;
  if (item >= p.full_items) {                 // split is 1 or 2
    const int j = item - p.full_items;
    tile = p.full_items + (j >> 1);
    it.w = block_n >> 1;
    it.n_off = (j & 1) * it.w;
  }
  it.m_unit = tile / p.n_tiles;
  it.n_tile = tile - it.m_unit * p.n_tiles;
  return it;
}

// CG = 1: one CTA per 128 x BLOCK_N tile.  CG = 2: a CTA PAIR (cluster of 2, tcgen05 cta_group::2) per 256 x BLOCK_N tile:
// each CTA stages its own 128 A rows and HALF of the B rows, so the per-SM shared-memory traffic per MMA cycle drops by a
// third -- with CG = 1 the UMMA operand reads + TMA writes (192 B/clk at 128x256x64) exceed what smem sustains and cap the
// main loop near 55 % of the tensor peak (measured, profiles/README.md).
//
// EPI = 0: the epilogue stores straight from registers (bf16 outputs: 64 KB per tile, far below what the LSU path moves).
// EPI = 1 (fp32 outputs, optionally + bf16 copy: 192 KB per tile): thread-per-row register stores top out near 23 GB/s per
// SM (tools/membench.cu: one sector per lane per instruction), which made the fp32 residual GEMMs epilogue-bound.  Here the
// two epilogue half-groups (4 warps = 128 rows each) stage 32-column slices in swizzled shared memory and one elected
// lane per half-group hands them to the TMA store engine.
// EPI = 3 (bf16 outputs without residual: QKV, to_q, GEGLU projections): the same idea for bf16 -- each half-group stages whole
// 64-column output slices (128 rows x 128 B, SWIZZLE_128B; a 32-column remainder as SWIZZLE_64B) and hands them to the TMA store
// engine.  Thread-per-row register stores (EPI 0) write one 32-byte sector per lane and instruction, ~12 B/clk per SM: 5 k cycles
// for the 64 KB of a 128 x 256 bf16 tile, and with the LayerNorm fold on top the epilogue took longer than the tile's main loop
// once the MMAs ran at the tensor-pipe rate (MMA warp waiting for a free accumulator 31 % of a QKV launch, profiles/README.md).
// EPI = 2 (fp32 residual GEMMs with a short K: attention out-projections): additionally the residual slices arrive by TMA
// load, one slice ahead, into the second of two fp32 staging slots (the thread reads its row, adds, and writes the result
// back in place); the main loop gives up two stages for them.  With register loads the residual reads (a sector per lane
// per instruction) were the critical path of those GEMMs (profiles/README.md).
template <int BLOCK_N, int CG = 1, int EPI = 0>
struct TcCfg {
  static constexpr int A_BYTES = 128 * 128;             // 128 rows x 64 bf16
  static constexpr int B_BYTES = (BLOCK_N / CG) * 128;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_BYTES = EPI ? 1024 : 256;
  // fp32-output epilogues: slice width per half-group and round.  EPI 2 (short K: the epilogue is the critical path) moves 32
  // columns per round -- half the barrier / TMA round trips per tile; EPI 1 (long K: the main loop is) keeps 16-column slices and
  // their smaller staging buffers (one more main-loop stage: measured, 6 vs 5 stages is worth 3-6 % on the K >= 2560 shapes).
  static constexpr int SLW = (EPI == 2) ? 32 : 16;
  static constexpr int EPI_F_BYTES = 128 * SLW * 4, EPI_H_BYTES = 128 * SLW * 2; // per half-group: fp32 / bf16 slice
  static constexpr int NBF = (EPI == 2) ? 2 : 1, NBH = 1;                        // fp32 slots per half-group (EPI 2: one holds the next residual)
  static constexpr int EPI3_SLICE = 128 * 128;                                   // EPI 3: 128 rows x 64 bf16 columns, EPI3_SLOTS slots per half-group
  static constexpr int EPI3_SLOTS = IA2P_EPI3_SLOTS;
  static constexpr int EPI_BYTES = EPI == 3 ? 2 * EPI3_SLOTS * EPI3_SLICE : EPI ? 2 * (NBF * EPI_F_BYTES + NBH * EPI_H_BYTES) : 0;
  static constexpr int BUDGET = 227 * 1024 - 1024 /*align slack*/ - BAR_BYTES - EPI_BYTES;
  static constexpr int STAGES = (BUDGET / STAGE_BYTES) > IA2P_MAX_STAGES ? IA2P_MAX_STAGES : (BUDGET / STAGE_BYTES);
  static constexpr int TMEM_COLS = (2 * BLOCK_N <= 256) ? 256 : 512;
  static constexpr int STAGE_OFF = STAGES * STAGE_BYTES + BAR_BYTES;            // epilogue staging, from smem_base
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + BAR_BYTES + EPI_BYTES;
  static_assert(STAGES >= 3, "pipeline too shallow");
};

constexpr int kEpiWarpsConst = 8;
constexpr int kMaxKSplit = 4;
// Split-K fix-up, run by the 8 epilogue warps before the normal epilogue (warp = TMEM lane quarter q x column half).
// Partial storage layout per (tile, split >= 1): [BLOCK_N / 32 chunks][4][128 rows][8 floats], so that lane r of a warp moves
// consecutive 32-byte pieces (fully coalesced both ways).  Returns true when this CTA only produced a partial.
template <int BLOCK_N>
__device__ __forceinline__ bool splitk_prepass(const TcParams& p, int unit, int sidx, uint32_t tmem_acc, int warp, int lane) {
  constexpr int NCH = BLOCK_N / 32, NCH0 = (NCH + 1) / 2;
  const int q = warp & 3, hf = (warp - 2) >> 2, row = q * 32 + lane;
  const int c_lo = hf == 0 ? 0 : NCH0, c_hi = hf == 0 ? NCH0 : NCH;
  const uint32_t t_row = tmem_acc + ((uint32_t)(q * 32) << 16);
  const size_t per_split = (size_t)NCH * 4 * 128 * 8;                       // floats per (tile, split)
  float* base = p.ws + (size_t)unit * (p.ksplit - 1) * per_split;
  if (sidx > 0) {
    float* dst = base + (size_t)(sidx - 1) * per_split;
    for (int c = c_lo; c < c_hi; ++c) {
      uint32_t v[32];
      tmem_ld_32x32(t_row + (uint32_t)(c * 32), v);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 4; ++i) stg256(dst + ((size_t)(c * 4 + i) * 128 + row) * 8, reinterpret_cast<const float*>(&v[8 * i]));
    }
    tc_fence_before();
    named_bar_sync(3, 32 * kEpiWarpsConst);
    if (warp == 2 && lane == 0) {
      __threadfence();
      atomicAdd(p.flags + unit, 1u);
    }
#ifdef IA2P_TC_TRACE
    if (warp == 2) TRACE_PUT(10, gtime_ns());
#endif
    return true;
  }
#ifdef IA2P_TC_TRACE
  if (warp == 2) TRACE_PUT(11, gtime_ns());
#endif
  if (warp == 2 && lane == 0) {
    long long t0 = clock64();
    while (ld_acquire_gpu(p.flags + unit) < (unsigned)(p.ksplit - 1)) {
      if (clock64() - t0 > 20000000000LL) __trap();                          // protocol bug -> launch failure, not a hang
    }
    p.flags[unit] = 0u;                                                      // every partial has arrived: re-arm for the next launch
  }
  named_bar_sync(3, 32 * kEpiWarpsConst);
#ifdef IA2P_TC_TRACE
  if (warp == 2) TRACE_PUT(12, gtime_ns());
#endif
  for (int c = c_lo; c < c_hi; ++c) {
    uint32_t v[32];
    tmem_ld_32x32(t_row + (uint32_t)(c * 32), v);
    tmem_ld_wait();
    // all partial pieces of this chunk are requested before the first add (<= 3 splits x 4 x 32 bytes in flight per thread)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float d[kMaxKSplit - 1][8];
#pragma unroll
      for (int sp = 0; sp < kMaxKSplit - 1; ++sp)
        if (sp + 1 < p.ksplit) ldg256_cg(base + (size_t)sp * per_split + ((size_t)(c * 4 + i) * 128 + row) * 8, d[sp]);
#pragma unroll
      for (int sp = 0; sp < kMaxKSplit - 1; ++sp)
        if (sp + 1 < p.ksplit) {
#pragma unroll
          for (int k = 0; k < 8; ++k) v[8 * i + k] = __float_as_uint(__uint_as_float(v[8 * i + k]) + d[sp][k]);
        }
    }
    tmem_st_32x32(t_row + (uint32_t)(c * 32), v);
  }
  tmem_st_wait();
  tc_fence_before();
  named_bar_sync(3, 32 * kEpiWarpsConst);                                    // other warps read these columns in the epilogue proper
  tc_fence_after();
#ifdef IA2P_TC_TRACE
  if (warp == 2) TRACE_PUT(13, gtime_ns());
#endif
  return false;
}

constexpr int kEpiWarps = 8;                            // two warps per TMEM lane quarter, each takes half of the columns
constexpr int kTcThreads = 64 + 32 * kEpiWarps;

template <int BLOCK_N, int CG, int EPI>
__global__ void __launch_bounds__(kTcThreads, 1)
tc_gemm_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ TcParams p) {
  using Cfg = TcCfg<BLOCK_N, CG, EPI>;
  const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;     // 0 = leader (issues the MMAs), 1 = peer
  constexpr int STAGES = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + STAGES * Cfg::STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (STAGES + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * STAGES + 2 + b); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * STAGES + 4);
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = warp_idx_uniform();
  const int lane = threadIdx.x & 31;
#ifdef IA2P_WITH_MC
  const uint32_t mc = (CG == 1 && p.mc > 1) ? (uint32_t)p.mc : 1u;      // A-multicast cluster size
#else
  constexpr uint32_t mc = 1u;
#endif
  const uint32_t crank = (mc > 1) ? cluster_ctarank() : 0u;
  pdl_launch_dependents();
#ifdef IA2P_TC_TRACE
  if (warp == 0) TRACE_PUT(0, gtime_ns());
#endif

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&maps.w);
    tma_prefetch_desc(&maps.w2);
    tma_prefetch_desc(&maps.a[0]);
    if (EPI >= 1) {
      tma_prefetch_desc(&maps.o);
      tma_prefetch_desc(&maps.o2);
    }
    if (EPI == 2) {
      tma_prefetch_desc(&maps.r);
      for (int i = 0; i < 8; ++i) mbar_init(bar_base + 8u * (2 * STAGES + 6 + i), 1);
    }
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);               // CG = 2: the leader expects BOTH CTAs' TMA bytes on its barrier
      mbar_init(empty_bar(s), mc);             // multicast: a stage is free once EVERY CTA of the cluster has consumed it
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), kEpiWarps * CG);   // CG = 2: both CTAs' epilogue warps release the leader's MMA warp
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    if (CG == 2) { tmem_alloc_2sm(tmem_slot, Cfg::TMEM_COLS); tmem_relinquish_2sm(); }
    else { tmem_alloc(tmem_slot, Cfg::TMEM_COLS); tmem_relinquish(); }
  }
  tc_fence_before();
  if (CG == 2 || mc > 1) cluster_sync_all(); else __syncthreads();   // peer barriers must be initialised before remote arrives
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // Programmatic dependent launch: everything above overlapped the previous kernel's tail.  The producer warp waits later: it
  // first issues the WEIGHT loads of its first k-blocks (p.early_b: the B operand is never written by a kernel of the same stream)
  const bool early_b = p.early_b != 0 && mc == 1;
  if (warp != 0 || !early_b) pdl_wait();
#ifdef IA2P_TC_TRACE
  if (warp == 0) TRACE_PUT(1, gtime_ns());
  if (threadIdx.x == 0 && g_tc_timeline != nullptr) atomicMin(g_tc_timeline + 2 * (size_t)p.trace_id, gtime_ns());
#endif

  // tile walk: CG = 2 steps over tile PAIRS (two consecutive m-tiles); this CTA owns m_tile = 2 * pair + rank
  const int total_tiles = p.total_items;
#ifdef IA2P_WITH_SPLITK                                          // experiment builds only (see the note at IA2P_WITH_SPLITK below)
  const bool splitk = (CG == 1) && p.ksplit > 1;                // one (tile, k-range) item per CTA
#else
  constexpr bool splitk = false;
#endif
  const int unit0 = splitk ? (int)blockIdx.x / p.ksplit : (int)blockIdx.x / CG;
  const int unit_step = splitk ? (1 << 30) : (int)gridDim.x / CG;
  const int sidx = splitk ? (int)blockIdx.x % p.ksplit : 0;
  const int kb0 = sidx * p.kb_per;                              // this CTA's k-block range [kb0, kb1)
  const int kb1 = splitk ? (kb0 + p.kb_per < p.num_kb ? kb0 + p.kb_per : p.num_kb) : p.num_kb;
  const int TB = 128 >> (p.tw_log2 + p.th_log2);

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    TRACE_DECL(tr_wait_empty);
    bool pf_done = (p.pf_ptr == nullptr);
    // multicast: first pixel of this CTA's slice inside the tile's (TB, TH, TW) box; rows are ordered (tb, th, tw)
    const int mc_row0 = (int)crank * (128 / (int)mc);
    const int mc_x = mc_row0 & ((1 << p.tw_log2) - 1);
    const int mc_y = (mc_row0 >> p.tw_log2) & ((1 << p.th_log2) - 1);
    const int mc_b = mc_row0 >> (p.tw_log2 + p.th_log2);
    // early_b: the first min(STAGES, k-blocks) stages of the first tile get their arrive + B (weight) load here, BEFORE
    // griddepcontrol.wait; the main loop below then only adds the A load for those stages.
    int pre = 0;
    if (early_b && !splitk && unit0 < total_tiles) {
      const TcItem ti = tc_decode_item(p, unit0, BLOCK_N);
      const int n0 = ti.n_tile * BLOCK_N + ti.n_off + (int)rank * (ti.w / CG);
      const CUtensorMap* wm = (ti.w == BLOCK_N) ? &maps.w : &maps.w2;
      const uint32_t stage_tx = (uint32_t)(Cfg::A_BYTES + (ti.w / CG) * 128);
      for (int e = 0; e < p.ntaps && pre < STAGES; ++e) {
        const TapEntry t = p.taps[e];
        for (int c = 0; c < t.nchunks && pre < STAGES; ++c, ++pre) {
          if (elect_one()) {
            const uint32_t a_dst = smem_base + pre * Cfg::STAGE_BYTES;
            if (CG == 2) {
              if (rank == 0) mbar_arrive_expect_tx(full_bar(pre), 2 * stage_tx);
              tma_load_2d_2sm(a_dst + Cfg::A_BYTES, wm, full_bar(pre), t.wk0 + c * 64, n0);
            } else {
              mbar_arrive_expect_tx(full_bar(pre), stage_tx);
              tma_load_2d(a_dst + Cfg::A_BYTES, wm, full_bar(pre), t.wk0 + c * 64, n0);
            }
          }
          __syncwarp();
        }
      }
    }
    if (early_b) pdl_wait();
    int issued = 0;                                     // k-blocks issued so far by this CTA
    for (int tile = unit0; tile < total_tiles; tile += unit_step) {
      const TcItem ti = tc_decode_item(p, tile, BLOCK_N);
      const int m_tile = ti.m_unit * CG + (int)rank;    // may be == m_tiles for the odd tail: TMA zero-fills (batch coord OOB)
      const int xt = m_tile % p.tiles_x;
      const int r = m_tile / p.tiles_x;
      const int yt = r % p.tiles_y, bt = r / p.tiles_y;
      const int x0 = xt << p.tw_log2, y0 = yt << p.th_log2, b0 = bt * TB;
      const int n0 = ti.n_tile * BLOCK_N + ti.n_off + (int)rank * (ti.w / CG);   // this CTA's slice of the B rows
      const CUtensorMap* wm = (ti.w == BLOCK_N) ? &maps.w : &maps.w2;
      const uint32_t stage_tx = (uint32_t)(Cfg::A_BYTES + (ti.w / CG) * 128);
      int kbi = 0;
      for (int e = 0; e < p.ntaps; ++e) {
        const TapEntry t = p.taps[e];
        const CUtensorMap* am = &maps.a[t.map_id];
        for (int c = 0; c < t.nchunks; ++c, ++kbi) {
          if (kbi < kb0 || kbi >= kb1) continue;          // split-K: another CTA owns this k-block
          const bool b_done = issued < pre;               // arrive + B load already issued ahead of griddepcontrol.wait
          ++issued;
          TRACE_T0(tw0);
          mbar_wait(empty_bar(stage), phase ^ 1u);
          TRACE_ADD(tr_wait_empty, tw0);
          if (b_done) {
            if (elect_one()) {
              const uint32_t a_dst = smem_base + stage * Cfg::STAGE_BYTES;
              if (CG == 2) tma_load_4d_2sm(a_dst, am, full_bar(stage), c * 64, x0 + t.dx, y0 + t.dy, b0);
              else tma_load_4d(a_dst, am, full_bar(stage), c * 64, x0 + t.dx, y0 + t.dy, b0);
            }
          } else if (elect_one()) {
            const uint32_t a_dst = smem_base + stage * Cfg::STAGE_BYTES;
            if (CG == 2) {
              // Both CTAs' loads complete on the LEADER's full barrier (peer-bit-masked address).  Only the leader arrives
              // (expecting the bytes of both CTAs): a remote arrive per k-block from the peer costs ~1 us of release latency
              // and starves the MMA (measured).  The signed tx-count makes early peer completions harmless, and the peer
              // cannot run a phase ahead because its stage is only freed by the leader's multicast commit.
              if (rank == 0) mbar_arrive_expect_tx(full_bar(stage), 2 * stage_tx);
              tma_load_4d_2sm(a_dst, am, full_bar(stage), c * 64, x0 + t.dx, y0 + t.dy, b0);
              tma_load_2d_2sm(a_dst + Cfg::A_BYTES, wm, full_bar(stage), t.wk0 + c * 64, n0);
            } else if (mc > 1) {
              // this CTA's slice of the A rows goes to every CTA of the cluster; the other slices arrive from the peers.  A
              // peer's bytes may land before the arrive below (signed tx-count), never a phase early: the peer's stage is
              // only freed by THIS CTA's multicast commit as well.
              mbar_arrive_expect_tx(full_bar(stage), stage_tx);
              tma_load_4d_mc(a_dst + crank * (uint32_t)(Cfg::A_BYTES / (int)mc), am, full_bar(stage), c * 64, x0 + t.dx + mc_x,
                             y0 + t.dy + mc_y, b0 + mc_b, (uint16_t)((1u << mc) - 1u));
              tma_load_2d(a_dst + Cfg::A_BYTES, wm, full_bar(stage), t.wk0 + c * 64, n0);
            } else {
              mbar_arrive_expect_tx(full_bar(stage), stage_tx);
              tma_load_4d(a_dst, am, full_bar(stage), c * 64, x0 + t.dx, y0 + t.dy, b0);
              tma_load_2d(a_dst + Cfg::A_BYTES, wm, full_bar(stage), t.wk0 + c * 64, n0);
            }
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
      if (!pf_done) {                                   // first tile's loads issued: now pull this CTA's slice of the next weights
        pf_done = true;
        if (elect_one()) {
          const long long per = ((p.pf_bytes / (long long)gridDim.x + 4095) / 4096) * 4096;
          const long long lo = per * (long long)blockIdx.x;
          long long hi = lo + per;
          if (hi > p.pf_bytes) hi = p.pf_bytes;
          for (long long o = lo; o < hi; o += 16384) {
            const long long n = (hi - o < 16384) ? ((hi - o) & ~15LL) : 16384;
            if (n > 0) bulk_prefetch_l2(p.pf_ptr + o, (uint32_t)n);
          }
        }
      }
    }
    TRACE_PUT(5, tr_wait_empty);
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer (CG = 2: leader CTA only)
    constexpr uint32_t idesc_full = umma_idesc_bf16(128 * CG, BLOCK_N);
    constexpr uint32_t idesc_half = umma_idesc_bf16(128 * CG, BLOCK_N / 2);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    TRACE_DECL(tr_wait_full);
    TRACE_DECL(tr_wait_tempty);
    TRACE_DECL(tr_loop);
    TRACE_T0(tl0);
    for (int tile = unit0; tile < total_tiles && rank == 0; tile += unit_step, ++it) {
      const int buf = it & 1;
      const uint32_t use = (uint32_t)(it >> 1);
      TRACE_T0(te0);
      mbar_wait(tempty_bar(buf), (use & 1u) ^ 1u);
      TRACE_ADD(tr_wait_tempty, te0);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BLOCK_N);
      const uint32_t idesc = (tile < p.full_items) ? idesc_full : idesc_half;
      const int nkb = kb1 - kb0;
      for (int kb = 0; kb < nkb; ++kb) {
        TRACE_T0(tf0);
        mbar_wait(full_bar(stage), phase);
        TRACE_ADD(tr_wait_full, tf0);
#ifdef IA2P_TC_TRACE
        if (it == 0 && kb == 0) TRACE_PUT(10, clock64() - tf0);        // cold start: TMA issue -> first operands landed
#endif
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_addr = smem_base + stage * Cfg::STAGE_BYTES;
          const uint64_t da = umma_desc_sw128(a_addr);
          const uint64_t db = umma_desc_sw128(a_addr + Cfg::A_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k) {   // 4 x UMMA_K(16) per 64-wide K block: +32 B inside the swizzle atom
            if (CG == 2) umma_bf16_2sm(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (uint32_t)((kb | k) != 0));
            else umma_bf16(d_tmem, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, (uint32_t)((kb | k) != 0));
          }
          if (CG == 2) {
            umma_commit_2sm_mc(empty_bar(stage), 3);             // frees this stage in BOTH CTAs
            if (kb == nkb - 1) umma_commit_2sm_mc(tfull_bar(buf), 3);
          } else {
            if (mc > 1) umma_commit_mc(empty_bar(stage), (uint16_t)((1u << mc) - 1u));   // frees this stage in every CTA of the cluster
            else umma_commit(empty_bar(stage));
            if (kb == nkb - 1) umma_commit(tfull_bar(buf));
          }
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
    TRACE_ADD(tr_loop, tl0);
#ifdef IA2P_TC_TRACE
    TRACE_PUT(15, gtime_ns());                                        // all MMAs issued
#endif
    TRACE_PUT(2, tr_wait_full);
    TRACE_PUT(3, tr_wait_tempty);
    TRACE_PUT(4, tr_loop);
    TRACE_PUT(9, it);
  } else if (EPI == 3) {
    // ------------------------------------------------------------ epilogue, bf16 output through shared memory + TMA store
    // Half-group h = warps {2..5} / {6..9} (each covers the tile's 128 rows) owns the 64-column OUTPUT slices h, h + 2, ...; a
    // thread turns its row's accumulator columns of the slice into bf16 (bias / row bias / LN fold / GEGLU), writes them into the
    // half-group's swizzled staging slot, and the elected thread issues one TMA store per slice (two slots: one drains while the
    // next is filled).  The two half-groups never synchronise with each other.
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const bool lead_warp = (warp == 2 + 4 * half);        // its elect.sync lane issues the half-group's TMA traffic (uniform operands)
    const int tw = row & ((1 << p.tw_log2) - 1);
    const int th = (row >> p.tw_log2) & ((1 << p.th_log2) - 1);
    const int tb = row >> (p.tw_log2 + p.th_log2);
    const uint32_t st_base = smem_base + Cfg::STAGE_OFF + half * (Cfg::EPI3_SLOTS * Cfg::EPI3_SLICE);
    const uint32_t sw128 = (uint32_t)row & 7u;             // SWIZZLE_128B: 16-B chunk ^= row % 8
    const uint32_t sw64 = (uint32_t)(row >> 1) & 3u;       // SWIZZLE_64B (32-column remainder slice): 16-B chunk ^= (row / 2) % 4
    const uint32_t tempty_leader0 = (CG == 2 && rank != 0) ? mapa_shared(tempty_bar(0), 0) : 0u;
    int it = 0;
    TRACE_DECL(tr_wait_tfull);
    TRACE_DECL(tr_busy);
    uint32_t g = 0;                                        // slices stored so far by this half-group (slot = g & 1)
    for (int tile = unit0; tile < total_tiles; tile += unit_step, ++it) {
      const int buf = it & 1;
      const uint32_t use = (uint32_t)(it >> 1);
      const TcItem ti = tc_decode_item(p, tile, BLOCK_N);
      const int m_tile = ti.m_unit * CG + (int)rank;
      const int xt = m_tile % p.tiles_x;
      const int r = m_tile / p.tiles_x;
      const int yt = r % p.tiles_y, bt = r / p.tiles_y;
      const int x0 = xt << p.tw_log2, y0 = yt << p.th_log2, b0 = bt * TB;
      const int x = x0 + tw, y = y0 + th, b = b0 + tb;
      const bool valid = (x < p.Wo) && (y < p.Ho) && (b < p.B) && (m_tile < p.m_tiles);
      const long long pix = ((long long)b * p.Ho + y) * p.Wo + x;
      const int n_base = ti.n_tile * BLOCK_N + ti.n_off;    // first accumulator column (index into N) of this item
      int aw = ti.w;                                        // accumulator columns of this item that exist
      if (p.N - n_base < aw) aw = p.N - n_base;
      const int ow = p.geglu ? aw >> 1 : aw;                // output columns, and the first one
      const int o_base = p.geglu ? n_base >> 1 : n_base;
      const int nsl = (ow + 63) >> 6;
      const float* rb = (p.rowbias != nullptr && valid) ? p.rowbias + (pix / p.rows_per_batch) * (long long)p.N : nullptr;
      float ln_mean = 0.f, ln_rstd = 1.f;
      if (p.ln_stats != nullptr && valid) {                 // LN-fold consumer: see the EPI 0 epilogue
        const float* sp = p.ln_stats + pix * (long long)p.ln_parts * 2;
        float s1 = 0.f, s2 = 0.f;
        if ((p.ln_parts & 3) == 0) {
          const int nq = p.ln_parts >> 2;
          for (int i0 = 0; i0 < nq; i0 += 3) {
            float v[3][8];
#pragma unroll
            for (int j = 0; j < 3; ++j)
              if (i0 + j < nq) ldg256(sp + (i0 + j) * 8, v[j]);
#pragma unroll
            for (int j = 0; j < 3; ++j)
              if (i0 + j < nq) {
                s1 += v[j][0]; s2 += v[j][1]; s1 += v[j][2]; s2 += v[j][3];
                s1 += v[j][4]; s2 += v[j][5]; s1 += v[j][6]; s2 += v[j][7];
              }
          }
        } else {
          for (int i = 0; i < p.ln_parts; ++i) {
            const float2 v = __ldg(reinterpret_cast<const float2*>(sp) + i);
            s1 += v.x;
            s2 += v.y;
          }
        }
        ln_mean = s1 * p.ln_inv_n;
        ln_rstd = rsqrtf(fmaxf(s2 * p.ln_inv_n - ln_mean * ln_mean, 0.f) + p.ln_eps);
      }
      const float ln_nm = -ln_mean * ln_rstd;               // rstd * (acc - mean * c1) + bias = acc * rstd + (c1 * (-mean * rstd) + bias)

      TRACE_T0(tq0);
      mbar_wait(tfull_bar(buf), use & 1u);
      TRACE_ADD(tr_wait_tfull, tq0);
      TRACE_T0(tb0);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BLOCK_N);
      auto release_acc = [&]() {                            // after this warp's last TMEM read of the item
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (CG == 2 && rank != 0) mbar_arrive_cluster(tempty_leader0 + 8u * buf);
          else mbar_arrive(tempty_bar(buf));
        }
      };
      if (half >= nsl) release_acc();                       // nothing to read for this half-group

#pragma unroll 1
      for (int sl = half; sl < nsl; sl += 2) {
        const int cols = (ow - 64 * sl) < 64 ? (ow - 64 * sl) : 64;      // 64, or 32 for a remainder slice
        const uint32_t slot = st_base + (Cfg::EPI3_SLOTS > 1 ? (g & 1u) * Cfg::EPI3_SLICE : 0u);
        uint32_t pk[32];                                                 // this row's slice: 64 bf16
#pragma unroll
        for (int pc = 0; pc < 2; ++pc) {
          if (pc * 32 < cols) {                                          // uniform over the half-group
            const int oc = 64 * sl + 32 * pc;                            // output column (within the item) of this 32-column piece
            float f[32];
            if (!p.geglu) {
              const int n = n_base + oc;
              uint32_t v[32];
              tmem_ld_32x32(t_row + (uint32_t)oc, v);
              tmem_ld_wait();
              if (sl + 2 >= nsl && (pc + 1) * 32 >= cols) release_acc();
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
                if (p.bias != nullptr) bv = __ldg(reinterpret_cast<const float4*>(p.bias + n + i));
                if (p.ln_stats != nullptr) {
                  const float4 cv = __ldg(reinterpret_cast<const float4*>(p.ln_c1 + n + i));
                  bv.x = fmaf(cv.x, ln_nm, bv.x); bv.y = fmaf(cv.y, ln_nm, bv.y); bv.z = fmaf(cv.z, ln_nm, bv.z); bv.w = fmaf(cv.w, ln_nm, bv.w);
                }
                if (rb != nullptr) {
                  const float4 rv = __ldg(reinterpret_cast<const float4*>(rb + n + i));
                  bv.x += rv.x; bv.y += rv.y; bv.z += rv.z; bv.w += rv.w;
                }
                f[i] = fmaf(__uint_as_float(v[i]), ln_rstd, bv.x); f[i + 1] = fmaf(__uint_as_float(v[i + 1]), ln_rstd, bv.y);
                f[i + 2] = fmaf(__uint_as_float(v[i + 2]), ln_rstd, bv.z); f[i + 3] = fmaf(__uint_as_float(v[i + 3]), ln_rstd, bv.w);
              }
              if (p.act == IA2P_EPI_GELU) {
#pragma unroll
                for (int i = 0; i < 32; ++i) f[i] = gelu_erf_f(f[i]);
              } else if (p.act == IA2P_EPI_QUICK_GELU) {
#pragma unroll
                for (int i = 0; i < 32; ++i) f[i] = quick_gelu_f(f[i]);
              }
            } else {
              // GEGLU: accumulator columns come in 64-wide groups [32 value | 32 gate] (W rows interleaved, packing.interleave_geglu)
              const int n = n_base + 2 * oc;
              uint32_t vv[32], vg[32];
              tmem_ld_32x32(t_row + (uint32_t)(2 * oc), vv);
              tmem_ld_32x32(t_row + (uint32_t)(2 * oc + 32), vg);
              tmem_ld_wait();
              if (sl + 2 >= nsl && (pc + 1) * 32 >= cols) release_acc();
#pragma unroll
              for (int i = 0; i < 32; i += 4) {
                float4 bv = make_float4(0.f, 0.f, 0.f, 0.f), bg = bv;
                if (p.bias != nullptr) {
                  bv = __ldg(reinterpret_cast<const float4*>(p.bias + n + i));
                  bg = __ldg(reinterpret_cast<const float4*>(p.bias + n + 32 + i));
                }
                if (p.ln_stats != nullptr) {
                  const float4 cv = __ldg(reinterpret_cast<const float4*>(p.ln_c1 + n + i));
                  const float4 cg = __ldg(reinterpret_cast<const float4*>(p.ln_c1 + n + 32 + i));
                  bv.x = fmaf(cv.x, ln_nm, bv.x); bv.y = fmaf(cv.y, ln_nm, bv.y); bv.z = fmaf(cv.z, ln_nm, bv.z); bv.w = fmaf(cv.w, ln_nm, bv.w);
                  bg.x = fmaf(cg.x, ln_nm, bg.x); bg.y = fmaf(cg.y, ln_nm, bg.y); bg.z = fmaf(cg.z, ln_nm, bg.z); bg.w = fmaf(cg.w, ln_nm, bg.w);
                }
                f[i + 0] = fmaf(__uint_as_float(vv[i + 0]), ln_rstd, bv.x) * gelu_erf_f(fmaf(__uint_as_float(vg[i + 0]), ln_rstd, bg.x));
                f[i + 1] = fmaf(__uint_as_float(vv[i + 1]), ln_rstd, bv.y) * gelu_erf_f(fmaf(__uint_as_float(vg[i + 1]), ln_rstd, bg.y));
                f[i + 2] = fmaf(__uint_as_float(vv[i + 2]), ln_rstd, bv.z) * gelu_erf_f(fmaf(__uint_as_float(vg[i + 2]), ln_rstd, bg.z));
                f[i + 3] = fmaf(__uint_as_float(vv[i + 3]), ln_rstd, bv.w) * gelu_erf_f(fmaf(__uint_as_float(vg[i + 3]), ln_rstd, bg.w));
              }
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) pk[16 * pc + i] = pack_bf16x2(f[2 * i], f[2 * i + 1]);
          }
        }
        // the slot must have been read out by its previous store (two slices ago): at most one group may still be pending
        if (lead_warp && elect_one()) {
          if (Cfg::EPI3_SLOTS > 1) bulk_wait_read_1(); else bulk_wait_read_all();
        }
        named_bar_sync(1 + half, 128);
        if (cols == 64) {
          const uint32_t d = slot + (uint32_t)row * 128u;
#pragma unroll
          for (uint32_t j = 0; j < 8; ++j) sts128u(d + ((j ^ sw128) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
        } else {
          const uint32_t d = slot + (uint32_t)row * 64u;
#pragma unroll
          for (uint32_t j = 0; j < 4; ++j) sts128u(d + ((j ^ sw64) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
        }
        fence_proxy_async();
        named_bar_sync(1 + half, 128);
        if (lead_warp && elect_one()) {
          tma_store_4d(cols == 64 ? &maps.o : &maps.o2, slot, o_base + 64 * sl, x0, y0, b0);   // rows / columns outside the output are clipped
          bulk_commit_group();
        }
        ++g;
      }
      TRACE_ADD(tr_busy, tb0);
    }
    if (lead_warp && elect_one()) bulk_wait_read_all();                          // staging memory must outlive the last store's read
    if (warp == 2) { TRACE_PUT(6, tr_wait_tfull); TRACE_PUT(7, tr_busy); }
#ifdef IA2P_TC_TRACE
    if (warp == 2) TRACE_PUT(11, gtime_ns());                          // this CTA's epilogue is done
#endif
  } else if (EPI >= 1) {
    // ------------------------------------------------------------ epilogue, TMA variants (fp32 out [+ bf16 copy + LN stats])
    // Half-group h = warps {2..5} / {6..9} (each covers the tile's 128 rows) owns the SLW-column slices h, h + 2, ... of the item:
    // per slice a thread reads its row's SLW (EPI 2: 32, EPI 1: 16) accumulator columns, applies bias / row bias / residual, writes the fp32 (and bf16)
    // values into the half-group's swizzled staging slot (128 B rows, SWIZZLE_128B; bf16 copy 64 B rows, SWIZZLE_64B), and the
    // half-group's elect.sync lane issues one TMA store per slot.  EPI 2: the residual slice of the NEXT slice is TMA-loaded into
    // the other fp32 slot meanwhile and summed in place.  The two half-groups never synchronise with each other.
    // (Round-2 history: with 16-column slices -- twice the barrier / TMA round trips per tile -- this epilogue needed 11 us per
    // 128 x 256 tile against 7 us of MMAs, i.e. the 126 attention out-projections of a step were epilogue-bound.)
    constexpr int NBF = Cfg::NBF, SLW = Cfg::SLW;
    constexpr uint32_t NCF = SLW / 4, NCH = SLW / 8;      // 16-byte chunks per staged fp32 / bf16 row
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int row = q * 32 + lane;
    const bool lead_warp = (warp == 2 + 4 * half);        // its elect.sync lane issues the half-group's TMA traffic (uniform operands)
    const int tw = row & ((1 << p.tw_log2) - 1);
    const int th = (row >> p.tw_log2) & ((1 << p.th_log2) - 1);
    const int tb = row >> (p.tw_log2 + p.th_log2);
    const uint32_t st_f = smem_base + Cfg::STAGE_OFF + half * (NBF * Cfg::EPI_F_BYTES);
    const uint32_t st_h = smem_base + Cfg::STAGE_OFF + 2 * NBF * Cfg::EPI_F_BYTES + half * Cfg::EPI_H_BYTES;
    // swizzle of the staged rows: 128-byte rows SWIZZLE_128B (16-B chunk ^= row % 8), 64-byte rows SWIZZLE_64B (^= (row / 2) % 4),
    // 32-byte rows SWIZZLE_32B (^= (row / 4) % 2)
    const uint32_t swf = (SLW == 32) ? ((uint32_t)row & 7u) : ((uint32_t)(row >> 1) & 3u);
    const uint32_t swh = (SLW == 32) ? ((uint32_t)(row >> 1) & 3u) : ((uint32_t)(row >> 2) & 1u);
    auto res_full = [&](uint32_t b) { return bar_base + 8u * (uint32_t)(2 * STAGES + 6 + half * 4) + 8u * b; };
    const uint32_t tempty_leader0 = (CG == 2 && rank != 0) ? mapa_shared(tempty_bar(0), 0) : 0u;
    int it = 0;
    TRACE_DECL(tr_wait_tfull);
    TRACE_DECL(tr_busy);
    uint32_t g = 0;                                       // slices processed so far by this half-group (EPI 2: ring position)
    for (int tile = unit0; tile < total_tiles; tile += unit_step, ++it) {
      const int buf = it & 1;
      const uint32_t use = (uint32_t)(it >> 1);
      const TcItem ti = tc_decode_item(p, tile, BLOCK_N);
      if (CG == 1 && splitk) {                               // sum the k-range partials first (or hand ours over and stop)
        mbar_wait(tfull_bar(buf), use & 1u);
        tc_fence_after();
        if (splitk_prepass<BLOCK_N>(p, tile, sidx, tmem_base + (uint32_t)(buf * BLOCK_N), warp, lane)) continue;
      }
      const int m_tile = ti.m_unit * CG + (int)rank;
      const int xt = m_tile % p.tiles_x;
      const int r = m_tile / p.tiles_x;
      const int yt = r % p.tiles_y, bt = r / p.tiles_y;
      const int x0 = xt << p.tw_log2, y0 = yt << p.th_log2, b0 = bt * TB;
      const int x = x0 + tw, y = y0 + th, b = b0 + tb;
      const bool valid = (x < p.Wo) && (y < p.Ho) && (b < p.B) && (m_tile < p.m_tiles);
      const long long pix = ((long long)b * p.Ho + y) * p.Wo + x;
      const int n_base = ti.n_tile * BLOCK_N + ti.n_off;
      int nsl = ti.w / SLW;                                 // SLW-column slices of this item that exist in the output
      if ((p.N - n_base) < ti.w) nsl = (p.N - n_base) / SLW;
      const float* rb = (p.rowbias != nullptr && valid) ? p.rowbias + (pix / p.rows_per_batch) * (long long)p.N : nullptr;
      const bool res32 = (EPI == 1) && (p.residual != nullptr) && p.res_f32 && valid;
      const bool res16 = (p.residual != nullptr) && !p.res_f32 && valid;
      const float* res_row = static_cast<const float*>(p.residual) + pix * p.ldr;
      float st_sum = 0.f, st_sq = 0.f;

      auto issue_res = [&](int sl, uint32_t gg) {           // elected lane, EPI == 2: residual slice -> fp32 slot gg & 1
        const uint32_t bb = gg & 1u;
        mbar_arrive_expect_tx(res_full(bb), Cfg::EPI_F_BYTES);
        tma_load_4d(st_f + bb * Cfg::EPI_F_BYTES, &maps.r, res_full(bb), n_base + sl * SLW, x0, y0, b0);
      };
      float rpre[2][SLW];                                   // EPI 1: fp32 residual of the next two slices of this half-group
      auto load_res = [&](int sl, float (&dst)[SLW]) {
#pragma unroll
        for (int i = 0; i < SLW / 8; ++i) ldg256(res_row + n_base + sl * SLW + i * 8, &dst[i * 8]);
      };
      if (EPI == 2) {
        if (half < nsl && lead_warp && elect_one()) {
          bulk_wait_read_all();                             // both fp32 slots are free again
          issue_res(half, g);
        }
      } else {
        if (res32 && half < nsl) {
          load_res(half, rpre[0]);
          if (half + 2 < nsl) load_res(half + 2, rpre[1]);
        }
        // pull the NEXT item's residual rows (this half-group's slices) into L2 while this one is processed
        if ((p.residual != nullptr) && p.res_f32 && tile + unit_step < total_tiles) {
          const TcItem ti2 = tc_decode_item(p, tile + unit_step, BLOCK_N);
          const int m_tile2 = ti2.m_unit * CG + (int)rank;
          const int xt2 = m_tile2 % p.tiles_x;
          const int r2 = m_tile2 / p.tiles_x;
          const int yt2 = r2 % p.tiles_y, bt2 = r2 / p.tiles_y;
          const int x2 = (xt2 << p.tw_log2) + tw, y2 = (yt2 << p.th_log2) + th, b2 = bt2 * TB + tb;
          if ((x2 < p.Wo) && (y2 < p.Ho) && (b2 < p.B) && (m_tile2 < p.m_tiles)) {
            const long long pix2 = ((long long)b2 * p.Ho + y2) * p.Wo + x2;
            const int col2 = ti2.n_tile * BLOCK_N + ti2.n_off + 16 * half;       // one 32-byte sector's line per 32 columns
            const float* rrow = static_cast<const float*>(p.residual) + pix2 * p.ldr + col2;
#pragma unroll
            for (int i = 0; i < BLOCK_N / 32; ++i)
              if (i < (ti2.w >> 5) && col2 + i * 32 < p.N)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(rrow + i * 32));
          }
        }
      }

      TRACE_T0(tq0);
      mbar_wait(tfull_bar(buf), use & 1u);
      TRACE_ADD(tr_wait_tfull, tq0);
      TRACE_T0(tb0);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BLOCK_N);
      auto release_acc = [&]() {                            // after this warp's last TMEM read of the item
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (CG == 2 && rank != 0) mbar_arrive_cluster(tempty_leader0 + 8u * buf);
          else mbar_arrive(tempty_bar(buf));
        }
      };
      if (half >= nsl) release_acc();                       // nothing to read for this half-group

      // (fully unrolled over the slices a half-group can own: lets the compiler hoist the next slice's loads over the barriers)
#pragma unroll
      for (int k = 0; k < (BLOCK_N / SLW + 1) / 2; ++k) {
        const int sl = half + 2 * k;
        const int pi = k & 1;                               // rpre slot of this slice
        if (sl >= nsl) break;                               // uniform over the half-group
        const int n = n_base + sl * SLW;
        const uint32_t f_slot = st_f + (NBF > 1 ? (g & 1u) * Cfg::EPI_F_BYTES : 0u);
        const uint32_t f_row = f_slot + (uint32_t)row * (uint32_t)(SLW * 4);
        const uint32_t h_row = st_h + (uint32_t)row * (uint32_t)(SLW * 2);
        float f[SLW];
        {
          uint32_t v[SLW];
          if constexpr (SLW == 32) tmem_ld_32x32(t_row + (uint32_t)(sl * SLW), v);
          else tmem_ld_32x16(t_row + (uint32_t)(sl * SLW), v);
          tmem_ld_wait();
          if (sl + 2 >= nsl) release_acc();                 // last TMEM read of this item: release the accumulator early
#pragma unroll
          for (int i = 0; i < SLW; ++i) f[i] = __uint_as_float(v[i]);
        }
        if (valid) {
          if (p.bias != nullptr) {
#pragma unroll
            for (int i = 0; i < SLW; i += 4) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + n + i));
              f[i] += bv.x; f[i + 1] += bv.y; f[i + 2] += bv.z; f[i + 3] += bv.w;
            }
          }
          if (rb != nullptr) {
#pragma unroll
            for (int i = 0; i < SLW; i += 4) {
              const float4 bv = __ldg(reinterpret_cast<const float4*>(rb + n + i));
              f[i] += bv.x; f[i + 1] += bv.y; f[i + 2] += bv.z; f[i + 3] += bv.w;
            }
          }
          if (res32) {
#pragma unroll
            for (int i = 0; i < SLW; ++i) f[i] += rpre[pi][i];
            if (sl + 4 < nsl) load_res(sl + 4, rpre[pi]);
          } else if (res16) {
            const uint4* rp = reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(p.residual) + pix * p.ldr + n);
#pragma unroll
            for (int i = 0; i < SLW / 8; ++i) {
              const uint4 rv = __ldg(rp + i);
              float2 t;
              t = unpack_bf16x2(rv.x); f[8 * i + 0] += t.x; f[8 * i + 1] += t.y;
              t = unpack_bf16x2(rv.y); f[8 * i + 2] += t.x; f[8 * i + 3] += t.y;
              t = unpack_bf16x2(rv.z); f[8 * i + 4] += t.x; f[8 * i + 5] += t.y;
              t = unpack_bf16x2(rv.w); f[8 * i + 6] += t.x; f[8 * i + 7] += t.y;
            }
          }
        }
        // every store issued so far must have been read out of shared memory: the fp32 slot written below (EPI 1: the only one;
        // EPI 2: the one whose residual is being consumed was free already, the OTHER one receives the next residual after the
        // barrier) and the single bf16 slot
        if (lead_warp && elect_one()) bulk_wait_read_all();
        named_bar_sync(1 + half, 128);
        if (EPI == 2) {
          // all threads have left the previous slice (incl. its column-statistics reads): the other slot may be refilled
          if (sl + 2 < nsl && lead_warp && elect_one()) issue_res(sl + 2, g + 1);
          mbar_wait(res_full(g & 1u), (g >> 1) & 1u);
#pragma unroll
          for (uint32_t j = 0; j < NCF; ++j) {
            const float4 rv = lds128(f_row + ((j ^ swf) << 4));
            f[4 * j] += rv.x; f[4 * j + 1] += rv.y; f[4 * j + 2] += rv.z; f[4 * j + 3] += rv.w;
          }
        }
        if (p.stats_out != nullptr && valid) {
#pragma unroll
          for (int i = 0; i < SLW; ++i) { st_sum += f[i]; st_sq += f[i] * f[i]; }
        }
        if (p.colstats != nullptr && !valid) {                // rows outside the output must not count in the column sums
#pragma unroll
          for (int i = 0; i < SLW; ++i) f[i] = 0.f;
        }
#pragma unroll
        for (uint32_t j = 0; j < NCF; ++j) sts128(f_row + ((j ^ swf) << 4), f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
        if (p.out2 != nullptr) {
#pragma unroll
          for (uint32_t j = 0; j < NCH; ++j)
            sts128u(h_row + ((j ^ swh) << 4), pack_bf16x2(f[8 * j], f[8 * j + 1]), pack_bf16x2(f[8 * j + 2], f[8 * j + 3]),
                    pack_bf16x2(f[8 * j + 4], f[8 * j + 5]), pack_bf16x2(f[8 * j + 6], f[8 * j + 7]));
        }
        fence_proxy_async();
        named_bar_sync(1 + half, 128);
        if (lead_warp && elect_one()) {
          tma_store_4d(&maps.o, f_slot, n, x0, y0, b0);
          if (p.out2 != nullptr) tma_store_4d(&maps.o2, st_h, n, x0, y0, b0);
          bulk_commit_group();
        }
        if (p.colstats != nullptr) {
          // GroupNorm statistics for free: column sums of the staged slice over the tile's 128 rows.  Warp wq of the half-group
          // owns NCF / 4 16-byte chunks (4 columns each); lane = (row phase 0..7, column 0..3) walks rows phase + 8 i of one
          // chunk, which the swizzled layout spreads over all 32 banks; three shuffles fold the 8 phases.
          const uint32_t wq = (uint32_t)(warp - 2) & 3u, cc = (uint32_t)lane & 3u, r0 = (uint32_t)lane >> 2;
#pragma unroll
          for (uint32_t ch = 0; ch < NCF / 4; ++ch) {
            const uint32_t chunk = (NCF / 4) * wq + ch;
            float cs = 0.f, cq = 0.f;
#pragma unroll
            for (uint32_t i = 0; i < 16; ++i) {
              const uint32_t rr = r0 + 8u * i;
              const uint32_t sw = (SLW == 32) ? (rr & 7u) : ((rr >> 1) & 3u);
              const float v = lds32(f_slot + rr * (uint32_t)(SLW * 4) + ((chunk ^ sw) << 4) + cc * 4u);
              cs += v;
              cq += v * v;
            }
#pragma unroll
            for (int o = 4; o <= 16; o <<= 1) {
              cs += __shfl_xor_sync(0xffffffffu, cs, o);
              cq += __shfl_xor_sync(0xffffffffu, cq, o);
            }
            if (lane < 4 && m_tile < p.m_tiles)
              *reinterpret_cast<float2*>(p.colstats + ((long long)m_tile * p.N + n + 4 * (int)chunk + lane) * 2) = make_float2(cs, cq);
          }
        }
        ++g;
      }
      if (p.stats_out != nullptr && valid) {
        float* sp = p.stats_out + (pix * p.n_tiles + ti.n_tile) * 8;
        if (ti.w == BLOCK_N) *reinterpret_cast<float4*>(sp + half * 4) = make_float4(st_sum, st_sq, 0.f, 0.f);
        else *reinterpret_cast<float2*>(sp + ((ti.n_off != 0 ? 2 : 0) + half) * 2) = make_float2(st_sum, st_sq);
      }
      TRACE_ADD(tr_busy, tb0);
    }
    if (lead_warp && elect_one()) bulk_wait_read_all();         // staging memory must outlive the last store's read
    if (warp == 2) { TRACE_PUT(6, tr_wait_tfull); TRACE_PUT(7, tr_busy); }
#ifdef IA2P_TC_TRACE
    if (warp == 2) TRACE_PUT(11, gtime_ns());                          // this CTA's epilogue is done
#endif
  } else {
    // ------------------------------------------------------------ epilogue (4 warps, one accumulator row per thread)
    // TMEM -> registers hands every thread one output row.  Shared memory is NOT used here on purpose: with
    // cta_group::1 the UMMA operand reads already run close to the smem bandwidth, and staging the tile through smem for
    // a transposed (fully coalesced) store measurably starves the MMA.  Instead each thread moves whole 32-byte sectors
    // with 256-bit global accesses, and the fp32 residual (independent of the accumulator) is fetched two 32-column
    // chunks ahead -- the first two before waiting for the MMA -- so its latency hides behind the main loop.
    const int q = warp & 3;                               // TMEM lane quarter this warp may read
    const int half = (warp - 2) >> 2;                     // 0: first half of the tile's 32-column chunks, 1: second half
    const int row = q * 32 + lane;
    const int tw = row & ((1 << p.tw_log2) - 1);
    const int th = (row >> p.tw_log2) & ((1 << p.th_log2) - 1);
    const int tb = row >> (p.tw_log2 + p.th_log2);
    constexpr int NCH = BLOCK_N / 32;
    constexpr int NCH0 = (NCH + 1) / 2;                   // chunks [0, NCH0) -> half 0, [NCH0, NCH) -> half 1 (full tile)
    const uint32_t tempty_leader0 = (CG == 2 && rank != 0) ? mapa_shared(tempty_bar(0), 0) : 0u;
    int it = 0;
    TRACE_DECL(tr_wait_tfull);
    TRACE_DECL(tr_busy);
    for (int tile = unit0; tile < total_tiles; tile += unit_step, ++it) {
      const int buf = it & 1;
      const uint32_t use = (uint32_t)(it >> 1);
      const TcItem ti = tc_decode_item(p, tile, BLOCK_N);
      if (CG == 1 && splitk) {                               // sum the k-range partials first (or hand ours over and stop)
        mbar_wait(tfull_bar(buf), use & 1u);
        tc_fence_after();
        if (splitk_prepass<BLOCK_N>(p, tile, sidx, tmem_base + (uint32_t)(buf * BLOCK_N), warp, lane)) continue;
      }
      const int n_tile = ti.n_tile;
      const int m_tile = ti.m_unit * CG + (int)rank;
      const int xt = m_tile % p.tiles_x;
      const int r = m_tile / p.tiles_x;
      const int yt = r % p.tiles_y, bt = r / p.tiles_y;
      const int x = (xt << p.tw_log2) + tw, y = (yt << p.th_log2) + th, b = bt * TB + tb;
      const bool valid = (x < p.Wo) && (y < p.Ho) && (b < p.B) && (m_tile < p.m_tiles);
      const long long pix = ((long long)b * p.Ho + y) * p.Wo + x;
      const int n0 = n_tile * BLOCK_N + ti.n_off;           // first output column of this item
      const int nch = ti.w >> 5, nch0 = (nch + 1) >> 1;     // 32-column chunks of this item, and of its first half
      const int c_lo = half == 0 ? 0 : nch0, c_hi = half == 0 ? nch0 : nch;
      const float* rb = (p.rowbias != nullptr && valid) ? p.rowbias + (pix / p.rows_per_batch) * (long long)p.N : nullptr;
      const bool res32 = (p.residual != nullptr) && p.res_f32 && valid && !p.geglu;
      const float* res_row = static_cast<const float*>(p.residual) + pix * p.ldr;
      // consumer side of the LN fold: this row's mean / rstd from the producer's partial sums (fixed order: reproducible)
      float ln_mean = 0.f, ln_rstd = 1.f;
      if (p.ln_stats != nullptr && valid) {
        // All partials of the row are requested before the first add: issued one by one inside a run-time loop, the ~20 dependent
        // L2 round trips (8 k cycles) made the epilogue of every LN-folded GEMM longer than its main loop (MMA warp waiting for a
        // free accumulator 24-31 % of the QKV / GEGLU launches, profiles/README.md).  Same summation order as before.
        const float* sp = p.ln_stats + pix * (long long)p.ln_parts * 2;
        float s1 = 0.f, s2 = 0.f;
        if ((p.ln_parts & 3) == 0) {                        // 4 partials = one 32-byte sector (ia2p_gemm_ln_parts: 4 per N tile)
          const int nq = p.ln_parts >> 2;
          for (int i0 = 0; i0 < nq; i0 += 3) {
            float v[3][8];
#pragma unroll
            for (int j = 0; j < 3; ++j)
              if (i0 + j < nq) ldg256(sp + (i0 + j) * 8, v[j]);
#pragma unroll
            for (int j = 0; j < 3; ++j)
              if (i0 + j < nq) {
                s1 += v[j][0]; s2 += v[j][1]; s1 += v[j][2]; s2 += v[j][3];
                s1 += v[j][4]; s2 += v[j][5]; s1 += v[j][6]; s2 += v[j][7];
              }
          }
        } else {
          for (int i = 0; i < p.ln_parts; ++i) {
            const float2 v = __ldg(reinterpret_cast<const float2*>(sp) + i);
            s1 += v.x;
            s2 += v.y;
          }
        }
        ln_mean = s1 * p.ln_inv_n;
        ln_rstd = rsqrtf(fmaxf(s2 * p.ln_inv_n - ln_mean * ln_mean, 0.f) + p.ln_eps);
      }
      float st_sum = 0.f, st_sq = 0.f;                      // producer side: partial row statistics of this column half

      float rpre[2][32];
      auto load_res = [&](int c, float (&dst)[32]) {
        if (n0 + c * 32 < p.N) {
#pragma unroll
          for (int i = 0; i < 4; ++i) ldg256(res_row + n0 + c * 32 + i * 8, &dst[i * 8]);
        }
      };
      if (res32) {
        load_res(c_lo, rpre[0]);
        if (c_lo + 1 < c_hi) load_res(c_lo + 1, rpre[1]);
      }
      // pull the NEXT tile's residual rows (this warp's column half) from DRAM into L2 while this tile is processed: the
      // epilogue of residual GEMMs with short K is latency-bound on these reads otherwise
      if ((p.residual != nullptr) && p.res_f32 && !p.geglu && tile + unit_step < total_tiles) {
        const int tile2 = tile + unit_step;
        const TcItem ti2 = tc_decode_item(p, tile2, BLOCK_N);
        const int m_tile2 = ti2.m_unit * CG + (int)rank;
        const int xt2 = m_tile2 % p.tiles_x;
        const int r2 = m_tile2 / p.tiles_x;
        const int yt2 = r2 % p.tiles_y, bt2 = r2 / p.tiles_y;
        const int x2 = (xt2 << p.tw_log2) + tw, y2 = (yt2 << p.th_log2) + th, b2 = bt2 * TB + tb;
        if ((x2 < p.Wo) && (y2 < p.Ho) && (b2 < p.B) && (m_tile2 < p.m_tiles)) {
          const long long pix2 = ((long long)b2 * p.Ho + y2) * p.Wo + x2;
          const int nch2 = ti2.w >> 5, nch20 = (nch2 + 1) >> 1;
          const int c2_lo = half == 0 ? 0 : nch20, c2_n = half == 0 ? nch20 : nch2 - nch20;
          const int col2 = ti2.n_tile * BLOCK_N + ti2.n_off + c2_lo * 32;
          const float* rrow = static_cast<const float*>(p.residual) + pix2 * p.ldr + col2;
#pragma unroll
          for (int i = 0; i < NCH0; ++i)
            if (i < c2_n && col2 + i * 32 < p.N)
              asm volatile("prefetch.global.L2 [%0];" ::"l"(rrow + i * 32));
        }
      }

      TRACE_T0(tq0);
      mbar_wait(tfull_bar(buf), use & 1u);
      TRACE_ADD(tr_wait_tfull, tq0);
      TRACE_T0(tb0);
      tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BLOCK_N);

      if (!p.geglu) {
#pragma unroll
        for (int cc = 0; cc < NCH0; ++cc) {
          const int c = c_lo + cc;
          const int n = n0 + c * 32;
          if (c < c_hi && n < p.N) {                             // warp-uniform
            uint32_t v[32];
            tmem_ld_32x32(t_row + (uint32_t)(c * 32), v);
            tmem_ld_wait();
            if (valid) {
              float f[32];
#pragma unroll
              for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
              if (p.ln_stats != nullptr) {      // rstd * (acc - mean * c1) + bias = acc * rstd + (c1 * (-mean * rstd) + bias)
                const float ln_nm = -ln_mean * ln_rstd;
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                  const float4 cv = __ldg(reinterpret_cast<const float4*>(p.ln_c1 + n + i));
                  float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
                  if (p.bias != nullptr) bv = __ldg(reinterpret_cast<const float4*>(p.bias + n + i));
                  f[i] = fmaf(f[i], ln_rstd, fmaf(cv.x, ln_nm, bv.x)); f[i + 1] = fmaf(f[i + 1], ln_rstd, fmaf(cv.y, ln_nm, bv.y));
                  f[i + 2] = fmaf(f[i + 2], ln_rstd, fmaf(cv.z, ln_nm, bv.z)); f[i + 3] = fmaf(f[i + 3], ln_rstd, fmaf(cv.w, ln_nm, bv.w));
                }
              } else if (p.bias != nullptr) {
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                  const float4 bv = __ldg(reinterpret_cast<const float4*>(p.bias + n + i));
                  f[i] += bv.x; f[i + 1] += bv.y; f[i + 2] += bv.z; f[i + 3] += bv.w;
                }
              }
              if (rb != nullptr) {
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                  const float4 bv = __ldg(reinterpret_cast<const float4*>(rb + n + i));
                  f[i] += bv.x; f[i + 1] += bv.y; f[i + 2] += bv.z; f[i + 3] += bv.w;
                }
              }
              if (res32) {
#pragma unroll
                for (int i = 0; i < 32; ++i) f[i] += rpre[cc & 1][i];
                if (c + 2 < c_hi) load_res(c + 2, rpre[cc & 1]);
              } else if (p.residual != nullptr) {
                if (p.res_f32) {   // (unreachable: res32 covers it) kept for clarity
                } else {
                  const uint4* rp = reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(p.residual) + pix * p.ldr + n);
#pragma unroll
                  for (int i = 0; i < 4; ++i) {
                    const uint4 rv = __ldg(rp + i);
                    float2 t;
                    t = unpack_bf16x2(rv.x); f[8 * i + 0] += t.x; f[8 * i + 1] += t.y;
                    t = unpack_bf16x2(rv.y); f[8 * i + 2] += t.x; f[8 * i + 3] += t.y;
                    t = unpack_bf16x2(rv.z); f[8 * i + 4] += t.x; f[8 * i + 5] += t.y;
                    t = unpack_bf16x2(rv.w); f[8 * i + 6] += t.x; f[8 * i + 7] += t.y;
                  }
                }
              }
              if (p.stats_out != nullptr) {
#pragma unroll
                for (int i = 0; i < 32; ++i) { st_sum += f[i]; st_sq += f[i] * f[i]; }
              }
              if (p.out2 != nullptr) {
                __nv_bfloat16* op2 = p.out2 + pix * p.ldo2 + n;
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                  float o[8];
#pragma unroll
                  for (int k = 0; k < 8; ++k) o[k] = __uint_as_float(pack_bf16x2(f[16 * i + 2 * k], f[16 * i + 2 * k + 1]));
                  stg256(reinterpret_cast<float*>(op2 + i * 16), o);
                }
              }
              if (p.out_f32) {
                float* op = static_cast<float*>(p.out) + pix * p.ldo + n;
#pragma unroll
                for (int i = 0; i < 4; ++i) stg256(op + i * 8, &f[i * 8]);
              } else {
                __nv_bfloat16* op = static_cast<__nv_bfloat16*>(p.out) + pix * p.ldo + n;
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                  float o[8];
#pragma unroll
                  for (int k = 0; k < 8; ++k) o[k] = __uint_as_float(pack_bf16x2(f[16 * i + 2 * k], f[16 * i + 2 * k + 1]));
                  stg256(reinterpret_cast<float*>(op + i * 16), o);
                }
              }
            }
          }
        }
      } else {
        // GEGLU: W rows interleaved in 32-row groups [value | gate]; out col = n/2 + i:  value * gelu_erf(gate)
#pragma unroll 1
        for (int c = half; c < (ti.w >> 6); c += 2) {            // value/gate chunk pairs alternate between the two halves
          const int n = n0 + c * 64;
          if (n >= p.N) break;                                   // warp-uniform
          uint32_t vv[32], vg[32];
          tmem_ld_32x32(t_row + (uint32_t)(c * 64), vv);
          tmem_ld_32x32(t_row + (uint32_t)(c * 64 + 32), vg);
          tmem_ld_wait();
          if (valid) {
            float f[32];
            // LN fold as two FMAs per element: rstd * (acc - mean * c1) + bias = acc * rstd + (c1 * (-mean * rstd) + bias)
            const float ln_nm = -ln_mean * ln_rstd;
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              float4 bv = make_float4(0.f, 0.f, 0.f, 0.f), bg = bv;
              if (p.bias != nullptr) {
                bv = __ldg(reinterpret_cast<const float4*>(p.bias + n + i));
                bg = __ldg(reinterpret_cast<const float4*>(p.bias + n + 32 + i));
              }
              if (p.ln_stats != nullptr) {
                const float4 cv = __ldg(reinterpret_cast<const float4*>(p.ln_c1 + n + i));
                const float4 cg = __ldg(reinterpret_cast<const float4*>(p.ln_c1 + n + 32 + i));
                bv.x = fmaf(cv.x, ln_nm, bv.x); bv.y = fmaf(cv.y, ln_nm, bv.y); bv.z = fmaf(cv.z, ln_nm, bv.z); bv.w = fmaf(cv.w, ln_nm, bv.w);
                bg.x = fmaf(cg.x, ln_nm, bg.x); bg.y = fmaf(cg.y, ln_nm, bg.y); bg.z = fmaf(cg.z, ln_nm, bg.z); bg.w = fmaf(cg.w, ln_nm, bg.w);
              }
              const float a0 = __uint_as_float(vv[i + 0]), a1 = __uint_as_float(vv[i + 1]), a2 = __uint_as_float(vv[i + 2]), a3 = __uint_as_float(vv[i + 3]);
              const float g0 = __uint_as_float(vg[i + 0]), g1 = __uint_as_float(vg[i + 1]), g2 = __uint_as_float(vg[i + 2]), g3 = __uint_as_float(vg[i + 3]);
              f[i + 0] = fmaf(a0, ln_rstd, bv.x) * gelu_erf_f(fmaf(g0, ln_rstd, bg.x));
              f[i + 1] = fmaf(a1, ln_rstd, bv.y) * gelu_erf_f(fmaf(g1, ln_rstd, bg.y));
              f[i + 2] = fmaf(a2, ln_rstd, bv.z) * gelu_erf_f(fmaf(g2, ln_rstd, bg.z));
              f[i + 3] = fmaf(a3, ln_rstd, bv.w) * gelu_erf_f(fmaf(g3, ln_rstd, bg.w));
            }
            __nv_bfloat16* op = static_cast<__nv_bfloat16*>(p.out) + pix * p.ldo + (n >> 1);
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              float o[8];
#pragma unroll
              for (int k = 0; k < 8; ++k) o[k] = __uint_as_float(pack_bf16x2(f[16 * i + 2 * k], f[16 * i + 2 * k + 1]));
              stg256(reinterpret_cast<float*>(op + i * 16), o);
            }
          }
        }
      }
      // four partial-sum slots per (row, n tile): a whole tile fills {half 0, -, half 1, -} (the unused ones with zeros), a
      // tail-split slice `sub` fills {2 sub + half}
      if (p.stats_out != nullptr && valid) {
        float* sp = p.stats_out + (pix * p.n_tiles + n_tile) * 8;
        if (ti.w == BLOCK_N) *reinterpret_cast<float4*>(sp + half * 4) = make_float4(st_sum, st_sq, 0.f, 0.f);
        else *reinterpret_cast<float2*>(sp + ((ti.n_off != 0 ? 2 : 0) + half) * 2) = make_float2(st_sum, st_sq);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CG == 2 && rank != 0) mbar_arrive_cluster(tempty_leader0 + 8u * buf);   // release the LEADER's MMA warp
        else mbar_arrive(tempty_bar(buf));
      }
      TRACE_ADD(tr_busy, tb0);
    }
    if (warp == 2) { TRACE_PUT(6, tr_wait_tfull); TRACE_PUT(7, tr_busy); }
#ifdef IA2P_TC_TRACE
    if (warp == 2) TRACE_PUT(11, gtime_ns());                          // this CTA's epilogue is done
#endif
  }

  // ------------------------------------------------------------ teardown
#ifdef IA2P_TC_TRACE
  if (warp == 0) TRACE_PUT(8, gtime_ns());
#endif
  tc_fence_before();
  if (CG == 2 || mc > 1) cluster_sync_all(); else __syncthreads();   // all CTAs done with TMEM / no remote arrive or multicast in flight
  if (warp == 1) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_2sm(tmem_base, Cfg::TMEM_COLS); else tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
#ifdef IA2P_TC_TRACE
  if (threadIdx.x == 0 && g_tc_timeline != nullptr) atomicMax(g_tc_timeline + 2 * (size_t)p.trace_id + 1, gtime_ns());
  if (warp == 0) TRACE_PUT(14, gtime_ns());                                 // after the final barrier: the CTA's true end
#endif
}

// ================================================================ host side
// Tensor map, rank <= 4, dims/strides innermost-first; strides in ELEMENTS (stride of dim 0 is 1).  Default: bf16 operand
// tiles with SWIZZLE_128B; the epilogue staging slices use fp32 / SWIZZLE_64B and bf16 / SWIZZLE_32B.
static int make_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_el,
                    const uint32_t* box, CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                    CUtensorMapSwizzle sw = CU_TENSOR_MAP_SWIZZLE_128B) {
  const uint64_t esz = (dt == CU_TENSOR_MAP_DATA_TYPE_FLOAT32) ? 4 : 2;
  EncodeTiledFn enc = tensor_map_encoder();
  IA2P_REQUIRE(enc != nullptr, IA2P_E_DRIVER, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t gdim[4], gstr[3];
  cuuint32_t bx[4], es[4];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) {
      gstr[i - 1] = strides_el[i] * esz;
      IA2P_REQUIRE(gstr[i - 1] % 16 == 0, IA2P_E_ALIGN, "tensor-map stride %llu B not a multiple of 16", (unsigned long long)gstr[i - 1]);
    }
  }
  IA2P_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0, IA2P_E_ALIGN, "tensor-map base not 16-byte aligned");
  CUresult r = enc(m, dt, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  IA2P_REQUIRE(r == CUDA_SUCCESS, IA2P_E_DRIVER, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
  return 0;
}

// Tile width: the widest of {256, 160, 128, 64} that divides N and still yields enough tiles to occupy the GPU; problems with
// few output rows (batch-1 512^2: M = 512 -> 4 row tiles) fall through to the narrowest one, so that e.g. the FF-out GEMM
// (N 1280, K 5120) streams its weights through 80 CTAs instead of 20.
constexpr int kMinTilesForWideBlock = 120;
constexpr int kSplitKMinKb = 40;                         // split-K only from K >= 2560 on
static bool splitk_enabled();
static int pick_block_n(int64_t N, bool geglu, int64_t m_tiles, int num_kb = 0) {
  if (const char* e = getenv("IA2P_GEMM_BN")) {          // experiments only
    const int v = atoi(e);
    if ((v == 64 || v == 128 || v == 160 || v == 256) && N % v == 0 && (!geglu || v % 64 == 0)) return v;
  }
  if (N == 1280 && !geglu) {                             // experiments only: tile width of the N = 1280 problems (out-proj, to_q, FF-out)
    static int bn1280 = -1;
    if (bn1280 < 0) { const char* e = getenv("IA2P_GEMM_BN1280"); bn1280 = e ? atoi(e) : 0; }
    if ((bn1280 == 128 || bn1280 == 160 || bn1280 == 64) && m_tiles * (N / bn1280) >= kMinTilesForWideBlock) return bn1280;
  }
  const int cand[4] = {256, 160, 128, 64};
  int last = 0, first = 0;
  for (int i = 0; i < 4; ++i) {
    const int c = cand[i];
    if (N % c != 0 || (geglu && c % 64 != 0)) continue;
    if (first == 0) first = c;
    last = c;
    if (m_tiles * (N / c) >= kMinTilesForWideBlock) return c;
  }
  // too few tiles at every width: with a split-K workspace keep the WIDEST tile (best operand reuse) and fill the SMs with
  // k-range splits instead of narrow tiles
  if (first != 0 && num_kb >= kSplitKMinKb && splitk_enabled() && m_tiles * (N / first) * 2 <= sm_count()) return first;
  return last != 0 ? last : 128;                         // 128 with a ragged last tile when nothing divides N
}

// Split-K workspace (ia2p_set_tc_workspace): [16 KB of tile flags, zero-initialised by the caller][partial accumulators]
static thread_local void* g_ws_ptr = nullptr;
static thread_local long long g_ws_bytes = 0;
constexpr long long kWsFlagBytes = 16384;
static bool splitk_enabled() {
#ifndef IA2P_WITH_SPLITK
  return false;
#endif
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("IA2P_GEMM_SPLITK");          // experiments only: 0 disables
    v = (e != nullptr && e[0] == '0') ? 0 : 1;
  }
  return v != 0 && g_ws_ptr != nullptr;
}
// k-range splits for a problem of `units` tiles (single-CTA kernel) and num_kb k-blocks; 1 = no split
static int pick_ksplit(long long units, int num_kb, int bn) {
  // A split costs a dump + a fix-up pass (~2 us + ~2 us per extra split) and saves (1 - 1/ks) of the K loop (~0.35 us per
  // k-block): worth it from ~16 k-blocks per split on (measured: 7 splits of a 20-k-block out-projection ran 2x SLOWER).
  if (!splitk_enabled() || units * 2 > sm_count() || num_kb < kSplitKMinKb || units > kWsFlagBytes / 4) return 1;
  int ks = (int)(sm_count() / units);
  if (ks > num_kb / 16) ks = num_kb / 16;
  if (ks > kMaxKSplit) ks = kMaxKSplit;
  const long long per = (long long)bn * 128 * 4;         // bytes of one partial tile
  while (ks > 1 && units * (ks - 1) * per > g_ws_bytes - kWsFlagBytes) --ks;
  return ks < 2 ? 1 : ks;
}

static thread_local const void* g_pf_ptr = nullptr;
static thread_local long long g_pf_bytes = 0;

static bool tail_split_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("IA2P_GEMM_TAILSPLIT");       // experiments only: 0 disables
    v = (e != nullptr && e[0] == '0') ? 0 : 1;
  }
  return v != 0;
}

template <int BN, int CG, int EPI>
static int launch_tc(const TcMaps& maps, TcParams& p, cudaStream_t st) {
  using Cfg = TcCfg<BN, CG, EPI>;
  IA2P_ONCE_PER_DEVICE(IA2P_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<BN, CG, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES)));
  p.n_tiles = (p.N + BN - 1) / BN;
  const int units = ((p.m_tiles + CG - 1) / CG) * p.n_tiles;
  const int max_units = sm_count() / CG;
  const int grid = (units < max_units ? units : max_units) * CG;
  // Tail split: with r = units mod G tiles left for a last wave that would occupy r of G CTAs (pairs), cut those tiles into
  // two column halves when both halves still fit in ONE wave (a half tile costs ~0.6 of a whole one: the main loop of a
  // narrower tile is bound by the A-operand traffic).  Needs BLOCK_N / 2 to be a whole number of 32-column epilogue chunks
  // (64-column value|gate groups for GEGLU) and N a multiple of BLOCK_N (no ragged last tile).
  p.full_items = units;
  p.total_items = units;
  p.split = 1;
  p.ksplit = 1;
  p.kb_per = p.num_kb;
  p.ws = nullptr;
  p.flags = nullptr;
  int grid_override = 0;
  if (CG == 1) {
    const int ks = pick_ksplit(units, p.num_kb, BN);
    if (ks > 1) {
      p.kb_per = (p.num_kb + ks - 1) / ks;
      p.ksplit = (p.num_kb + p.kb_per - 1) / p.kb_per;
      p.flags = static_cast<unsigned*>(g_ws_ptr);
      p.ws = reinterpret_cast<float*>(static_cast<char*>(g_ws_ptr) + kWsFlagBytes);
      grid_override = units * p.ksplit;
    }
  }
  const int rem = units % max_units;
  IA2P_REQUIRE(p.mc <= 1 || (CG == 1 && p.ksplit == 1 && units <= max_units && p.n_tiles % p.mc == 0), IA2P_E_ARG,
               "tc launch: A-multicast picked for a launch that cannot run it (internal)");
  const bool can_split = p.ksplit == 1 && p.mc <= 1 && tail_split_enabled() && (BN % 64 == 0) && (!p.geglu || BN % 128 == 0) && (p.N % BN == 0);
  if (can_split && units > max_units && rem != 0 && 2 * rem <= max_units) {
    p.split = 2;
    p.full_items = units - rem;
    p.total_items = p.full_items + 2 * rem;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(grid_override ? grid_override : grid));
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (CG == 1 && p.mc > 1) ? p.mc : CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 2 : 1;
#ifdef IA2P_TC_TRACE
  p.trace_id = g_tc_launch_id++;
#endif
  p.early_b = pdl_enabled() ? 1 : 0;
  p.pf_ptr = static_cast<const char*>(g_pf_ptr);       // one-shot hint: consumed by this launch
  p.pf_bytes = g_pf_bytes;
  g_pf_ptr = nullptr;
  g_pf_bytes = 0;
  IA2P_CUDA(cudaLaunchKernelEx(&cfg, tc_gemm_kernel<BN, CG, EPI>, maps, p));
  IA2P_LAUNCH_CHECK();
  return 0;
}

// CTA-pair (cta_group::2) kernel is the default: it halves the L2->smem traffic of the B operand (48 -> 32 KB per CTA and
// k-block), which is what bounds the single-CTA main loop (~15 TB/s of L2->SM reads at 128x256 tiles, profiles/README.md); in the
// power-capped full step it is worth ~1-2 %.  Tiles with a short main loop (K <= 768) stay on the single-CTA kernel: the pair
// protocol's per-tile hand-offs (remote tmem_empty arrives, multicast commits) cost more than the B traffic saves there
// (measured: M 32768, N 5120, K 640 GEGLU 653 -> 535 TFLOP/s with pairs).  IA2P_GEMM_CG=1 / 2 force one kernel (experiments).
static bool use_pair(int m_tiles, int num_kb, int64_t N, int bn) {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("IA2P_GEMM_CG");
    v = (e != nullptr && e[0] == '1') ? 1 : (e != nullptr && e[0] == '2') ? 2 : 0;
  }
  if (m_tiles < 2 || bn == 64) return false;                      // BLOCK_N 64 exists for small problems only: single CTA
  if (pick_ksplit((int64_t)m_tiles * ((N + bn - 1) / bn), num_kb, bn) > 1) return false;   // split-K runs on the single-CTA kernel
  if (v == 0 && (int64_t)m_tiles * ((N + bn - 1) / bn) < 2 * sm_count()) return false;   // too few tiles to pair up
  static int min_kb = -1;
  if (min_kb < 0) {
    const char* e = getenv("IA2P_GEMM_PAIR_MINKB");      // experiments: pairs from this many k-blocks on (default 13)
    min_kb = (e != nullptr && atoi(e) > 0) ? atoi(e) : 13;
  }
  return v == 2 || (v == 0 && num_kb >= min_kb);
}

// A-operand multicast (TcParams::mc), OPT-IN (IA2P_GEMM_MC=2 | 4 = largest cluster): for problems that fit in ONE wave of
// single-CTA tiles (few output rows: batch-1 512^2, a single interactive request) every row tile's A block is fetched by all
// of its n-tiles; clusters of mc CTAs (consecutive n-tiles of one row tile) fetch each A block once and multicast it.  Needs
// n_tiles % mc == 0 and all clusters co-resident (one CTA per SM: floor(SMs per GPC / mc) clusters per GPC; the cap below is
// conservative).  Measured on B200 (tools/small_m_graph.py, profiles/README.md section 9): NO gain -- M 512 / 2048, N 1280,
// K 5120: 33.6 / 39.1 us without, 34.2 / 40.0 us with clusters of 4 -- the few-row main loop is bound by MMA issue (>= 94
// cycles per tcgen05.mma whatever its N) and by shared-memory bandwidth (every CTA still receives the whole A tile), not by the
// L2 -> SM traffic multicast removes.  Hence off by default.
static int pick_mc(int bn, int64_t m_tiles, int64_t N, int num_kb) {
#ifndef IA2P_WITH_MC
  return 1;
#endif
  const char* e = getenv("IA2P_GEMM_MC");                // read per call (tests toggle it); a few ns next to a launch
  const int cap = (e != nullptr && (e[0] == '2' || e[0] == '4')) ? (e[0] - '0') : 1;
  if (cap <= 1 || N % bn != 0 || use_pair((int)m_tiles, num_kb, N, bn)) return 1;
  const int64_t n_tiles = N / bn, units = m_tiles * n_tiles;
  if (units > sm_count() || pick_ksplit(units, num_kb, bn) > 1) return 1;
  for (int mc = cap; mc >= 2; mc >>= 1) {
    const int64_t resident = (mc == 4) ? (sm_count() / 18) * 4 * 4 : (sm_count() / 18) * 9 * 2;   // 8 GPCs x floor(18 / mc) clusters
    if (n_tiles % mc == 0 && units <= resident) return mc;
  }
  return 1;
}
// shrink an A-operand pixel box {64, TW, TH, TB} (128 rows ordered (tb, th, tw)) to one of mc row slices
static void slice_box(uint32_t* box, int mc) {
  int rows = 128 / mc;
  for (int d = 1; d < 4; ++d) {
    const uint32_t take = box[d] < (uint32_t)rows ? box[d] : (uint32_t)rows;
    rows /= (int)take;
    box[d] = take;
  }
}

// fp32 outputs go through the TMA-store epilogue (EPI = 1); IA2P_GEMM_EPI=0 forces the register-store epilogue (experiments)
static bool tma_epilogue(const TcParams& p) {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("IA2P_GEMM_EPI");
    v = (e != nullptr && e[0] == '0') ? 0 : 1;
  }
  return v != 0 && p.out_f32 && !p.geglu;
}

// EPI = 2 (TMA-loaded residual, one main-loop stage fewer) pays when the main loop of a tile is short: K <= 1536
static bool tma_residual(const TcParams& p) {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("IA2P_GEMM_EPI");
    v = (e != nullptr && e[0] == '1') ? 0 : 1;
  }
  return v != 0 && tma_epilogue(p) && p.residual != nullptr && p.res_f32 && p.num_kb <= 24;
}

// bf16 outputs without residual / LN-producer extras go through the TMA-store epilogue (EPI = 3); IA2P_GEMM_EPI3=0 keeps them on the
// register-store epilogue (experiments)
static bool tma_epilogue_bf16(const TcParams& p) {
#ifdef IA2P_WITH_SPLITK
  return false;                                          // the split-K fix-up pass lives in the EPI 0 / 1 epilogues only
#endif
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("IA2P_GEMM_EPI3");
    v = (e != nullptr && e[0] == '0') ? 0 : 1;
  }
  return v != 0 && !p.out_f32 && p.residual == nullptr && p.out2 == nullptr && p.stats_out == nullptr && p.colstats == nullptr;
}

template <int BN>
static int dispatch_bn(const TcMaps& maps, TcParams& p, cudaStream_t st) {
  const bool pair = use_pair(p.m_tiles, p.num_kb, p.N, BN);
  if (tma_epilogue_bf16(p)) return pair ? launch_tc<BN, 2, 3>(maps, p, st) : launch_tc<BN, 1, 3>(maps, p, st);
  if (tma_residual(p)) return pair ? launch_tc<BN, 2, 2>(maps, p, st) : launch_tc<BN, 1, 2>(maps, p, st);
  if (tma_epilogue(p)) return pair ? launch_tc<BN, 2, 1>(maps, p, st) : launch_tc<BN, 1, 1>(maps, p, st);
  return pair ? launch_tc<BN, 2, 0>(maps, p, st) : launch_tc<BN, 1, 0>(maps, p, st);
}

static int dispatch_tc(TcMaps& maps, TcParams& p, int bn, cudaStream_t st) {
  if (tma_epilogue(p)) {
    // output maps: same pixel-box geometry as the A operand, 32 columns wide (fp32: 128-byte rows, bf16 copy: 64-byte rows)
    const int TW = 1 << p.tw_log2, TH = 1 << p.th_log2, TB = 128 >> (p.tw_log2 + p.th_log2);
    const bool wide = tma_residual(p);                  // EPI 2: 32-column slices, EPI 1: 16 (TcCfg::SLW)
    const uint32_t box[4] = {wide ? 32u : 16u, (uint32_t)TW, (uint32_t)TH, (uint32_t)TB};
    const CUtensorMapSwizzle sw_f = wide ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    const CUtensorMapSwizzle sw_h = wide ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    const uint64_t dims[4] = {(uint64_t)p.N, (uint64_t)p.Wo, (uint64_t)p.Ho, (uint64_t)p.B};
    const uint64_t str[4] = {1, (uint64_t)(p.ost_x ? p.ost_x : p.ldo), (uint64_t)(p.ost_y ? p.ost_y : p.ldo * p.Wo),
                             (uint64_t)(p.ost_b ? p.ost_b : p.ldo * p.Wo * p.Ho)};
    if (int e = make_map(&maps.o, p.out, 4, dims, str, box, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sw_f)) return e;
    maps.o2 = maps.o;
    if (p.out2 != nullptr) {
      const uint64_t str2[4] = {1, (uint64_t)p.ldo2, (uint64_t)p.ldo2 * p.Wo, (uint64_t)p.ldo2 * p.Wo * p.Ho};
      if (int e = make_map(&maps.o2, p.out2, 4, dims, str2, box, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, sw_h)) return e;
    }
    maps.r = maps.o;
    if (tma_residual(p)) {
      const uint64_t strr[4] = {1, (uint64_t)p.ldr, (uint64_t)p.ldr * p.Wo, (uint64_t)p.ldr * p.Wo * p.Ho};
      if (int e = make_map(&maps.r, p.residual, 4, dims, strr, box, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, sw_f)) return e;
    }
  } else if (tma_epilogue_bf16(p)) {
    // bf16 output maps: the A operand's pixel-box geometry, 64 columns (SWIZZLE_128B) and 32 columns (remainder slice, SWIZZLE_64B)
    const int TW = 1 << p.tw_log2, TH = 1 << p.th_log2, TB = 128 >> (p.tw_log2 + p.th_log2);
    const uint64_t n_out = (uint64_t)(p.geglu ? p.N / 2 : p.N);
    const uint64_t dims[4] = {n_out, (uint64_t)p.Wo, (uint64_t)p.Ho, (uint64_t)p.B};
    const uint64_t str[4] = {1, (uint64_t)(p.ost_x ? p.ost_x : p.ldo), (uint64_t)(p.ost_y ? p.ost_y : p.ldo * p.Wo),
                             (uint64_t)(p.ost_b ? p.ost_b : p.ldo * p.Wo * p.Ho)};
    const uint32_t box64[4] = {64, (uint32_t)TW, (uint32_t)TH, (uint32_t)TB}, box32[4] = {32, (uint32_t)TW, (uint32_t)TH, (uint32_t)TB};
    if (n_out >= 64) {
      if (int e = make_map(&maps.o, p.out, 4, dims, str, box64, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_128B)) return e;
    }
    if (int e = make_map(&maps.o2, p.out, 4, dims, str, box32, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, CU_TENSOR_MAP_SWIZZLE_64B)) return e;
    if (n_out < 64) maps.o = maps.o2;
    maps.r = maps.o2;
  } else {
    maps.o = maps.w;                 // unused: keep the kernel parameter defined
    maps.o2 = maps.w;
    maps.r = maps.w;
  }
  switch (bn) {
    case 256: return dispatch_bn<256>(maps, p, st);
    case 160: return dispatch_bn<160>(maps, p, st);
    case 64:
      if (tma_epilogue_bf16(p)) return launch_tc<64, 1, 3>(maps, p, st);
      if (tma_residual(p)) return launch_tc<64, 1, 2>(maps, p, st);
      if (tma_epilogue(p)) return launch_tc<64, 1, 1>(maps, p, st);
      return launch_tc<64, 1, 0>(maps, p, st);
    default: return dispatch_bn<128>(maps, p, st);
  }
}

static int make_w_map(TcMaps& maps, const void* W, int64_t N, int64_t Ktot, int bn, int m_tiles) {
  const bool pair = use_pair(m_tiles, (int)(Ktot / 64), N, bn);   // must mirror dispatch_bn: a CTA of a pair loads BN/2 rows
  const uint64_t dims[2] = {(uint64_t)Ktot, (uint64_t)N};
  const uint64_t str[2] = {1, (uint64_t)Ktot};
  const uint32_t box[2] = {64, (uint32_t)(pair ? bn / 2 : bn)};
  if (int e = make_map(&maps.w, W, 2, dims, str, box)) return e;
  const uint32_t box2[2] = {64, (uint32_t)((bn % 64 == 0) ? box[1] / 2 : box[1])};   // half tiles (tail split)
  return make_map(&maps.w2, W, 2, dims, str, box2);
}

static int ilog2_exact(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

}  // namespace ia2p

using namespace ia2p;

#ifdef IA2P_TC_TRACE
extern "C" int ia2p_debug_set_timeline(void* dev_buffer) {    // also resets the launch-id counter; returns nothing useful
  unsigned long long* p = static_cast<unsigned long long*>(dev_buffer);
  g_tc_launch_id = 0;
  return (int)cudaMemcpyToSymbol(g_tc_timeline, &p, sizeof(p));
}
extern "C" int ia2p_debug_next_launch_id(void) { return g_tc_launch_id; }
extern "C" int ia2p_debug_set_trace(void* dev_buffer) {       // debug build only; not part of include/ia2p.h
  unsigned long long* p = static_cast<unsigned long long*>(dev_buffer);
  return (int)cudaMemcpyToSymbol(g_tc_trace, &p, sizeof(p));
}
extern "C" int ia2p_debug_set_trace_stride(int rows_per_launch) {   // > 0: trace row = launch id * rows_per_launch + blockIdx.x
  return (int)cudaMemcpyToSymbol(g_tc_trace_stride, &rows_per_launch, sizeof(int));
}
#endif

extern "C" int ia2p_tc_features(void) {
  int f = 0;
#ifdef IA2P_WITH_SPLITK
  f |= 1;
#endif
#ifdef IA2P_WITH_MC
  f |= 2;
#endif
  return f;
}

extern "C" int64_t ia2p_tc_workspace_bytes(void) { return 64ll << 20; }

extern "C" int ia2p_set_tc_workspace(void* workspace, int64_t bytes) {
  if (workspace == nullptr || bytes <= kWsFlagBytes || (reinterpret_cast<uintptr_t>(workspace) & 255) != 0) {
    g_ws_ptr = nullptr;
    g_ws_bytes = 0;
    return workspace == nullptr ? 0 : IA2P_E_ARG;
  }
  g_ws_ptr = workspace;
  g_ws_bytes = bytes;
  return 0;
}

extern "C" int ia2p_tc_prefetch_hint(const void* next_weights, int64_t bytes) {
  g_pf_ptr = (bytes >= 16 && (reinterpret_cast<uintptr_t>(next_weights) & 15) == 0) ? next_weights : nullptr;
  g_pf_bytes = g_pf_ptr ? (bytes & ~15LL) : 0;
  return 0;
}

extern "C" int ia2p_gemm_bf16(const void* A, int64_t lda, int64_t K1, const void* A2, int64_t lda2, int64_t K2,
                              const void* W, void* out, int64_t ldo, int64_t M, int64_t N,
                              const float* bias, const float* rowbias, int64_t rows_per_batch,
                              const void* residual, int64_t ldr, int res_dtype, int out_dtype, int epilogue, void* stream) {
  return ia2p_gemm_ln_bf16(A, lda, K1, A2, lda2, K2, W, out, ldo, M, N, bias, rowbias, rows_per_batch, residual, ldr, res_dtype,
                           out_dtype, epilogue, nullptr, 0, nullptr, nullptr, nullptr, 0, nullptr, 0.f, stream);
}

extern "C" int64_t ia2p_gemm_ln_parts(int64_t M, int64_t N, int64_t K) {
  const int bn = pick_block_n(N, false, (M + 127) / 128, (int)(K / 64));
  return 4 * ((N + bn - 1) / bn);
}

extern "C" int ia2p_gemm_ln_bf16(const void* A, int64_t lda, int64_t K1, const void* A2, int64_t lda2, int64_t K2,
                                 const void* W, void* out, int64_t ldo, int64_t M, int64_t N,
                                 const float* bias, const float* rowbias, int64_t rows_per_batch,
                                 const void* residual, int64_t ldr, int res_dtype, int out_dtype, int epilogue,
                                 void* out_bf16, int64_t ldo2, float* stats_out, float* colstats,
                                 const float* ln_stats, int64_t ln_parts, const float* ln_c1, float ln_eps, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE((ln_stats == nullptr) == (ln_c1 == nullptr) && (ln_stats == nullptr || (ln_parts > 0 && ln_parts <= 256)), IA2P_E_ARG,
               "gemm: ln_stats, ln_c1 and ln_parts must be given together");
  IA2P_REQUIRE(ln_stats == nullptr || (ln_parts % 4 != 0) || (reinterpret_cast<uintptr_t>(ln_stats) & 31) == 0, IA2P_E_ALIGN,
               "gemm: ln_stats must be 32-byte aligned");
  IA2P_REQUIRE((out_bf16 == nullptr && stats_out == nullptr) || epilogue != IA2P_EPI_GEGLU, IA2P_E_ARG,
               "gemm: the GEGLU epilogue cannot also produce LN statistics");
  IA2P_REQUIRE(out_bf16 == nullptr || ((reinterpret_cast<uintptr_t>(out_bf16) & 31) == 0 && ldo2 % 16 == 0), IA2P_E_ALIGN,
               "gemm: out_bf16 must be 32-byte aligned with ldo2 %% 16 == 0");
  IA2P_REQUIRE(A && W && out && M > 0 && N > 0 && K1 > 0, IA2P_E_ARG, "gemm: null pointer or empty shape");
  IA2P_REQUIRE((out_dtype == IA2P_BF16 || out_dtype == IA2P_F32) && (residual == nullptr || res_dtype == IA2P_BF16 || res_dtype == IA2P_F32),
               IA2P_E_ARG, "gemm: out/residual dtype must be bf16 or f32");
  IA2P_REQUIRE(K1 % 64 == 0 && K2 % 64 == 0 && K2 >= 0, IA2P_E_SHAPE, "gemm: K1=%lld K2=%lld must be multiples of 64", (long long)K1, (long long)K2);
  IA2P_REQUIRE(N % 32 == 0, IA2P_E_SHAPE, "gemm: N=%lld must be a multiple of 32", (long long)N);
  IA2P_REQUIRE(lda % 8 == 0 && ldo % 8 == 0 && (A2 == nullptr || lda2 % 8 == 0) && (residual == nullptr || ldr % 8 == 0),
               IA2P_E_ALIGN, "gemm: leading dimensions must be multiples of 8 elements");
  IA2P_REQUIRE((A2 == nullptr) == (K2 == 0), IA2P_E_ARG, "gemm: A2 and K2 must be given together");
  // the epilogue moves 32-byte sectors (256-bit global accesses)
  IA2P_REQUIRE((reinterpret_cast<uintptr_t>(out) & 31) == 0 && (ldo * (out_dtype == IA2P_F32 ? 4 : 2)) % 32 == 0, IA2P_E_ALIGN,
               "gemm: out must be 32-byte aligned with a 32-byte-multiple row pitch (ldo=%lld)", (long long)ldo);
  IA2P_REQUIRE(residual == nullptr || res_dtype != IA2P_F32 || ((reinterpret_cast<uintptr_t>(residual) & 31) == 0 && ldr % 8 == 0),
               IA2P_E_ALIGN, "gemm: fp32 residual must be 32-byte aligned with ldr%%8==0");
  const bool geglu = epilogue == IA2P_EPI_GEGLU;
  IA2P_REQUIRE(!geglu || (N % 64 == 0 && residual == nullptr && rowbias == nullptr && out_dtype == IA2P_BF16), IA2P_E_ARG, "gemm: GEGLU needs N%%64==0, bf16 output and no residual/rowbias");
  const bool act = epilogue == IA2P_EPI_GELU || epilogue == IA2P_EPI_QUICK_GELU;
  IA2P_REQUIRE(!act || (residual == nullptr && rowbias == nullptr && out_dtype == IA2P_BF16 && out_bf16 == nullptr &&
                        stats_out == nullptr && colstats == nullptr), IA2P_E_ARG,
               "gemm: GELU / quick-GELU epilogues need bf16 output and no residual, rowbias, LN statistics or column statistics");
  IA2P_REQUIRE(rowbias == nullptr || rows_per_batch > 0, IA2P_E_ARG, "gemm: rowbias needs rows_per_batch");
  IA2P_REQUIRE(M < (1ll << 31) && N < (1ll << 31), IA2P_E_SHAPE, "gemm: M/N too large");

  const int bn = pick_block_n(N, geglu, (M + 127) / 128, (int)((K1 + K2) / 64));
  TcMaps maps;
  TcParams p{};
  p.mc = pick_mc(bn, (M + 127) / 128, N, (int)((K1 + K2) / 64));
  uint32_t box[4] = {64, 128, 1, 1};
  slice_box(box, p.mc);
  {
    const uint64_t dims[4] = {(uint64_t)K1, (uint64_t)M, 1, 1};
    const uint64_t str[4] = {1, (uint64_t)lda, (uint64_t)lda * (uint64_t)M, (uint64_t)lda * (uint64_t)M};
    if (int e = make_map(&maps.a[0], A, 4, dims, str, box)) return e;
    maps.a[1] = maps.a[0]; maps.a[2] = maps.a[0]; maps.a[3] = maps.a[0];
  }
  p.taps[0] = TapEntry{0, 0, 0, (int16_t)(K1 / 64), 0};
  p.ntaps = 1;
  if (A2 != nullptr) {
    const uint64_t dims[4] = {(uint64_t)K2, (uint64_t)M, 1, 1};
    const uint64_t str[4] = {1, (uint64_t)lda2, (uint64_t)lda2 * (uint64_t)M, (uint64_t)lda2 * (uint64_t)M};
    if (int e = make_map(&maps.a[1], A2, 4, dims, str, box)) return e;
    p.taps[1] = TapEntry{1, 0, 0, (int16_t)(K2 / 64), (int32_t)K1};
    p.ntaps = 2;
  }
  if (int e = make_w_map(maps, W, N, K1 + K2, bn, (int)((M + 127) / 128))) return e;
  p.num_kb = (int)((K1 + K2) / 64);
  p.tw_log2 = 7; p.th_log2 = 0;
  p.tiles_x = (int)((M + 127) / 128); p.tiles_y = 1;
  p.m_tiles = p.tiles_x;
  p.Wo = (int)M; p.Ho = 1; p.B = 1;
  p.N = (int)N;
  p.rows_per_batch = rowbias ? (int)rows_per_batch : 1;
  p.bias = bias; p.rowbias = rowbias;
  p.residual = residual;
  p.out = out;
  p.ldo = ldo; p.ldr = ldr; p.geglu = geglu ? 1 : 0;
  p.out_f32 = out_dtype == IA2P_F32; p.res_f32 = res_dtype == IA2P_F32;
  p.out2 = static_cast<__nv_bfloat16*>(out_bf16); p.ldo2 = ldo2; p.stats_out = stats_out;
  IA2P_REQUIRE(colstats == nullptr || (out_dtype == IA2P_F32 && !geglu), IA2P_E_ARG, "gemm: column statistics need the fp32-output epilogue");
  p.colstats = colstats;
  p.ln_stats = ln_stats; p.ln_c1 = ln_c1; p.ln_parts = (int)ln_parts;
  p.ln_inv_n = 1.0f / (float)(K1 + K2); p.ln_eps = ln_eps;
  p.act = act ? epilogue : 0;
  IA2P_REQUIRE(!act || tma_epilogue_bf16(p), IA2P_E_ARG, "gemm: GELU / quick-GELU epilogues need the bf16 TMA-store epilogue");
  return dispatch_tc(maps, p, bn, static_cast<cudaStream_t>(stream));
}

static int conv3x3_impl(const void* x, int64_t B, int64_t H, int64_t W, int64_t Cin, int stride, bool pad_end,
                        const void* w, const void* sc_a, int64_t sc_ca, const void* sc_b, int64_t sc_cb,
                        void* out, int out_dtype, int64_t Cout, const float* bias, const float* rowbias,
                        const void* residual, int res_dtype, float* colstats, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE((out_dtype == IA2P_BF16 || out_dtype == IA2P_F32) && (residual == nullptr || res_dtype == IA2P_BF16 || res_dtype == IA2P_F32),
               IA2P_E_ARG, "conv3x3: out/residual dtype must be bf16 or f32");
  IA2P_REQUIRE(x && w && out && B > 0 && H > 0 && W > 0, IA2P_E_ARG, "conv3x3: null pointer or empty shape");
  IA2P_REQUIRE(stride == 1 || stride == 2, IA2P_E_ARG, "conv3x3: stride must be 1 or 2");
  IA2P_REQUIRE(Cin % 64 == 0 && sc_ca % 64 == 0 && sc_cb % 64 == 0, IA2P_E_SHAPE, "conv3x3: channel counts must be multiples of 64 (Cin=%lld)", (long long)Cin);
  IA2P_REQUIRE(Cout % 32 == 0, IA2P_E_SHAPE, "conv3x3: Cout=%lld must be a multiple of 32", (long long)Cout);
  IA2P_REQUIRE((sc_a == nullptr) == (sc_ca == 0) && (sc_b == nullptr) == (sc_cb == 0) && (sc_b == nullptr || sc_a != nullptr),
               IA2P_E_ARG, "conv3x3: inconsistent shortcut sources");
  IA2P_REQUIRE(stride == 1 || (sc_a == nullptr && H % 2 == 0 && W % 2 == 0), IA2P_E_ARG, "conv3x3: stride 2 needs even H,W and no shortcut");
  IA2P_REQUIRE((reinterpret_cast<uintptr_t>(out) & 31) == 0 && (residual == nullptr || (reinterpret_cast<uintptr_t>(residual) & 31) == 0),
               IA2P_E_ALIGN, "conv3x3: out/residual must be 32-byte aligned");
  const int64_t Ho = H / stride, Wo = W / stride;
  // tile: largest power-of-two divisors
  int TW = 1; while (TW < 128 && Wo % (TW * 2) == 0) TW *= 2;
  int TH = 1; while (TW * TH < 128 && Ho % (TH * 2) == 0) TH *= 2;
  const int TB = 128 / (TW * TH);
  const int64_t Ktot = 9 * Cin + sc_ca + sc_cb;
  const int bn = pick_block_n(Cout, false, (Wo / TW) * (Ho / TH) * ((B + TB - 1) / TB), (int)(Ktot / 64));

  TcMaps maps;
  TcParams p{};
  p.mc = pick_mc(bn, (Wo / TW) * (Ho / TH) * ((B + TB - 1) / TB), Cout, (int)(Ktot / 64));
  uint32_t box[4] = {64, (uint32_t)TW, (uint32_t)TH, (uint32_t)TB};
  slice_box(box, p.mc);
  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(x);
  int nt = 0;
  if (stride == 1) {
    const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)B};
    const uint64_t str[4] = {1, (uint64_t)Cin, (uint64_t)(W * Cin), (uint64_t)(H * W * Cin)};
    if (int e = make_map(&maps.a[0], xb, 4, dims, str, box)) return e;
    maps.a[1] = maps.a[0]; maps.a[2] = maps.a[0]; maps.a[3] = maps.a[0];
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx)
        p.taps[nt++] = TapEntry{0, (int16_t)(kx - 1), (int16_t)(ky - 1), (int16_t)(Cin / 64), (int32_t)((ky * 3 + kx) * Cin)};
    const void* srcs[2] = {sc_a, sc_b};
    const int64_t cs[2] = {sc_ca, sc_cb};
    int64_t koff = 9 * Cin;
    for (int s = 0; s < 2; ++s) {
      if (srcs[s] == nullptr) continue;
      const uint64_t d2[4] = {(uint64_t)cs[s], (uint64_t)W, (uint64_t)H, (uint64_t)B};
      const uint64_t s2[4] = {1, (uint64_t)cs[s], (uint64_t)(W * cs[s]), (uint64_t)(H * W * cs[s])};
      if (int e = make_map(&maps.a[1 + s], srcs[s], 4, d2, s2, box)) return e;
      p.taps[nt++] = TapEntry{(int16_t)(1 + s), 0, 0, (int16_t)(cs[s] / 64), (int32_t)koff};
      koff += cs[s];
    }
  } else {
    // x = 2*xo + px: one decimated view per parity (py, px).  pad 1 (UNet Downsample2D): input index 2*xo + k - 1, so tap k in
    // {0,1,2} reads parity (k==1 ? 0 : 1) at offset (k==0 ? -1 : 0).  pad_end (VAE encoder Downsample2D: padding 0 after
    // F.pad(0,1,0,1)): input index 2*xo + k, so tap k reads parity (k & 1) at offset (k==2 ? +1 : 0).
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)B};
        const uint64_t str[4] = {1, (uint64_t)(2 * Cin), (uint64_t)(2 * W * Cin), (uint64_t)(H * W * Cin)};
        if (int e = make_map(&maps.a[py * 2 + px], xb + (py * W + px) * Cin, 4, dims, str, box)) return e;
      }
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) {
        const int py = pad_end ? (ky & 1) : (ky == 1 ? 0 : 1), px = pad_end ? (kx & 1) : (kx == 1 ? 0 : 1);
        const int ox = pad_end ? (kx == 2 ? 1 : 0) : (kx == 0 ? -1 : 0), oy = pad_end ? (ky == 2 ? 1 : 0) : (ky == 0 ? -1 : 0);
        p.taps[nt++] = TapEntry{(int16_t)(py * 2 + px), (int16_t)ox, (int16_t)oy, (int16_t)(Cin / 64), (int32_t)((ky * 3 + kx) * Cin)};
      }
  }
  p.ntaps = nt;
  if (int e = make_w_map(maps, w, Cout, Ktot, bn, (int)((Wo / TW) * (Ho / TH) * ((B + TB - 1) / TB)))) return e;
  p.num_kb = (int)(Ktot / 64);
  p.tw_log2 = ilog2_exact(TW); p.th_log2 = ilog2_exact(TH);
  p.tiles_x = (int)(Wo / TW); p.tiles_y = (int)(Ho / TH);
  p.m_tiles = p.tiles_x * p.tiles_y * (int)((B + TB - 1) / TB);
  p.Wo = (int)Wo; p.Ho = (int)Ho; p.B = (int)B;
  p.N = (int)Cout;
  p.rows_per_batch = (int)(Ho * Wo);
  p.bias = bias; p.rowbias = rowbias;
  p.residual = residual;
  p.out = out;
  p.ldo = Cout; p.ldr = Cout; p.geglu = 0;
  p.out_f32 = out_dtype == IA2P_F32; p.res_f32 = res_dtype == IA2P_F32;
  IA2P_REQUIRE(colstats == nullptr || (p.out_f32 && tma_epilogue(p)), IA2P_E_ARG, "conv3x3: column statistics need the fp32-output epilogue");
  p.colstats = colstats;
  return dispatch_tc(maps, p, bn, static_cast<cudaStream_t>(stream));
}

extern "C" int ia2p_conv3x3_nhwc_bf16(const void* x, int64_t B, int64_t H, int64_t W, int64_t Cin, int stride,
                                      const void* w, const void* sc_a, int64_t sc_ca, const void* sc_b, int64_t sc_cb,
                                      void* out, int out_dtype, int64_t Cout, const float* bias, const float* rowbias,
                                      const void* residual, int res_dtype, float* colstats, void* stream) {
  return conv3x3_impl(x, B, H, W, Cin, stride, false, w, sc_a, sc_ca, sc_b, sc_cb, out, out_dtype, Cout, bias, rowbias, residual,
                      res_dtype, colstats, stream);
}

extern "C" int ia2p_conv3x3_s2_padend_nhwc_bf16(const void* x, int64_t B, int64_t H, int64_t W, int64_t Cin, const void* w,
                                                void* out, int out_dtype, int64_t Cout, const float* bias, void* stream) {
  return conv3x3_impl(x, B, H, W, Cin, 2, true, w, nullptr, 0, nullptr, 0, out, out_dtype, Cout, bias, nullptr, nullptr, IA2P_BF16,
                      nullptr, stream);
}

// Nearest-2x upsample folded into the following 3x3 conv ([3P] Upsample2D: F.interpolate(x, scale 2, "nearest") -> conv).  An output
// pixel of parity (py, px) only ever sees a 2x2 neighbourhood of the LOW-resolution map (up[i] = in[i >> 1]), so the conv
// splits into four 2x2 convs over the low-res input with pre-summed weights: 4/9 of the MACs, no upsampled tensor in HBM.
// w4: [4 parities (py*2+px)][Cout][4*Cin] bf16, tap order (row tap, col tap); out: [B, 2H, 2W, Cout] fp32 (TMA-store epilogue
// with a stride-2 output map per parity).
extern "C" int ia2p_conv_up2x_nhwc_bf16(const void* x, int64_t B, int64_t H, int64_t W, int64_t Cin, const void* w4, void* out,
                                        int64_t Cout, const float* bias, float* colstats, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x && w4 && out && B > 0 && H > 0 && W > 0, IA2P_E_ARG, "conv_up2x: null pointer or empty shape");
  IA2P_REQUIRE(Cin % 64 == 0 && Cout % 32 == 0, IA2P_E_SHAPE, "conv_up2x: Cin %% 64 == 0 and Cout %% 32 == 0 required");
  IA2P_REQUIRE((reinterpret_cast<uintptr_t>(out) & 31) == 0, IA2P_E_ALIGN, "conv_up2x: out must be 32-byte aligned");
  int TW = 1; while (TW < 128 && W % (TW * 2) == 0) TW *= 2;
  int TH = 1; while (TW * TH < 128 && H % (TH * 2) == 0) TH *= 2;
  const int TB = 128 / (TW * TH);
  const int64_t Ktot = 4 * Cin;
  const int bn = pick_block_n(Cout, false, (W / TW) * (H / TH) * ((B + TB - 1) / TB), (int)(Ktot / 64));
  const int mc = pick_mc(bn, (W / TW) * (H / TH) * ((B + TB - 1) / TB), Cout, (int)(Ktot / 64));
  uint32_t box[4] = {64, (uint32_t)TW, (uint32_t)TH, (uint32_t)TB};
  slice_box(box, mc);
  const __nv_bfloat16* xb = static_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* wb = static_cast<const __nv_bfloat16*>(w4);
  for (int par = 0; par < 4; ++par) {
    const int py = par >> 1, px = par & 1;
    TcMaps maps;
    TcParams p{};
    p.mc = mc;
    const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)W, (uint64_t)H, (uint64_t)B};
    const uint64_t str[4] = {1, (uint64_t)Cin, (uint64_t)(W * Cin), (uint64_t)(H * W * Cin)};
    if (int e = make_map(&maps.a[0], xb, 4, dims, str, box)) return e;
    maps.a[1] = maps.a[0]; maps.a[2] = maps.a[0]; maps.a[3] = maps.a[0];
    int nt = 0;
    for (int i = 0; i < 2; ++i)
      for (int j = 0; j < 2; ++j)
        p.taps[nt++] = TapEntry{0, (int16_t)(px == 0 ? j - 1 : j), (int16_t)(py == 0 ? i - 1 : i), (int16_t)(Cin / 64),
                                (int32_t)((i * 2 + j) * Cin)};
    p.ntaps = nt;
    p.num_kb = (int)(Ktot / 64);
    p.tw_log2 = ilog2_exact(TW); p.th_log2 = ilog2_exact(TH);
    p.tiles_x = (int)(W / TW); p.tiles_y = (int)(H / TH);
    p.m_tiles = p.tiles_x * p.tiles_y * (int)((B + TB - 1) / TB);
    if (int e = make_w_map(maps, wb + (size_t)par * Cout * Ktot, Cout, Ktot, bn, p.m_tiles)) return e;
    p.Wo = (int)W; p.Ho = (int)H; p.B = (int)B;
    p.N = (int)Cout;
    p.rows_per_batch = (int)(H * W);
    p.bias = bias;
    p.out = static_cast<float*>(out) + ((int64_t)py * 2 * W + px) * Cout;
    p.ldo = Cout; p.ldr = Cout;
    p.ost_x = 2 * Cout; p.ost_y = 4 * W * Cout; p.ost_b = 4 * H * W * Cout;
    p.out_f32 = 1; p.res_f32 = 0; p.geglu = 0;
    p.colstats = colstats == nullptr ? nullptr : colstats + (size_t)par * p.m_tiles * Cout * 2;   // one segment per output parity
    IA2P_REQUIRE(tma_epilogue(p), IA2P_E_ARG, "conv_up2x needs the TMA-store epilogue (IA2P_GEMM_EPI=0 is set)");
    if (int e = dispatch_tc(maps, p, bn, static_cast<cudaStream_t>(stream))) return e;
  }
  return 0;
}

// Row tiles the conv kernels cut a [B, Ho, Wo] output pixel grid into, i.e. the first dimension of a `colstats` buffer -- or 0 when
// a tile would span several images (Ho * Wo has too few factors of two for a 128-pixel tile), in which case the column
// statistics cannot serve a per-image GroupNorm and must not be requested.  Plain GEMMs use ceil(M / 128) row tiles.
extern "C" int64_t ia2p_conv_colstats_tiles(int64_t B, int64_t Ho, int64_t Wo) {
  if (B <= 0 || Ho <= 0 || Wo <= 0) return 0;
  int TW = 1; while (TW < 128 && Wo % (TW * 2) == 0) TW *= 2;
  int TH = 1; while (TW * TH < 128 && Ho % (TH * 2) == 0) TH *= 2;
  if (TW * TH != 128) return 0;
  return (Wo / TW) * (Ho / TH) * B;
}
