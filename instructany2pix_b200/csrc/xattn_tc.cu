// tcgen05 / TMEM / TMA decoupled cross-attention for sm_100a, head_dim 64 (IPAttnProcessor2_0.__call__,
// diffusion/ip_adapter/attention_processor.py:371-397: softmax(Q Kt^T) Vt + scale * softmax(Q Ki^T) Vi in ONE pass).
//
// All keys of a (batch, head) fit one MMA: text keys padded to T1 (multiple of 16) followed by the IP keys padded to T2 (0 | 16);
// TK = T1 + T2 <= 128.  Work item = 128 query rows of one (batch, head); a persistent grid of two CTAs per SM strides over the
// items.  CTA = 6 warps: w0 TMA producer (per item: Q tile + the K / V rows of its head, 2-stage ring; K/V come from L2),
// w1 tcgen05.mma issuer, w2..w5 softmax + epilogue (one query row per thread):
//   MMA1: S(TMEM, TK cols fp32) = Q K^T                                     [M128 N=TK K64]   4 instructions
//   softmax warps: the whole S row (<= 128 fp32) goes to registers in one round of TMEM loads (S is free for the next MMA1 at
//       once), then the maxima of the two branches, then p = 2^(s*scale - m): text p's are packed unnormalised while l_text accumulates, the <= 16 IP p's wait
//       in registers until l_text is known and are packed times scale * l_text / l_ip, so that ONE common 1 / l_text in the
//       epilogue finishes both branches; P -> TMEM as bf16 pairs (the A operand of MMA2)
//   MMA2: O(TMEM, 64 cols) = P V                                             [M128 N64 K=TK]   TK / 16 instructions
//   epilogue: O / l_text -> bf16 -> swizzled staging tile in shared memory -> ONE TMA store per item (thread-per-row register
//       stores move a 32-byte sector per lane and instruction: ~0.7 us per 16 KB tile, more than the two MMAs together).
// MMA1 of item i+1 is issued before MMA2 of item i, and the second CTA on the SM fills the tensor pipe while this one does its
// softmax.  Cost model (tools/mmabench.cu: >= 94 cycles per tcgen05.mma): (4 + TK/16) x ~94 cycles per item = 940 at TK 96,
// next to 768 cycles of exponentials; the warp-level mma.sync kernel this replaces (attn.cu) ran at 23 % of the HBM roofline.
#include <cuda.h>

#include <mutex>

#include "common.cuh"
#include "tensormap.cuh"

namespace ia2p {

struct alignas(64) XaMaps {
  CUtensorMap q, kt, vt, ki, vi, o;   // 3-D {heads*64, tokens, batch}; boxes {64, 128 | T1 | 16, 1}, SWIZZLE_128B
};

constexpr int kXaQ = 128 * 128;    // bytes of a Q tile: 128 rows x 64 bf16

// ROWS = true: batch row b weighs its IP branch by ip_rows[b] (one request per row) instead of ip_scale
template <int T1, int T2, bool ROWS>
__global__ void __launch_bounds__(192, 2)
xattn_tc_kernel(const __grid_constant__ XaMaps maps, int n_q, int n_text, int n_ip,
                int heads, int n_items, float ip_scale, float scale_log2, const float* __restrict__ ip_rows) {
  constexpr int TK = T1 + T2;
  constexpr int KV = TK * 128;                          // bytes of the K (or V) rows of one head
  constexpr int STAGE = kXaQ + 2 * KV;
  constexpr int NCH = (TK + 31) / 32;                   // 32-column chunks of S
  static_assert(T1 % 16 == 0 && (T2 == 0 || T2 == 16) && TK <= 128, "key padding");
  static_assert(!ROWS || T2 > 0, "per-row IP scales need IP keys");
  pdl_launch_dependents();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t tiles = (raw + 128u + 1023u) & ~1023u;      // >= 128 B of barriers in front
  const uint32_t bars = raw;
  const uint32_t full = bars, empty = bars + 16, s_full = bars + 32, s_empty = bars + 40, p_full = bars + 48, o_full = bars + 56,
                 tmem_slot = bars + 64;
  const int warp = warp_idx_uniform(), lane = threadIdx.x & 31;
  const int n_qtiles = (n_q + 127) >> 7;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&maps.q); tma_prefetch_desc(&maps.kt); tma_prefetch_desc(&maps.vt); tma_prefetch_desc(&maps.o);
    if (T2 > 0) { tma_prefetch_desc(&maps.ki); tma_prefetch_desc(&maps.vi); }
    for (int s = 0; s < 2; ++s) { mbar_init(full + 8 * s, 1); mbar_init(empty + 8 * s, 1); }
    mbar_init(s_full, 1); mbar_init(s_empty, 4); mbar_init(p_full, 4); mbar_init(o_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, 256); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(smem_raw + (tmem_slot - raw));
  const uint32_t tS = tmem_base, tO = tmem_base + 128, tP = tmem_base + 192;   // S <= 128 | O 64 | P <= 64 (bf16 pairs) columns
  pdl_wait();

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    int it = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x, ++it) {
      const int st = it & 1;
      const int qt = w % n_qtiles, bh = w / n_qtiles, h = bh % heads, b = bh / heads;
      mbar_wait(empty + 8 * st, (uint32_t)(((it >> 1) & 1) ^ 1));
      if (elect_one()) {
        const uint32_t sQ = tiles + st * STAGE, sK = sQ + kXaQ, sV = sK + KV;
        mbar_arrive_expect_tx(full + 8 * st, STAGE);
        tma_load_3d(sQ, &maps.q, full + 8 * st, h * 64, qt * 128, b);
        tma_load_3d(sK, &maps.kt, full + 8 * st, h * 64, 0, b);            // rows >= n_text: zero-filled
        tma_load_3d(sV, &maps.vt, full + 8 * st, h * 64, 0, b);
        if (T2 > 0) {
          tma_load_3d(sK + T1 * 128, &maps.ki, full + 8 * st, h * 64, 0, b);
          tma_load_3d(sV + T1 * 128, &maps.vi, full + 8 * st, h * 64, 0, b);
        }
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc_qk = umma_idesc_bf16(128, TK, 0);
    constexpr uint32_t idesc_pv = umma_idesc_bf16(128, 64, 1);
    const int n_mine = (n_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    auto issue_qk = [&](int it) {
      const int st = it & 1;
      mbar_wait(full + 8 * st, (uint32_t)((it >> 1) & 1));
      if (it > 0) mbar_wait(s_empty, (uint32_t)((it - 1) & 1));              // softmax finished reading S of the previous item
      tc_fence_after();
      if (elect_one()) {
        const uint32_t sQ = tiles + st * STAGE;
        const uint64_t da = umma_desc_sw128(sQ), db = umma_desc_sw128(sQ + kXaQ);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(tS, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc_qk, (uint32_t)(k != 0));
        umma_commit(s_full);
      }
      __syncwarp();
    };
    if (n_mine > 0) issue_qk(0);
    for (int it = 0; it < n_mine; ++it) {
      if (it + 1 < n_mine) issue_qk(it + 1);                                  // overlaps the softmax of item it
      const int st = it & 1;
      mbar_wait(p_full, (uint32_t)(it & 1));                                  // P written; O of the previous item read out
      tc_fence_after();
      if (elect_one()) {
        const uint32_t sV = tiles + st * STAGE + kXaQ + KV;
#pragma unroll
        for (int ks = 0; ks < TK / 16; ++ks)
          umma_bf16_ts(tO, tP + (uint32_t)(ks * 8), umma_desc_sw128_mn(sV + ks * 2048, KV), idesc_pv, (uint32_t)(ks != 0));
        umma_commit(empty + 8 * st);                                          // Q, K, V of this stage are consumed
        umma_commit(o_full);
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------ softmax + epilogue: one query row per thread
    const int qd = warp & 3;
    const int row = qd * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(qd * 32) << 16;
    const bool elected = (warp == 2) && lane == 0;
    const uint32_t sO = tiles + 2 * STAGE;                                     // 16 KB output staging tile
    int it = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x, ++it) {
      const int qt = w % n_qtiles, bh = w / n_qtiles, h = bh % heads, b = bh / heads;
      mbar_wait(s_full, (uint32_t)(it & 1));
      tc_fence_after();
      // the whole S row (TK <= 128 columns) goes to registers in ONE round of TMEM loads (all in flight together), which also
      // frees S for MMA1 of the next item before any math starts; v[] dies pair by pair as the packed P is produced
      uint32_t v[NCH][32];
#pragma unroll
      for (int c = 0; c < NCH; ++c) tmem_ld_32x32(tS + lane_sel + (uint32_t)(c * 32), v[c]);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_empty);                                    // S may be overwritten by MMA1 of the next item
      // row maxima of the two branches (raw scores; scale > 0)
      float mt = -INFINITY, mi = -INFINITY;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          const int j = c * 32 + i;
          if (j < T1) { if (j < n_text) mt = fmaxf(mt, __uint_as_float(v[c][i])); }
          else if (j < TK) { if (j - T1 < n_ip) mi = fmaxf(mi, __uint_as_float(v[c][i])); }
        }
      }
      const float nmt = -mt * scale_log2, nmi = (mi == -INFINITY) ? 0.f : -mi * scale_log2;
      // exponentials; text pairs are packed at once, the IP values wait for l_text
      uint32_t pk[64];
      float pip[T2 > 0 ? T2 : 1];
      float lt = 0.f, li = 0.f;
#pragma unroll
      for (int i = TK / 2; i < 64; ++i) pk[i] = 0u;
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
          const int j = c * 32 + i;
          if (j < T1) {
            const float p0 = (j < n_text) ? ex2_approx(fmaf(__uint_as_float(v[c][i]), scale_log2, nmt)) : 0.f;
            const float p1 = (j + 1 < n_text) ? ex2_approx(fmaf(__uint_as_float(v[c][i + 1]), scale_log2, nmt)) : 0.f;
            lt += p0 + p1;
            pk[j >> 1] = pack_bf16x2(p0, p1);
          } else if (j < TK) {
            const float p0 = (j - T1 < n_ip) ? ex2_approx(fmaf(__uint_as_float(v[c][i]), scale_log2, nmi)) : 0.f;
            const float p1 = (j + 1 - T1 < n_ip) ? ex2_approx(fmaf(__uint_as_float(v[c][i + 1]), scale_log2, nmi)) : 0.f;
            li += p0 + p1;
            pip[(j - T1) % (T2 > 0 ? T2 : 1)] = p0;
            pip[(j + 1 - T1) % (T2 > 0 ? T2 : 1)] = p1;
          }
        }
      }
      if (T2 > 0) {
        const float s = ROWS ? __ldg(ip_rows + b) : ip_scale;
        const float f = (li > 0.f) ? s * lt / li : 0.f;
#pragma unroll
        for (int i = 0; i < T2; i += 2) pk[(T1 + i) >> 1] = pack_bf16x2(pip[i] * f, pip[i + 1] * f);
      }
      // P / O are free: MMA2 of the previous item completed (o_full waited below in the previous iteration) and its O was read
      {
        uint32_t (&plo)[32] = *reinterpret_cast<uint32_t (*)[32]>(&pk[0]);
        tmem_st_32x32(tP + lane_sel, plo);
        if (TK > 64) {
          uint32_t (&phi)[32] = *reinterpret_cast<uint32_t (*)[32]>(&pk[32]);
          tmem_st_32x32(tP + lane_sel + 32u, phi);
        }
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
      // epilogue: O / l_text -> bf16 -> staging tile (SWIZZLE_128B: 16-byte chunk ^= row % 8) -> one TMA store (rows >= n_q clipped)
      mbar_wait(o_full, (uint32_t)(it & 1));
      tc_fence_after();
      const float inv = 1.f / lt;
      if (elected) bulk_wait_read_all();                                       // the previous item's store has left the staging tile
      named_bar_sync(1, 128);
      {
        uint32_t o[2][32];
        tmem_ld_32x32(tO + lane_sel, o[0]);
        tmem_ld_32x32(tO + lane_sel + 32u, o[1]);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
          for (int i = 0; i < 4; ++i)
            sts128u(sO + (uint32_t)row * 128u + ((uint32_t)((c * 4 + i) ^ (row & 7)) << 4),
                    pack_bf16x2(__uint_as_float(o[c][8 * i + 0]) * inv, __uint_as_float(o[c][8 * i + 1]) * inv),
                    pack_bf16x2(__uint_as_float(o[c][8 * i + 2]) * inv, __uint_as_float(o[c][8 * i + 3]) * inv),
                    pack_bf16x2(__uint_as_float(o[c][8 * i + 4]) * inv, __uint_as_float(o[c][8 * i + 5]) * inv),
                    pack_bf16x2(__uint_as_float(o[c][8 * i + 6]) * inv, __uint_as_float(o[c][8 * i + 7]) * inv));
      }
      tc_fence_before();
      fence_proxy_async();
      named_bar_sync(1, 128);
      if (elected) {
        tma_store_3d(&maps.o, sO, h * 64, qt * 128, b);
        bulk_commit_group();
      }
    }
    if (elected) bulk_wait_read_all();                                         // staging memory must outlive the last store's read
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

template <int T1, int T2, bool ROWS>
static int launch_xa(const void* q, int64_t ldq, const void* kt, const void* vt, int64_t ldkv, int n_text, const void* ki,
                     const void* vi, int64_t ldkv_ip, int n_ip, float ip_scale, const float* ip_rows, void* out, int64_t ldo,
                     int64_t batch, int64_t n_q, int heads, float scale, cudaStream_t st) {
  constexpr int TK = T1 + T2;
  constexpr int smem = 2 * (kXaQ + 2 * TK * 128) + kXaQ + 1024 + 128;
  XaMaps maps;
  if (int e = make_map_3d_bf16(&maps.q, q, heads * 64, ldq, n_q, batch, 128, "cross_attn")) return e;
  if (int e = make_map_3d_bf16(&maps.kt, kt, heads * 64, ldkv, n_text, batch, T1, "cross_attn")) return e;
  if (int e = make_map_3d_bf16(&maps.vt, vt, heads * 64, ldkv, n_text, batch, T1, "cross_attn")) return e;
  if (int e = make_map_3d_bf16(&maps.o, out, heads * 64, ldo, n_q, batch, 128, "cross_attn")) return e;
  maps.ki = maps.kt;
  maps.vi = maps.vt;
  if (T2 > 0) {
    if (int e = make_map_3d_bf16(&maps.ki, ki, heads * 64, ldkv_ip, n_ip, batch, T2, "cross_attn")) return e;
    if (int e = make_map_3d_bf16(&maps.vi, vi, heads * 64, ldkv_ip, n_ip, batch, T2, "cross_attn")) return e;
  }
  IA2P_ONCE_PER_DEVICE(
      IA2P_CUDA(cudaFuncSetAttribute(xattn_tc_kernel<T1, T2, ROWS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      IA2P_CUDA(cudaFuncSetAttribute(xattn_tc_kernel<T1, T2, ROWS>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)));
  const long long n_items = (long long)((n_q + 127) / 128) * heads * batch;
  IA2P_REQUIRE(n_items < (1ll << 31), IA2P_E_SHAPE, "cross_attn: too many work items");
  const long long resident = 2LL * sm_count();
  const dim3 grid((unsigned)(n_items < resident ? n_items : resident));
  launch_pdl(xattn_tc_kernel<T1, T2, ROWS>, dim3(grid), dim3(192), smem, st, maps, (int)n_q, n_text, n_ip, heads, (int)n_items,
             ip_scale, scale * 1.4426950408889634f, ip_rows);
  IA2P_LAUNCH_CHECK();
  return 0;
}

// -> 0 launched | < 0 / > 0 error; *handled = false: shape outside this kernel (caller falls back to the mma.sync kernel).
// ip_rows (nullable, used only when n_ip > 0): per-batch-row IP scales in device memory instead of ip_scale.
int launch_xattn_tc(const void* q, int64_t ldq, const void* kt, const void* vt, int64_t ldkv, int n_text, const void* ki,
                    const void* vi, int64_t ldkv_ip, int n_ip, float ip_scale, const float* ip_rows, void* out, int64_t ldo,
                    int64_t batch, int64_t n_q, int heads, float scale, cudaStream_t st, bool* handled) {
  *handled = true;
  const int t1 = n_text <= 80 ? 80 : (n_text <= 96 ? 96 : (n_text <= 112 ? 112 : 128));
#define IA2P_XA(T1_, T2_, ROWS_) \
  return launch_xa<T1_, T2_, ROWS_>(q, ldq, kt, vt, ldkv, n_text, ki, vi, ldkv_ip, n_ip, ip_scale, ip_rows, out, ldo, batch, n_q, heads, \
                                    scale, st)
  if (n_ip > 0 && ip_rows != nullptr) {
    if (t1 == 80) IA2P_XA(80, 16, true);
    if (t1 == 96) IA2P_XA(96, 16, true);
    if (t1 == 112) IA2P_XA(112, 16, true);
  } else if (n_ip > 0) {
    if (t1 == 80) IA2P_XA(80, 16, false);
    if (t1 == 96) IA2P_XA(96, 16, false);
    if (t1 == 112) IA2P_XA(112, 16, false);
  } else {
    if (t1 == 80) IA2P_XA(80, 0, false);
    if (t1 == 96) IA2P_XA(96, 0, false);
    if (t1 == 112) IA2P_XA(112, 0, false);
    IA2P_XA(128, 0, false);
  }
#undef IA2P_XA
  *handled = false;                       // 112 < n_text <= 128 together with IP keys: more than 128 key columns
  return 0;
}

}  // namespace ia2p
