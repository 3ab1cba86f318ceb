// Attention kernels, head_dim 64, bf16 in / fp32 softmax / bf16 out.
//   * flash self-attention (online softmax over 64-key tiles, cp.async double buffering)
//   * decoupled cross-attention: text branch + IP image-token branch, two independent softmaxes, ONE P.V pass
//     and one output write (replaces two SDPA calls + add; attention_processor.py:371-397)
// Round-1 implementation uses warp-level mma.sync m16n8k16 tiles (legacy tensor path, HMMA); the tcgen05/TMEM
// version is the planned replacement for the self-attention kernel (DESIGN.md, "next").
#include <cstdlib>

#include "common.cuh"

namespace ia2p {

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// tile of rows x 64 bf16 (128 B per row), 16-byte chunks XOR-swizzled by (row & 7)
__device__ __forceinline__ uint32_t tile_off(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }

// copy `rows` rows (64 bf16 each) global -> swizzled smem tile; rows >= valid_rows are zero-filled
__device__ __forceinline__ void load_tile(uint32_t smem, const __nv_bfloat16* g, long long ld, int rows, int valid_rows,
                                          int tid, int nthreads) {
  for (int id = tid; id < rows * 8; id += nthreads) {
    const int r = id >> 3, ch = id & 7;
    const bool ok = r < valid_rows;
    cp_async16(smem + tile_off(r, ch), g + (ok ? (long long)r * ld + ch * 8 : 0), ok ? 16 : 0);
  }
}

constexpr float kLog2e = 1.4426950408889634f;

// ================================================================ flash self-attention
// grid (ceil(N/128), heads, batch), 256 threads: warp w owns query rows [16w, 16w+16) of the 128-row tile.
__global__ void __launch_bounds__(256)
flash_self_attn_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                       const __nv_bfloat16* __restrict__ v, long long ld, __nv_bfloat16* __restrict__ out, long long ldo,
                       int n_tokens, float scale_log2) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sQ = smem_u32(smem);            // 128 x 64
  const uint32_t sK = sQ + 128 * 128;            // 2 x (64 x 64)
  const uint32_t sV = sK + 2 * 64 * 128;         // 2 x (64 x 64)
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int q0 = blockIdx.x * 128;
  const int h = blockIdx.y;
  const long long tok0 = (long long)blockIdx.z * n_tokens;
  const __nv_bfloat16* qg = q + (tok0 + q0) * ld + h * 64;
  const __nv_bfloat16* kg = k + tok0 * ld + h * 64;
  const __nv_bfloat16* vg = v + tok0 * ld + h * 64;

  const int n_kv_tiles = (n_tokens + 63) / 64;
  load_tile(sQ, qg, ld, 128, min(128, n_tokens - q0), tid, 256);
  load_tile(sK, kg, ld, 64, min(64, n_tokens), tid, 256);
  load_tile(sV, vg, ld, 64, min(64, n_tokens), tid, 256);
  cp_async_commit();

  uint32_t qf[4][4];
  float o[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;

  for (int j = 0; j < n_kv_tiles; ++j) {
    const int buf = j & 1;
    cp_async_wait<0>();
    __syncthreads();
    if (j + 1 < n_kv_tiles) {   // prefetch next K/V tile into the other buffer (its previous readers passed the barrier)
      const int kv0 = (j + 1) * 64;
      load_tile(sK + (buf ^ 1) * 64 * 128, kg + (long long)kv0 * ld, ld, 64, min(64, n_tokens - kv0), tid, 256);
      load_tile(sV + (buf ^ 1) * 64 * 128, vg + (long long)kv0 * ld, ld, 64, min(64, n_tokens - kv0), tid, 256);
      cp_async_commit();
    }
    if (j == 0) {
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const int r = warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
        ldsm_x4(sQ + tile_off(r, kk * 2 + (lane >> 4)), qf[kk][0], qf[kk][1], qf[kk][2], qf[kk][3]);
      }
    }
    const uint32_t kb = sK + buf * 64 * 128, vb = sV + buf * 64 * 128;
    float s[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
      for (int kp = 0; kp < 2; ++kp) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4(kb + tile_off(nt * 8 + (lane & 7), kp * 4 + (lane >> 3)), b0, b1, b2, b3);
        mma_bf16(s[nt], qf[kp * 2], b0, b1);
        mma_bf16(s[nt], qf[kp * 2 + 1], b2, b3);
      }
    }
    // online softmax (rows g and g+8 of this warp's 16)
    const int key_base = j * 64 + 2 * t;
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const bool ok = key_base + nt * 8 + e < n_tokens;
        s[nt][e] = ok ? s[nt][e] * scale_log2 : -INFINITY;
        s[nt][2 + e] = ok ? s[nt][2 + e] * scale_log2 : -INFINITY;
        mx0 = fmaxf(mx0, s[nt][e]);
        mx1 = fmaxf(mx1, s[nt][2 + e]);
      }
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
    const float a0 = exp2f(m0 - mn0), a1 = exp2f(m1 - mn1);
    m0 = mn0; m1 = mn1;
    float rs0 = 0.f, rs1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      s[nt][0] = exp2f(s[nt][0] - mn0); s[nt][1] = exp2f(s[nt][1] - mn0);
      s[nt][2] = exp2f(s[nt][2] - mn1); s[nt][3] = exp2f(s[nt][3] - mn1);
      rs0 += s[nt][0] + s[nt][1];
      rs1 += s[nt][2] + s[nt][3];
    }
    l0 = l0 * a0 + rs0;
    l1 = l1 * a1 + rs1;
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) { o[dt][0] *= a0; o[dt][1] *= a0; o[dt][2] *= a1; o[dt][3] *= a1; }
    // O += P V
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      uint32_t pa[4];
      pa[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
      pa[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
      pa[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      pa[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
      for (int dp = 0; dp < 4; ++dp) {
        uint32_t b0, b1, b2, b3;
        const int r = kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
        ldsm_x4_t(vb + tile_off(r, dp * 2 + (lane >> 4)), b0, b1, b2, b3);
        mma_bf16(o[2 * dp], pa, b0, b1);
        mma_bf16(o[2 * dp + 1], pa, b2, b3);
      }
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.f / l0, i1 = 1.f / l1;
  // stage the warp's 16x64 tile through (its own rows of) the Q buffer for 16-byte coalesced stores
  __syncwarp();
  uint8_t* sq = smem;
#pragma unroll
  for (int dt = 0; dt < 8; ++dt) {
    const int r0 = warp * 16 + g, r1 = r0 + 8;
    *reinterpret_cast<uint32_t*>(sq + tile_off(r0, dt) + t * 4) = pack_bf16x2(o[dt][0] * i0, o[dt][1] * i0);
    *reinterpret_cast<uint32_t*>(sq + tile_off(r1, dt) + t * 4) = pack_bf16x2(o[dt][2] * i1, o[dt][3] * i1);
  }
  __syncwarp();
  __nv_bfloat16* og = out + (tok0 + q0) * ldo + h * 64;
  for (int id = lane; id < 16 * 8; id += 32) {
    const int r = warp * 16 + (id >> 3), ch = id & 7;
    if (q0 + r < n_tokens)
      *reinterpret_cast<uint4*>(og + (long long)r * ldo + ch * 8) = *reinterpret_cast<const uint4*>(sq + tile_off(r, ch));
  }
}

// ================================================================ decoupled cross-attention
// All keys resident in smem: text keys padded to T1 (multiple of 16), IP keys padded to T2 (0 or 16).
// ip_rows (nullable): per-batch-row IP scales in device memory, used instead of ip_scale.
template <int T1, int T2>
__global__ void __launch_bounds__(256, (T1 <= 96) ? 3 : 1)
cross_attn_kernel(const __nv_bfloat16* __restrict__ q, long long ldq, const __nv_bfloat16* __restrict__ kt,
                  const __nv_bfloat16* __restrict__ vt, long long ldkv, int n_text, const __nv_bfloat16* __restrict__ ki,
                  const __nv_bfloat16* __restrict__ vi, long long ldkv_ip, int n_ip, float ip_scale,
                  const float* __restrict__ ip_rows, __nv_bfloat16* __restrict__ out, long long ldo, int n_q, float scale_log2) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  constexpr int TK = T1 + T2;
  constexpr int NT = TK / 8, NT1 = T1 / 8;
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sQ0 = smem_u32(smem);       // 2 x (128 x 64): double-buffered Q tiles
  const uint32_t sK = sQ0 + 2 * 128 * 128;   // TK x 64
  const uint32_t sV = sK + TK * 128;         // TK x 64
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int h = blockIdx.y;
  const long long b = blockIdx.z;
  const int n_qtiles = (n_q + 127) >> 7;
  const float ips = ip_rows != nullptr ? __ldg(ip_rows + b) : ip_scale;
  // K/V of this (batch, head) are loaded ONCE per CTA; the CTA then walks its query tiles with the next Q tile in flight
  load_tile(sK, kt + b * n_text * ldkv + h * 64, ldkv, T1, n_text, tid, 256);
  load_tile(sV, vt + b * n_text * ldkv + h * 64, ldkv, T1, n_text, tid, 256);
  if (T2 > 0) {
    load_tile(sK + T1 * 128, ki + b * n_ip * ldkv_ip + h * 64, ldkv_ip, T2, n_ip, tid, 256);
    load_tile(sV + T1 * 128, vi + b * n_ip * ldkv_ip + h * 64, ldkv_ip, T2, n_ip, tid, 256);
  }
  {
    const int q0 = blockIdx.x * 128;
    load_tile(sQ0, q + (b * n_q + q0) * ldq + h * 64, ldq, 128, min(128, n_q - q0), tid, 256);
  }
  cp_async_commit();

  int it = 0;
  for (int qt = blockIdx.x; qt < n_qtiles; qt += gridDim.x, ++it) {
    const int q0 = qt * 128;
    const uint32_t sQ = sQ0 + (it & 1) * 128 * 128;
    const int qn = qt + gridDim.x;
    if (qn < n_qtiles) {                      // prefetch the next Q tile into the other buffer
      load_tile(sQ0 + ((it + 1) & 1) * 128 * 128, q + (b * n_q + qn * 128) * ldq + h * 64, ldq, 128, min(128, n_q - qn * 128), tid, 256);
      cp_async_commit();
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();

    uint32_t qf[4][4];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const int r = warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
      ldsm_x4(sQ + tile_off(r, kk * 2 + (lane >> 4)), qf[kk][0], qf[kk][1], qf[kk][2], qf[kk][3]);
    }
    float s[NT][4];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
      for (int kp = 0; kp < 2; ++kp) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4(sK + tile_off(nt * 8 + (lane & 7), kp * 4 + (lane >> 3)), b0, b1, b2, b3);
        mma_bf16(s[nt], qf[kp * 2], b0, b1);
        mma_bf16(s[nt], qf[kp * 2 + 1], b2, b3);
      }
    }
    // two independent softmaxes: text keys [0, n_text) and IP keys [T1, T1 + n_ip)
    float mx[2][2] = {{-INFINITY, -INFINITY}, {-INFINITY, -INFINITY}};
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int br = nt < NT1 ? 0 : 1;
      const int lim = br == 0 ? n_text : n_ip;
      const int kidx = (br == 0 ? nt * 8 : nt * 8 - T1) + 2 * t;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const bool ok = kidx + e < lim;
        s[nt][e] = ok ? s[nt][e] * scale_log2 : -INFINITY;
        s[nt][2 + e] = ok ? s[nt][2 + e] * scale_log2 : -INFINITY;
        mx[br][0] = fmaxf(mx[br][0], s[nt][e]);
        mx[br][1] = fmaxf(mx[br][1], s[nt][2 + e]);
      }
    }
    float sum[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
#pragma unroll
    for (int br = 0; br < 2; ++br)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        mx[br][r] = fmaxf(mx[br][r], __shfl_xor_sync(0xffffffffu, mx[br][r], 1));
        mx[br][r] = fmaxf(mx[br][r], __shfl_xor_sync(0xffffffffu, mx[br][r], 2));
        if (mx[br][r] == -INFINITY) mx[br][r] = 0.f;   // empty branch (n_ip == 0): exp2(-inf - 0) = 0
      }
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int br = nt < NT1 ? 0 : 1;
      s[nt][0] = ex2_approx(s[nt][0] - mx[br][0]); s[nt][1] = ex2_approx(s[nt][1] - mx[br][0]);
      s[nt][2] = ex2_approx(s[nt][2] - mx[br][1]); s[nt][3] = ex2_approx(s[nt][3] - mx[br][1]);
      sum[br][0] += s[nt][0] + s[nt][1];
      sum[br][1] += s[nt][2] + s[nt][3];
    }
    float w[2][2];
#pragma unroll
    for (int br = 0; br < 2; ++br)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        sum[br][r] += __shfl_xor_sync(0xffffffffu, sum[br][r], 1);
        sum[br][r] += __shfl_xor_sync(0xffffffffu, sum[br][r], 2);
        const float inv = sum[br][r] > 0.f ? 1.f / sum[br][r] : 0.f;
        w[br][r] = br == 0 ? inv : inv * ips;
      }
    float o[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < TK / 16; ++kk) {
      const int br = (2 * kk) < NT1 ? 0 : 1;      // T1 is a multiple of 16: a 16-key step never straddles branches
      uint32_t pa[4];
      pa[0] = pack_bf16x2(s[2 * kk][0] * w[br][0], s[2 * kk][1] * w[br][0]);
      pa[1] = pack_bf16x2(s[2 * kk][2] * w[br][1], s[2 * kk][3] * w[br][1]);
      pa[2] = pack_bf16x2(s[2 * kk + 1][0] * w[br][0], s[2 * kk + 1][1] * w[br][0]);
      pa[3] = pack_bf16x2(s[2 * kk + 1][2] * w[br][1], s[2 * kk + 1][3] * w[br][1]);
#pragma unroll
      for (int dp = 0; dp < 4; ++dp) {
        uint32_t b0, b1, b2, b3;
        const int r = kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
        ldsm_x4_t(sV + tile_off(r, dp * 2 + (lane >> 4)), b0, b1, b2, b3);
        mma_bf16(o[2 * dp], pa, b0, b1);
        mma_bf16(o[2 * dp + 1], pa, b2, b3);
      }
    }
    // stage this warp's 16 x 64 tile through its own rows of the (consumed) Q buffer for 16-byte coalesced stores
    __syncwarp();
    uint8_t* sq = smem + (it & 1) * 128 * 128;
#pragma unroll
    for (int dt = 0; dt < 8; ++dt) {
      const int r0 = warp * 16 + g, r1 = r0 + 8;
      *reinterpret_cast<uint32_t*>(sq + tile_off(r0, dt) + t * 4) = pack_bf16x2(o[dt][0], o[dt][1]);
      *reinterpret_cast<uint32_t*>(sq + tile_off(r1, dt) + t * 4) = pack_bf16x2(o[dt][2], o[dt][3]);
    }
    __syncwarp();
    __nv_bfloat16* og = out + (b * n_q + q0) * ldo + h * 64;
    for (int id = lane; id < 16 * 8; id += 32) {
      const int r = warp * 16 + (id >> 3), ch = id & 7;
      if (q0 + r < n_q)
        *reinterpret_cast<uint4*>(og + (long long)r * ldo + ch * 8) = *reinterpret_cast<const uint4*>(sq + tile_off(r, ch));
    }
    __syncthreads();      // buffer (it & 1) is refilled by the prefetch issued at the top of the next iteration
  }
}

template <int T1, int T2>
static int launch_cross(const void* q, int64_t ldq, const void* kt, const void* vt, int64_t ldkv, int n_text, const void* ki,
                        const void* vi, int64_t ldkv_ip, int n_ip, float ip_scale, const float* ip_rows, void* out, int64_t ldo,
                        int64_t batch, int64_t n_q, int heads, float scale, cudaStream_t st) {
  constexpr int smem = 2 * 128 * 128 + 2 * (T1 + T2) * 128;
  IA2P_ONCE_PER_DEVICE(IA2P_CUDA(cudaFuncSetAttribute(cross_attn_kernel<T1, T2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)));
  // query tiles per (batch, head) are split over the fewest CTAs that still fill the GPU (~3 CTAs per SM): K/V loads amortise
  const int n_qtiles = (int)((n_q + 127) / 128);
  int split = n_qtiles;
  for (int d = 1; d <= n_qtiles; ++d)
    if (n_qtiles % d == 0 && (long long)d * heads * batch >= 3LL * sm_count()) { split = d; break; }
  if (const char* e = getenv("IA2P_XATTN_SPLIT")) {      // experiments only
    const int v = atoi(e);
    if (v >= 1 && v <= n_qtiles && n_qtiles % v == 0) split = v;
  }
  const dim3 grid((unsigned)split, (unsigned)heads, (unsigned)batch);
  launch_pdl(cross_attn_kernel<T1, T2>, dim3(grid), dim3(256), smem, st, 
      static_cast<const __nv_bfloat16*>(q), ldq, static_cast<const __nv_bfloat16*>(kt), static_cast<const __nv_bfloat16*>(vt),
      ldkv, n_text, static_cast<const __nv_bfloat16*>(ki), static_cast<const __nv_bfloat16*>(vi), ldkv_ip, n_ip, ip_scale,
      ip_rows, static_cast<__nv_bfloat16*>(out), ldo, (int)n_q, scale * kLog2e);
  IA2P_LAUNCH_CHECK();
  return 0;
}

// ================================================================ causal self-attention, T <= 128 (CLIP text towers)
// One CTA per (head, sequence) holds the whole sequence: Q, K, V padded to TK rows (multiple of 16, zero-filled) in smem.  Warp w
// owns query rows [16w, 16w + 16) and, causally, only the key tiles [0, 16w + 16): the MMAs past the diagonal are skipped.  Keys
// j > i are set to -inf before the exponentials (exactly 0 after them), the softmax is fp32 over the whole row at once (all keys
// are resident: no online rescaling), P is normalised before the bf16 pack.  mma.sync rather than tcgen05: a 77-token head is
// 5 x 16 query rows, far below one 128-row UMMA tile, and the whole problem of a CFG pair (2 x 20 heads) is 40 CTAs.
template <int TK>
__global__ void __launch_bounds__(TK * 2)
causal_self_attn_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                        const __nv_bfloat16* __restrict__ v, long long ld, __nv_bfloat16* __restrict__ out, long long ldo,
                        int T, float scale_log2) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  constexpr int NT = TK / 8;
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t sQ = smem_u32(smem);        // TK x 64 each
  const uint32_t sK = sQ + TK * 128;
  const uint32_t sV = sK + TK * 128;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int h = blockIdx.x;
  const long long tok0 = (long long)blockIdx.y * T;
  load_tile(sQ, q + tok0 * ld + h * 64, ld, TK, T, tid, TK * 2);
  load_tile(sK, k + tok0 * ld + h * 64, ld, TK, T, tid, TK * 2);
  load_tile(sV, v + tok0 * ld + h * 64, ld, TK, T, tid, TK * 2);
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();
  const int r0 = warp * 16;
  if (r0 >= T) return;                        // no barrier follows

  uint32_t qf[4][4];
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    const int r = r0 + (lane & 7) + ((lane >> 3) & 1) * 8;
    ldsm_x4(sQ + tile_off(r, kk * 2 + (lane >> 4)), qf[kk][0], qf[kk][1], qf[kk][2], qf[kk][3]);
  }
  float s[NT][4];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
    if (nt < 2 * warp + 2) {                  // warp-uniform: key tiles at or left of the diagonal
#pragma unroll
      for (int kp = 0; kp < 2; ++kp) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4(sK + tile_off(nt * 8 + (lane & 7), kp * 4 + (lane >> 3)), b0, b1, b2, b3);
        mma_bf16(s[nt], qf[kp * 2], b0, b1);
        mma_bf16(s[nt], qf[kp * 2 + 1], b2, b3);
      }
    }
  }
  const int row0 = r0 + g, row1 = row0 + 8;
  float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int key = nt * 8 + 2 * t + e;
      s[nt][e] = key <= row0 ? s[nt][e] * scale_log2 : -INFINITY;
      s[nt][2 + e] = key <= row1 ? s[nt][2 + e] * scale_log2 : -INFINITY;
      mx0 = fmaxf(mx0, s[nt][e]);
      mx1 = fmaxf(mx1, s[nt][2 + e]);
    }
  }
  mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
  mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
  float l0 = 0.f, l1 = 0.f;                   // key 0 is never masked: the row maxima are finite
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) {
    s[nt][0] = ex2_approx(s[nt][0] - mx0); s[nt][1] = ex2_approx(s[nt][1] - mx0);
    s[nt][2] = ex2_approx(s[nt][2] - mx1); s[nt][3] = ex2_approx(s[nt][3] - mx1);
    l0 += s[nt][0] + s[nt][1];
    l1 += s[nt][2] + s[nt][3];
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1); l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1); l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.f / l0, i1 = 1.f / l1;
  float o[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
#pragma unroll
  for (int kk = 0; kk < TK / 16; ++kk) {
    if (kk <= warp) {                         // 16-key steps at or left of the diagonal
      uint32_t pa[4];
      pa[0] = pack_bf16x2(s[2 * kk][0] * i0, s[2 * kk][1] * i0);
      pa[1] = pack_bf16x2(s[2 * kk][2] * i1, s[2 * kk][3] * i1);
      pa[2] = pack_bf16x2(s[2 * kk + 1][0] * i0, s[2 * kk + 1][1] * i0);
      pa[3] = pack_bf16x2(s[2 * kk + 1][2] * i1, s[2 * kk + 1][3] * i1);
#pragma unroll
      for (int dp = 0; dp < 4; ++dp) {
        uint32_t b0, b1, b2, b3;
        const int r = kk * 16 + (lane & 7) + ((lane >> 3) & 1) * 8;
        ldsm_x4_t(sV + tile_off(r, dp * 2 + (lane >> 4)), b0, b1, b2, b3);
        mma_bf16(o[2 * dp], pa, b0, b1);
        mma_bf16(o[2 * dp + 1], pa, b2, b3);
      }
    }
  }
  // stage this warp's 16 x 64 tile through its own (consumed) rows of the Q tile for 16-byte coalesced stores
  __syncwarp();
#pragma unroll
  for (int dt = 0; dt < 8; ++dt) {
    *reinterpret_cast<uint32_t*>(smem + tile_off(row0, dt) + t * 4) = pack_bf16x2(o[dt][0], o[dt][1]);
    *reinterpret_cast<uint32_t*>(smem + tile_off(row1, dt) + t * 4) = pack_bf16x2(o[dt][2], o[dt][3]);
  }
  __syncwarp();
  __nv_bfloat16* og = out + tok0 * ldo + h * 64;
  for (int id = lane; id < 16 * 8; id += 32) {
    const int r = r0 + (id >> 3), ch = id & 7;
    if (r < T) *reinterpret_cast<uint4*>(og + (long long)r * ldo + ch * 8) = *reinterpret_cast<const uint4*>(smem + tile_off(r, ch));
  }
}

template <int TK>
static int launch_causal(const void* q, const void* k, const void* v, int64_t ld, void* out, int64_t ldo, int64_t n, int64_t T,
                         int heads, float scale, cudaStream_t st) {
  constexpr int smem = 3 * TK * 128;
  IA2P_ONCE_PER_DEVICE(IA2P_CUDA(cudaFuncSetAttribute(causal_self_attn_kernel<TK>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)));
  launch_pdl(causal_self_attn_kernel<TK>, dim3((unsigned)heads, (unsigned)n), dim3(TK * 2), smem, st,
             static_cast<const __nv_bfloat16*>(q), static_cast<const __nv_bfloat16*>(k), static_cast<const __nv_bfloat16*>(v), ld,
             static_cast<__nv_bfloat16*>(out), ldo, (int)T, scale * kLog2e);
  IA2P_LAUNCH_CHECK();
  return 0;
}

}  // namespace ia2p

namespace ia2p {
int launch_fa_tc(const void* q, const void* k, const void* v, int64_t ld, void* out, int64_t ldo, int64_t batch,
                 int64_t n_tokens, int heads, float softmax_scale, cudaStream_t st);
int launch_xattn_tc(const void* q, int64_t ldq, const void* kt, const void* vt, int64_t ldkv, int n_text, const void* ki,
                    const void* vi, int64_t ldkv_ip, int n_ip, float ip_scale, const float* ip_rows, void* out, int64_t ldo,
                    int64_t batch, int64_t n_q, int heads, float scale, cudaStream_t st, bool* handled);
}
using namespace ia2p;

// IA2P_ATTN_IMPL=mma selects the round-1 warp-level mma.sync kernel (kept for A/B measurements); default is tcgen05.
static bool use_legacy_attn() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("IA2P_ATTN_IMPL");
    v = (e != nullptr && e[0] == 'm') ? 1 : 0;
  }
  return v == 1;
}

extern "C" int ia2p_flash_self_attn_bf16(const void* q, const void* k, const void* v, int64_t ld, void* out, int64_t ldo,
                                         int64_t batch, int64_t n_tokens, int heads, float softmax_scale, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(q && k && v && out && batch > 0 && n_tokens > 0 && heads > 0, IA2P_E_ARG, "flash_self_attn: bad arguments");
  IA2P_REQUIRE(ld % 8 == 0 && ldo % 8 == 0, IA2P_E_ALIGN, "flash_self_attn: ld/ldo must be multiples of 8");
  IA2P_REQUIRE(heads <= 65535 && batch <= 65535, IA2P_E_SHAPE, "flash_self_attn: heads/batch too large");
  if (!use_legacy_attn())
    return launch_fa_tc(q, k, v, ld, out, ldo, batch, n_tokens, heads, softmax_scale, static_cast<cudaStream_t>(stream));
  constexpr int smem = 128 * 128 + 4 * 64 * 128;
  IA2P_ONCE_PER_DEVICE(IA2P_CUDA(cudaFuncSetAttribute(flash_self_attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)));
  const dim3 grid((unsigned)((n_tokens + 127) / 128), (unsigned)heads, (unsigned)batch);
  flash_self_attn_kernel<<<grid, 256, smem, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(q), static_cast<const __nv_bfloat16*>(k), static_cast<const __nv_bfloat16*>(v), ld,
      static_cast<__nv_bfloat16*>(out), ldo, (int)n_tokens, softmax_scale * kLog2e);
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_causal_self_attn_bf16(const void* q, const void* k, const void* v, int64_t ld, void* out, int64_t ldo,
                                          int64_t n, int64_t T, int heads, float softmax_scale, void* stream) {
  IA2P_REQUIRE(q && k && v && out && n > 0 && heads > 0, IA2P_E_ARG, "causal_self_attn: bad arguments");
  IA2P_REQUIRE(T >= 1 && T <= 128, IA2P_E_SHAPE, "causal_self_attn: T=%lld must be in [1, 128]", (long long)T);
  IA2P_REQUIRE(heads <= 65535 && n <= 65535, IA2P_E_SHAPE, "causal_self_attn: heads/n too large");
  IA2P_REQUIRE(ld % 8 == 0 && ldo % 8 == 0 && ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) |
               reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(out)) & 15) == 0,
               IA2P_E_ALIGN, "causal_self_attn: ld/ldo must be multiples of 8 and q/k/v/out 16-byte aligned");
  if (int e = check_device()) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (T <= 32) return launch_causal<32>(q, k, v, ld, out, ldo, n, T, heads, softmax_scale, st);
  if (T <= 80) return launch_causal<80>(q, k, v, ld, out, ldo, n, T, heads, softmax_scale, st);
  return launch_causal<128>(q, k, v, ld, out, ldo, n, T, heads, softmax_scale, st);
}

// ip_rows == nullptr: one IP scale for the batch (ia2p_decoupled_cross_attn_bf16); else ip_rows[batch] on the device
static int cross_attn_launch(const void* q, int64_t ldq, const void* k_text, const void* v_text, int64_t ldkv, int n_text,
                             const void* k_ip, const void* v_ip, int64_t ldkv_ip, int n_ip, float ip_scale, const float* ip_rows,
                             void* out, int64_t ldo, int64_t batch, int64_t n_q, int heads, float softmax_scale, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(q && k_text && v_text && out && batch > 0 && n_q > 0 && heads > 0, IA2P_E_ARG, "cross_attn: bad arguments");
  IA2P_REQUIRE(n_text > 0 && n_text <= 128 && n_ip >= 0 && n_ip <= 16, IA2P_E_SHAPE, "cross_attn: n_text=%d (<=128) n_ip=%d (<=16)", n_text, n_ip);
  IA2P_REQUIRE(n_ip == 0 || (k_ip && v_ip), IA2P_E_ARG, "cross_attn: k_ip/v_ip required when n_ip > 0");
  IA2P_REQUIRE(ldq % 8 == 0 && ldkv % 8 == 0 && ldo % 8 == 0 && (n_ip == 0 || ldkv_ip % 8 == 0), IA2P_E_ALIGN, "cross_attn: leading dims must be multiples of 8");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  static const bool legacy_cross = [] { const char* e = getenv("IA2P_XATTN_IMPL"); return e != nullptr && e[0] == 'm'; }();   // A/B only
  if (!use_legacy_attn() && !legacy_cross) {                  // tcgen05 kernel (xattn_tc.cu) whenever all keys fit 128 columns
    bool handled = false;
    const int e = launch_xattn_tc(q, ldq, k_text, v_text, ldkv, n_text, k_ip, v_ip, ldkv_ip, n_ip, ip_scale, ip_rows, out, ldo, batch,
                                  n_q, heads, softmax_scale, st, &handled);
    if (e != 0 || handled) return e;
  }
  const int t1 = n_text <= 80 ? 80 : (n_text <= 96 ? 96 : 128);
#define IA2P_CROSS(T1_, T2_) \
  return launch_cross<T1_, T2_>(q, ldq, k_text, v_text, ldkv, n_text, k_ip, v_ip, ldkv_ip, n_ip, ip_scale, ip_rows, out, ldo, batch, n_q, \
                                heads, softmax_scale, st)
  if (n_ip > 0) {
    if (t1 == 80) IA2P_CROSS(80, 16);
    if (t1 == 96) IA2P_CROSS(96, 16);
    IA2P_CROSS(128, 16);
  } else {
    if (t1 == 80) IA2P_CROSS(80, 0);
    if (t1 == 96) IA2P_CROSS(96, 0);
    IA2P_CROSS(128, 0);
  }
#undef IA2P_CROSS
}

extern "C" int ia2p_decoupled_cross_attn_bf16(const void* q, int64_t ldq, const void* k_text, const void* v_text, int64_t ldkv,
                                              int n_text, const void* k_ip, const void* v_ip, int64_t ldkv_ip, int n_ip,
                                              float ip_scale, void* out, int64_t ldo, int64_t batch, int64_t n_q, int heads,
                                              float softmax_scale, void* stream) {
  return cross_attn_launch(q, ldq, k_text, v_text, ldkv, n_text, k_ip, v_ip, ldkv_ip, n_ip, ip_scale, nullptr, out, ldo, batch, n_q,
                           heads, softmax_scale, stream);
}

extern "C" int ia2p_decoupled_cross_attn_rows_bf16(const void* q, int64_t ldq, const void* k_text, const void* v_text,
                                                   int64_t ldkv, int n_text, const void* k_ip, const void* v_ip, int64_t ldkv_ip,
                                                   int n_ip, const float* ip_scale, void* out, int64_t ldo, int64_t batch,
                                                   int64_t n_q, int heads, float softmax_scale, void* stream) {
  IA2P_REQUIRE(ip_scale != nullptr, IA2P_E_ARG, "cross_attn_rows: null IP-scale array");
  IA2P_REQUIRE((reinterpret_cast<uintptr_t>(ip_scale) & 3) == 0, IA2P_E_ALIGN, "cross_attn_rows: ip_scale must be 4-byte aligned");
  return cross_attn_launch(q, ldq, k_text, v_text, ldkv, n_text, k_ip, v_ip, ldkv_ip, n_ip, 0.f, ip_scale, out, ldo, batch, n_q,
                           heads, softmax_scale, stream);
}
