// HBM-bound normalisation kernels: GroupNorm (NHWC, optional two-source channel concat, optional fused SiLU) and
// LayerNorm (warp per row, two-pass statistics in registers).  bf16 I/O, fp32 math, fp64 cross-CTA accumulation.
#include "common.cuh"

namespace ia2p {

// ---------------------------------------------------------------- 8-element vector load/store helpers
template <typename T> struct Vec8;
template <> struct Vec8<__nv_bfloat16> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&f)[8]) {
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
    float2 t;
    t = unpack_bf16x2(v.x); f[0] = t.x; f[1] = t.y;
    t = unpack_bf16x2(v.y); f[2] = t.x; f[3] = t.y;
    t = unpack_bf16x2(v.z); f[4] = t.x; f[5] = t.y;
    t = unpack_bf16x2(v.w); f[6] = t.x; f[7] = t.y;
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, const float (&f)[8]) {
    uint4 o;
    o.x = pack_bf16x2(f[0], f[1]); o.y = pack_bf16x2(f[2], f[3]);
    o.z = pack_bf16x2(f[4], f[5]); o.w = pack_bf16x2(f[6], f[7]);
    *reinterpret_cast<uint4*>(p) = o;
  }
};
template <> struct Vec8<float> {
  // one full 32-byte sector per lane per instruction (LDG.256 / STG.256); rows are 32-byte aligned (cols % 8 == 0)
  static __device__ __forceinline__ void load(const float* p, float (&f)[8]) { ldg256(p, f); }
  static __device__ __forceinline__ void store(float* p, const float (&f)[8]) { stg256(p, f); }
};

// ---------------------------------------------------------------- GroupNorm statistics
// grid (slabs, batch); block (CV = C/8 vector lanes, ROWS pixel lanes).  Every thread owns one 8-channel vector
// column and strides over the slab's pixels.  Deterministic by construction (no atomics): per-thread partials go to
// shared memory, one thread per group folds them in a fixed order, and the per-slab results are written to
// partials[b][slab][group] which the apply kernel sums in slab order.
constexpr int kGnMaxSlabs = 128;

template <typename T>
__global__ void __launch_bounds__(512, 2) gn_stats_kernel(const T* __restrict__ xa, int ca, const T* __restrict__ xb, int cb,
                                long long hw, int groups, int pix_per_slab, double* __restrict__ partials) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  extern __shared__ float sm[];   // [ROWS][2][C]
  const int C = ca + cb;
  const int c0 = threadIdx.x * 8;
  const long long b = blockIdx.y;
  const long long p_begin = (long long)blockIdx.x * pix_per_slab;
  long long p_end = p_begin + pix_per_slab;
  if (p_end > hw) p_end = hw;

  float s[8], ss[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = ss[j] = 0.f;
  const bool from_a = c0 < ca;
  const T* src = from_a ? xa + b * hw * ca + c0 : xb + b * hw * cb + (c0 - ca);
  const int ld = from_a ? ca : cb;
  {
    const long long step = blockDim.y;
    long long p = p_begin + threadIdx.y;
    for (; p + 3 * step < p_end; p += 4 * step) {          // 4 independent loads in flight per thread
      float f0[8], f1[8], f2[8], f3[8];
      Vec8<T>::load(src + p * ld, f0);
      Vec8<T>::load(src + (p + step) * ld, f1);
      Vec8<T>::load(src + (p + 2 * step) * ld, f2);
      Vec8<T>::load(src + (p + 3 * step) * ld, f3);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s[j] += (f0[j] + f1[j]) + (f2[j] + f3[j]);
        ss[j] += (f0[j] * f0[j] + f1[j] * f1[j]) + (f2[j] * f2[j] + f3[j] * f3[j]);
      }
    }
    for (; p < p_end; p += step) {
      float f[8];
      Vec8<T>::load(src + p * ld, f);
#pragma unroll
      for (int j = 0; j < 8; ++j) { s[j] += f[j]; ss[j] += f[j] * f[j]; }
    }
  }
  float* mine = sm + (size_t)threadIdx.y * 2 * C;
#pragma unroll
  for (int j = 0; j < 8; ++j) { mine[c0 + j] = s[j]; mine[C + c0 + j] = ss[j]; }
  __syncthreads();
  const int cpg = C / groups;
  for (int g = threadIdx.y * blockDim.x + threadIdx.x; g < groups; g += blockDim.x * blockDim.y) {
    double a = 0.0, q = 0.0;
    for (int r = 0; r < (int)blockDim.y; ++r) {
      const float* row = sm + (size_t)r * 2 * C;
      for (int c = g * cpg; c < (g + 1) * cpg; ++c) { a += (double)row[c]; q += (double)row[C + c]; }
    }
    double* dst = partials + ((b * gridDim.x + blockIdx.x) * groups + g) * 2;
    dst[0] = a;
    dst[1] = q;
  }
}

// ---------------------------------------------------------------- GroupNorm statistics from the producers' column sums
// The tcgen05 GEMM / conv epilogue can emit per-tile (128 pixels) per-channel (sum, sum of squares) of its fp32 output
// (TcParams::colstats); this kernel folds them into the per-(image, group) partials gn_apply_kernel expects (one "slab"), so the
// statistics pass over the activation disappears.  One CTA per (group, image); fixed summation order -> bit-reproducible.
__global__ void __launch_bounds__(128) gn_colstats_reduce_kernel(const float* __restrict__ csa, int ca, int sega,
                                                                 const float* __restrict__ csb, int cb, int segb, int tiles_per_image,
                                                                 int batch, int groups, double* __restrict__ partials) {
  pdl_launch_dependents();
  pdl_wait();
  const int g = blockIdx.x, b = blockIdx.y;
  const int C = ca + cb, cpg = C / groups;
  double s = 0.0, q = 0.0;
  // work items: (tile of the image, channel of the group); a channel lives in source a or b
  const int items = tiles_per_image * cpg;
  for (int it = threadIdx.x; it < items; it += blockDim.x) {
    const int t = it / cpg, c = g * cpg + (it - t * cpg);
    const bool in_a = c < ca;
    const float* cs = in_a ? csa : csb;
    const int cw = in_a ? ca : cb, cc = in_a ? c : c - ca, seg = in_a ? sega : segb;
    const int tps = tiles_per_image / seg;                          // tiles of one image inside one segment
    const int sidx = t / tps, tin = t - sidx * tps;
    const long long tile = (long long)sidx * batch * tps + (long long)b * tps + tin;
    const float2 v = *reinterpret_cast<const float2*>(cs + (tile * cw + cc) * 2);
    s += (double)v.x;
    q += (double)v.y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  __shared__ double red[2][4];
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s; red[1][threadIdx.x >> 5] = q; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double* dst = partials + ((long long)b * groups + g) * 2;
    dst[0] = (red[0][0] + red[0][1]) + (red[0][2] + red[0][3]);
    dst[1] = (red[1][0] + red[1][1]) + (red[1][2] + red[1][3]);
  }
}

// ---------------------------------------------------------------- GroupNorm apply (+SiLU)
template <typename T>
__global__ void __launch_bounds__(512, 2) gn_apply_kernel(const T* __restrict__ xa, int ca, const T* __restrict__ xb, int cb,
                                const float* __restrict__ gamma, const float* __restrict__ beta,
                                __nv_bfloat16* __restrict__ y, __nv_bfloat16* __restrict__ raw, long long hw, int groups,
                                float eps, int silu, int pix_per_slab, const double* __restrict__ partials, int nslabs) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  extern __shared__ float sm[];   // scale[C], shift[C], then mean[groups], rstd[groups]
  const int C = ca + cb;
  const int cpg = C / groups;
  const long long b = blockIdx.y;
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  const int nthr = blockDim.x * blockDim.y;
  const double cnt = (double)hw * cpg;
  float* gmean = sm + 2 * C;
  float* grstd = gmean + groups;
  // per-group totals from the per-slab partials: warp w takes groups w, w+nwarps, ...; lanes stride over the slabs and a
  // fixed-order shuffle tree folds them (bit-reproducible, and every load of the reduction is in flight at once)
  {
    const int lane = tid & 31, wid = tid >> 5, nwarps = (nthr + 31) >> 5;
    for (int g = wid; g < groups; g += nwarps) {
      double a = 0.0, q = 0.0;
      for (int sl = lane; sl < nslabs; sl += 32) {
        const double2 v = *reinterpret_cast<const double2*>(partials + ((b * nslabs + sl) * groups + g) * 2);
        a += v.x;
        q += v.y;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
      }
      if (lane == 0) {
        const double mean = a / cnt;
        double var = q / cnt - mean * mean;
        if (var < 0.0) var = 0.0;
        gmean[g] = (float)mean;
        grstd[g] = (float)(1.0 / sqrt(var + (double)eps));
      }
    }
  }
  __syncthreads();
  for (int c = tid; c < C; c += nthr) {
    const int g = c / cpg;
    const float sc = grstd[g] * gamma[c];
    sm[c] = sc;
    sm[C + c] = beta[c] - gmean[g] * sc;
  }
  __syncthreads();
  const int c0 = threadIdx.x * 8;
  const bool from_a = c0 < ca;
  const T* src = from_a ? xa + b * hw * ca + c0 : xb + b * hw * cb + (c0 - ca);
  const int ld = from_a ? ca : cb;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { sc[j] = sm[c0 + j]; sh[j] = sm[C + c0 + j]; }
  const long long p_begin = (long long)blockIdx.x * pix_per_slab;
  long long p_end = p_begin + pix_per_slab;
  if (p_end > hw) p_end = hw;
  auto emit = [&](long long p, float (&f)[8]) {
    if (raw != nullptr) Vec8<__nv_bfloat16>::store(raw + (b * hw + p) * C + c0, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      f[j] = f[j] * sc[j] + sh[j];
      if (silu) f[j] = silu_f(f[j]);
    }
    Vec8<__nv_bfloat16>::store(y + (b * hw + p) * C + c0, f);
  };
  {
    const long long step = blockDim.y;
    long long p = p_begin + threadIdx.y;
    for (; p + step < p_end; p += 2 * step) {              // 2 independent loads in flight (register budget: 2 CTAs/SM)
      float f0[8], f1[8];
      Vec8<T>::load(src + p * ld, f0);
      Vec8<T>::load(src + (p + step) * ld, f1);
      emit(p, f0); emit(p + step, f1);
    }
    for (; p < p_end; p += step) {
      float f[8];
      Vec8<T>::load(src + p * ld, f);
      emit(p, f);
    }
  }
}

// ---------------------------------------------------------------- LayerNorm (warp per row)
template <typename T, typename TO, int MAXV>
__global__ void layernorm_kernel(const T* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                                 TO* __restrict__ y, long long rows, int cols, float eps) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (row >= rows) return;
  const int nv = cols / 8;
  float f[MAXV][8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nv) {
      Vec8<T>::load(x + row * cols + v * 8, f[i]);
#pragma unroll
      for (int j = 0; j < 8; ++j) s += f[i][j];
    }
  }
  const float mean = warp_sum(s) / (float)cols;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nv) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { const float d = f[i][j] - mean; q += d * d; }
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)cols + eps);
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int v = lane + i * 32;
    if (v < nv) {
      float o[8];
      const float4 g0 = __ldg(reinterpret_cast<const float4*>(gamma + v * 8)), g1 = __ldg(reinterpret_cast<const float4*>(gamma + v * 8) + 1);
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(beta + v * 8)), b1 = __ldg(reinterpret_cast<const float4*>(beta + v * 8) + 1);
      const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (f[i][j] - mean) * rstd * g[j] + bb[j];
      Vec8<TO>::store(y + row * cols + v * 8, o);
    }
  }
}

template <typename T, typename TO>
static int launch_ln(const void* x, const float* gamma, const float* beta, void* y, int64_t rows, int64_t cols, float eps,
                     cudaStream_t st) {
  const int block = 256;
  const long long grid = (rows * 32 + block - 1) / block;
  const T* xp = static_cast<const T*>(x);
  TO* yp = static_cast<TO*>(y);
  if (cols <= 8 * 32 * 2) launch_pdl(layernorm_kernel<T, TO, 2>, dim3((unsigned)grid), dim3(block), 0, st, xp, gamma, beta, yp, rows, (int)cols, eps);
  else if (cols <= 8 * 32 * 5) launch_pdl(layernorm_kernel<T, TO, 5>, dim3((unsigned)grid), dim3(block), 0, st, xp, gamma, beta, yp, rows, (int)cols, eps);
  else launch_pdl(layernorm_kernel<T, TO, 8>, dim3((unsigned)grid), dim3(block), 0, st, xp, gamma, beta, yp, rows, (int)cols, eps);
  IA2P_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------- CLIP token + position embedding (warp per row)
// out[r] = tok[ids[r]] + pos[r % T] in fp32; an id outside [0, V) reads nothing and yields a NaN row.  Optionally the bf16 copy
// and the row's (sum, sum of squares) in the producer format of ia2p_gemm_ln_bf16 (one part per row).
__global__ void clip_embed_kernel(const long long* __restrict__ ids, const __nv_bfloat16* __restrict__ tok, long long V,
                                  const float* __restrict__ pos, float* __restrict__ out, __nv_bfloat16* __restrict__ out_bf16,
                                  float* __restrict__ stats, long long rows, int T, int cols) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  if (row >= rows) return;
  const long long id = __ldg(ids + row);
  const bool ok = id >= 0 && id < V;
  const float* pr = pos + (row % T) * cols;
  float s = 0.f, q = 0.f;
  for (int v = lane; v < cols / 8; v += 32) {
    float a[8], b[8];
    if (ok) {
      Vec8<__nv_bfloat16>::load(tok + id * cols + v * 8, a);
      Vec8<float>::load(pr + v * 8, b);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] += b[j];
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] = __int_as_float(0x7fffffff);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) { s += a[j]; q = fmaf(a[j], a[j], q); }
    Vec8<float>::store(out + row * cols + v * 8, a);
    if (out_bf16 != nullptr) Vec8<__nv_bfloat16>::store(out_bf16 + row * cols + v * 8, a);
  }
  if (stats != nullptr) {
    s = warp_sum(s);
    q = warp_sum(q);
    if (lane == 0) { stats[2 * row] = s; stats[2 * row + 1] = q; }
  }
}

}  // namespace ia2p

using namespace ia2p;

extern "C" int64_t ia2p_groupnorm_workspace_bytes(int64_t batch, int groups) {
  return batch * kGnMaxSlabs * groups * 2 * (int64_t)sizeof(double);
}

extern "C" int ia2p_groupnorm_nhwc(const void* xa, int64_t ca, const void* xb, int64_t cb, int x_dtype, const float* gamma,
                                   const float* beta, void* y, void* raw, int64_t batch, int64_t hw, int groups, float eps,
                                   int silu, const float* cs_a, int64_t cs_a_segments, const float* cs_b, int64_t cs_b_segments,
                                   void* workspace, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x_dtype == IA2P_BF16 || x_dtype == IA2P_F32, IA2P_E_ARG, "groupnorm: x_dtype must be bf16 or f32");
  IA2P_REQUIRE(xa && gamma && beta && y && workspace && batch > 0 && hw > 0 && groups > 0, IA2P_E_ARG, "groupnorm: bad arguments");
  IA2P_REQUIRE((xb == nullptr) == (cb == 0), IA2P_E_ARG, "groupnorm: xb and cb must be given together");
  const int64_t C = ca + cb;
  IA2P_REQUIRE(ca % 8 == 0 && cb % 8 == 0 && C % groups == 0, IA2P_E_SHAPE, "groupnorm: ca=%lld cb=%lld groups=%d unsupported", (long long)ca, (long long)cb, groups);
  IA2P_REQUIRE(C / 8 <= 1024 && C <= 4096 && groups <= 64, IA2P_E_SHAPE, "groupnorm: C=%lld / groups=%d too large", (long long)C, groups);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int cv = (int)(C / 8);
  int rows = 512 / cv;
  if (rows < 1) rows = 1;
  if (rows > 32) rows = 32;
  // enough slabs for ~4 CTAs per SM, at least `rows*4` pixels each
  long long slabs = ((long long)sm_count() * 4 + batch - 1) / batch;
  long long max_slabs = (hw + rows * 4 - 1) / (rows * 4);
  if (slabs > max_slabs) slabs = max_slabs;
  if (slabs > kGnMaxSlabs) slabs = kGnMaxSlabs;
  if (slabs < 1) slabs = 1;
  const int pps = (int)((hw + slabs - 1) / slabs);
  slabs = (hw + pps - 1) / pps;
  const dim3 block(cv, rows), grid((unsigned)slabs, (unsigned)batch);
  const size_t smem_stats = (size_t)rows * 2 * C * sizeof(float);           // <= 32 KB (rows * C <= 4096)
  const size_t smem = (2 * C + 2 * groups) * sizeof(float);
  double* stats = static_cast<double*>(workspace);
  __nv_bfloat16* yp = static_cast<__nv_bfloat16*>(y);
  __nv_bfloat16* rp = static_cast<__nv_bfloat16*>(raw);
  // statistics: either from the producers' column sums (one reduction CTA per (group, image), nslabs = 1) or by a pass over x
  const bool from_cs = cs_a != nullptr;
  int nslabs = (int)slabs;
  if (from_cs) {
    IA2P_REQUIRE(cb == 0 || cs_b != nullptr, IA2P_E_ARG, "groupnorm: column statistics must be given for both sources");
    const int64_t sa = cs_a_segments > 0 ? cs_a_segments : 1, sb = cs_b_segments > 0 ? cs_b_segments : 1;
    IA2P_REQUIRE(hw % (128 * sa) == 0 && hw % (128 * sb) == 0, IA2P_E_SHAPE, "groupnorm: column statistics need hw %% (128 * segments) == 0");
    IA2P_CUDA(launch_pdl(gn_colstats_reduce_kernel, dim3((unsigned)groups, (unsigned)batch), dim3(128), 0, st, cs_a, (int)ca, (int)sa,
                         cs_b, (int)cb, (int)sb, (int)(hw / 128), (int)batch, groups, stats));
    nslabs = 1;
  }
  if (x_dtype == IA2P_BF16) {
    const __nv_bfloat16 *a = static_cast<const __nv_bfloat16*>(xa), *b = static_cast<const __nv_bfloat16*>(xb);
    if (!from_cs) launch_pdl(gn_stats_kernel<__nv_bfloat16>, dim3(grid), dim3(block), smem_stats, st, a, (int)ca, b, (int)cb, hw, groups, pps, stats);
    IA2P_LAUNCH_CHECK();
    launch_pdl(gn_apply_kernel<__nv_bfloat16>, dim3(grid), dim3(block), smem, st, a, (int)ca, b, (int)cb, gamma, beta, yp, rp, hw, groups, eps, silu, pps, (const double*)stats, nslabs);
  } else {
    const float *a = static_cast<const float*>(xa), *b = static_cast<const float*>(xb);
    if (!from_cs) launch_pdl(gn_stats_kernel<float>, dim3(grid), dim3(block), smem_stats, st, a, (int)ca, b, (int)cb, hw, groups, pps, stats);
    IA2P_LAUNCH_CHECK();
    launch_pdl(gn_apply_kernel<float>, dim3(grid), dim3(block), smem, st, a, (int)ca, b, (int)cb, gamma, beta, yp, rp, hw, groups, eps, silu, pps, (const double*)stats, nslabs);
  }
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_layernorm(const void* x, int x_dtype, const float* gamma, const float* beta, void* y, int y_dtype,
                              int64_t rows, int64_t cols, float eps, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x && gamma && beta && y && rows > 0 && cols > 0, IA2P_E_ARG, "layernorm: bad arguments");
  IA2P_REQUIRE(cols % 8 == 0 && cols <= 2048, IA2P_E_SHAPE, "layernorm: cols=%lld must be a multiple of 8 and <= 2048", (long long)cols);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x_dtype == IA2P_BF16 && y_dtype == IA2P_BF16) return launch_ln<__nv_bfloat16, __nv_bfloat16>(x, gamma, beta, y, rows, cols, eps, st);
  if (x_dtype == IA2P_F32 && y_dtype == IA2P_BF16) return launch_ln<float, __nv_bfloat16>(x, gamma, beta, y, rows, cols, eps, st);
  if (x_dtype == IA2P_F32 && y_dtype == IA2P_F32) return launch_ln<float, float>(x, gamma, beta, y, rows, cols, eps, st);
  set_error("layernorm: unsupported dtype pair (%d -> %d)", x_dtype, y_dtype);
  return IA2P_E_ARG;
}

extern "C" int ia2p_clip_embed(const int64_t* ids, int64_t n, int64_t T, const void* tok, int64_t V, const float* pos, int64_t P,
                               int64_t C, float* out, void* out_bf16, float* stats, void* stream) {
  IA2P_REQUIRE(ids && tok && pos && out && n > 0 && T > 0 && V > 0 && C > 0, IA2P_E_ARG, "clip_embed: bad arguments");
  IA2P_REQUIRE((out_bf16 == nullptr) == (stats == nullptr), IA2P_E_ARG, "clip_embed: out_bf16 and stats must be given together");
  IA2P_REQUIRE(T <= P, IA2P_E_SHAPE, "clip_embed: T=%lld exceeds the %lld positions of the table", (long long)T, (long long)P);
  IA2P_REQUIRE(C % 8 == 0, IA2P_E_SHAPE, "clip_embed: C=%lld must be a multiple of 8", (long long)C);
  IA2P_REQUIRE((reinterpret_cast<uintptr_t>(tok) & 15) == 0 && (reinterpret_cast<uintptr_t>(out_bf16) & 15) == 0 &&
               (reinterpret_cast<uintptr_t>(pos) & 31) == 0 && (reinterpret_cast<uintptr_t>(out) & 31) == 0 &&
               (reinterpret_cast<uintptr_t>(ids) & 7) == 0, IA2P_E_ALIGN, "clip_embed: misaligned table or output");
  if (int e = check_device()) return e;
  const long long rows = n * T;
  const int block = 256;
  launch_pdl(clip_embed_kernel, dim3((unsigned)((rows * 32 + block - 1) / block)), dim3(block), 0, static_cast<cudaStream_t>(stream),
             reinterpret_cast<const long long*>(ids), static_cast<const __nv_bfloat16*>(tok), (long long)V, pos, out,
             static_cast<__nv_bfloat16*>(out_bf16), stats, rows, (int)T, (int)C);
  IA2P_LAUNCH_CHECK();
  return 0;
}
