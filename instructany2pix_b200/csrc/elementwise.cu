// HBM-bound elementwise kernels: fused CFG + DDIM update, inverse-DDIM axpby, prior CFG + DDPM step,
// sinusoidal embeddings, nearest 2x upsample, conv_in / conv_out (few-channel 3x3 convs at the NCHW boundary).
#include <type_traits>

#include "common.cuh"

namespace ia2p {

// ---------------------------------------------------------------- 128-bit accesses for the one-pass elementwise kernels
// Eight consecutive elements per thread and iteration: two LDG.128 / STG.128 for fp32, one for bf16 / fp16 (north_star: "vectorised
// 128-bit coalesced epilogues").  Callers guarantee 16-byte alignment and a multiple-of-8 element count (else the scalar kernels run).
template <typename T> __device__ __forceinline__ void load8(const T* p, float (&v)[8]);
template <> __device__ __forceinline__ void load8<float>(const float* p, float (&v)[8]) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <> __device__ __forceinline__ void load8<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
  float2 t;
  t = unpack_bf16x2(a.x); v[0] = t.x; v[1] = t.y; t = unpack_bf16x2(a.y); v[2] = t.x; v[3] = t.y;
  t = unpack_bf16x2(a.z); v[4] = t.x; v[5] = t.y; t = unpack_bf16x2(a.w); v[6] = t.x; v[7] = t.y;
}
template <> __device__ __forceinline__ void load8<__half>(const __half* p, float (&v)[8]) {
  const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
  const __half2* h = reinterpret_cast<const __half2*>(&a);
#pragma unroll
  for (int i = 0; i < 4; ++i) { const float2 t = __half22float2(h[i]); v[2 * i] = t.x; v[2 * i + 1] = t.y; }
}
template <typename T> __device__ __forceinline__ void store8(T* p, const float (&v)[8]);
template <> __device__ __forceinline__ void store8<float>(float* p, const float (&v)[8]) {
  reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
  reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
}
template <> __device__ __forceinline__ void store8<__nv_bfloat16>(__nv_bfloat16* p, const float (&v)[8]) {
  *reinterpret_cast<uint4*>(p) = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}
template <> __device__ __forceinline__ void store8<__half>(__half* p, const float (&v)[8]) {
  uint4 a;
  __half2* h = reinterpret_cast<__half2*>(&a);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
  *reinterpret_cast<uint4*>(p) = a;
}

// v rounded to T's precision and back (what a later load of a stored T reads)
template <typename T> __device__ __forceinline__ float round_to(float v);
template <> __device__ __forceinline__ float round_to<float>(float v) { return v; }
template <> __device__ __forceinline__ float round_to<__nv_bfloat16>(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
template <> __device__ __forceinline__ float round_to<__half>(float v) { return __half2float(__float2half_rn(v)); }

// ---------------------------------------------------------------- CFG + DDIM (one pass over the latents)
// VEC = true: 8 elements per thread and iteration through 128-bit loads / stores; VEC = false: scalar fallback for unaligned or
// ragged sizes.  total = batch * n; eps_u at [i], eps_c at [total + i].
// ROWS = true: the guidance scale of sample i / n is g_rows[i / n] (one request per batch row); the VEC variant needs n % 8 == 0,
// so the eight elements of a thread belong to one sample and one load serves them.  ROWS = false compiles to the scalar-g kernel.
// COEF = true (with ROWS): c_x and c_e are per row too (cx_rows / ce_rows), and x_in2 is the NEXT UNet input of the batch rows
// (not duplicated): x_in2[i] = s_rows[row] * x_out[i], with x_out[i] read back at TX precision -- bitwise axpby(x_out, x_out, s, 0)
// for finite values.  The arithmetic of x_out is the scalar kernel's, so row b is bitwise the scalar kernel at that row's values.
template <typename TE, typename TX, typename TI, bool VEC, bool ROWS, bool COEF = false>
__global__ void cfg_ddim_kernel(const TE* __restrict__ eps2, const TX* __restrict__ x, TX* __restrict__ x_out,
                                TI* __restrict__ x_in2, long long total, float g_scalar, float cx, float ce,
                                const float* __restrict__ g_rows, long long n, const float* __restrict__ cx_rows,
                                const float* __restrict__ ce_rows, const float* __restrict__ s_rows) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  constexpr int W = VEC ? 8 : 1;
  for (long long i = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * W; i < total; i += (long long)gridDim.x * blockDim.x * W) {
    const float g = ROWS ? __ldg(g_rows + i / n) : g_scalar;
    if constexpr (COEF) {
      cx = __ldg(cx_rows + i / n);
      ce = __ldg(ce_rows + i / n);
    }
    if constexpr (VEC) {
      float eu[8], ec[8], xv[8], v[8];
      load8(eps2 + i, eu);
      load8(eps2 + total + i, ec);
      load8(x + i, xv);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = cx * xv[j] + ce * (eu[j] + g * (ec[j] - eu[j]));
      store8(x_out + i, v);
      if constexpr (COEF) {
        if (x_in2 != nullptr) {
          const float s = __ldg(s_rows + i / n);
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = s * round_to<TX>(v[j]);
          store8(x_in2 + i, v);
        }
      } else if (x_in2 != nullptr) {
        store8(x_in2 + i, v);
        store8(x_in2 + total + i, v);
      }
    } else {
      const float eu = load_as_float(eps2 + i), ec = load_as_float(eps2 + total + i);
      const float v = cx * load_as_float(x + i) + ce * (eu + g * (ec - eu));
      store_from_float(x_out + i, v);
      if constexpr (COEF) {
        if (x_in2 != nullptr) store_from_float(x_in2 + i, __ldg(s_rows + i / n) * round_to<TX>(v));
      } else if (x_in2 != nullptr) {
        store_from_float(x_in2 + i, v);
        store_from_float(x_in2 + total + i, v);
      }
    }
  }
}

template <typename TE, typename TX, bool VEC>
__global__ void axpby_kernel(const TE* __restrict__ eps, const TX* __restrict__ x, TX* __restrict__ out, long long n,
                             float cx, float ce) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  constexpr int W = VEC ? 8 : 1;
  for (long long i = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * W; i < n; i += (long long)gridDim.x * blockDim.x * W) {
    if constexpr (VEC) {
      float e[8], xv[8], v[8];
      load8(eps + i, e);
      load8(x + i, xv);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = cx * xv[j] + ce * e[j];
      store8(out + i, v);
    } else {
      store_from_float(out + i, cx * load_as_float(x + i) + ce * load_as_float(eps + i));
    }
  }
}

// ---------------------------------------------------------------- continuous batching: per-slot time-embedding rows
// Slot s of an S-slot CFG batch owns UNet rows s (uncond) and S + s (cond).  tables[s] is [rows, 2 * sumC]: per step the blocked
// rowbias of a CFG pair (block r = the [2, C_r] bias of ResnetBlock r); step[s] selects the row.  The kernel writes the blocked
// [2S, C_r] blocks of the UNet batch and the slot's ncoef per-step coefficients to coef[j * S + s].  Grid (x, S, blocks).
constexpr int kMaxRowbiasBlocks = 64;
struct RowbiasBlocks { int lo[kMaxRowbiasBlocks + 1]; };

__global__ void rowbias_gather_kernel(const float* __restrict__ tables, const float* __restrict__ coef_tables,
                                      const int* __restrict__ step, float* __restrict__ rowbias, float* __restrict__ coef, int S,
                                      int rows, int ncoef, RowbiasBlocks blk) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  const int s = blockIdx.y, r = blockIdx.z;
  const int lo = blk.lo[r], C = blk.lo[r + 1] - lo, width = 2 * blk.lo[gridDim.z];
  const int k = min(max(step[s], 0), rows - 1);
  const float* src = tables + ((long long)s * rows + k) * width + 2LL * lo;
  float* dst = rowbias + 2LL * S * lo;
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
    dst[(long long)s * C + c] = src[c];
    dst[(long long)(S + s) * C + c] = src[C + c];
  }
  if (blockIdx.x == 0 && r == 0 && threadIdx.x < ncoef)
    coef[threadIdx.x * S + s] = coef_tables[((long long)s * rows + k) * ncoef + threadIdx.x];
}

// runs after the gather: every slot moves to its next row; the last row is the sentinel an idle slot stays on
__global__ void step_advance_kernel(int* __restrict__ step, int S, int last) {
  pdl_launch_dependents();
  pdl_wait();
  for (int s = threadIdx.x; s < S; s += blockDim.x)
    if (step[s] < last) step[s] += 1;
}

__global__ void prior_step_kernel(const float* __restrict__ x0_pair, const float* __restrict__ x,
                                  const float* __restrict__ noise, float* __restrict__ out, long long n, float sqrt_a,
                                  float sqrt_1ma, float g, float c_x0, float c_x, float sigma) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float xv = x[i];
    const float ec = (xv - sqrt_a * x0_pair[i]) / sqrt_1ma;        // get_eps, cond half first
    const float eu = (xv - sqrt_a * x0_pair[n + i]) / sqrt_1ma;
    const float e = eu + g * (ec - eu);
    const float x0 = (xv - sqrt_1ma * e) / sqrt_a;
    float v = c_x0 * x0 + c_x * xv;
    if (noise != nullptr) v += sigma * noise[i];
    out[i] = v;
  }
}

// ---------------------------------------------------------------- inpainting blend ([3P] StableDiffusionXLInpaintPipeline loop tail)
// out = (1 - m) * (c_x * x0 + c_e * noise) + m * lat: the known region is reset to the (re-noised) original latents after every
// step; m: [B, 1, hw] broadcast over the C channels.  noise may be NULL (last step: the clean original).
__global__ void inpaint_blend_kernel(const float* __restrict__ lat, const float* __restrict__ x0, const float* __restrict__ noise,
                                     const float* __restrict__ mask, float* __restrict__ out, long long B, int C, long long hw,
                                     float c_x, float c_e) {
  pdl_launch_dependents();
  pdl_wait();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < B * C * hw; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / (C * hw), p = i % hw;
    const float m = mask[b * hw + p];
    float keep = c_x * x0[i];
    if (noise != nullptr) keep += c_e * noise[i];
    out[i] = (1.f - m) * keep + m * lat[i];
  }
}

// ---------------------------------------------------------------- polar interpolation of two latents (pipeline.py:295-300)
// out = ll / |ll| * (alpha |x| + (1 - alpha) |y|),  ll = alpha x + (1 - alpha) y;  norms over the WHOLE tensor.
// Pass 1: per-block partial sums of x^2, y^2, ll^2 (fp64, fixed order -> bit-reproducible); pass 2: every block re-reduces the
// partials in the same order and applies the scale.
constexpr int kPolarMaxBlocks = 256;
__global__ void __launch_bounds__(256) polar_partials_kernel(const float* __restrict__ x, const float* __restrict__ y, long long n,
                                                             float alpha, double* __restrict__ partials) {
  pdl_launch_dependents();
  pdl_wait();
  float sx = 0.f, sy = 0.f, sl = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float a = x[i], b = y[i], l = a * alpha + b * (1.f - alpha);
    sx += a * a;
    sy += b * b;
    sl += l * l;
  }
  __shared__ double red[3][8];
  double dx = sx, dy = sy, dl = sl;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    dx += __shfl_xor_sync(0xffffffffu, dx, o);
    dy += __shfl_xor_sync(0xffffffffu, dy, o);
    dl += __shfl_xor_sync(0xffffffffu, dl, o);
  }
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { red[0][w] = dx; red[1][w] = dy; red[2][w] = dl; }
  __syncthreads();
  if (threadIdx.x < 3) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[threadIdx.x][i];
    partials[blockIdx.x * 3 + threadIdx.x] = t;
  }
}
__global__ void __launch_bounds__(256) polar_apply_kernel(const float* __restrict__ x, const float* __restrict__ y, float* __restrict__ out,
                                                          long long n, float alpha, const double* __restrict__ partials, int nparts) {
  pdl_launch_dependents();
  pdl_wait();
  __shared__ float s_scale;
  if (threadIdx.x == 0) {
    double t[3] = {0.0, 0.0, 0.0};
    for (int i = 0; i < nparts; ++i)
      for (int k = 0; k < 3; ++k) t[k] += partials[i * 3 + k];
    const double target = sqrt(t[0]) * (double)alpha + sqrt(t[1]) * (double)(1.f - alpha);
    s_scale = (float)(target / sqrt(t[2]));
  }
  __syncthreads();
  const float sc = s_scale;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = (x[i] * alpha + y[i] * (1.f - alpha)) * sc;
}

template <typename TO>
__global__ void timestep_embedding_kernel(const float* __restrict__ t, long long n, int dim, int flip, float shift,
                                          TO* __restrict__ out) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  const int half = dim / 2;
  const long long total = n * (long long)dim;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long r = idx / dim;
    const int c = (int)(idx - r * dim);
    float v = 0.f;
    if (c < 2 * half) {
      const int i = c < half ? c : c - half;
      const bool is_sin = flip ? (c >= half) : (c < half);
      const float freq = expf(-9.210340371976184f * (float)i / ((float)half - shift));
      const float a = t[r] * freq;
      v = is_sin ? sinf(a) : cosf(a);
    }
    store_from_float(out + idx, v);
  }
}

__device__ __forceinline__ uint4 load8_as_bf16(const __nv_bfloat16* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ uint4 load8_as_bf16(const float* p) {
  const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
  uint4 o;
  o.x = pack_bf16x2(a.x, a.y); o.y = pack_bf16x2(a.z, a.w); o.z = pack_bf16x2(b.x, b.y); o.w = pack_bf16x2(b.z, b.w);
  return o;
}
__device__ __forceinline__ uint4 load8_as_bf16(const __half* p) {
  uint4 o;
  o.x = pack_bf16x2(__half2float(p[0]), __half2float(p[1])); o.y = pack_bf16x2(__half2float(p[2]), __half2float(p[3]));
  o.z = pack_bf16x2(__half2float(p[4]), __half2float(p[5])); o.w = pack_bf16x2(__half2float(p[6]), __half2float(p[7]));
  return o;
}

template <typename T>
__global__ void upsample2x_kernel(const T* __restrict__ x, uint4* __restrict__ y, long long batch, int h, int w, int cv) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  // cv = C/8 vectors per pixel; output pixel (oy, ox) <- input (oy>>1, ox>>1); output bf16 (conv operand)
  const long long total = batch * (long long)(2 * h) * (2 * w) * cv;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % cv);
    long long pix = idx / cv;
    const int ox = (int)(pix % (2 * w));
    pix /= (2 * w);
    const int oy = (int)(pix % (2 * h));
    const long long b = pix / (2 * h);
    y[idx] = load8_as_bf16(x + (((b * h + (oy >> 1)) * w + (ox >> 1)) * cv + c) * 8);
  }
}

template <typename T>
__global__ void cast_bf16_kernel(const T* __restrict__ x, uint4* __restrict__ y, long long nvec) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x)
    y[i] = load8_as_bf16(x + i * 8);
}

// ---------------------------------------------------------------- conv_in: NCHW (few channels) -> NHWC (bf16|fp32)
// fp32 CUDA-core conv (K = 9*Cin = 36 is too shallow for tensor cores and the input latents stay unrounded).
// Block = 64 output pixels: weights transposed to smem [K][Cout], the 64 input patches to smem [64][K]; each thread
// produces channel quads (float4 weight reads conflict-free, patch reads broadcast), stores are fully coalesced.
constexpr int kConvInTile = 64;
template <typename TX, typename TO>
__global__ void __launch_bounds__(256)
conv_in_kernel(const TX* __restrict__ x, long long in_batch, long long B, int H, int W, int Cin,
               const float* __restrict__ w, const float* __restrict__ bias, TO* __restrict__ out, int Cout) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  extern __shared__ float sm[];
  const int K = Cin * 9;
  float* sw = sm;                       // [K][Cout]
  float* sp = sm + (size_t)K * Cout;    // [tile][K]
  const long long npix = B * (long long)H * W;
  for (int i = threadIdx.x; i < K * Cout; i += blockDim.x) {     // weights staged ONCE per CTA; the CTA then walks its pixel tiles
    const int co = i / K, k = i - co * K;              // w is [Cout][Cin][3][3] = [Cout][K]
    sw[k * Cout + co] = w[i];
  }
  const long long ntiles = (npix + kConvInTile - 1) / kConvInTile;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long pix0 = tile * kConvInTile;
    __syncthreads();                                   // previous tile's patch fully consumed (and weights visible)
    for (int i = threadIdx.x; i < kConvInTile * K; i += blockDim.x) {
      const int p = i / K, k = i - p * K;
      const int ci = k / 9, tap = k - ci * 9;
      const long long pix = pix0 + p;
      float v = 0.f;
      if (pix < npix) {
        const int xx = (int)(pix % W), yy = (int)((pix / W) % H);
        const long long b = pix / ((long long)W * H);
        const int iy = yy + tap / 3 - 1, ix = xx + tap % 3 - 1;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W)
          v = load_as_float(x + (((b % in_batch) * Cin + ci) * H + iy) * (long long)W + ix);
      }
      sp[i] = v;
    }
    __syncthreads();
    // register tile: 4 pixels (p, p+16, p+32, p+48) x 4 output channels per thread, so one 16-byte weight read feeds 16 FMAs
    // (the one-pixel version was bound by shared-memory bandwidth: 5 wavefronts per 4 FMAs)
    const int cq_n = Cout / 4;
    for (int idx = threadIdx.x; idx < (kConvInTile / 4) * cq_n; idx += blockDim.x) {
      const int pg = idx / cq_n, cq = idx - pg * cq_n;
      const float4 b4 = bias ? *reinterpret_cast<const float4*>(bias + cq * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 acc[4] = {b4, b4, b4, b4};
      const float* pp = sp + pg * K;
      for (int k = 0; k < K; ++k) {
        const float4 wv = *reinterpret_cast<const float4*>(sw + k * Cout + cq * 4);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float v = pp[j * (kConvInTile / 4) * K + k];
          acc[j].x += v * wv.x; acc[j].y += v * wv.y; acc[j].z += v * wv.z; acc[j].w += v * wv.w;
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const long long pix = pix0 + pg + j * (kConvInTile / 4);
        if (pix >= npix) continue;
        TO* o = out + pix * Cout + cq * 4;
        if constexpr (sizeof(TO) == 4) {
          *reinterpret_cast<float4*>(o) = acc[j];                                  // one 16-byte store per thread, coalesced
        } else if constexpr (sizeof(TO) == 2 && std::is_same<TO, __nv_bfloat16>::value) {
          *reinterpret_cast<uint2*>(o) = make_uint2(pack_bf16x2(acc[j].x, acc[j].y), pack_bf16x2(acc[j].z, acc[j].w));
        } else {
          store_from_float(o, acc[j].x); store_from_float(o + 1, acc[j].y); store_from_float(o + 2, acc[j].z); store_from_float(o + 3, acc[j].w);
        }
      }
    }
  }
}

// ---------------------------------------------------------------- conv_out: NHWC bf16 -> NCHW, Cout <= 8
// one warp = one output pixel; lanes split the (tap, channel) reduction with 16-byte loads; weights [Cout,3,3,Cin] fp32.
template <typename TO, int COUT>
__global__ void conv_out_kernel(const __nv_bfloat16* __restrict__ x, long long B, int H, int W, int Cin,
                                const float* __restrict__ w, const float* __restrict__ bias, TO* __restrict__ out) {
  pdl_launch_dependents();   // programmatic dependent launch: see common.cuh
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const long long warp_global = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
  const int cv = Cin / 8;
  for (long long pix = warp_global; pix < B * (long long)H * W; pix += nwarps) {
    const int xx = (int)(pix % W);
    const int yy = (int)((pix / W) % H);
    const long long b = pix / ((long long)W * H);
    float acc[COUT];
#pragma unroll
    for (int j = 0; j < COUT; ++j) acc[j] = 0.f;
    for (int tap = 0; tap < 9; ++tap) {
      const int iy = yy + tap / 3 - 1, ix = xx + tap % 3 - 1;
      if (iy < 0 || iy >= H || ix < 0 || ix >= W) continue;   // warp-uniform
      const uint4* xp = reinterpret_cast<const uint4*>(x + ((b * H + iy) * (long long)W + ix) * Cin);
      for (int v = lane; v < cv; v += 32) {
        const uint4 xv = __ldg(xp + v);
        float f[8];
        float2 t;
        t = unpack_bf16x2(xv.x); f[0] = t.x; f[1] = t.y;
        t = unpack_bf16x2(xv.y); f[2] = t.x; f[3] = t.y;
        t = unpack_bf16x2(xv.z); f[4] = t.x; f[5] = t.y;
        t = unpack_bf16x2(xv.w); f[6] = t.x; f[7] = t.y;
#pragma unroll
        for (int j = 0; j < COUT; ++j) {
          const float4* wp = reinterpret_cast<const float4*>(w + ((long long)(j * 9 + tap)) * Cin + v * 8);
          const float4 w0 = __ldg(wp), w1 = __ldg(wp + 1);
          acc[j] += f[0] * w0.x + f[1] * w0.y + f[2] * w0.z + f[3] * w0.w + f[4] * w1.x + f[5] * w1.y + f[6] * w1.z + f[7] * w1.w;
        }
      }
    }
#pragma unroll
    for (int j = 0; j < COUT; ++j) acc[j] = warp_sum(acc[j]);
    if (lane == 0) {
#pragma unroll
      for (int j = 0; j < COUT; ++j)
        store_from_float(out + ((b * COUT + j) * H + yy) * (long long)W + xx, acc[j] + (bias ? bias[j] : 0.f));
    }
  }
}

// ---------------------------------------------------------------- VAE boundary helpers
// 1x1 conv over few channels, NCHW fp32 -> NCHW fp32: out[b,co,p] = scale * sum_ci w[co,ci] x[b,ci,p] + bias[co]
// ([3P] AutoencoderKL.post_quant_conv / quant_conv, with the 1/scaling_factor of sdxl_pipeline.py:866 folded into `scale`).
__global__ void conv1x1_nchw_small_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                                          float* __restrict__ out, long long B, int Cin, int Cout, long long HW, float scale) {
  pdl_launch_dependents();
  pdl_wait();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < B * HW; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / HW, p = i - b * HW;
    float v[8];
    for (int ci = 0; ci < Cin; ++ci) v[ci] = x[(b * Cin + ci) * HW + p];
    for (int co = 0; co < Cout; ++co) {
      float a = 0.f;
      for (int ci = 0; ci < Cin; ++ci) a += w[co * Cin + ci] * v[ci];
      out[(b * Cout + co) * HW + p] = a * scale + (bias ? bias[co] : 0.f);
    }
  }
}

__global__ void gaussian_sample_kernel(const float* __restrict__ moments, const float* __restrict__ noise, float* __restrict__ out,
                                       long long B, long long CHW, float scale) {
  pdl_launch_dependents();
  pdl_wait();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < B * CHW; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / CHW, r = i - b * CHW;
    const float mean = moments[b * 2 * CHW + r];
    float v = mean;
    if (noise != nullptr) v += expf(0.5f * fminf(fmaxf(moments[b * 2 * CHW + CHW + r], -30.f), 20.f)) * noise[i];
    out[i] = v * scale;
  }
}

// out[b, c, p] = x[(b * hw + p) * ld + c], c < C <= 8: the first C channels of an NHWC fp32 tensor as NCHW.  Used after a
// few-output-channel 3x3 conv that ran on the tensor cores with its output channels zero-padded to 32 (conv_out of the UNet /
// VAE): thread = pixel, reads one 16/32-byte prefix of its row, writes C plane elements (coalesced per plane).
__global__ void nhwc_prefix_to_nchw_kernel(const float* __restrict__ x, long long ld, float* __restrict__ out, long long B, long long hw,
                                           int C) {
  pdl_launch_dependents();
  pdl_wait();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < B * hw; i += (long long)gridDim.x * blockDim.x) {
    const long long b = i / hw, p = i - b * hw;
    const float4 v0 = *reinterpret_cast<const float4*>(x + i * ld);
    float v[8] = {v0.x, v0.y, v0.z, v0.w, 0.f, 0.f, 0.f, 0.f};
    if (C > 4) {
      const float4 v1 = *reinterpret_cast<const float4*>(x + i * ld + 4);
      v[4] = v1.x; v[5] = v1.y; v[6] = v1.z; v[7] = v1.w;
    }
    for (int c = 0; c < C; ++c) out[(b * C + c) * hw + p] = v[c];
  }
}

// Row softmax of an fp32 score matrix [rows, cols] (row pitch ld) -> bf16 probabilities: p = softmax(scale * s).  One CTA per
// row, three passes over the row (max, sum, write); the row (<= 64 KB) stays in L1/L2 between them.  Used by the VAE's single
// 512-wide attention head (16 384 tokens at 1024^2), which runs once per image as GEMM -> softmax -> GEMM.
__global__ void __launch_bounds__(256) softmax_rows_kernel(const float* __restrict__ s, long long ld, __nv_bfloat16* __restrict__ out,
                                                           long long ldo, int cols, float scale_log2) {
  pdl_launch_dependents();
  pdl_wait();
  const float4* row = reinterpret_cast<const float4*>(s + blockIdx.x * ld);
  const int nv = cols >> 2;
  __shared__ float red[8];
  __shared__ float bcast;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float mx = -INFINITY;
  for (int i = threadIdx.x; i < nv; i += 256) {
    const float4 v = row[i];
    mx = fmaxf(mx, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
  }
  mx = warp_max(mx);
  if (lane == 0) red[w] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    float m = red[0];
    for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]);
    bcast = m * scale_log2;
  }
  __syncthreads();
  const float m = bcast;
  float sum = 0.f;
  for (int i = threadIdx.x; i < nv; i += 256) {
    const float4 v = row[i];
    sum += exp2f(fmaf(v.x, scale_log2, -m)) + exp2f(fmaf(v.y, scale_log2, -m)) + exp2f(fmaf(v.z, scale_log2, -m)) +
           exp2f(fmaf(v.w, scale_log2, -m));
  }
  sum = warp_sum(sum);
  __syncthreads();
  if (lane == 0) red[w] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    bcast = 1.f / t;
  }
  __syncthreads();
  const float inv = bcast;
  uint2* orow = reinterpret_cast<uint2*>(out + blockIdx.x * ldo);
  for (int i = threadIdx.x; i < nv; i += 256) {
    const float4 v = row[i];
    uint2 o;
    o.x = pack_bf16x2(exp2f(fmaf(v.x, scale_log2, -m)) * inv, exp2f(fmaf(v.y, scale_log2, -m)) * inv);
    o.y = pack_bf16x2(exp2f(fmaf(v.z, scale_log2, -m)) * inv, exp2f(fmaf(v.w, scale_log2, -m)) * inv);
    orow[i] = o;
  }
}

static int grid_for(long long work_items, int block) {
  long long g = (work_items + block - 1) / block;
  const long long cap = (long long)sm_count() * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace ia2p

using namespace ia2p;

#define DISPATCH_DTYPE(code, T, ...)                                   \
  switch (code) {                                                      \
    case IA2P_F32: { using T = float; __VA_ARGS__; break; }            \
    case IA2P_BF16: { using T = __nv_bfloat16; __VA_ARGS__; break; }   \
    case IA2P_F16: { using T = __half; __VA_ARGS__; break; }           \
    default: set_error("unknown dtype code %d", (int)(code)); return IA2P_E_ARG; \
  }

// g_rows == nullptr: one guidance scale `g` for the batch (ia2p_cfg_ddim_step); else g_rows[batch] on the device
static int cfg_ddim_launch(const void* eps2, int eps_dtype, const void* x, void* x_out, int x_dtype, void* x_in_next2,
                           int xin_dtype, int64_t batch, int64_t n, float g, const float* g_rows, float c_x, float c_e,
                           void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(eps2 && x && x_out && batch > 0 && n > 0, IA2P_E_ARG, "cfg_ddim_step: null pointer or empty shape");
  const long long total = batch * n;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x_in_next2 == nullptr) xin_dtype = x_dtype;
  auto esz = [](int dt) { return dt == IA2P_F32 ? 4ll : 2ll; };
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  // 128-bit path: every 8-element group of every array starts on a 16-byte boundary (the second halves start at `total`); with
  // per-row scales a group must also lie inside one sample
  const bool vec = total % 8 == 0 && al16(eps2) && al16(x) && al16(x_out) && (x_in_next2 == nullptr || al16(x_in_next2)) &&
                   (total * esz(eps_dtype)) % 16 == 0 && (total * esz(xin_dtype)) % 16 == 0 && (g_rows == nullptr || n % 8 == 0);
  const int grid = grid_for(vec ? total / 8 : total, 256);
#define IA2P_CFG_DDIM(VEC_, ROWS_)                                                                                              \
  DISPATCH_DTYPE(eps_dtype, TE, DISPATCH_DTYPE(x_dtype, TX, DISPATCH_DTYPE(xin_dtype, TI,                                       \
      (launch_pdl(cfg_ddim_kernel<TE, TX, TI, VEC_, ROWS_>, dim3(grid), dim3(256), 0, st, static_cast<const TE*>(eps2),         \
                  static_cast<const TX*>(x), static_cast<TX*>(x_out), static_cast<TI*>(x_in_next2), total, g, c_x, c_e, g_rows, \
                  (long long)n, nullptr, nullptr, nullptr)))))
  if (g_rows == nullptr) {
    if (vec) { IA2P_CFG_DDIM(true, false); } else { IA2P_CFG_DDIM(false, false); }
  } else {
    if (vec) { IA2P_CFG_DDIM(true, true); } else { IA2P_CFG_DDIM(false, true); }
  }
#undef IA2P_CFG_DDIM
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_cfg_ddim_step(const void* eps2, int eps_dtype, const void* x, void* x_out, int x_dtype,
                                  void* x_in_next2, int xin_dtype, int64_t batch, int64_t n, float g, float c_x,
                                  float c_e, void* stream) {
  return cfg_ddim_launch(eps2, eps_dtype, x, x_out, x_dtype, x_in_next2, xin_dtype, batch, n, g, nullptr, c_x, c_e, stream);
}

extern "C" int ia2p_cfg_ddim_step_rows(const void* eps2, int eps_dtype, const void* x, void* x_out, int x_dtype,
                                       void* x_in_next2, int xin_dtype, int64_t batch, int64_t n, const float* g,
                                       float c_x, float c_e, void* stream) {
  IA2P_REQUIRE(g != nullptr, IA2P_E_ARG, "cfg_ddim_step_rows: null guidance-scale array");
  IA2P_REQUIRE((reinterpret_cast<uintptr_t>(g) & 3) == 0, IA2P_E_ALIGN, "cfg_ddim_step_rows: g must be 4-byte aligned");
  return cfg_ddim_launch(eps2, eps_dtype, x, x_out, x_dtype, x_in_next2, xin_dtype, batch, n, 0.f, g, c_x, c_e, stream);
}

extern "C" int ia2p_cfg_step_coef_rows(const void* eps2, int eps_dtype, const void* x, void* x_out, int x_dtype,
                                       void* x_in_next, int xin_dtype, int64_t batch, int64_t n, const float* g,
                                       const float* c_x, const float* c_e, const float* s_in, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(eps2 && x && x_out && batch > 0 && n > 0, IA2P_E_ARG, "cfg_step_coef_rows: null pointer or empty shape");
  IA2P_REQUIRE(g && c_x && c_e, IA2P_E_ARG, "cfg_step_coef_rows: null coefficient array");
  IA2P_REQUIRE((x_in_next == nullptr) == (s_in == nullptr), IA2P_E_ARG, "cfg_step_coef_rows: x_in_next and s_in go together");
  auto al4 = [](const float* p) { return (reinterpret_cast<uintptr_t>(p) & 3) == 0; };
  IA2P_REQUIRE(al4(g) && al4(c_x) && al4(c_e) && (s_in == nullptr || al4(s_in)), IA2P_E_ALIGN,
               "cfg_step_coef_rows: coefficient arrays must be 4-byte aligned");
  const long long total = batch * n;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (x_in_next == nullptr) xin_dtype = x_dtype;
  auto esz = [](int dt) { return dt == IA2P_F32 ? 4ll : 2ll; };
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  // 128-bit path: as in cfg_ddim_launch, and every 8-element group lies inside one row
  const bool vec = n % 8 == 0 && al16(eps2) && al16(x) && al16(x_out) && (x_in_next == nullptr || al16(x_in_next)) &&
                   (total * esz(eps_dtype)) % 16 == 0;
  const int grid = grid_for(vec ? total / 8 : total, 256);
#define IA2P_CFG_COEF(VEC_)                                                                                                     \
  DISPATCH_DTYPE(eps_dtype, TE, DISPATCH_DTYPE(x_dtype, TX, DISPATCH_DTYPE(xin_dtype, TI,                                       \
      (launch_pdl(cfg_ddim_kernel<TE, TX, TI, VEC_, true, true>, dim3(grid), dim3(256), 0, st, static_cast<const TE*>(eps2),    \
                  static_cast<const TX*>(x), static_cast<TX*>(x_out), static_cast<TI*>(x_in_next), total, 0.f, 1.f, 0.f, g,    \
                  (long long)n, c_x, c_e, s_in)))))
  if (vec) { IA2P_CFG_COEF(true); } else { IA2P_CFG_COEF(false); }
#undef IA2P_CFG_COEF
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_rowbias_gather(const float* tables, const float* coef_tables, int* step, float* rowbias, float* coef,
                                   int64_t slots, int64_t rows, const int64_t* block_lo, int64_t nblocks, int64_t ncoef,
                                   void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(tables && coef_tables && step && rowbias && coef && block_lo, IA2P_E_ARG, "rowbias_gather: null pointer");
  IA2P_REQUIRE(slots > 0 && slots <= 65535 && rows > 0 && ncoef > 0 && ncoef <= 256, IA2P_E_ARG,
               "rowbias_gather: bad slots / rows / ncoef");
  IA2P_REQUIRE(nblocks > 0 && nblocks <= kMaxRowbiasBlocks, IA2P_E_ARG, "rowbias_gather: 1..%d ResnetBlocks", kMaxRowbiasBlocks);
  RowbiasBlocks blk;
  int max_c = 0;
  IA2P_REQUIRE(block_lo[0] == 0, IA2P_E_ARG, "rowbias_gather: the first block starts at column 0");
  for (int r = 0; r <= nblocks; ++r) {
    IA2P_REQUIRE(r == 0 || (block_lo[r] > block_lo[r - 1] && block_lo[r] < (1ll << 28)), IA2P_E_ARG,
                 "rowbias_gather: block offsets must increase");
    blk.lo[r] = (int)block_lo[r];
    if (r && blk.lo[r] - blk.lo[r - 1] > max_c) max_c = blk.lo[r] - blk.lo[r - 1];
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const dim3 grid((max_c + 255) / 256, (unsigned)slots, (unsigned)nblocks);
  IA2P_CUDA(launch_pdl(rowbias_gather_kernel, grid, dim3(256), 0, st, tables, coef_tables, (const int*)step, rowbias, coef,
                       (int)slots, (int)rows, (int)ncoef, blk));
  IA2P_LAUNCH_CHECK();
  IA2P_CUDA(launch_pdl(step_advance_kernel, dim3(1), dim3(128), 0, st, step, (int)slots, (int)rows - 1));
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_axpby(const void* eps, int eps_dtype, const void* x, void* x_out, int x_dtype, int64_t n, float c_x,
                          float c_e, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(eps && x && x_out && n > 0, IA2P_E_ARG, "axpby: null pointer or empty shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  const bool vec = n % 8 == 0 && al16(eps) && al16(x) && al16(x_out);
  const int grid = grid_for(vec ? n / 8 : n, 256);
  if (vec) {
    DISPATCH_DTYPE(eps_dtype, TE, DISPATCH_DTYPE(x_dtype, TX,
        (launch_pdl(axpby_kernel<TE, TX, true>, dim3(grid), dim3(256), 0, st, static_cast<const TE*>(eps), static_cast<const TX*>(x),
                    static_cast<TX*>(x_out), n, c_x, c_e))));
  } else {
    DISPATCH_DTYPE(eps_dtype, TE, DISPATCH_DTYPE(x_dtype, TX,
        (launch_pdl(axpby_kernel<TE, TX, false>, dim3(grid), dim3(256), 0, st, static_cast<const TE*>(eps), static_cast<const TX*>(x),
                    static_cast<TX*>(x_out), n, c_x, c_e))));
  }
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_inpaint_blend(const float* latents, const float* orig_latents, const float* noise, const float* mask, float* out,
                                  int64_t B, int64_t C, int64_t HW, float c_x, float c_e, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(latents && orig_latents && mask && out && B > 0 && C > 0 && HW > 0, IA2P_E_ARG, "inpaint_blend: bad arguments");
  IA2P_CUDA(launch_pdl(inpaint_blend_kernel, dim3(grid_for(B * C * HW, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream), latents,
                       orig_latents, noise, mask, out, (long long)B, (int)C, (long long)HW, c_x, c_e));
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int64_t ia2p_polar_workspace_bytes(void) { return (int64_t)kPolarMaxBlocks * 3 * sizeof(double); }

extern "C" int ia2p_polar_interpolate(const float* x, const float* y, float* out, int64_t n, float alpha, void* workspace, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x && y && out && workspace && n > 0, IA2P_E_ARG, "polar_interpolate: null pointer or empty shape");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int grid = grid_for(n, 256);
  if (grid > kPolarMaxBlocks) grid = kPolarMaxBlocks;
  double* parts = static_cast<double*>(workspace);
  IA2P_CUDA(launch_pdl(polar_partials_kernel, dim3(grid), dim3(256), 0, st, x, y, (long long)n, alpha, parts));
  IA2P_CUDA(launch_pdl(polar_apply_kernel, dim3(grid), dim3(256), 0, st, x, y, out, (long long)n, alpha, (const double*)parts, grid));
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_prior_cfg_ddpm_step(const float* x0_pair, const float* x, const float* noise, float* x_out, int64_t n,
                                        float sqrt_a, float sqrt_1ma, float g, float c_x0, float c_x, float sigma,
                                        void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x0_pair && x && x_out && n > 0, IA2P_E_ARG, "prior_cfg_ddpm_step: null pointer or empty shape");
  prior_step_kernel<<<grid_for(n, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x0_pair, x, noise, x_out, n, sqrt_a,
                                                                                     sqrt_1ma, g, c_x0, c_x, sigma);
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_timestep_embedding(const float* t, int64_t n, int dim, int flip_sin_to_cos, float shift, void* out,
                                       int out_dtype, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(t && out && n > 0 && dim > 1, IA2P_E_ARG, "timestep_embedding: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = grid_for(n * dim, 256);
  DISPATCH_DTYPE(out_dtype, TO,
      (launch_pdl(timestep_embedding_kernel<TO>, dim3(grid), dim3(256), 0, st, t, n, dim, flip_sin_to_cos, shift, static_cast<TO*>(out))));
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_upsample2x_nhwc(const void* x, int x_dtype, void* y, int64_t batch, int64_t h, int64_t w, int64_t c, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x && y && batch > 0 && h > 0 && w > 0 && c > 0, IA2P_E_ARG, "upsample2x: bad arguments");
  IA2P_REQUIRE(c % 8 == 0, IA2P_E_SHAPE, "upsample2x: C=%lld must be a multiple of 8", (long long)c);
  const long long total = batch * 4 * h * w * (c / 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = grid_for(total, 256);
  DISPATCH_DTYPE(x_dtype, TX, (launch_pdl(upsample2x_kernel<TX>, dim3(grid), dim3(256), 0, st, static_cast<const TX*>(x), static_cast<uint4*>(y),
                                                                          batch, (int)h, (int)w, (int)(c / 8))));
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_cast_to_bf16(const void* x, int x_dtype, void* y, int64_t n, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x && y && n > 0, IA2P_E_ARG, "cast_to_bf16: bad arguments");
  IA2P_REQUIRE(n % 8 == 0, IA2P_E_SHAPE, "cast_to_bf16: n=%lld must be a multiple of 8", (long long)n);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = grid_for(n / 8, 256);
  DISPATCH_DTYPE(x_dtype, TX, (launch_pdl(cast_bf16_kernel<TX>, dim3(grid), dim3(256), 0, st, static_cast<const TX*>(x), static_cast<uint4*>(y), n / 8)));
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_conv_in_nchw(const void* x, int x_dtype, int64_t in_batch, int64_t B, int64_t H, int64_t W, int64_t Cin,
                                 const float* w, const float* bias, void* out, int out_dtype, int64_t Cout, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x && w && out && B > 0 && in_batch > 0 && H > 0 && W > 0, IA2P_E_ARG, "conv_in: bad arguments");
  IA2P_REQUIRE(out_dtype == IA2P_BF16 || out_dtype == IA2P_F32, IA2P_E_ARG, "conv_in: out_dtype must be bf16 or f32");
  // Cin = 4: latents; 8 / 9: inpainting UNets (latents + mask + masked-image latents, [3P] StableDiffusionXLInpaintPipeline)
  IA2P_REQUIRE(Cin >= 1 && Cin <= 16 && Cout % 8 == 0 && Cout <= 640, IA2P_E_SHAPE, "conv_in: Cin<=16, Cout%%8==0, Cout<=640 required");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long npix = B * H * W;
  const size_t smem = (size_t)Cin * 9 * (Cout + kConvInTile) * sizeof(float);
  const long long ntiles = (npix + kConvInTile - 1) / kConvInTile;
  const long long resident = (long long)sm_count() * (smem <= 56 * 1024 ? 4 : (smem <= 100 * 1024 ? 2 : 1));
  const unsigned grid = (unsigned)(ntiles < resident ? ntiles : resident);      // persistent: weights are staged once per CTA
  IA2P_REQUIRE(smem <= 200 * 1024, IA2P_E_SHAPE, "conv_in: shared-memory footprint too large");
#define IA2P_CONV_IN(TX_, TO_)                                                                                           \
  do {                                                                                                                   \
    if (smem > 48 * 1024)                                                                                                \
      IA2P_CUDA(cudaFuncSetAttribute(conv_in_kernel<TX_, TO_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    launch_pdl(conv_in_kernel<TX_, TO_>, dim3(grid), dim3(256), smem, st, static_cast<const TX_*>(x), in_batch, B, (int)H, (int)W, (int)Cin, w, \
                                                      bias, static_cast<TO_*>(out), (int)Cout);                         \
  } while (0)
  if (out_dtype == IA2P_BF16) {
    DISPATCH_DTYPE(x_dtype, TX, IA2P_CONV_IN(TX, __nv_bfloat16));
  } else {
    DISPATCH_DTYPE(x_dtype, TX, IA2P_CONV_IN(TX, float));
  }
#undef IA2P_CONV_IN
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_conv_out_nhwc(const void* x, int64_t B, int64_t H, int64_t W, int64_t Cin, const float* w,
                                  const float* bias, void* out, int out_dtype, int64_t Cout, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x && w && out && B > 0 && H > 0 && W > 0, IA2P_E_ARG, "conv_out: bad arguments");
  IA2P_REQUIRE(Cin % 8 == 0 && (Cout == 4 || Cout == 3 || Cout == 8), IA2P_E_SHAPE,
               "conv_out: Cin%%8==0 and Cout in {3, 4, 8} required (got %lld, %lld)", (long long)Cin, (long long)Cout);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int grid = grid_for(B * H * W * 32, 256);
#define IA2P_CONV_OUT(CO_)                                                                                                      \
  DISPATCH_DTYPE(out_dtype, TO,                                                                                                 \
      (launch_pdl(conv_out_kernel<TO, CO_>, dim3(grid), dim3(256), 0, st, static_cast<const __nv_bfloat16*>(x), B, (int)H, (int)W, \
                  (int)Cin, w, bias, static_cast<TO*>(out))))
  if (Cout == 4) { IA2P_CONV_OUT(4); }
  else if (Cout == 3) { IA2P_CONV_OUT(3); }
  else { IA2P_CONV_OUT(8); }
#undef IA2P_CONV_OUT
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_conv1x1_nchw_small(const float* x, const float* w, const float* bias, float* out, int64_t B, int64_t Cin,
                                       int64_t Cout, int64_t HW, float scale, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x && w && out && B > 0 && HW > 0, IA2P_E_ARG, "conv1x1_nchw_small: bad arguments");
  IA2P_REQUIRE(Cin >= 1 && Cin <= 8 && Cout >= 1 && Cout <= 8, IA2P_E_SHAPE, "conv1x1_nchw_small: channel counts must be in [1, 8]");
  IA2P_CUDA(launch_pdl(conv1x1_nchw_small_kernel, dim3(grid_for(B * HW, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream), x, w, bias, out,
                       (long long)B, (int)Cin, (int)Cout, (long long)HW, scale));
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_nhwc_prefix_to_nchw(const float* x, int64_t ld, float* out, int64_t B, int64_t HW, int64_t C, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(x && out && B > 0 && HW > 0 && C >= 1 && C <= 8, IA2P_E_ARG, "nhwc_prefix_to_nchw: bad arguments");
  IA2P_REQUIRE(ld % 4 == 0 && ld >= 8 && (reinterpret_cast<uintptr_t>(x) & 15) == 0, IA2P_E_ALIGN, "nhwc_prefix_to_nchw: ld %% 4 == 0, ld >= 8, 16-byte base");
  IA2P_CUDA(launch_pdl(nhwc_prefix_to_nchw_kernel, dim3(grid_for(B * HW, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream), x, (long long)ld,
                       out, (long long)B, (long long)HW, (int)C));
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_gaussian_sample(const float* moments, const float* noise, float* out, int64_t B, int64_t C, int64_t HW,
                                    float scale, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(moments && out && B > 0 && C > 0 && HW > 0, IA2P_E_ARG, "gaussian_sample: bad arguments");
  IA2P_CUDA(launch_pdl(gaussian_sample_kernel, dim3(grid_for(B * C * HW, 256)), dim3(256), 0, static_cast<cudaStream_t>(stream), moments,
                       noise, out, (long long)B, (long long)(C * HW), scale));
  IA2P_LAUNCH_CHECK();
  return 0;
}

extern "C" int ia2p_softmax_rows_f32_bf16(const float* scores, int64_t ld, void* out, int64_t ldo, int64_t rows, int64_t cols,
                                          float scale, void* stream) {
  if (int e = check_device()) return e;
  IA2P_REQUIRE(scores && out && rows > 0 && cols > 0, IA2P_E_ARG, "softmax_rows: bad arguments");
  IA2P_REQUIRE(cols % 4 == 0 && ld % 4 == 0 && ldo % 4 == 0 && (reinterpret_cast<uintptr_t>(scores) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(out) & 7) == 0,
               IA2P_E_ALIGN, "softmax_rows: cols / pitches must be multiples of 4 and the bases 16 / 8-byte aligned");
  IA2P_REQUIRE(rows < (1ll << 31), IA2P_E_SHAPE, "softmax_rows: too many rows");
  IA2P_CUDA(launch_pdl(softmax_rows_kernel, dim3((unsigned)rows), dim3(256), 0, static_cast<cudaStream_t>(stream), scores, (long long)ld,
                       static_cast<__nv_bfloat16*>(out), (long long)ldo, (int)cols, scale * 1.4426950408889634f));
  IA2P_LAUNCH_CHECK();
  return 0;
}
