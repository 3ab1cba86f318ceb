// Shared device helpers (sm_100a inline PTX: mbarrier, TMA, tcgen05/TMEM) and host-side error plumbing.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <stdint.h>

#include "../../include/ia2p.h"

namespace ia2p {

// ---------------------------------------------------------------- host error plumbing
void set_error(const char* fmt, ...);
int check_device();                       // 0 or IA2P_E_DEVICE (cached per device)
int sm_count();
#define IA2P_REQUIRE(cond, code, ...)            \
  do {                                           \
    if (!(cond)) {                               \
      ::ia2p::set_error(__VA_ARGS__);            \
      return (code);                             \
    }                                            \
  } while (0)
#define IA2P_CUDA(expr)                                                                   \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::ia2p::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return (int)_e;                                                                     \
    }                                                                                     \
  } while (0)
#define IA2P_LAUNCH_CHECK() IA2P_CUDA(cudaGetLastError())
bool pdl_enabled();                        // IA2P_PDL=1 enables programmatic dependent launch (off by default, see below)
// Kernel function attributes (dynamic shared-memory limit, carve-out) belong to the DEVICE: set them once per device this
// process launches on, not once per process.  `stmts` may use IA2P_CUDA (returns the error code from the enclosing function).
#define IA2P_ONCE_PER_DEVICE(stmts)                                            \
  do {                                                                         \
    static std::atomic<unsigned long long> _done{0};                           \
    int _dev = 0;                                                              \
    IA2P_CUDA(cudaGetDevice(&_dev));                                           \
    const unsigned long long _bit = 1ull << (_dev & 63);                       \
    if (!(_done.load(std::memory_order_acquire) & _bit)) {                     \
      stmts;                                                                   \
      _done.fetch_or(_bit, std::memory_order_release);                         \
    }                                                                          \
  } while (0)

// kernel<<<grid, block, smem, stream>>>(args...) with the programmatic-stream-serialisation attribute
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------- small device utilities
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }
// Warp index as a value the compiler KNOWS is warp-uniform (a shuffle from lane 0): role branches on it are uniform branches, so
// everything computed inside them from uniform inputs can live in uniform registers.
__device__ __forceinline__ int warp_idx_uniform() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }
// One lane of a converged warp (elect.sync).  Unlike `lane == 0`, ptxas treats the guarded region as single-lane code with uniform
// operands: tcgen05.mma / tcgen05.commit / TMA issue compile to ONE instruction with uniform-register operands instead of a
// per-lane "waterfall" loop (ELECT + 7 x R2UR.BROADCAST + branch around every UTCHMMA -- measured ~150 clk of issue per MMA,
// which made the single issuing thread, not the tensor pipe, the bottleneck of the GEMM main loop).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ float silu_f(float v) { return v / (1.0f + __expf(-v)); }
// Exact (erf) GELU, v * Phi(v), with Phi(-|v|) = 0.5 erfc(|v| / sqrt 2) from Abramowitz & Stegun 7.1.26 (|error| <= 1.5e-7 in
// erf; measured max |error| of the whole expression 4.2e-7 over [-10, 10], tests/test_kernels_gpu.py::test_gelu_accuracy).
// 17 instructions incl. one MUFU.RCP and one MUFU.EX2 instead of ~46 for erff(): in the GEGLU GEMM the erff() version kept
// the 8 epilogue warps busy 80 % of the time and slowed the concurrent tcgen05 main loop by 12 % (tools/trace_gemm.py).
__device__ __forceinline__ float gelu_erf_f(float v) {
  const float a = fabsf(v);
  float t, e;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f * 0.70710678118654752440f, a, 1.0f)));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  p = p * t;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(a * a * (-0.5f * 1.4426950408889634f)));
  const float q = 0.5f * p * e;
  return v * (v >= 0.f ? 1.0f - q : q);
}
// CLIP's quick_gelu, v * sigmoid(1.702 v)
__device__ __forceinline__ float quick_gelu_f(float v) { return v / (1.0f + __expf(-1.702f * v)); }
__device__ __forceinline__ float gelu_new_f(float v) {
  return 0.5f * v * (1.0f + tanhf(0.79788456080286535588f * (v + 0.044715f * v * v * v)));
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 r = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&r);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t v) {
  __nv_bfloat162 r = *reinterpret_cast<__nv_bfloat162*>(&v);
  return __bfloat1622float2(r);
}

template <typename T> __device__ __forceinline__ float load_as_float(const T* p);
template <> __device__ __forceinline__ float load_as_float<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float load_as_float<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <> __device__ __forceinline__ float load_as_float<__half>(const __half* p) { return __half2float(*p); }
template <typename T> __device__ __forceinline__ void store_from_float(T* p, float v);
template <> __device__ __forceinline__ void store_from_float<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void store_from_float<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ void store_from_float<__half>(__half* p, float v) { *p = __float2half_rn(v); }

// 256-bit global accesses (sm_100: LDG.256 / STG.256): one full 32-byte sector per thread per instruction.
__device__ __forceinline__ void ldg256(const float* p, float* d) {
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3]), "=f"(d[4]), "=f"(d[5]), "=f"(d[6]), "=f"(d[7]) : "l"(p));
}
__device__ __forceinline__ void stg256(float* p, const float* d) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
               ::"l"(p), "f"(d[0]), "f"(d[1]), "f"(d[2]), "f"(d[3]), "f"(d[4]), "f"(d[5]), "f"(d[6]), "f"(d[7]) : "memory");
}

// 32-byte load / store that bypass the (non-coherent) L1: data another CTA of the same kernel wrote (split-K partials)
__device__ __forceinline__ void ldg256_cg(const float* p, float* d) {
  asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3]) : "l"(p) : "memory");
  asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(d[4]), "=f"(d[5]), "=f"(d[6]), "=f"(d[7]) : "l"(p + 4) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---------------------------------------------------------------- programmatic dependent launch
// With IA2P_PDL=1 every kernel of the library is launched with programmatic stream serialisation (launch_pdl above): its CTAs
// may be scheduled while the previous kernel of the stream is still draining, so the set-up part (barrier init, TMEM
// allocation, descriptor prefetch, index arithmetic) overlaps that tail.  Measured on B200: back-to-back eager GEMMs gain
// 1.3-2.4 us per launch, but inside the CUDA-graph UNet step (power-capped, kernels already queued by the graph) the step time
// does not improve (70.1 vs 70.2 ms GEMM-only PDL; 71.6 vs 72.6 ms with every kernel) -- so it is OFF by default.  pdl_wait() blocks until the previous kernel has completed and
// its writes are visible; EVERY CTA must execute it before touching global memory (and before exiting), which also keeps
// completion transitive along the stream.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------- debug-build tracing (tools/trace_gemm.py, -DIA2P_TC_TRACE)
#ifdef IA2P_TC_TRACE
// each .cu that traces defines its own `__device__ unsigned long long* IA2P_TRACE_BUF` (no relocatable device code here)
__device__ __forceinline__ unsigned long long gtime_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define TRACE_DECL(name) long long name = 0
#define TRACE_T0(v) const long long v = clock64()
#define TRACE_ADD(acc, v) acc += clock64() - v
// IA2P_TRACE_ROW: row of this CTA in the trace buffer (default: blockIdx.x, i.e. the buffer describes the LAST launch; a kernel may
// define it as launch_id * stride + blockIdx.x to keep one row per (launch, CTA) of a whole CUDA-graph step)
#ifndef IA2P_TRACE_ROW
#define IA2P_TRACE_ROW ((size_t)blockIdx.x)
#endif
#define TRACE_PUT_AT(cta, slot, val) do { if (IA2P_TRACE_BUF != nullptr && lane == 0) IA2P_TRACE_BUF[(size_t)(cta) * 16 + (slot)] = (unsigned long long)(val); } while (0)
#define TRACE_PUT(slot, val) TRACE_PUT_AT(IA2P_TRACE_ROW, slot, val)
#else
#define TRACE_DECL(name)
#define TRACE_T0(v)
#define TRACE_ADD(acc, v)
#define TRACE_PUT_AT(cta, slot, val)
#define TRACE_PUT(slot, val)
#endif

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trap (-> cudaErrorLaunchFailure), never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 20000000000LL) __trap();   // ~10 s at 2 GHz
  }
}

// ---------------------------------------------------------------- thread-block clusters / CTA pairs
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx_cluster(uint32_t cluster_addr, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.release.cluster.shared::cluster.b64 _, [%0], %1;" ::"r"(cluster_addr), "r"(bytes) : "memory");
}

// ---------------------------------------------------------------- TMA (cp.async.bulk.tensor)
__device__ __forceinline__ void tma_prefetch_desc(const void* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// Multicast TMA load: the box lands at the SAME shared-memory offset in every CTA of `cta_mask` (cluster ranks) and completes
// tx bytes on the mbarrier at the same offset in each of them.
__device__ __forceinline__ void tma_load_4d_mc(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2, int c3, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "h"(cta_mask)
      : "memory");
}

// TMA store (shared::cta -> global, bulk async-group completion) of one 4-D box; out-of-bounds parts of the box are clipped.
__device__ __forceinline__ void tma_store_4d(const void* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const void* map, uint32_t src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// all bulk groups committed by THIS thread have finished READING their shared-memory source
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// ... all but the most recent one
__device__ __forceinline__ void bulk_wait_read_1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float lds32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void sts128u(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// L2 prefetch of a contiguous global range (no shared memory involved, no completion to wait for); bytes % 16 == 0
__device__ __forceinline__ void bulk_prefetch_l2(const void* gptr, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gptr), "r"(bytes) : "memory");
}

// CTA-pair (cta_group::2) loads: data lands in THIS CTA's smem, the completion is signalled on the LEADER CTA's mbarrier
// (same smem offset, peer bit cleared -- the addressing CUTLASS's SM100_TMA_2SM_LOAD uses).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const void* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// CTA-pair MMA (issued by the leader CTA only): M = 256 split over the two CTAs' TMEM, each CTA supplies its A rows and
// its half of B from its own smem (same descriptors / offsets in both CTAs).
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit -> arrive on the barrier at this smem offset in every CTA of `cta_mask`
__device__ __forceinline__ void umma_commit_2sm_mc(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem desc] * B[smem desc]; kind::f16 covers bf16 inputs with fp32 accumulation.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same with the A operand in TMEM (lane = row, each 32-bit column holds two consecutive K elements): D (+)= A[tmem] * B[smem desc]
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same, arriving on the barrier at this offset in every CTA of `cta_mask` (single-CTA MMAs inside a cluster that shares operands).
__device__ __forceinline__ void umma_commit_mc(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(cta_mask) : "memory");
}
// Arrive on an mbarrier when all tcgen05 ops previously issued by this thread have completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 32 columns (fp32) -> 32 registers per thread; thread i of the warp reads TMEM lane (base_lane + i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 16 columns
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// single-instruction exp2 (MUFU.EX2, flush-to-zero): exp2f() without fast-math adds 3 range-fixup instructions per call
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// 2^x on the FMA / ALU pipes instead of the SFU (Cody-Waite range reduction + a degree-3 minimax polynomial on [-0.5, 0.5],
// max relative error 7.5e-5 -- far below the bf16 rounding the result gets in the attention kernels): x + 1.5 * 2^23 leaves
// round(x) in the low mantissa bits, which are shifted straight into the exponent field of the polynomial's value.  Valid for
// -125 <= x < 100 (smaller x is clamped).  The flash-attention softmax is bound by the 16 MUFU lanes of an SM; evaluating a
// quarter of the exponentials here runs them on otherwise idle pipes (FlashAttention-4's trick).
__device__ __forceinline__ float ex2_poly3(float x) {
  x = fmaxf(x, -125.f);
  const float xf = x + 12582912.f;
  const float f = x - (xf - 12582912.f);
  float p = fmaf(0.0551716685f, f, 0.2426111400f);
  p = fmaf(p, f, 0.6932609677f);
  p = fmaf(p, f, 0.9999280572f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(xf) << 23));
}
// Packed fp32 pairs (sm_100 FFMA2 / FADD2: one issue slot for two fp32 operations on an aligned 64-bit register pair).  The
// flash-attention softmax is bound by ISSUE slots next to the MUFU lanes, so the scale-subtract, the row sum and the polynomial run
// on pairs of neighbouring keys.
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f2_sub(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// ex2_poly3 on a pair: 2 FMNMX + 3 FADD2 + 3 FFMA2 + 2 shift-adds = 5 issue slots per exponential (scalar form: 8)
__device__ __forceinline__ uint64_t ex2_poly3_x2(uint64_t x2) {
  float x0, x1;
  f2_unpack(x2, x0, x1);
  x2 = f2_pack(fmaxf(x0, -125.f), fmaxf(x1, -125.f));
  const uint64_t magic = f2_pack(12582912.f, 12582912.f);
  const uint64_t xf = f2_add(x2, magic);
  const uint64_t f = f2_sub(x2, f2_sub(xf, magic));
  uint64_t p = f2_fma(f2_pack(0.0551716685f, 0.0551716685f), f, f2_pack(0.2426111400f, 0.2426111400f));
  p = f2_fma(p, f, f2_pack(0.6932609677f, 0.6932609677f));
  p = f2_fma(p, f, f2_pack(0.9999280572f, 0.9999280572f));
  float p0, p1, n0, n1;
  f2_unpack(p, p0, p1);
  f2_unpack(xf, n0, n1);
  return f2_pack(__int_as_float(__float_as_int(p0) + (__float_as_int(n0) << 23)), __int_as_float(__float_as_int(p1) + (__float_as_int(n1) << 23)));
}
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor, K-major operand, SWIZZLE_128B, rows of 64 bf16 (128 B), 8-row groups 1024 B apart
// (bit layout: cute/arch/mma_sm100_desc.hpp SmemDescriptor; version=1 for sm_100).
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);      // start address  [0,14)
  d |= (uint64_t)1 << 16;                           // leading byte offset (unused for swizzled K-major) [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;                 // stride byte offset [32,46)
  d |= (uint64_t)1 << 46;                           // descriptor version [46,48)
  d |= (uint64_t)2 << 61;                           // SWIZZLE_128B [61,64)
  return d;
}
// Same for an MN-major operand (rows = K index, 64 MN elements = 128 B contiguous per row, e.g. V[key][d] as the B operand of
// P.V): 8-row K groups 1024 B apart (SBO); LBO = distance between 64-element MN atoms (unused when the MN extent is 64).
__device__ __forceinline__ uint64_t umma_desc_sw128_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor: D=f32, A=B=bf16, both K-major, dense (cute InstrDescriptor bit layout).
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n, int b_mn_major = 0) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(b_mn_major & 1) << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(m >> 4) << 24);
}

}  // namespace ia2p
