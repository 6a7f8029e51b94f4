// Shared helpers for libvatlq (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include <type_traits>

#include "../../include/vatlq.h"

namespace vatlq {

extern thread_local char g_err[512];
extern std::atomic<uint64_t> g_launches;

#define VQ_REQUIRE(cond, msg)                                                       \
  do {                                                                              \
    if (!(cond)) {                                                                  \
      snprintf(::vatlq::g_err, sizeof(::vatlq::g_err), "%s: %s", __func__, msg);    \
      return VATLQ_EINVAL;                                                          \
    }                                                                               \
  } while (0)

#define VQ_CUDA(expr)                                                              \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) {                                                       \
      snprintf(::vatlq::g_err, sizeof(::vatlq::g_err), "%s:%d %s -> %s", __FILE__, \
               __LINE__, #expr, cudaGetErrorString(_e));                           \
      return (int)_e;                                                              \
    }                                                                              \
  } while (0)

// count + check a kernel launch
#define VQ_LAUNCHED()                     \
  do {                                    \
    ::vatlq::g_launches.fetch_add(1);     \
    VQ_CUDA(cudaGetLastError());          \
  } while (0)

inline int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
int fill_f64(double* p, long long n, double v, cudaStream_t stream);
// canonical |x|^2 of every row (coreset.cu); a 16-bit X gives the bits of its fp32 upcast
int vq_launch_norms(const float* X, int64_t n, int d, double* xx, cudaStream_t stream);
int vq_launch_norms(const __half* X, int64_t n, int d, double* xx, cudaStream_t stream);
int vq_launch_norms(const __nv_bfloat16* X, int64_t n, int d, double* xx, cudaStream_t stream);

// ---------------------------------------------------------------- device helpers
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}

// ---------------------------------------------------------------- heat-map element types (VATLQ_F32 / F16 / BF16)
// Every fp16 and bf16 value is exactly representable in fp32, so a 16-bit heat map is read through an exact
// conversion at the load and everything after it is the fp32 arithmetic.  A "quad" is four consecutive pixels:
// one float4 (16 B) in fp32, one uint2 (8 B) in 16 bits; a lane that owns quad q owns the same four pixels in
// either form, so every accumulation chain sees the same values in the same order as on the fp32 upcast.
__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(__half x) { return __half2float(x); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 x) { return __bfloat162float(x); }

template <typename T> struct QuadOf { using type = uint2; };
template <> struct QuadOf<float> { using type = float4; };

__device__ __forceinline__ float4 quad_f32(float4 v, const float*) { return v; }
__device__ __forceinline__ float4 quad_f32(uint2 v, const __half*) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ float4 quad_f32(uint2 v, const __nv_bfloat16*) {   // bf16 = the top half of an fp32
  return make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xffff0000u), __uint_as_float(v.y << 16),
                     __uint_as_float(v.y & 0xffff0000u));
}
// quad q of p (shared or global memory, plain load)
template <typename T>
__device__ __forceinline__ float4 load_quad(const T* p, size_t q) {
  return quad_f32(reinterpret_cast<const typename QuadOf<T>::type*>(p)[q], p);
}
// quad q of p through the read-only path (__ldg)
template <typename T>
__device__ __forceinline__ float4 ldg_quad(const T* p, size_t q) {
  return quad_f32(__ldg(reinterpret_cast<const typename QuadOf<T>::type*>(p) + q), p);
}
__device__ __forceinline__ float ldg_f32(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ldg_f32(const __half* p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ float ldg_f32(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }

__device__ __forceinline__ uint2 ldg_stream(const uint2* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
// quad q of p, streamed (read once: no L1 allocation)
template <typename T>
__device__ __forceinline__ float4 ldg_stream_quad(const T* p, size_t q) {
  return quad_f32(ldg_stream(reinterpret_cast<const typename QuadOf<T>::type*>(p) + q), p);
}

// host side: element size of a VATLQ_* dtype code (0: unknown code)
inline size_t dtype_size(int dtype) {
  return dtype == VATLQ_F32 ? 4 : (dtype == VATLQ_F16 || dtype == VATLQ_BF16) ? 2 : 0;
}
// host side: p suits the quad loads of a dtype (16 B in fp32, 8 B in 16 bits)
inline bool quad_aligned(const void* p, int dtype) { return ((uintptr_t)p & (4 * dtype_size(dtype) - 1)) == 0; }

// call f(T*) with H cast to the element type of dtype (dtype already validated)
template <typename F>
inline int with_dtype(int dtype, F&& f) {
  if (dtype == VATLQ_F16) return f((const __half*)nullptr);
  if (dtype == VATLQ_BF16) return f((const __nv_bfloat16*)nullptr);
  return f((const float*)nullptr);
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// fixed-order butterfly: every lane ends with the same bits
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---------------------------------------------------------------- programmatic dependent launch
// Chains of short kernels (a core-set round: candidate tiles + planner, segment filter, pass; a
// k-means++ step: seven kernels) are launched with cudaLaunchAttributeProgrammaticStreamSerialization.  Each starts with pdl_enter(): wait until
// the previous kernel has completed and flushed (so the data flow is exactly the stream order), then let the NEXT
// kernel's CTAs be scheduled as SMs free up — they sit in their own pdl_enter() until this grid is done.  What is
// saved is the launch / scheduling latency of every kernel boundary of the round.  Without the launch attribute both
// instructions are no-ops.
__device__ __forceinline__ void pdl_enter() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// launch `kernel` as a programmatic dependent of the previous kernel in `stream` (pdl = false: plain launch)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, bool pdl,
                              Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at{};
  at.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &at;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------- mbarrier / TMA bulk copy (sm_90+)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  const uint32_t a = smem_u32(bar);
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(a), "r"(parity)
        : "memory");
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

}  // namespace vatlq
