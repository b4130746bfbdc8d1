// Shared helpers for libpsld_b200.so (sm_100a only).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/psld_b200.h"

namespace psld {

void set_error(const char* fmt, ...);

#define PSLD_CHECK_ARG(cond, ...)            \
  do {                                       \
    if (!(cond)) {                           \
      ::psld::set_error(__VA_ARGS__);        \
      return PSLD_EINVAL;                    \
    }                                        \
  } while (0)

#define PSLD_CHECK_CUDA(expr)                                                          \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      ::psld::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                        __LINE__);                                                     \
      return PSLD_ECUDA;                                                               \
    }                                                                                  \
  } while (0)

#define PSLD_CHECK_LAUNCH() PSLD_CHECK_CUDA(cudaGetLastError())

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- programmatic dependent launch (PDL) ---------------------------------------------------
// Every kernel of the per-step program is launched with the programmatic-stream-serialization
// attribute: its CTAs may become resident while the previous kernel in the stream is still
// draining (one launch per ~50 us of work makes launch latency, the prologue and the first
// weight fetch a visible share of a step).  Contract: a kernel launched through launch_pdl()
// executes pdl_wait() before it reads or writes ANY global memory another kernel may touch
// (weights / constant tables are exempt); kernels that fit the GPU in a single wave may call
// pdl_launch_dependents() early.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
// Memory-bound / tiny kernels trigger at their first instruction: the dependent grid is launched by
// the hardware once EVERY block of this grid has started (so it never competes with unscheduled
// blocks), its prologue (barrier init, TMEM allocation, descriptor prefetch) and launch latency then
// overlap this kernel's last wave; correctness still rests on the dependent's pdl_wait().
__device__ __forceinline__ void pdl_trigger_early() { pdl_launch_dependents(); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t s, int cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  unsigned n = 0;
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = (unsigned)cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[n].val.programmaticStreamSerializationAllowed = 1;
  ++n;
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- "split bf16" activations (PSLD_BF16S): value = hi + lo, both bf16; a pixel row of C
// channels is stored as [C hi | C lo] (row stride 2C, lo at +C).  Pointers to bf16s advance in
// bf16 units; every accessor below takes the lo offset (= the row's channel count) as `lo`.
struct __align__(2) bf16s { __nv_bfloat16 v; };

template <typename T> struct Elt { static constexpr int kMul = 1; };      // row stride = kMul * C
template <> struct Elt<bf16s> { static constexpr int kMul = 2; };

__device__ __forceinline__ float2 bf2_to_f2(uint32_t w) {
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w));
}
__device__ __forceinline__ uint32_t f2_to_bf2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
// (a, b) -> packed hi pair and lo pair; a - hi is exact in fp32
__device__ __forceinline__ void split_bf2(float a, float b, uint32_t& hi, uint32_t& lo) {
  hi = f2_to_bf2(a, b);
  const float2 h = bf2_to_f2(hi);
  lo = f2_to_bf2(a - h.x, b - h.y);
}

// ---- element-type helpers: 4-wide vector load / store with fp32 math ----------------
template <typename T>
struct Vec4;

template <>
struct Vec4<float> {
  static __device__ __forceinline__ float4 load(const float* p, int = 0) {
    return *reinterpret_cast<const float4*>(p);
  }
  static __device__ __forceinline__ void store(float* p, float4 v, int = 0) {
    *reinterpret_cast<float4*>(p) = v;
  }
};

template <>
struct Vec4<__nv_bfloat16> {
  static __device__ __forceinline__ float4 load(const __nv_bfloat16* p, int = 0) {
    uint2 r = *reinterpret_cast<const uint2*>(p);
    const float2 fa = bf2_to_f2(r.x), fb = bf2_to_f2(r.y);
    return make_float4(fa.x, fa.y, fb.x, fb.y);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* p, float4 v, int = 0) {
    uint2 r;
    r.x = f2_to_bf2(v.x, v.y);
    r.y = f2_to_bf2(v.z, v.w);
    *reinterpret_cast<uint2*>(p) = r;
  }
};

template <>
struct Vec4<bf16s> {
  static __device__ __forceinline__ float4 load(const bf16s* p, int lo) {
    const uint2 h = *reinterpret_cast<const uint2*>(p);
    const uint2 l = *reinterpret_cast<const uint2*>(p + lo);
    const float2 ha = bf2_to_f2(h.x), hb = bf2_to_f2(h.y), la = bf2_to_f2(l.x), lb = bf2_to_f2(l.y);
    return make_float4(ha.x + la.x, ha.y + la.y, hb.x + lb.x, hb.y + lb.y);
  }
  static __device__ __forceinline__ void store(bf16s* p, float4 v, int lo) {
    uint2 h, l;
    split_bf2(v.x, v.y, h.x, l.x);
    split_bf2(v.z, v.w, h.y, l.y);
    *reinterpret_cast<uint2*>(p) = h;
    *reinterpret_cast<uint2*>(p + lo) = l;
  }
};

// scalar element access: p points at channel c of a pixel row, `lo` = the row's channel count
template <typename T>
__device__ __forceinline__ float ld_elt(const T* p, int lo);
template <>
__device__ __forceinline__ float ld_elt<float>(const float* p, int) { return *p; }
template <>
__device__ __forceinline__ float ld_elt<__nv_bfloat16>(const __nv_bfloat16* p, int) {
  return __bfloat162float(*p);
}
template <>
__device__ __forceinline__ float ld_elt<bf16s>(const bf16s* p, int lo) {
  return __bfloat162float(p[0].v) + __bfloat162float(p[lo].v);
}
template <typename T>
__device__ __forceinline__ void st_elt(T* p, float v, int lo);
template <>
__device__ __forceinline__ void st_elt<float>(float* p, float v, int) { *p = v; }
template <>
__device__ __forceinline__ void st_elt<__nv_bfloat16>(__nv_bfloat16* p, float v, int) {
  *p = __float2bfloat16_rn(v);
}
template <>
__device__ __forceinline__ void st_elt<bf16s>(bf16s* p, float v, int lo) {
  const __nv_bfloat16 h = __float2bfloat16_rn(v);
  p[0].v = h;
  p[lo].v = __float2bfloat16_rn(v - __bfloat162float(h));
}

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) {
  return __bfloat162float(v);
}
template <typename T>
__device__ __forceinline__ T from_f32(float v);
template <>
__device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) {
  return __float2bfloat16_rn(v);
}

__device__ __forceinline__ float silu_f(float x) { return x / (1.0f + expf(-x)); }

// bytes per logical element (split bf16 = two bf16)
static inline size_t dtype_size(int dt) { return dt == PSLD_BF16 ? 2 : (dt == PSLD_F64 ? 8 : 4); }

// per-op entry points (implemented in the .cu files, dispatched from capi.cu)
int run_layout(const psld_op& op, cudaStream_t s);
int run_axpby(const psld_op& op, cudaStream_t s);
int launch_axpby(float* out, float a, const float* x, float b, const float* y, int64_t n,
                 cudaStream_t s);
int run_temb(const psld_op& op, cudaStream_t s);
int run_gn(const psld_op& op, cudaStream_t s);
int run_fir(const psld_op& op, cudaStream_t s);
int run_conv_simt(const psld_op& op, cudaStream_t s);
int run_attn_simt(const psld_op& op, cudaStream_t s);
int prepare_conv_tc(psld_op& op);
int release_conv_tc(psld_op& op);
int run_conv_tc(const psld_op& op, cudaStream_t s);
int prepare_conv_gn_tc(psld_op& op);
int release_conv_gn_tc(psld_op& op);
int run_conv_gn_tc(const psld_op& op, cudaStream_t s);
int prepare_attn_tc(psld_op& op);
int release_attn_tc(psld_op& op);
int run_attn_tc(const psld_op& op, cudaStream_t s);
// tensor-core attention over more than 256 tokens runs the key-streaming kernel (attn_stream_tc.cu);
// prepare_attn_tc hands it the shapes it takes (HW % 128 == 0, HW >= 512)
inline bool attn_streams_keys(int HW) { return HW > 256; }
int prepare_attn_stream_tc(psld_op& op);
int release_attn_stream_tc(psld_op& op);
int run_attn_stream_tc(const psld_op& op, cudaStream_t s);

int launch_step_inc(int* step_ptr, cudaStream_t s);
int launch_sscs_table(void* u, int state_dtype, float* net_in, const float* eps,
                      const psld_sscs_coeffs* table, const int* step_ptr, int stages, uint64_t seed,
                      int64_t B, int64_t chw, cudaStream_t s);
int launch_em_table(void* u, int state_dtype, float* net_in, const float* eps,
                    const psld_score_step* table, const int* step_ptr, uint64_t seed, int64_t B,
                    int64_t chw, cudaStream_t s);

}  // namespace psld
