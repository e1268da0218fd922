// Shared helpers for the unidefense_b200 CUDA kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#define UD_OK 0
#define UD_ERR_INVALID (-1)
#define UD_ERR_UNSUPPORTED (-2)
#define UD_ERR_CUDA (-3)
#define UD_ERR_WORKSPACE (-4)

// thread-local last error (ud_api.cu)
void ud_set_error(const char* fmt, ...);
int ud_check_launch(const char* what);   // also counts the launch (ud_launch_count)
void ud_count_launch(void);

#define UD_REQUIRE(cond, code, ...)            \
  do {                                         \
    if (!(cond)) {                             \
      ud_set_error(__VA_ARGS__);               \
      return (code);                           \
    }                                          \
  } while (0)

#define UD_CUDA(call)                                                        \
  do {                                                                       \
    cudaError_t e_ = (call);                                                 \
    if (e_ != cudaSuccess) {                                                 \
      ud_set_error("%s failed: %s", #call, cudaGetErrorString(e_));          \
      return UD_ERR_CUDA;                                                    \
    }                                                                        \
  } while (0)

static inline int ud_cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline size_t ud_align_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

#define UD_NUM_SMS 148
#define UD_SMEM_CTA_MAX (227u << 10)   // dynamic shared memory one CTA may use on sm_100a

// Lets `kernel` launch with `bytes` of dynamic shared memory: UD_ERR_UNSUPPORTED above UD_SMEM_CTA_MAX, UD_ERR_CUDA
// when the attribute cannot be set (dynamic plus static bytes over the limit).  `what` names the op in the message.
template <class K>
static int ud_set_smem(K kernel, size_t bytes, const char* what) {
  UD_REQUIRE(bytes <= UD_SMEM_CTA_MAX, UD_ERR_UNSUPPORTED, "%s: needs %zu bytes of shared memory per CTA (> 227 KB)",
             what, bytes);
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  UD_REQUIRE(e == cudaSuccess, UD_ERR_CUDA, "%s: cudaFuncSetAttribute(smem=%zu) failed: %s", what, bytes,
             cudaGetErrorString(e));
  return UD_OK;
}

__device__ __forceinline__ float ud_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float ud_warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide sum, result broadcast to every thread.  `red` = >=33 floats of shared memory.
// Deterministic (fixed tree).  All threads of the block must call it.
__device__ __forceinline__ float ud_block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nwarps = (blockDim.x + 31) >> 5;
  v = ud_warp_sum(v);
  __syncthreads();  // protect `red` from a previous use
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (warp == 0) {
    float t = (lane < nwarps) ? red[lane] : 0.f;
    t = ud_warp_sum(t);
    if (lane == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}

__device__ __forceinline__ float ud_sigmoid(float x) { return 1.f / (1.f + __expf(-x)); }
// Flush-to-zero forms of the two special-function instructions (MUFU.EX2 / MUFU.RCP, <= 2 ulp): without .ftz the
// compiler wraps each in a denormal range check + rescale (3-4 extra instructions), which made the issue-bound
// epilogue kernels pay ~12 instructions per swish instead of 5.  A flushed denormal here is a sigmoid of |z| > 87.
__device__ __forceinline__ float ud_ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float ud_rcp_ftz(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float ud_sigmoid_fast(float x) { return ud_rcp_ftz(1.f + ud_ex2_ftz(-1.4426950408889634f * x)); }
__device__ __forceinline__ float ud_sign(float x) { return (x > 0.f) ? 1.f : ((x < 0.f) ? -1.f : 0.f); }

// cp.async (LDGSTS): global -> shared without staging in registers, so a CTA can put its whole tile in
// flight before it starts computing.  4- and 8-byte forms (cache at all levels), 16-byte form bypasses L1.
__device__ __forceinline__ void ud_cp_async4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}
__device__ __forceinline__ void ud_cp_async8(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}
__device__ __forceinline__ void ud_cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc));
}
__device__ __forceinline__ void ud_cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void ud_cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// activation codes shared with the host API
#define UD_ACT_NONE 0
#define UD_ACT_RELU 1
#define UD_ACT_SWISH 2

__device__ __forceinline__ float ud_act_fwd(float z, int act) {
  if (act == UD_ACT_RELU) return fmaxf(z, 0.f);
  if (act == UD_ACT_SWISH) return z * ud_sigmoid(z);
  return z;
}
// d act(z) / dz     (swish: reference efficientnet/utils.py:73-77: s*(1+z*(1-s)))
__device__ __forceinline__ float ud_act_grad(float z, int act) {
  if (act == UD_ACT_RELU) return z > 0.f ? 1.f : 0.f;
  if (act == UD_ACT_SWISH) {
    const float s = ud_sigmoid(z);
    return s * (1.f + z * (1.f - s));
  }
  return 1.f;
}

// align_corners=True bilinear source coordinate, exactly as ATen computes it in fp32:
// scale = (in-1)/(out-1) (float division), src = scale * dst; i0 = (int)src; l1 = src - i0.
struct UdLerp {
  int i0, i1;
  float l0, l1;
};
__device__ __forceinline__ UdLerp ud_lerp_ac(int dst, int in_size, float scale) {
  UdLerp r;
  const float src = scale * (float)dst;
  r.i0 = (int)src;
  r.i1 = r.i0 + ((r.i0 < in_size - 1) ? 1 : 0);
  r.l1 = src - (float)r.i0;
  r.l0 = 1.f - r.l1;
  return r;
}
// The same taps from an entry t of a host-built table (ud_lerp_table: t = {__int_as_float(i0), l1}).
__device__ __forceinline__ void ud_lerp_tab(const float2 t, int in_size, int& i0, int& i1, float& l0, float& l1) {
  i0 = __float_as_int(t.x);
  i1 = i0 + ((i0 < in_size - 1) ? 1 : 0);
  l1 = t.y;
  l0 = 1.f - l1;
}
static inline float ud_ac_scale(int in_size, int out_size) {
  return out_size > 1 ? (float)(in_size - 1) / (float)(out_size - 1) : 0.f;
}
