// Shared device helpers for the xlstm_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#define XL_WARP 32

namespace xl {

// ---- programmatic dependent launch (PDL) -----------------------------------------------------------
// Every kernel of the step is launched with cudaLaunchAttributeProgrammaticStreamSerialization: its CTAs may
// become resident while the previous kernel N of the stream is still running. Every thread of a kernel runs
//     [prologue]  pdl_wait();  pdl_trigger();  [body]
// pdl_wait() returns when kernel N has completed and its writes are visible; pdl_trigger() then lets the NEXT
// kernel start launching. Because the trigger comes after the wait, a kernel's prologue runs only when every
// kernel up to N-1 is complete: the prologue may read weights and anything written by kernels <= N-1 (the
// recurrent state of the previous env step, activations two kernels back), set up barriers / TMEM / tensor
// maps and prefetch; anything kernel N itself writes is read, and every global write is done, after the wait.
// Both are no-ops when the kernel was launched without the attribute.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

extern int g_use_pdl;   // xl_set_option("pdl", 0/1); defined in xl_elementwise.cu

template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s,
                            Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_use_pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Opt a kernel in to `smem` bytes of dynamic shared memory (> 48 KB needs cudaFuncAttributeMaxDynamicSharedMemorySize).
// The attribute belongs to (kernel, device/context): the "already configured" high-water mark is kept per kernel
// instantiation (the kernel is a template argument) AND per device, and updated atomically, so several handles on
// different GPUs or threads of one process all get their opt-in.
constexpr int kMaxDevices = 64;
template <auto Kernel>
inline cudaError_t ensure_dyn_smem(size_t smem) {
  static std::atomic<size_t> configured[kMaxDevices];
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const bool tracked = dev >= 0 && dev < kMaxDevices;
  if (tracked && smem <= configured[dev].load(std::memory_order_acquire)) return cudaSuccess;
  if (smem <= 48 * 1024 && tracked && configured[dev].load(std::memory_order_acquire) == 0) return cudaSuccess;
  e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  if (tracked) {
    size_t cur = configured[dev].load(std::memory_order_relaxed);
    while (cur < smem && !configured[dev].compare_exchange_weak(cur, smem, std::memory_order_release)) {
    }
  }
  return cudaSuccess;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum over the whole CTA; result valid in every thread. `red` = >= 32 floats of shared memory.
// Fixed order (lane tree, then warp 0 tree) -> deterministic for a given block size.
__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();  // protect `red` from a previous use
  if (lane == 0) red[wid] = v;
  __syncthreads();
  float r = (lane < nw) ? red[lane] : 0.f;
  r = warp_sum(r);
  return r;
}

// numerically stable log-sigmoid, the form ATen uses: min(x,0) - log1p(exp(-|x|))
__device__ __forceinline__ float log_sigmoid(float x) { return fminf(x, 0.f) - log1pf(expf(-fabsf(x))); }

__device__ __forceinline__ float silu(float x) { return x / (1.f + expf(-x)); }
// SFU version (ex2.approx + rcp.approx, ~2 ulp): used where SiLU sits on a latency-critical tail
__device__ __forceinline__ float silu_fast(float x) { return __fdividef(x, 1.f + __expf(-x)); }

// ---- packed fp32 pairs: sm_100 FFMA2 / FMUL2 / FADD2 (two IEEE fp32 results per instruction and lane) -------------
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpk2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 bc2(float x) { return pk2(x, x); }   // ptxas folds this into a scalar (broadcast) operand
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// x0*w0 + x1*w1 + x2*w2 + x3*w3 per half, contracted the way nvcc contracts the scalar expression
__device__ __forceinline__ f32x2 dot4_bc(const float (&x)[4], const float4& wa, const float4& wb) {
  f32x2 t = mul2(bc2(x[1]), pk2(wa.z, wa.w));
  t = fma2(bc2(x[0]), pk2(wa.x, wa.y), t);
  t = fma2(bc2(x[2]), pk2(wb.x, wb.y), t);
  return fma2(bc2(x[3]), pk2(wb.z, wb.w), t);
}

// streaming (evict-first) 128-bit accesses for the once-touched state stream
__device__ __forceinline__ float4 ld_stream(const float4* p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream(float4* p, const float4& v) { __stcs(p, v); }

// L2-coherent load (bypasses the non-coherent L1) for data written by other CTAs of the same launch
__device__ __forceinline__ float ld_cg(const float* p) { return __ldcg(p); }

__device__ __forceinline__ float bf16_bits_to_float(uint16_t b) { return __uint_as_float(((uint32_t)b) << 16); }

// torch.argmax of lg[0..n) by one warp (result valid in every lane): first index of the maximum; NaN counts as the
// maximum (first NaN wins). Used by the argmax action kernel and as the sampler's fallback, which must agree.
__device__ __forceinline__ int warp_argmax(const float* __restrict__ lg, int n, int lane) {
  float best = -INFINITY;
  int bi = 0x7fffffff;
  bool best_nan = false;
  for (int i = lane; i < n; i += 32) {
    const float v = lg[i];
    const bool vn = (v != v);
    bool take;
    if (best_nan) take = false;                       // earlier NaN in this lane wins (smaller index)
    else if (vn) take = true;
    else take = (bi == 0x7fffffff) || (v > best);
    if (take) { best = v; bi = i; best_nan = vn; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    const int on = __shfl_xor_sync(0xffffffffu, (int)best_nan, o);
    bool take;
    if (oi == 0x7fffffff) take = false;
    else if (bi == 0x7fffffff) take = true;
    else if (best_nan && on) take = oi < bi;
    else if (on) take = true;
    else if (best_nan) take = false;
    else take = (ov > best) || (ov == best && oi < bi);
    if (take) { best = ov; bi = oi; best_nan = (on != 0); }
  }
  return bi;
}

}  // namespace xl
