// Shared device/host helpers for libsnb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/snb200.h"

#define SNB_LRELU_SLOPE 0.2f

// ---- error reporting (thread-local, no global mutable state shared between host threads)
int snb_fail(const char* fmt, ...);
#define SNB_REQUIRE(cond, ...) do { if (!(cond)) return snb_fail(__VA_ARGS__); } while (0)
#define SNB_LAUNCH_CHECK(name) do { cudaError_t _e = cudaGetLastError(); \
  if (_e != cudaSuccess) return snb_fail("%s: %s", name, cudaGetErrorString(_e)); } while (0)
#define SNB_CUDA(call) do { cudaError_t _e = (call); \
  if (_e != cudaSuccess) return snb_fail("%s: %s", #call, cudaGetErrorString(_e)); } while (0)

// ---- programmatic dependent launch (PDL).  Every kernel of the library is launched with the programmatic-stream-
// serialization attribute and starts with pdl_launch() (lets the NEXT kernel's CTAs be scheduled as soon as all CTAs of this
// one have started and SM resources free up) followed — before it touches any global memory — by pdl_wait() (blocks until the
// PREVIOUS kernel has completed and its writes are visible).  Correctness is the plain stream order; what is gained is the
// launch latency / ramp-up of kernel N+1 overlapping the tail of kernel N (34 dependent launches per forward, ~390 per
// adaptation step).  SNB200_PDL=0 launches without the attribute (both instructions are then no-ops).
bool snb_pdl_enabled();
template <class... KA, class... A>
static inline void snb_launch(void (*kern)(KA...), dim3 grid, dim3 block, size_t smem, void* stream, A&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = snb_pdl_enabled() ? 1 : 0;
  (void)cudaLaunchKernelEx(&cfg, kern, static_cast<KA>(args)...);     // errors are picked up by SNB_LAUNCH_CHECK
}
// same, as clusters of two CTAs (tcgen05 cta_group::2 kernels); grid.x must be even
template <class... KA, class... A>
static inline void snb_launch_cluster2(void (*kern)(KA...), dim3 grid, dim3 block, size_t smem, void* stream, A&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = snb_pdl_enabled() ? 2 : 1;
  (void)cudaLaunchKernelEx(&cfg, kern, static_cast<KA>(args)...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }
#endif

static inline int snb_ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---- one entry of the batched weight preparation with the table passed by value (conv_c32_tc.cu; used by the whole-model
// prepare of model.cu).  cfg = nwin | mode << 8 | kind << 16 | a << 24 | b << 28 as in snb_prep_conv_weights_tc_batch, plus
// kind 3 (C4 image), 4 (eval-mode BatchNorm fold: aux = {beta, running_mean, running_var}), 5 (copy of `count` floats) and 6
// (flipped disparity-channel taps of the refinement input layer, used by the adaptation step's backward).
struct snb_prep_item { const float* src; const float* aux[3]; float* out; int cfg; int count; };
int snb_prep_param_launch(const snb_prep_item* items, int n, void* stream);

// ---- small device helpers
__device__ __forceinline__ float lrelu(float v) { return v > 0.f ? v : SNB_LRELU_SLOPE * v; }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 16-byte cp.async with zero fill when !valid (src-size 0). `src` must be a valid address either way.
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, bool valid) {
  uint32_t d = smem_u32(smem_dst);
  int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" :: "r"(d), "l"(gsrc), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" :: "n"(N) : "memory"); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// PyTorch upsample_bilinear2d source index, align_corners=False (area_pixel_compute_source_index, cubic=false).
__device__ __forceinline__ void bilinear_src(int dst, float scale, int in_size, int& i0, int& i1, float& l1) {
  float s = scale * (dst + 0.5f) - 0.5f;
  s = s < 0.f ? 0.f : s;
  i0 = (int)s;
  if (i0 > in_size - 1) i0 = in_size - 1;
  i1 = i0 + ((i0 < in_size - 1) ? 1 : 0);
  l1 = s - (float)i0;
}

__device__ __forceinline__ float bilinear_sample(const float* __restrict__ p, int h, int w, int y, int x, float sh, float sw) {
  int y0, y1, x0, x1; float ly, lx;
  bilinear_src(y, sh, h, y0, y1, ly);
  bilinear_src(x, sw, w, x0, x1, lx);
  float hy = 1.f - ly, hx = 1.f - lx;
  return hy * (hx * p[y0 * w + x0] + lx * p[y0 * w + x1]) + ly * (hx * p[y1 * w + x0] + lx * p[y1 * w + x1]);
}

// ---- packed fp32 FMA (Blackwell FFMA2: two fp32 FMAs per instruction, same rounding as two scalar fmaf)
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  return (unsigned long long)__float_as_uint(lo) | ((unsigned long long)__float_as_uint(hi) << 32);
}
__device__ __forceinline__ float lo2(unsigned long long v) { return __uint_as_float((unsigned)(v & 0xffffffffull)); }
__device__ __forceinline__ float hi2(unsigned long long v) { return __uint_as_float((unsigned)(v >> 32)); }
__device__ __forceinline__ void ffma2(unsigned long long& acc, unsigned long long a, unsigned long long b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}

// ---- mbarrier / TMA bulk-copy helpers (Hopper+/Blackwell async proxy)
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded: a protocol bug (e.g. a byte count that never completes) traps and surfaces as a launch failure instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000ll) __trap();     // ~2 s at 1.9 GHz
  }
}
// 1-D TMA bulk copy global -> shared, completing `bytes` on the mbarrier (bytes % 16 == 0, 16-B aligned).
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
               :: "r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
