// Shared tcgen05 / TMEM / mbarrier helpers of the tensor-core convolution kernels (sm_100a).
#pragma once
#include "common.cuh"
#include <cuda_fp16.h>
#include <cuda.h>

// ---- host: cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*snb_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                        const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                        CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline snb_encode_tiled_fn snb_get_encode_tiled() {
  static snb_encode_tiled_fn fn = []() -> snb_encode_tiled_fn {       // thread-safe one-time lookup of a driver entry point
    void* p = nullptr;
    cudaDriverEntryPointQueryResult st;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &st) != cudaSuccess || st != cudaDriverEntryPointSuccess) return nullptr;
    return reinterpret_cast<snb_encode_tiled_fn>(p);
  }();
  return fn;
}


namespace tc {

constexpr int NSTAGE = 3;
constexpr int A_BYTES = 128 * 128;                       // one 128x32 fp32 operand image (hi or lo)
constexpr int B_BYTES = 96 * 128;                        // one 96x32 fp32 operand image (hi or lo)
constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;   // A_hi | A_lo | B_hi | B_lo = 56 KB (multiple of 1024)
constexpr int OUT_BYTES = 3 * 128 * 128;                  // Y0 | Y1 | Y2 staging tiles (128 x 32 fp32 each)
constexpr int NACC = 4;                                  // TMEM accumulator slots of 128 columns (96 used)
constexpr int NUM_LOADER_WARPS = 7;                      // 7 + 1 MMA + 8 epilogue = 16 warps = 4 per SMSP -> 128 regs/thread, no spills
constexpr int LROWS = (128 + NUM_LOADER_WARPS * 4 - 1) / (NUM_LOADER_WARPS * 4);   // tile rows per loader thread (5)
constexpr int LSTRIDE = NUM_LOADER_WARPS * 4;             // row stride between a loader thread's rows (28)
constexpr int NUM_EPI_WARPS = 8;                         // two per TMEM lane quadrant (16 of the 32 columns each)
constexpr int NTHREADS = (NUM_LOADER_WARPS + 1 + NUM_EPI_WARPS) * 32;
constexpr int SMEM_BYTES = NSTAGE * STAGE_BYTES + OUT_BYTES + 3072 /*barriers, misc*/ + 1024 /*alignment slack*/;
constexpr int WIMG_FLOATS_PER_WINDOW = 2 * B_BYTES / 4;  // hi + lo

// instruction descriptor, kind::tf32: D=f32 (bits 4-5 = 1), A=B=tf32 (bits 7-9 = 10-12 = 2), K-major A and B,
// N>>3 at bits 17-22, M>>4 at bits 24-28   (cute::UMMA::InstrDescriptor)
constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((96u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  // K-major, SWIZZLE_128B: start>>4 | LBO(16 B, unused)<<16 | SBO(1024 B = 8 rows x 128 B)<<32 | version 1<<46 | layout 2<<61
  return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}

// One elected lane of a CONVERGED warp.  The MMA-issuing warp runs its whole loop warp-uniformly (waits, descriptor math in
// the uniform datapath) and only the tcgen05 instruction itself is predicated on the elected lane: issuing from inside an
// `if (lane == 0)` region instead makes nvcc wrap every UTCHMMA in an ELECT/branch loop (~12 SASS instructions and
// 80+ cycles per MMA on the issuing thread — measured: the issue thread, not the tensor pipe, bounded the kernel).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  if (elect_one())
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accumulate) : "memory");
}
// A operand from TMEM (lanes = M rows, 8 consecutive 32-bit columns = K), B from shared memory
__device__ __forceinline__ void mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t accumulate) {
  if (elect_one())
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}\n" :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(IDESC), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  if (elect_one())
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// two 32-column loads in flight, one wait
__device__ __forceinline__ void tmem_ld32x2(uint32_t t0, uint32_t t1, float (&a)[32], float (&b)[32]) {
  uint32_t r[64];
#define SNB_LD32(OFF, ADDR) \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 " \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, " \
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n" \
      : "=r"(r[OFF+0]), "=r"(r[OFF+1]), "=r"(r[OFF+2]), "=r"(r[OFF+3]), "=r"(r[OFF+4]), "=r"(r[OFF+5]), "=r"(r[OFF+6]), "=r"(r[OFF+7]), \
        "=r"(r[OFF+8]), "=r"(r[OFF+9]), "=r"(r[OFF+10]), "=r"(r[OFF+11]), "=r"(r[OFF+12]), "=r"(r[OFF+13]), "=r"(r[OFF+14]), "=r"(r[OFF+15]), \
        "=r"(r[OFF+16]), "=r"(r[OFF+17]), "=r"(r[OFF+18]), "=r"(r[OFF+19]), "=r"(r[OFF+20]), "=r"(r[OFF+21]), "=r"(r[OFF+22]), "=r"(r[OFF+23]), \
        "=r"(r[OFF+24]), "=r"(r[OFF+25]), "=r"(r[OFF+26]), "=r"(r[OFF+27]), "=r"(r[OFF+28]), "=r"(r[OFF+29]), "=r"(r[OFF+30]), "=r"(r[OFF+31]) \
      : "r"(ADDR) : "memory")
  SNB_LD32(0, t0); SNB_LD32(32, t1);
#undef SNB_LD32
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) { a[i] = __uint_as_float(r[i]); b[i] = __uint_as_float(r[32 + i]); }
}

// registers -> TMEM: lane (32*quadrant + laneid) gets 32 consecutive 32-bit columns starting at taddr's column
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n"
      :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
         "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
         "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
         "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }
// registers -> TMEM, 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n"
      :: "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
         "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// Bounded mbarrier wait: a protocol bug traps (reported as a launch failure) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(40);                                 // back off: spinning warps must not steal issue slots from working ones
    if (clock64() - t0 > 4000000000ll) __trap();     // ~2 s at 1.9 GHz
  }
}
// latency-critical variant for the single MMA-issuing thread (no sleep)
__device__ __forceinline__ void mbar_wait_spin(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}
// Un-predicated variants for use INSIDE one `if (elect_one()) { ... }` block that issues a whole batch of MMAs + commits: one
// ELECT / divergence check per batch instead of one per instruction.
__device__ __forceinline__ void mma_tf32_ts_raw(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}\n" :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(IDESC), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_tf32_raw(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" :: "r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(IDESC), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mma_commit_raw(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" :: "r"(smem_u32(bar)) : "memory");
}

// ---- fp16-split operands (kind::f16, M128 N96 K16, fp32 accumulate): instruction descriptor with A = B = f16 (format 0),
// D = f32, K-major A and B.  The A operand sits in TMEM as packed pairs: 32-bit column j of lane m = {k = 2j (low half), 2j + 1}.
constexpr uint32_t IDESC_F16 = (1u << 4) | ((96u >> 3) << 17) | ((128u >> 4) << 24);
__device__ __forceinline__ void mma_f16_ts_raw(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(IDESC_F16), "r"(accumulate) : "memory");
}
// Float index (from the start of a weight image) of the spare slot that carries 2^-s, the inverse of the power-of-two scale the
// fp16-split weights were multiplied with: image Q (second 12 KB block of window 0), row 0, logical 16-B chunk 4 (never an operand).
constexpr int WIMG_SCALE_SLOT = B_BYTES / 4 + 16;
// {lo, hi} -> packed f16x2 (lo in the low half), round to nearest, saturating to +-65504 instead of overflowing to inf
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ float2 unpack_f16x2(uint32_t v) {
  return __half22float2(*reinterpret_cast<const __half2*>(&v));
}
// 32 fp32 channels of one position -> 16 packed xh words | 16 packed xl' words, xh = fp16(x), xl' = fp16((x - xh) * 2^11)
__device__ __forceinline__ void split_f16(const float4 (&v)[8], uint32_t (&hl)[32]) {
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const uint32_t h0 = pack_f16x2(v[c].x, v[c].y), h1 = pack_f16x2(v[c].z, v[c].w);
    const float2 f0 = unpack_f16x2(h0), f1 = unpack_f16x2(h1);
    hl[2 * c] = h0; hl[2 * c + 1] = h1;
    hl[16 + 2 * c] = pack_f16x2((v[c].x - f0.x) * 2048.f, (v[c].y - f0.y) * 2048.f);
    hl[16 + 2 * c + 1] = pack_f16x2((v[c].z - f1.x) * 2048.f, (v[c].w - f1.y) * 2048.f);
  }
}
// 32 fp32 channels of one position -> the 16 packed xh words only (single-product operands: no xl')
__device__ __forceinline__ void hi_f16(const float4 (&v)[8], uint32_t (&h)[16]) {
#pragma unroll
  for (int c = 0; c < 8; ++c) { h[2 * c] = pack_f16x2(v[c].x, v[c].y); h[2 * c + 1] = pack_f16x2(v[c].z, v[c].w); }
}

// mbarrier.arrive that is data-dependent on `dep`: the arrive cannot ISSUE before the instructions that produced `dep` have
// their operands, i.e. before the shared-memory loads feeding them have returned.  A consumer that releases a TMA-filled smem
// slot right after issuing its LDS instructions (values "in registers" only once they arrive) lets the producer's next TMA
// write race the loads still in flight — seen as rare, large errors in back-to-back launches of the 2-D kernel.
__device__ __forceinline__ void mbar_arrive_after(uint64_t* bar, uint32_t dep) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %1, 0x7fc12345;\n@p mbarrier.arrive.shared::cta.b64 _, [%0];\n"
               "@!p mbarrier.arrive.shared::cta.b64 _, [%0];\n}\n" :: "r"(smem_u32(bar)), "r"(dep) : "memory");
}
__device__ __forceinline__ uint32_t xor_all(const float4 (&v)[8]) {
  uint32_t x = 0;
#pragma unroll
  for (int c = 0; c < 8; ++c)
    x ^= __float_as_uint(v[c].x) ^ __float_as_uint(v[c].y) ^ __float_as_uint(v[c].z) ^ __float_as_uint(v[c].w);
  return x;
}

// M128 N32 K8 variant (small-Cin im2col convolutions, 32->1 tap contractions), A from TMEM; call inside one elected region
constexpr uint32_t IDESC_N32 = (1u << 4) | (2u << 7) | (2u << 10) | ((32u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ void mma_n32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}\n" :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(IDESC_N32), "r"(accumulate) : "memory");
}

// Warp-uniform wait for the CONVERGED MMA-issuing warp: every lane polls and the loop exits on a warp vote, so the loop
// is provably non-divergent and nvcc keeps the loop-carried state (stage counters, smem/TMEM addresses, descriptors) in
// the uniform datapath — with a per-lane exit condition they live in vector registers and every tcgen05.mma pays
// R2UR / VOTEU / ELECT round trips (~13 SASS instructions, ~80 cycles per MMA on the issuing warp, measured).
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity) {
  if (__all_sync(0xffffffffu, mbar_try_wait(bar, parity))) return;
  const long long t0 = clock64();
  while (!__all_sync(0xffffffffu, mbar_try_wait(bar, parity))) {
    __nanosleep(20);                                 // a spinning warp must not take issue slots from the epilogue warps it waits for
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}
// three 16-column TMEM loads in flight, one wait
__device__ __forceinline__ void tmem_ld16x3(uint32_t t0, uint32_t t1, uint32_t t2, float (&a)[16], float (&b)[16], float (&c)[16]) {
  uint32_t r[48];
#define SNB_LD16(ARR, OFF, ADDR) \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n" \
      : "=r"(ARR[OFF+0]), "=r"(ARR[OFF+1]), "=r"(ARR[OFF+2]), "=r"(ARR[OFF+3]), "=r"(ARR[OFF+4]), "=r"(ARR[OFF+5]), "=r"(ARR[OFF+6]), "=r"(ARR[OFF+7]), \
        "=r"(ARR[OFF+8]), "=r"(ARR[OFF+9]), "=r"(ARR[OFF+10]), "=r"(ARR[OFF+11]), "=r"(ARR[OFF+12]), "=r"(ARR[OFF+13]), "=r"(ARR[OFF+14]), "=r"(ARR[OFF+15]) \
      : "r"(ADDR) : "memory")
  SNB_LD16(r, 0, t0); SNB_LD16(r, 16, t1); SNB_LD16(r, 32, t2);
#undef SNB_LD16
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) { a[i] = __uint_as_float(r[i]); b[i] = __uint_as_float(r[16 + i]); c[i] = __uint_as_float(r[32 + i]); }
}

template <bool PROF>
__device__ __forceinline__ long long mbar_wait_timed(uint64_t* bar, uint32_t parity) {
  if (!PROF) { mbar_wait(bar, parity); return 0; }
  const long long t0 = clock64();
  mbar_wait(bar, parity);
  return clock64() - t0;
}
template <bool PROF> __device__ __forceinline__ long long prof_clock() { return PROF ? clock64() : 0; }

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, 256;\n" ::: "memory"); }


__device__ __forceinline__ int floordiv(int a, int b) { int q = a / b; return (a % b < 0) ? q - 1 : q; }

// 3xTF32 operand split: hi = x rounded to nearest TF32 (11-bit significand; ties away from zero, done on the bit pattern),
// lo = x - hi (exact in fp32, |lo| <= 2^-12 |x|; the tensor core reads its top 19 bits).  Rounding instead of truncating hi
// halves |lo|, so both the dropped lo*lo term and the truncation of lo are 4x smaller (~2^-22 relative per product).
__device__ __forceinline__ uint32_t tf32_hi_bits(float x) { return (__float_as_uint(x) + 0x1000u) & 0xffffe000u; }
__device__ __forceinline__ void split_tf32(const float4& x, float4& hi, float4& lo) {
  hi.x = __uint_as_float(tf32_hi_bits(x.x));
  hi.y = __uint_as_float(tf32_hi_bits(x.y));
  hi.z = __uint_as_float(tf32_hi_bits(x.z));
  hi.w = __uint_as_float(tf32_hi_bits(x.w));
  lo = make_float4(x.x - hi.x, x.y - hi.y, x.z - hi.z, x.w - hi.w);
}

}  // namespace tc
