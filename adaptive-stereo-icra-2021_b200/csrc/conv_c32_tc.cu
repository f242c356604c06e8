// 32->32 stride-1 3x3 (dilated, 2-D) / 3x3x3 (3-D) convolution as an implicit GEMM on the 5th-gen tensor cores.
// Replaces the nn.Conv3d cost-filter layers (stereo_net.py:155-160,185-186) and the nn.Conv2d of every BasicBlock
// (stereo_net.py:37-39,44-51; feature extractor :73-77 and refinement :96-100), incl. folded BN, LeakyReLU, residual.
//
// GEMM view (per (b,d) slice, "flat padded" pixel index q = h*P + w with pitch P = W + dil, columns >= W read as zero):
//   M tile  = 128 consecutive q               (TMEM lanes)
//   K       = (kd,kh) windows x 32 cin        (one window = one pipeline stage: A tile 128 x 32 fp32 = 16 KB)
//   N       = 96 = 3 kw x 32 cout             (kw is folded into N: the three kw taps share one un-shifted A window, so
//                                              the 128x32 A tile is read from smem once per window, not three times —
//                                              with N = 32 the MMA would be bound by the A-operand smem feed)
//   Y_kw[m] accumulates in TMEM (3 x 32 fp32 columns); the epilogue forms out[m] = Y0[m-dil] + Y1[m] + Y2[m+dil] in
//   smem, so a tile yields 128 - 2*dil output positions (tiles overlap by 2*dil rows).
// Operands are TF32 (tcgen05.mma.kind::tf32, fp32 accumulate in TMEM).  passes = 3 runs the error-compensated split
//   x*w ~= xh*wh + xl*wh + xh*wl   (xh = top 19 bits, xl = x - xh)  -> ~2^-21 relative, i.e. fp32-grade results;
// passes = 1 is plain single-pass TF32 (reported separately, north star).
//
// Warp roles (512 threads = 4 warps per SM sub-partition -> 128 registers/thread; 1 CTA/SM, persistent over tiles):
//   warps 0-6  loaders : LDG.128 channels-last rows -> hi/lo split -> STS into the SWIZZLE_128B K-major A image,
//                        zero rows for padding; warp 0 also issues the TMA bulk copy of the window's B image (3-D)
//   warp  7    MMA     : one elected thread issues tcgen05.mma (M128 N96 K8) and tcgen05.commit on the mbarriers
//   warps 8-15 epilogue: tcgen05.ld TMEM -> smem (Y0|Y1|Y2) -> shift-add + bias/BN/LeakyReLU/residual/stats -> coalesced STG
#include "tc_common.cuh"

namespace tc {

struct Params {
  const float* x; const float* wimg; float* y;
  int B, D, H, W;          // stride-1 "same" conv: output dims = input dims
  int nwin;                // 3 (2-D: kh) or 9 (3-D: kd,kh)
  int dil, P;              // dilation, flat pitch W + dil
  int tiles_per_slice, ntiles, step;   // step = 128 - 2*dil output positions per tile
  int passes;              // 1 or 3
  snb_conv_epilogue e;
  long long* dbg;          // optional [grid][8] cycle counters (diagnostics), or NULL
};


// PROF = true adds clock64() timers around every wait (snb_conv_c32_tc_profile); the product path is PROF = false.
template <bool PROF>
__global__ void __launch_bounds__(NTHREADS, 1)
conv_c32_tc_kernel(const Params p) {
  extern __shared__ unsigned char smem_dyn[];
  const uint32_t base_u32 = (smem_u32(smem_dyn) + 1023u) & ~1023u;
  unsigned char* base = smem_dyn + (base_u32 - smem_u32(smem_dyn));
  unsigned char* sOutB = base + NSTAGE * STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sOutB + OUT_BYTES);
  uint64_t* full = bars;                 // [NSTAGE]  loaders (+TMA bytes) -> MMA
  uint64_t* empty = bars + NSTAGE;       // [NSTAGE]  MMA commit -> loaders
  uint64_t* tfull = bars + 2 * NSTAGE;   // [NACC]    MMA commit -> epilogue
  uint64_t* tempty = tfull + NACC;       // [NACC]    epilogue -> MMA
  uint64_t* wbar = tempty + NACC;        // resident-weights barrier (2-D)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wbar + 1);
  float* sRed = reinterpret_cast<float*>(tmem_slot + 2);   // [8 warps][64]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool stream_b = p.nwin > NSTAGE;       // 3-D: weights do not fit next to the A ring -> streamed per window

  if (warp == NUM_LOADER_WARPS) {
    if (lane == 0) {
      for (int i = 0; i < NSTAGE; ++i) { mbar_init(&full[i], NUM_LOADER_WARPS + 1); mbar_init(&empty[i], 1); }
      for (int i = 0; i < NACC; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], NUM_EPI_WARPS); }
      mbar_init(wbar, 1);
      mbar_fence_init();
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" :: "r"(smem_u32(tmem_slot)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch();                                    // dependents only once this CTA owns its TMEM columns (no alloc dead-lock with an early dependent)
  pdl_wait();                                      // everything above touched no global memory

  if (warp < NUM_LOADER_WARPS) {
    // =============================================================== loaders
    // Software-pipelined: the global loads of window i+PF are in flight (registers) while window i is split and
    // stored to smem, so a loader thread never sits out a full L2/HBM round trip per window.
    constexpr int PF = 3;
    const int chunk = tid & 7, rgrp = tid >> 3;            // 8 lanes cover one 128-B row; rows rgrp + LSTRIDE*j (< 128)
    const int my_tiles = (p.ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int n_items = my_tiles * p.nwin;                 // item = (tile, window)
    // ---- load cursor state
    int l_item = 0, l_widx = 0, l_b = 0, l_d = 0;
    int l_tile = blockIdx.x;
    int h0[LROWS], w0[LROWS];
    auto decode_tile = [&]() {
      const int slice = l_tile / p.tiles_per_slice, tt = l_tile - slice * p.tiles_per_slice;
      l_b = slice / p.D; l_d = slice - l_b * p.D;
      const int q = tt * p.step - p.dil + rgrp;
      int h = floordiv(q, p.P), w = q - h * p.P;
#pragma unroll
      for (int j = 0; j < LROWS; ++j) {  // rows rgrp + LSTRIDE*j: one division per tile, then increments
        h0[j] = h; w0[j] = w;
        w += LSTRIDE;
        while (w >= p.P) { w -= p.P; ++h; }
      }
    };
    auto issue_loads = [&](float4 (&v)[LROWS]) {
      if (l_widx == 0) decode_tile();
      const int kd = (p.nwin == 9) ? l_widx / 3 : 0, kh = l_widx - kd * 3;
      const int di = (p.nwin == 9) ? l_d + kd - 1 : l_d;
      const bool slice_ok = (unsigned)di < (unsigned)p.D;
#pragma unroll
      for (int j = 0; j < LROWS; ++j) {
        const int h = h0[j] + (kh - 1) * p.dil;
        const bool ok = slice_ok && rgrp + LSTRIDE * j < 128 && w0[j] < p.W && (unsigned)h < (unsigned)p.H;
        v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (ok) v[j] = __ldcg(reinterpret_cast<const float4*>(
                       p.x + ((((size_t)l_b * p.D + di) * p.H + h) * p.W + w0[j]) * 32 + chunk * 4));
      }
      ++l_item;
      if (++l_widx == p.nwin) { l_widx = 0; l_tile += gridDim.x; }
    };
    float4 v[PF][LROWS];
#pragma unroll
    for (int k = 0; k < PF; ++k)
      if (l_item < n_items) issue_loads(v[k]);

    uint32_t stage = 0, phase = 0;
    int s_widx = 0;
    long long t_wait = 0; const long long t_begin = prof_clock<PROF>();
    for (int item0 = 0; item0 < n_items; item0 += PF) {
#pragma unroll
      for (int k = 0; k < PF; ++k) {
        if (item0 + k >= n_items) break;
        unsigned char* st = base + stage * STAGE_BYTES;
        t_wait += mbar_wait_timed<PROF>(&empty[stage], phase ^ 1);
        if (tid == 0) {
          if (stream_b) {
            mbar_expect_tx(&full[stage], 2 * B_BYTES);
            bulk_g2s(st + 2 * A_BYTES, p.wimg + (size_t)s_widx * WIMG_FLOATS_PER_WINDOW, 2 * B_BYTES, &full[stage]);
          } else {
            mbar_arrive(&full[stage]);
          }
        }
#pragma unroll
        for (int j = 0; j < LROWS; ++j) {
          const int r = rgrp + LSTRIDE * j;
          if (r < 128) {
            const uint32_t off = r * 128 + ((chunk ^ (r & 7)) << 4);
            float4 hi, lo;
            split_tf32(v[k][j], hi, lo);
            *reinterpret_cast<float4*>(st + off) = hi;
            if (p.passes == 3) *reinterpret_cast<float4*>(st + A_BYTES + off) = lo;
          }
        }
        fence_async_smem();            // generic-proxy smem writes -> visible to the tensor-core (async) proxy
        __syncwarp();
        if (lane == 0) mbar_arrive(&full[stage]);
        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
        if (++s_widx == p.nwin) s_widx = 0;
        if (l_item < n_items) issue_loads(v[k]);   // refill this register slot with window item+PF
      }
    }
    if (PROF && p.dbg && tid == 0) { p.dbg[blockIdx.x * 16 + 0] = t_wait; p.dbg[blockIdx.x * 16 + 1] = prof_clock<PROF>() - t_begin; }
  } else if (warp == NUM_LOADER_WARPS) {
    // =============================================================== MMA issuer (converged warp, elected lane)
    {
      if (!stream_b) {       // 2-D: window kh always lands in stage kh -> keep its B image resident there
        if (lane == 0) {
          mbar_expect_tx(wbar, (uint32_t)p.nwin * 2 * B_BYTES);
          for (int w = 0; w < p.nwin; ++w)
            bulk_g2s(base + w * STAGE_BYTES + 2 * A_BYTES, p.wimg + (size_t)w * WIMG_FLOATS_PER_WINDOW, 2 * B_BYTES, wbar);
        }
        __syncwarp();
        mbar_wait_spin(wbar, 0);
      }
      uint32_t stage = 0, phase = 0;
      int it = 0;
      long long t_full = 0, t_tempty = 0; const long long t_begin = prof_clock<PROF>();
      for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++it) {
        const int acc = it & (NACC - 1);
        const uint32_t accphase = (it / NACC) & 1;
        t_tempty += mbar_wait_timed<PROF>(&tempty[acc], accphase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + acc * 128;
        for (int widx = 0; widx < p.nwin; ++widx) {
          t_full += mbar_wait_timed<PROF>(&full[stage], phase);
          tc_fence_after();
          const uint32_t sa = base_u32 + stage * STAGE_BYTES;
          const uint32_t sb = sa + 2 * A_BYTES;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {           // K = 8 tf32 = 32 bytes per MMA
            const uint64_t ah = make_desc(sa + ks * 32), bh = make_desc(sb + ks * 32);
            mma_tf32(tmem_d, ah, bh, (widx | ks) != 0);
            if (p.passes == 3) {
              mma_tf32(tmem_d, make_desc(sa + A_BYTES + ks * 32), bh, 1);
              mma_tf32(tmem_d, ah, make_desc(sb + B_BYTES + ks * 32), 1);
            }
          }
          mma_commit(&empty[stage]);                 // smem slot reusable once these MMAs have read it
          if (widx == p.nwin - 1) mma_commit(&tfull[acc]);
          if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
        }
      }
      if (PROF && p.dbg && lane == 0) { p.dbg[blockIdx.x * 16 + 2] = t_full; p.dbg[blockIdx.x * 16 + 3] = t_tempty; p.dbg[blockIdx.x * 16 + 4] = prof_clock<PROF>() - t_begin; }
    }
    __syncwarp();
  } else {
    // =============================================================== epilogue (8 warps; TMEM lane quadrant = warp % 4)
    // Step 1: TMEM -> smem, the three kw partials Y0|Y1|Y2 as separate 128x32 tiles (row = TMEM lane, 16-B chunks
    //         XOR-swizzled).  Step 2 (after one barrier): every thread owns one 16-B chunk of 4 rows and forms
    //         out[r] = Y0[r-dil] + Y1[r] + Y2[r+dil] + bias -> stats -> BN scale/shift -> LeakyReLU -> + residual -> STG,
    //         8 lanes per 128-B position so global traffic is fully coalesced.
    const int ew = warp - (NUM_LOADER_WARPS + 1);    // 0..7
    const int quad = warp & 3;
    const int half = ew >> 2;                        // which 16 of the 32 output channels this warp moves out of TMEM
    const int m = quad * 32 + lane;                  // TMEM lane == tile row
    const int et = tid - (NUM_LOADER_WARPS + 1) * 32;
    const int chunk = et & 7, rg = et >> 3;          // step 2: rows rg + 32*j, 16-B chunk `chunk`
    float* sY = reinterpret_cast<float*>(sOutB);
    const snb_conv_epilogue& e = p.e;
    const bool has_res = e.residual != nullptr, has_stats = e.stats != nullptr;
    float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f), sc4 = make_float4(1.f, 1.f, 1.f, 1.f), sh4 = bias4;
    if (e.bias) bias4 = reinterpret_cast<const float4*>(e.bias)[chunk];
    if (e.scale) { sc4 = reinterpret_cast<const float4*>(e.scale)[chunk]; sh4 = reinterpret_cast<const float4*>(e.shift)[chunk]; }
    int it = 0;
    long long t_tfull = 0, t_bar = 0, t_pre = 0, t_tmem = 0, t_out = 0; const long long t_begin = prof_clock<PROF>();
    for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, ++it) {
      const int acc = it & (NACC - 1);
      const uint32_t accphase = (it / NACC) & 1;
      const int slice = tile / p.tiles_per_slice, tt = tile - slice * p.tiles_per_slice;
      const int q0 = tt * p.step - p.dil;
      const long long tA = prof_clock<PROF>();
      // coordinates of this thread's 4 output rows (one division per tile, then increments)
      int hh[4], ww[4]; bool okr[4];
      {
        int q = q0 + rg;
        int h = floordiv(q, p.P), w = q - h * p.P;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = rg + 32 * j;
          hh[j] = h; ww[j] = w;
          okr[j] = r >= p.dil && r < 128 - p.dil && h >= 0 && h < p.H && w < p.W;
          w += 32;
          while (w >= p.P) { w -= p.P; ++h; }
        }
      }
      // residual rows do not depend on the MMA: put their loads in flight before waiting on TMEM
      float4 res[4];
      if (has_res) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          res[j] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (okr[j]) res[j] = __ldcg(reinterpret_cast<const float4*>(
                               e.residual + (((size_t)slice * p.H + hh[j]) * p.W + ww[j]) * 32 + chunk * 4));
        }
      }
      t_pre += prof_clock<PROF>() - tA;
      t_tfull += mbar_wait_timed<PROF>(&tfull[acc], accphase);
      tc_fence_after();
      const long long tB = prof_clock<PROF>();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * 128 + half * 16;
      {
        float v0[16], v1[16], v2[16];
        tmem_ld16x3(taddr, taddr + 32, taddr + 64, v0, v1, v2);
        float* row = sY + m * 32;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int o = ((half * 4 + c) ^ (m & 7)) << 2;
          *reinterpret_cast<float4*>(row + o) = make_float4(v0[4 * c], v0[4 * c + 1], v0[4 * c + 2], v0[4 * c + 3]);
          *reinterpret_cast<float4*>(row + 128 * 32 + o) = make_float4(v1[4 * c], v1[4 * c + 1], v1[4 * c + 2], v1[4 * c + 3]);
          *reinterpret_cast<float4*>(row + 2 * 128 * 32 + o) = make_float4(v2[4 * c], v2[4 * c + 1], v2[4 * c + 2], v2[4 * c + 3]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[acc]);      // this warp is done with the TMEM slot
      t_tmem += prof_clock<PROF>() - tB;
      { const long long tb = prof_clock<PROF>(); epi_bar(); t_bar += prof_clock<PROF>() - tb; }
      const long long tC = prof_clock<PROF>();
      float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < 4; ++j) {       // branch-free: out-of-range rows read clamped smem rows and skip only the store
        const int r = rg + 32 * j;
        const int r0 = max(r - p.dil, 0), r2 = min(r + p.dil, 127);    // kw=0 reads input w-dil: Y0[r-dil]; kw=2: Y2[r+dil]
        const float4 a = *reinterpret_cast<const float4*>(sY + r0 * 32 + ((chunk ^ (r0 & 7)) << 2));
        const float4 b = *reinterpret_cast<const float4*>(sY + 128 * 32 + r * 32 + ((chunk ^ (r & 7)) << 2));
        const float4 c = *reinterpret_cast<const float4*>(sY + 2 * 128 * 32 + r2 * 32 + ((chunk ^ (r2 & 7)) << 2));
        float4 o;
        o.x = (a.x + b.x) + c.x + bias4.x; o.y = (a.y + b.y) + c.y + bias4.y;
        o.z = (a.z + b.z) + c.z + bias4.z; o.w = (a.w + b.w) + c.w + bias4.w;
        if (has_stats && okr[j]) {
          s1[0] += o.x; s1[1] += o.y; s1[2] += o.z; s1[3] += o.w;
          s2[0] = fmaf(o.x, o.x, s2[0]); s2[1] = fmaf(o.y, o.y, s2[1]); s2[2] = fmaf(o.z, o.z, s2[2]); s2[3] = fmaf(o.w, o.w, s2[3]);
        }
        if (e.scale) { o.x = fmaf(o.x, sc4.x, sh4.x); o.y = fmaf(o.y, sc4.y, sh4.y); o.z = fmaf(o.z, sc4.z, sh4.z); o.w = fmaf(o.w, sc4.w, sh4.w); }
        if (e.lrelu) { o.x = lrelu(o.x); o.y = lrelu(o.y); o.z = lrelu(o.z); o.w = lrelu(o.w); }
        if (has_res) { o.x += res[j].x; o.y += res[j].y; o.z += res[j].z; o.w += res[j].w; }
        if (okr[j]) __stcg(reinterpret_cast<float4*>(p.y + (((size_t)slice * p.H + hh[j]) * p.W + ww[j]) * 32 + chunk * 4), o);
      }
      if (has_stats) {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          s1[c] += __shfl_xor_sync(0xffffffffu, s1[c], 8); s1[c] += __shfl_xor_sync(0xffffffffu, s1[c], 16);
          s2[c] += __shfl_xor_sync(0xffffffffu, s2[c], 8); s2[c] += __shfl_xor_sync(0xffffffffu, s2[c], 16);
        }
        if (lane < 8) {
#pragma unroll
          for (int c = 0; c < 4; ++c) { sRed[ew * 64 + lane * 4 + c] = s1[c]; sRed[ew * 64 + 32 + lane * 4 + c] = s2[c]; }
        }
        epi_bar();
        if (et < 64) {
          float a = 0.f;
#pragma unroll
          for (int wq = 0; wq < NUM_EPI_WARPS; ++wq) a += sRed[wq * 64 + et];
          e.stats[(size_t)tile * 64 + et] = a;
        }
      }
      t_out += prof_clock<PROF>() - tC;
      { const long long tb = prof_clock<PROF>(); epi_bar(); t_bar += prof_clock<PROF>() - tb; }     // sY / sRed are rewritten by the next tile
    }
    if (PROF && p.dbg && et == 0) { p.dbg[blockIdx.x * 16 + 5] = t_tfull; p.dbg[blockIdx.x * 16 + 6] = prof_clock<PROF>() - t_begin; p.dbg[blockIdx.x * 16 + 7] = t_bar; p.dbg[blockIdx.x * 16 + 8] = t_pre; p.dbg[blockIdx.x * 16 + 9] = t_tmem; p.dbg[blockIdx.x * 16 + 10] = t_out; }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == NUM_LOADER_WARPS) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" :: "r"(tmem_base) : "memory");
  }
}

// ---- fp16-split weight image (SNB_CONV_F16).  Per (kd,kh) window two 12 KB blocks of 96 rows x 128 B, SWIZZLE_128B K-major:
//   P: row n = [wh(n, cin 0..31) 64 B | wl(n, cin 0..31) 64 B]      Q: row n = [2^-11 wh 64 B | unused]
// with w' = w * 2^s, wh = fp16(w'), wl = fp16(w' - wh).  2^-s sits in the spare slot WIMG_SCALE_SLOT of the image (written by
// weight_scale_kernel, which must run before the prep kernel on the same stream).
__device__ __forceinline__ void store_f16_split(float* __restrict__ out, int win, int n, int k, float v, float scale) {
  const float vs = v * scale;
  const __half wh = __float2half_rn(vs);
  const float whf = __half2float(wh);
  const __half wl = __float2half_rn(vs - whf);
  const __half whs = __float2half_rn(whf * (1.f / 2048.f));
  __half* img = reinterpret_cast<__half*>(out + (size_t)win * WIMG_FLOATS_PER_WINDOW);
  const int sw = n & 7;
  img[n * 64 + ((((k >> 3)) ^ sw) << 3) + (k & 7)] = wh;                       // logical 16-B chunks 0..3
  img[n * 64 + ((((k >> 3) + 4) ^ sw) << 3) + (k & 7)] = wl;                   // logical chunks 4..7
  img[B_BYTES / 2 + n * 64 + ((((k >> 3)) ^ sw) << 3) + (k & 7)] = whs;
  if (win != 0 || n != 0 || k >= 2)                                            // the other half of Q is never an operand; keep it
    img[B_BYTES / 2 + n * 64 + ((((k >> 3) + 4) ^ sw) << 3) + (k & 7)] = __float2half_rn(0.f);   // defined (halfs 32,33 of row 0 = the 2^-s slot)
}

// ---- weight images of conv_c32_ws.cu (SNB_CONV_WS): one image per (window, kw), rows = [kz = 2 | kz = 1 | kz = 0] x 32 cout, where
// kz is the kernel axis the CTA walks along (2-D: kh, one window; 3-D: kd, window = kh).  2-D image = P [wh | wl] + Q [2^-11 wh | -]
// (24 KB, 2^-s in the same spare slot as above); 3-D image = [wh | wl''] with wl'' = 2^11 (w' - wh) (12 KB; 2^-s after the 9 images).
__device__ __forceinline__ void store_ws_split(float* __restrict__ out, bool d3, int win, int n, int k, float v, float scale) {
  const int kw = n >> 5, co = n & 31;
  const float vs = v * scale;
  const __half wh = __float2half_rn(vs);
  const float whf = __half2float(wh);
  const int sw = co & 7;                                  // row = blk * 32 + co: row & 7 == co & 7
  const int c0 = ((((k >> 3)) ^ sw) << 3) + (k & 7), c1 = ((((k >> 3) + 4) ^ sw) << 3) + (k & 7);
  if (d3) {
    const int kd = win / 3, kh = win - kd * 3;
    __half* img = reinterpret_cast<__half*>(out) + (size_t)(kh * 3 + kw) * (B_BYTES / 2);
    const int row = (2 - kd) * 32 + co;
    img[row * 64 + c0] = wh;
    img[row * 64 + c1] = __float2half_rn((vs - whf) * 2048.f);
  } else {
    __half* img = reinterpret_cast<__half*>(out) + (size_t)kw * B_BYTES;        // 24 KB per image = B_BYTES halfs
    const int row = (2 - win) * 32 + co;
    img[row * 64 + c0] = wh;
    img[row * 64 + c1] = __float2half_rn(vs - whf);
    img[B_BYTES / 2 + row * 64 + c0] = __float2half_rn(whf * (1.f / 2048.f));
    if (kw != 0 || row != 0 || k >= 2) img[B_BYTES / 2 + row * 64 + c1] = __float2half_rn(0.f);
  }
}
__device__ __forceinline__ int scale_slot_of(int mode_bits, int nwin) {
  return ((mode_bits & SNB_CONV_WS) && nwin >= 9) ? nwin * (B_BYTES / 4) : WIMG_SCALE_SLOT;      // nwin 9: 3-D set, 10: the P4 set below
}

// ---- the ten-image set of a 5x5 stride-2 layer for conv_c32_ws.cu MODE_P4 (forward only): phase (a,b) = window a*2+b contributes
// the images kw' = 0..(b ? 1 : 2) (first image 0 / 3 / 5 / 8), each 12 KB [wh | wl''] with rows [kz' = 2 | 1 | 0] x 32 cout holding
// w[cout][cin][2 kz' + a][2 kw' + b] (zero past the 5x5 support); ONE scale 2^-s for the whole layer after the ten images.
__device__ __forceinline__ void store_p4_images(const float* __restrict__ w, float* __restrict__ out, float scale, int first, int step) {
  for (int i = first; i < 10 * 96 * 32; i += step) {
    const int k = i & 31, row = (i >> 5) % 96, img = i / (96 * 32);
    const int win = img < 3 ? 0 : (img < 5 ? 1 : (img < 8 ? 2 : 3));
    const int kwp = img - (win == 0 ? 0 : win == 1 ? 3 : win == 2 ? 5 : 8);
    const int kz = 2 - (row >> 5), co = row & 31;
    const int y5 = 2 * kz + (win >> 1), x5 = 2 * kwp + (win & 1);
    const float v = (y5 < 5 && x5 < 5) ? w[((size_t)co * 32 + k) * 25 + y5 * 5 + x5] : 0.f;
    const float vs = v * scale;
    const __half wh = __float2half_rn(vs);
    const float whf = __half2float(wh);
    __half* im = reinterpret_cast<__half*>(out) + (size_t)img * (B_BYTES / 2);
    const int sw = co & 7;
    im[row * 64 + ((((k >> 3)) ^ sw) << 3) + (k & 7)] = wh;
    im[row * 64 + ((((k >> 3) + 4) ^ sw) << 3) + (k & 7)] = __float2half_rn((vs - whf) * 2048.f);
  }
}
__global__ void prep_weights_p4_kernel(const float* __restrict__ w, float* __restrict__ out) {
  pdl_wait();            // no early trigger: see WEIGHT-IMAGE WRITERS below
  store_p4_images(w, out, 1.f / out[10 * (B_BYTES / 4)], blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

// WEIGHT-IMAGE WRITERS never call griddepcontrol.launch_dependents: the launch after one of these kernels therefore starts only
// when it has completed, and — launches forming a chain — so does every later one.  That is what lets conv_c32_ws.cu fetch its
// resident weight images BEFORE its own griddepcontrol.wait, under the tail of whatever kernel precedes it.
// 2^-s for one weight tensor of `numel` floats: s = 13 - floor(log2 max|w|), i.e. max|w * 2^s| in [2^13, 2^14) — far from the
// fp16 overflow (65504) and with the low parts wl ~ 2^-11 w' of everything above 2^-16 max|w| still normal fp16 numbers.
__device__ __forceinline__ void weight_scale_block(const float* __restrict__ w, int numel, float* __restrict__ slot) {
  __shared__ float smax[32];
  float m = 0.f;
  for (int i = threadIdx.x; i < numel; i += blockDim.x) m = fmaxf(m, fabsf(w[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) smax[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) m = fmaxf(m, smax[i]);
    int s = 0;
    if (m > 0.f && m <= 3.0e38f) s = 13 - ilogbf(m);
    s = s < -20 ? -20 : (s > 40 ? 40 : s);
    *slot = ldexpf(1.f, -s);
  }
}
__global__ void weight_scale_kernel(const float* __restrict__ w, int numel, float* __restrict__ slot) {
  pdl_wait();            // no early trigger: see WEIGHT-IMAGE WRITERS below
  weight_scale_block(w, numel, slot);
}
// Entry kinds of the batched preparation (config bits 16..23, see snb_prep_conv_weights_tc_batch):
//   0, 1, 2  the tensor-core images described in snb200.h;
//   3        the C4 image of the refinement's input layer from its [32][4][3][3] weight: the "ws" image of the [32][32][3][3] tensor
//            W'[co][kw*4 + ch][kh][0] = w[co][ch][kh][kw] (zero elsewhere), nwin = 3, mode = SNB_CONV_WS (what ops.refine_in_weights_ws
//            builds with torch layout ops);
//   4        eval-mode BatchNorm fold: src = gamma, aux = {beta, running_mean, running_var}; out[0:32] = scale, out[64:96] = shift;
//   5        plain copy of `count` floats;
//   6        the data-gradient taps of the refinement input layer's disparity channel from its [32][4][3][3] weight:
//            out[c*9 + t] = w[c][0][8 - t] (RefineHead.backward's flipped [32][9] weight).
// Kinds 4 and 5 need the aux pointers / count of snb_prep_item, i.e. the by-value table of snb_prep_param_launch.
__device__ __forceinline__ int weight_numel_of(int kind, int nwin) {
  return kind == 0 ? 1024 * nwin * 3 : (kind == 3 ? 32 * 4 * 9 : 1024 * 25);
}
__device__ __forceinline__ void weight_scale_entry(const float* w, float* out, int cfg) {
  if (((cfg >> 8) & (SNB_CONV_F16 | SNB_CONV_WS)) == 0) return;
  const int nwin = cfg & 0xff, kind = (cfg >> 16) & 0xff;
  weight_scale_block(w, weight_numel_of(kind, nwin), out + scale_slot_of(cfg >> 8, nwin));
}
__global__ void weight_scale_batch_kernel(const long long* __restrict__ table) {
  pdl_wait();            // no early trigger: see WEIGHT-IMAGE WRITERS below
  const long long* e = table + 4 * blockIdx.x;
  weight_scale_entry(reinterpret_cast<const float*>(e[0]), reinterpret_cast<float*>(e[1]), (int)e[2]);
}

// w [32 cout][32 cin][kd*kh*kw taps] -> per (kd,kh) window: B_hi[n = kw*32 + cout][k = cin] then B_lo, each in the
// SWIZZLE_128B K-major smem image (row n = 128 B, 16-B chunk c stored at c ^ (n & 7)).  mode 1: data-gradient weights.
// mode | SNB_CONV_F16: the fp16-split format above.
__global__ void prep_weights_tc_kernel(const float* __restrict__ w, float* __restrict__ out, int nwin, int mode) {
  pdl_wait();            // no early trigger: see WEIGHT-IMAGE WRITERS below
  const bool f16 = (mode & SNB_CONV_F16) != 0, ws = (mode & SNB_CONV_WS) != 0;
  const float scale = (f16 || ws) ? 1.f / out[scale_slot_of(mode, nwin)] : 1.f;
  mode &= 0xf;
  const int taps = nwin * 3;
  const int total = nwin * 96 * 32;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int k = i & 31;                 // K index (input channel of this GEMM)
    const int n = (i >> 5) % 96;          // N index = kw*32 + output channel of this GEMM
    const int win = i / (96 * 32);
    const int kw = n >> 5, co = n & 31;
    const int tap = win * 3 + kw;
    float v;
    if (mode == 0) v = w[((size_t)co * 32 + k) * taps + tap];
    else           v = w[((size_t)k * 32 + co) * taps + (taps - 1 - tap)];   // dgrad: swap channels, flip taps
    if (ws) { store_ws_split(out, nwin == 9, win, n, k, v, scale); continue; }
    if (f16) { store_f16_split(out, win, n, k, v, scale); continue; }
    const float hi = __uint_as_float(tc::tf32_hi_bits(v));
    const size_t o = (size_t)win * WIMG_FLOATS_PER_WINDOW + n * 32 + (((k >> 2) ^ (n & 7)) << 2) + (k & 3);
    out[o] = hi;
    out[o + B_BYTES / 4] = v - hi;
  }
}

// One table entry (kinds above) over the flat index range first, first + step, ...
__device__ __forceinline__ void prep_entry(const float* __restrict__ w, const float* const* aux, float* __restrict__ out, int cfg,
                                           int count, int first, int step) {
  const int nwin = cfg & 0xff, mode = (cfg >> 8) & 0xf, kind = (cfg >> 16) & 0xff, pa = (cfg >> 24) & 0xf, pb = (cfg >> 28) & 0xf;
  if (kind == 4) {
    if (aux == nullptr) return;
    // bit for bit what autograd.fused.bn_fold computes with torch ops, one rounding per op and no FMA contraction:
    // scale = gamma * rsqrt(var + eps), shift = beta - mean * scale
    for (int c = first; c < 32; c += step) {
      const float sc = __fmul_rn(w[c], rsqrtf(__fadd_rn(aux[2][c], 1e-5f)));
      out[c] = sc;
      out[64 + c] = __fsub_rn(aux[0][c], __fmul_rn(aux[1][c], sc));
    }
    return;
  }
  if (kind == 5) {
    for (int i = first; i < count; i += step) out[i] = w[i];
    return;
  }
  if (kind == 6) {
    for (int i = first; i < 32 * 9; i += step) out[i] = w[(i / 9) * 36 + 8 - i % 9];
    return;
  }
  const bool f16 = ((cfg >> 8) & SNB_CONV_F16) != 0, ws = ((cfg >> 8) & SNB_CONV_WS) != 0;
  const float scale = (f16 || ws) ? 1.f / out[scale_slot_of(cfg >> 8, nwin)] : 1.f;
  if (kind == 2) { store_p4_images(w, out, scale, first, step); return; }
  const int taps = nwin * 3;
  const int total = nwin * 96 * 32;
  for (int i = first; i < total; i += step) {
    const int k = i & 31;
    const int n = (i >> 5) % 96;
    const int win = i / (96 * 32);
    const int kw = n >> 5, co = n & 31;
    int tap = win * 3 + kw;
    const int oc = mode == 0 ? co : k, ic = mode == 0 ? k : co;        // dgrad: swap channels, flip taps
    if (mode != 0) tap = taps - 1 - tap;
    float v;
    if (kind == 0) {
      v = w[((size_t)oc * 32 + ic) * taps + tap];
    } else if (kind == 3) {
      v = (tap % 3 == 0 && ic < 12) ? w[((oc * 4 + (ic & 3)) * 3 + tap / 3) * 3 + (ic >> 2)] : 0.f;
    } else {
      const int y5 = 2 * (tap / 3) + pa, x5 = 2 * (tap % 3) + pb;
      v = (y5 < 5 && x5 < 5) ? w[((size_t)oc * 32 + ic) * 25 + y5 * 5 + x5] : 0.f;
    }
    if (ws) { store_ws_split(out, nwin == 9, win, n, k, v, scale); continue; }
    if (f16) { store_f16_split(out, win, n, k, v, scale); continue; }
    const float hi = __uint_as_float(tc::tf32_hi_bits(v));
    const size_t o = (size_t)win * WIMG_FLOATS_PER_WINDOW + n * 32 + (((k >> 2) ^ (n & 7)) << 2) + (k & 3);
    out[o] = hi;
    out[o + B_BYTES / 4] = v - hi;
  }
}

// Batched variant: blockIdx.y picks a table entry {w, out, config, 0} (see snb_prep_conv_weights_tc_batch in snb200.h).
__global__ void prep_weights_tc_batch_kernel(const long long* __restrict__ table) {
  pdl_wait();            // no early trigger: see WEIGHT-IMAGE WRITERS below
  const long long* e = table + 4 * blockIdx.y;
  prep_entry(reinterpret_cast<const float*>(e[0]), nullptr, reinterpret_cast<float*>(e[1]), (int)e[2], 0,
             blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

// The same pair of kernels over a table passed BY VALUE (snb_prep_param_launch): no table upload, so a caller's preparation is one
// capturable launch pair with no host-to-device copy.  PREP_PARAM_MAX entries keep the parameter block under 4 KB.
constexpr int PREP_PARAM_MAX = 80;
struct PrepParamTable { snb_prep_item it[PREP_PARAM_MAX]; int n; };
static_assert(sizeof(PrepParamTable) <= 4096, "kernel parameter block");

__global__ void weight_scale_param_kernel(const __grid_constant__ PrepParamTable t) {
  pdl_wait();            // no early trigger: see WEIGHT-IMAGE WRITERS below
  const snb_prep_item& e = t.it[blockIdx.x];
  weight_scale_entry(e.src, e.out, e.cfg);
}

__global__ void prep_weights_param_kernel(const __grid_constant__ PrepParamTable t) {
  pdl_wait();            // no early trigger: see WEIGHT-IMAGE WRITERS below
  const snb_prep_item& e = t.it[blockIdx.y];
  prep_entry(e.src, e.aux, e.out, e.cfg, e.count, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x);
}

}  // namespace tc

static int tc_setup(const snb_conv_geom* g, tc::Params& p, const char* who) {
  SNB_REQUIRE(g != nullptr, "%s: null geometry", who);
  SNB_REQUIRE(g->transposed == 0 && g->stride == 1 && g->KH == 3 && g->KW == 3 && (g->KD == 1 || g->KD == 3), "%s: needs a stride-1 3x3(x3) conv", who);
  SNB_REQUIRE(g->OD == g->D && g->OH == g->H && g->OW == g->W && g->ph == g->dil && g->pw == g->dil &&
              g->pd == (g->KD == 3 ? 1 : 0), "%s: needs 'same' padding", who);
  SNB_REQUIRE(g->dil >= 1 && g->dil <= 16, "%s: dilation out of range", who);
  p.B = g->B; p.D = g->D; p.H = g->H; p.W = g->W;
  p.nwin = g->KD * 3; p.dil = g->dil; p.P = g->W + g->dil;
  p.step = 128 - 2 * g->dil;
  p.tiles_per_slice = snb_ceil_div((long long)g->H * p.P, p.step);
  const long long nt = (long long)g->B * g->D * p.tiles_per_slice;
  SNB_REQUIRE(nt < (1ll << 30), "%s: too many tiles", who);
  p.ntiles = (int)nt;
  return 0;
}

// 3-D product path: TMA producer + A operand in TMEM (conv3d_c32_tma.cu).  This file keeps the loader-warp kernel: the 2-D
// `flat` variant used by tests / A-B measurements, and the older 3-D kernel behind passes | 0x400.
int snb_conv3d_tma_num_tiles(const snb_conv_geom* g);
int snb_conv3d_tma_launch(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                          int passes, long long* dbg, void* stream);

extern "C" int snb_conv_c32_tc_num_tiles(const snb_conv_geom* g) {
  if (g && g->KD == 3) return snb_conv3d_tma_num_tiles(g);
  tc::Params p;
  if (tc_setup(g, p, "snb_conv_c32_tc_num_tiles")) return -1;
  return p.ntiles;
}

extern "C" int snb_conv_weights_tc_floats(int kd) { return kd * 3 * tc::WIMG_FLOATS_PER_WINDOW; }

extern "C" int snb_prep_conv_weights_tc(const float* w, float* out, int kd, int mode, void* stream) {
  SNB_REQUIRE(w && out && (kd == 1 || kd == 3) && ((mode & 0xf) == 0 || (mode & 0xf) == 1) && (mode & ~0x3f) == 0 &&
              (mode & (SNB_CONV_F16 | SNB_CONV_WS)) != (SNB_CONV_F16 | SNB_CONV_WS), "snb_prep_conv_weights_tc: bad args");
  const int nwin = kd * 3;
  if (mode & (SNB_CONV_F16 | SNB_CONV_WS)) {
    const int slot = ((mode & SNB_CONV_WS) && kd == 3) ? 9 * (tc::B_BYTES / 4) : tc::WIMG_SCALE_SLOT;
    snb_launch(tc::weight_scale_kernel, 1, 256, 0, stream, w, 1024 * nwin * 3, out + slot);
    SNB_LAUNCH_CHECK("weight_scale_kernel");
  }
  snb_launch(tc::prep_weights_tc_kernel, snb_ceil_div(nwin * 96 * 32, 256), 256, 0, stream, w, out, nwin, mode);
  SNB_LAUNCH_CHECK("prep_weights_tc_kernel");
  return 0;
}

extern "C" int snb_prep_conv5x5s2_weights_ws(const float* w, float* out, void* stream) {
  SNB_REQUIRE(w && out, "snb_prep_conv5x5s2_weights_ws: null pointer");
  snb_launch(tc::weight_scale_kernel, 1, 256, 0, stream, w, 1024 * 25, out + 10 * (tc::B_BYTES / 4));
  SNB_LAUNCH_CHECK("weight_scale_kernel");
  snb_launch(tc::prep_weights_p4_kernel, 36, 256, 0, stream, w, out);
  SNB_LAUNCH_CHECK("prep_weights_p4_kernel");
  return 0;
}

extern "C" int snb_prep_conv_weights_tc_batch(const long long* table, int n, void* stream) {
  SNB_REQUIRE(table && n > 0 && n <= 65535, "snb_prep_conv_weights_tc_batch: bad args");
  snb_launch(tc::weight_scale_batch_kernel, n, 256, 0, stream, table);       // no-op blocks for TF32-format entries
  SNB_LAUNCH_CHECK("weight_scale_batch_kernel");
  snb_launch(tc::prep_weights_tc_batch_kernel, dim3(36, n), 256, 0, stream, table);
  SNB_LAUNCH_CHECK("prep_weights_tc_batch_kernel");
  return 0;
}

int snb_prep_param_launch(const snb_prep_item* items, int n, void* stream) {
  SNB_REQUIRE(items && n > 0, "snb_prep_param_launch: bad args");
  for (int base = 0; base < n; base += tc::PREP_PARAM_MAX) {
    tc::PrepParamTable t;
    t.n = n - base < tc::PREP_PARAM_MAX ? n - base : tc::PREP_PARAM_MAX;
    for (int i = 0; i < t.n; ++i) t.it[i] = items[base + i];
    snb_launch(tc::weight_scale_param_kernel, t.n, 256, 0, stream, t);      // no-op blocks for the kinds without a scale
    SNB_LAUNCH_CHECK("weight_scale_param_kernel");
    snb_launch(tc::prep_weights_param_kernel, dim3(36, t.n), 256, 0, stream, t);
    SNB_LAUNCH_CHECK("prep_weights_param_kernel");
  }
  return 0;
}

static int conv_c32_tc_launch(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                              int passes, long long* dbg, void* stream);

extern "C" int snb_conv_c32_tc(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                               int passes, void* stream) {
  return conv_c32_tc_launch(x, wimg, y, g, e, passes, nullptr, stream);
}

extern "C" int snb_conv_c32_tc_profile(const float* x, const float* wimg, float* y, const snb_conv_geom* g,
                                       const snb_conv_epilogue* e, int passes, long long* counters, void* stream) {
  SNB_REQUIRE(counters != nullptr, "snb_conv_c32_tc_profile: null counters");
  return conv_c32_tc_launch(x, wimg, y, g, e, passes, counters, stream);
}

static int conv_c32_tc_launch(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                              int passes, long long* dbg, void* stream) {
  tc::Params p;
  if (int rc = tc_setup(g, p, "snb_conv_c32_tc")) return rc;
  SNB_REQUIRE(x && wimg && y && e, "snb_conv_c32_tc: null pointer");
  if (g->KD == 3 && (passes & 0x400) == 0) {                            // 3-D product path (dbg: per-role wait counters)
    SNB_REQUIRE((passes & 0xef) == 1 || (passes & 0xef) == 3, "snb_conv_c32_tc: passes must be 1 or 3");
    SNB_REQUIRE((passes & SNB_CONV_F16) == 0 || (passes & 0xf) == 3, "snb_conv_c32_tc: the fp16 split has 3 passes");
    SNB_REQUIRE(!e->scale || e->shift, "snb_conv_c32_tc: scale without shift");
    return snb_conv3d_tma_launch(x, wimg, y, g, e, passes & 0xff, dbg, stream);
  }
  SNB_REQUIRE(g->KD != 3 || e->stats == nullptr, "snb_conv_c32_tc: the loader-warp 3-D kernel (diagnostics) does not emit BN statistics");
  passes &= 0xff;
  SNB_REQUIRE(passes == 1 || passes == 3, "snb_conv_c32_tc: passes must be 1 or 3");
  SNB_REQUIRE(!e->scale || e->shift, "snb_conv_c32_tc: scale without shift");
  p.x = x; p.wimg = wimg; p.y = y; p.passes = passes; p.e = *e; p.dbg = dbg;
  int dev = 0, sms = 148;
  SNB_CUDA(cudaGetDevice(&dev));
  SNB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int grid = p.ntiles < sms ? p.ntiles : sms;
  if (dbg) {
    SNB_CUDA(cudaFuncSetAttribute(tc::conv_c32_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
    snb_launch(tc::conv_c32_tc_kernel<true>, grid, tc::NTHREADS, tc::SMEM_BYTES, stream, p);
  } else {
    SNB_CUDA(cudaFuncSetAttribute(tc::conv_c32_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM_BYTES));
    snb_launch(tc::conv_c32_tc_kernel<false>, grid, tc::NTHREADS, tc::SMEM_BYTES, stream, p);
  }
  SNB_LAUNCH_CHECK("conv_c32_tc_kernel");
  return 0;
}
