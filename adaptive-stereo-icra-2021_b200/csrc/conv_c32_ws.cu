// 32->32 stride-1 3x3 (dilated, 2-D) / 3x3x3 (3-D) 'same' convolution on the tcgen05 tensor cores — the round-2 product kernel:
// "walk + shifted operand copies + folded accumulator ring".  Replaces nn.Conv2d of every BasicBlock / conv_alone / the polyphase
// pieces of downsample[1:] (stereo_net.py:37-51,64-77,96-100) and the nn.Conv3d cost-filter layers (stereo_net.py:155-160,185-186),
// incl. bias, folded BatchNorm, LeakyReLU, the residual add and the train-mode BN partial sums.
//
// GEMM view.  M = 128 output positions (2-D: pixels of one image row; 3-D: consecutive positions of the un-padded flat index
// q = h*W + w of one (b,d) slice).  The CTA WALKS along the slowest kernel axis z (2-D: image rows in steps of `dil`; 3-D: the
// disparity axis): walk step u brings the raw input of position-row z0 + u - 1 on chip ONCE and it feeds the three output tiles
// u (kz = 0), u-1 (kz = 1), u-2 (kz = 2), whose accumulators sit side by side in a RING of 32-column blocks in TMEM.
//   raw windows  one TMA tile load per walk step (3-D: three, kh = 0,1,2, shifted by (kh-1)*W flat positions) of
//                128 + 2*dil position rows x 32 ch fp32 (SWIZZLE_128B, zero fill outside the row / slice / volume)
//   converters   thread = output position m: for kw = 0,1,2 read raw row m + kw*dil, split it into the fp16 pair (xh | xl')
//                (tc_common.cuh: x = xh + 2^-11 xl') and tcgen05.st it into A slot [kw] — the kw shift happens on the way INTO the
//                tensor core, so the accumulator is the convolution output itself (round 1 un-shifted three N = 96 partial
//                outputs in the epilogue: 48 KB of TMEM -> smem -> register traffic per tile, and that bounded the kernel).
//                3-D: the kw = 0 / 2 copies are zeroed where the flat index wrapped into the neighbouring image row.
//   MMA          per (window, kw, k-step): ONE M128 N96 K16 kind::f16 MMA per product of the split covers the three tiles'
//                kz taps at once: D = ring blocks [tile u-2 | u-1 | u], B rows = [kz = 2 | 1 | 0] x 32 cout (the weight image is
//                laid out that way).  N = 32 MMAs (one per tile) run at ~26 cycles instead of 16 — they are bound by the 4 KB
//                A-operand read from TMEM — so folding kz into N is worth 1.5x on the tensor pipe.  Where the ring wraps, or at
//                the ends of a strip, the MMA is issued as N = 64 + 32 / N = 32; a tile's very first MMA is a separate N = 32
//                one with accumulate = 0.
//   split        2-D: out = 2^-s (xh.wh + xl'.(2^-11 wh) + xh.wl), three weight images per kw (72 KB resident).
//                3-D: 27 taps x three images do not fit, so the two correction products go to a SECOND accumulator ring:
//                D1 = xh.wh, D2 = xl'.wh + xh.wl'' (wl'' = 2^11 wl), out = 2^-s (D1 + 2^-11 D2): two images per tap, all nine
//                (kh,kw) images resident (108 KB) — round 1 streamed 24 KB of weights per window and re-read every input
//                position nine times: 351 MB of L2 -> SM traffic per layer, the actual bound of that kernel (6.5 TB/s).
//   epilogue     two groups of four warps on alternating tiles: tcgen05.ld -> acc * alpha + beta (alpha = scale 2^-s,
//                beta = scale bias + shift) -> LeakyReLU -> + residual -> swizzled 16 KB tile in smem -> ONE TMA tile store.
//   residual     BasicBlock's `x + ...` (stereo_net.py:50) adds the layer's own input: the converter of the tile's centre row
//                holds x[m] in registers and parks it in TMEM next to the accumulator (2-D).  A residual that is not the input
//                (data gradients of the residual blocks) is TMA-loaded into the staging buffer and added in place (RES2).
// What bounds it now: shared-memory wavefronts (B-operand fetch + TMA write + converter reads + epilogue staging ~ 1300 per
// 2-D tile) about level with the tensor pipe (~950 cycles per 2-D tile).
// Warps: 0 producer, 1 MMA issuer (+ resident weights), 2-9 converters (two groups of four, alternating windows),
// 10-17 epilogue (two groups, alternating tiles).
#include <cuda.h>
#include <stdlib.h>
#include <mutex>
#include <vector>
#include "tc_common.cuh"

namespace wsk {

using namespace tc;

constexpr int NTHREADS_WS = 18 * 32;
constexpr int CONV_WARP0 = 2, EPI_WARP0 = 10;
constexpr int RING = 4;                                  // accumulator ring: 32-column blocks, tile t sits in block t % RING
constexpr int NR = 4;                                    // raw window ring depth
constexpr int STG_BYTES = 128 * 128;                     // one output tile, fp32

// MODE 0: 2-D 3x3 (dilated).  MODE 1: 3-D 3x3x3.  MODE 2: 5x5 stride-2 pad-2 conv written over the four polyphase images of its
// input (x[2i+a][2j+b] -> phase a*2+b, output-sized): out = sum over phases of a 3x3 'same' conv with the sub-kernel
// w[2kz+a][2kw+b] — the four phase rows of one walk step are four raw windows feeding ONE accumulator ring, so the whole layer is
// one launch instead of four chained ones that re-read and re-write the output (round 2, first half: 80 us per KITTI layer).
// MODE 3: 3x3 conv of a FOUR-channel channels-last image (the refinement's input layer: [disparity, r, g, b] -> 32,
// stereo_net.py:105-117).  A raw row is 16 B per pixel, so the three kw taps of a pixel are 48 contiguous bytes: they go into ONE
// K = 16 slice (k = kw*4 + ch, 12 used), and a walk step costs 3 MMAs instead of 18 — the layer becomes a store-bound kernel.
constexpr int MODE_2D = 0, MODE_3D = 1, MODE_P4 = 2, MODE_C4 = 3;
template <int MODE> struct Cfg {
  static constexpr bool TWO = MODE == MODE_3D || MODE == MODE_P4;      // two accumulator rings D1 / D2 and [wh | wl''] images
  static constexpr bool FLAT = MODE == MODE_3D;          // positions = un-padded flat index of a (b,d) slice, walk along d
  static constexpr bool ONCE = TWO;                      // converters: split every raw row ONCE, in place, then read it three times
  static constexpr int NWIN = MODE == MODE_3D ? 3 : (MODE == MODE_P4 ? 4 : 1);     // raw windows per walk step (3-D: kh; P4: phase)
  static constexpr int NIMG = MODE == MODE_3D ? 9 : (MODE == MODE_P4 ? 10 : (MODE == MODE_C4 ? 1 : 3));    // resident weight images
  static constexpr int NKS = MODE == MODE_C4 ? 1 : 2;    // K = 16 slices per (window, kw)
  static constexpr int IMG_BYTES = TWO ? B_BYTES : 2 * B_BYTES;     // TWO: [wh | wl''] 12 KB; 2-D: P [wh | wl] + Q [2^-11 wh | -] 24 KB
  static constexpr int RAW_BYTES = MODE == MODE_C4 ? 3 * 1024 : (TWO ? 17 * 1024 : 20 * 1024);     // 130 / up to 160 position rows of 128 B (C4: 16 B)
  static constexpr int NSTG = TWO ? 1 : 2;               // staging tiles per epilogue group
  static constexpr int NA = TWO ? 2 : 3;                 // A slots of 96 columns = 3 kw x (xh 16 | xl' 16)
  static constexpr int NRES = 3;                         // 2-D: residual slots of 32 columns
  static constexpr int D1_BASE = 0, D2_BASE = RING * 32, RES_BASE = RING * 32, A_BASE = TWO ? 2 * RING * 32 : RING * 32 + NRES * 32;
  static constexpr int SMEM_BYTES = NR * RAW_BYTES + 2 * NSTG * STG_BYTES + NIMG * IMG_BYTES + 4096 + 1024;
  // first weight image of a window and its number of kw taps (P4: odd-column phases have taps kw' = 0, 1 only: x5 = 2 kw' + 1 < 5)
  __host__ __device__ static constexpr int img_base(int win) { return MODE == MODE_P4 ? (win == 0 ? 0 : win == 1 ? 3 : win == 2 ? 5 : 8) : win * 3; }
  __host__ __device__ static constexpr int nkw(int win) { return MODE == MODE_C4 ? 1 : ((MODE == MODE_P4 && (win & 1)) ? 2 : 3); }
  static_assert(A_BASE + NA * 96 <= 512, "TMEM budget");
  static_assert(SMEM_BYTES <= 227 * 1024, "smem budget");
};

struct Params {
  const float* wimg; float* y;
  int B, D, H, W, dil;
  int ncb;                  // 2-D: column blocks of 128 pixels per row.  3-D: 128-position tiles per (b,d) slice
  int cmax;                 // longest chain (2-D: ceil(H/dil) rows, 3-D: D slices)
  int La, nsa, Lb;          // every chain = nsa long strips of La tiles + one short strip of Lb tiles (Lb may be 0)
  int nchains, nlong;       // nlong = nchains * nsa; strips [0, nlong) are the long ones, [nlong, nstrips) the short ones
  int nstrips;
  int res_mode;             // 0: none, 1: residual == input (on-chip, 2-D), 2: residual from global memory
  snb_conv_epilogue e;
  long long* dbg;
};

#define WSWAIT(acc, call) do { const long long _t0 = p.dbg ? clock64() : 0; call; if (p.dbg) acc += clock64() - _t0; } while (0)

// strip = a chain of `ntiles` output tiles along the walk axis.  2-D: rows z0, z0 + dil, ... of column block `cb`, image b.
// 3-D: slices z0, z0 + 1, ... of position tile `cb`, volume b.
struct Strip { int b, cb, z0, ntiles; };

template <bool D3>      // D3 = flat 3-D geometry
__device__ __forceinline__ Strip decode_strip(const Params& p, int sid) {
  Strip s;
  int j0, cap;
  if (sid < p.nlong) { const int seg = sid / p.nchains; sid -= seg * p.nchains; j0 = seg * p.La; cap = p.La; }
  else               { sid -= p.nlong; j0 = p.nsa * p.La; cap = p.Lb; }
  if (D3) {
    s.cb = sid % p.ncb; s.b = sid / p.ncb;
    s.ntiles = p.D - j0; if (s.ntiles > cap) s.ntiles = cap; if (s.ntiles < 0) s.ntiles = 0;
    s.z0 = j0;
  } else {
    const int rho = sid % p.dil; sid /= p.dil;
    s.cb = sid % p.ncb; s.b = sid / p.ncb;
    const int chain = (rho < p.H) ? (p.H - rho + p.dil - 1) / p.dil : 0;
    s.ntiles = chain - j0; if (s.ntiles > cap) s.ntiles = cap; if (s.ntiles < 0) s.ntiles = 0;
    s.z0 = rho + j0 * p.dil;
  }
  return s;
}
// Strips are dealt to the CTAs in rounds of gridDim.x, every other round in reverse order ("snake"): the long strips come first,
// so the CTAs that got the short ones at the end of a round are the first to get a second strip.  All four roles walk the same
// sequence.  (sid_k >= k * gridDim.x, so the first invalid k ends the sequence.)
__device__ __forceinline__ int strip_at(int k) {
  const int G = (int)gridDim.x, b = (int)blockIdx.x;
  return k * G + ((k & 1) ? G - 1 - b : b);
}
#define WS_FOR_STRIPS(sid) for (int _k = 0, sid = strip_at(0); sid < p.nstrips; sid = strip_at(++_k))

__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n"
      :: "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void group_bar(int id) { asm volatile("bar.sync %0, 128;\n" :: "r"(id) : "memory"); }     // 4 warps of one group

// M128 N{32,64,96} K16 kind::f16, A from TMEM, fp32 accumulate; idesc_n(b): instruction descriptor for N = 32 b
__device__ __forceinline__ uint32_t idesc_n(int nblk) { return (1u << 4) | ((uint32_t)(nblk * 4) << 17) | ((128u >> 4) << 24); }
__device__ __forceinline__ void mma_f16_i(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" :: "r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}

// All MMAs of one raw window (3 kw x 2 k-steps x 3 products of the split) for NG accumulator groups, straight-line: every
// descriptor is (per-group base) + (compile-time offset), so an MMA costs its UTCHMMA plus a couple of uniform adds — the single
// issuing thread is slow (a version with per-MMA loops / predicates over runtime group tables ran 2x slower end to end).
// SKIP_FIRST: the first product(s) of (kw = 0, ks = 0) were issued by the caller (new tile, accumulate = 0).
// SINGLE: the single-product variant, xh . wh only (see conv_c32_ws_kernel).
template <int MODE, int NG, bool SKIP_FIRST, int NKW, bool SINGLE>
__device__ __forceinline__ void issue_window(uint32_t d1, uint32_t d2, const uint32_t (&g_d)[3], uint32_t ta, uint32_t img0,
                                             const uint32_t (&g_b)[3], const uint32_t (&g_i)[3]) {
  using C = Cfg<MODE>;
  constexpr bool D3 = C::TWO;
  uint64_t bd[NG]; uint32_t dd1[NG], dd2[NG];
#pragma unroll
  for (int g = 0; g < NG; ++g) { bd[g] = make_desc(img0 + g_b[g]); dd1[g] = d1 + g_d[g]; dd2[g] = d2 + g_d[g]; }
#pragma unroll
  for (int kw = 0; kw < NKW; ++kw) {
#pragma unroll
    for (int ks = 0; ks < C::NKS; ++ks) {
      const uint32_t a = ta + kw * 32 + ks * 8;
      constexpr int Q_OFF = D3 ? 0 : B_BYTES;                 // second product's B: 3-D wh again, 2-D the 2^-11 wh image
      const uint64_t o1 = (uint64_t)((kw * C::IMG_BYTES + ks * 32) >> 4);
      const uint64_t o2 = (uint64_t)((kw * C::IMG_BYTES + Q_OFF + ks * 32) >> 4);
      const uint64_t o3 = (uint64_t)((kw * C::IMG_BYTES + 64 + ks * 32) >> 4);
      const bool skip = SKIP_FIRST && kw == 0 && ks == 0;
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        if (!skip) mma_f16_i(dd1[g], a, bd[g] + o1, g_i[g], 1);                      // xh . wh
        if (SINGLE) continue;
        if (!(skip && D3)) mma_f16_i(dd2[g], a + 16, bd[g] + o2, g_i[g], 1);         // xl' . (3-D: wh -> D2; 2-D: 2^-11 wh)
        mma_f16_i(dd2[g], a, bd[g] + o3, g_i[g], 1);                                 // xh . (3-D: wl'' -> D2; 2-D: wl)
      }
    }
  }
}

// FOLD (the product setting): one N = 96 MMA over the three ring blocks per product (see above) instead of three N = 32 MMAs:
// 37 / 40 / 44 us against 41 / 44 / 48 us per KITTI refinement block (dilation 1 / 4 / 8), 55 against 61 us per 3-D filter layer.
// SINGLE (MODE_2D / MODE_3D, inference only, no statistics): the reduced-precision variant that keeps only the first product of the
// split, out = 2^-s (xh . wh) — 10 explicit mantissa bits per operand instead of fp32-grade.  The converters write only the xh half
// of an A slot, the MMA warp issues one product per (window, kw, k-step) instead of three, the 3-D D2 ring is neither written nor
// read, and only the wh half of the same weight images is used (2-D: the P block of each image is all that is fetched).
template <int MODE, bool FOLD, bool RES2, bool SINGLE>      // RES2: a residual that is not the layer's input (p.res_mode == 2), added from a TMA-loaded tile
__global__ void __launch_bounds__(NTHREADS_WS, 1)
conv_c32_ws_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_out,
                   const __grid_constant__ CUtensorMap tmap_res, const __grid_constant__ CUtensorMap tmap_p1,
                   const __grid_constant__ CUtensorMap tmap_p2, const __grid_constant__ CUtensorMap tmap_p3, const Params p) {
  // tmap_p1..3 (MODE_P4 only): the polyphase images 1..3 of the input (tmap = image 0) — four sub-tensors of a split input, or
  // four STRIDED views (element strides 2 in x and y) of the un-split input, which needs no split pass at all.
  using C = Cfg<MODE>;
  constexpr int NA = C::NA, NRES = C::NRES, NWIN = C::NWIN;
  constexpr bool D3 = C::FLAT, TWO = C::TWO;
  static_assert(!SINGLE || MODE == MODE_2D || MODE == MODE_3D, "single-product variant: 2-D and 3-D layers only");
  constexpr int WLOAD = (SINGLE && !TWO) ? B_BYTES : C::IMG_BYTES;     // bytes fetched per weight image (2-D single: P only)
  extern __shared__ unsigned char smem_dyn[];
  const uint32_t base_u32 = (smem_u32(smem_dyn) + 1023u) & ~1023u;
  unsigned char* base = smem_dyn + (base_u32 - smem_u32(smem_dyn));
  unsigned char* sStg = base + NR * C::RAW_BYTES;           // [2 epilogue groups][NSTG] output tiles (1024-B aligned: TMA store source)
  unsigned char* sB = sStg + 2 * C::NSTG * STG_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sB + C::NIMG * C::IMG_BYTES);
  uint64_t* rfull = bars;                // [NR]    TMA (raw window) -> converters
  uint64_t* rempty = rfull + NR;         // [NR]    converters -> producer
  uint64_t* afull = rempty + NR;         // [NA]    converters -> MMA (A slot in TMEM)
  uint64_t* aempty = afull + NA;         // [NA]    MMA commit -> converters
  uint64_t* tfull = aempty + NA;         // [RING]  MMA commit -> epilogue
  uint64_t* tempty = tfull + RING;       // [RING]  epilogue -> MMA
  uint64_t* rsempty = tempty + RING;     // [NRES]  epilogue -> converters (residual slot drained)
  uint64_t* wbar = rsempty + NRES;
  uint64_t* resfull = wbar + 1;          // [2 groups][2]  TMA (global residual tile) -> epilogue group
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(resfull + 4);
  float* sPar = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(bars) + 512);    // [64] alpha | beta (16-B aligned)
  float* sRed = sPar + 96;                                  // [2 groups][4 warps][64]

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long t_entry = p.dbg ? clock64() : 0;
  const int RW = 128 + 2 * p.dil;                           // rows of a raw window
  const int HW = p.H * p.W;

  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < NR; ++i) { mbar_init(&rfull[i], 1); mbar_init(&rempty[i], 4); }
      for (int i = 0; i < NA; ++i) { mbar_init(&afull[i], 4); mbar_init(&aempty[i], 1); }
      for (int i = 0; i < RING; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 4); }      // a tile is drained by ONE epilogue group
      for (int i = 0; i < NRES; ++i) mbar_init(&rsempty[i], 4);
      for (int i = 0; i < 4; ++i) mbar_init(&resfull[i], 1);
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
  // The resident weight images are fetched BEFORE the grid-dependency wait, under the tail of the previous kernel: their only
  // writers (the weight preparation kernels, conv_c32_tc.cu "WEIGHT-IMAGE WRITERS") never trigger their dependents early, so
  // every launch that follows one of them starts after it has completed.  Everything else this kernel reads comes after the wait.
  if (warp == 1 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];\n" :: "l"(reinterpret_cast<uint64_t>(&tmap)) : "memory");
    asm volatile("prefetch.tensormap [%0];\n" :: "l"(reinterpret_cast<uint64_t>(&tmap_out)) : "memory");
    mbar_expect_tx(wbar, C::NIMG * WLOAD);
    for (int w = 0; w < C::NIMG; ++w)
      bulk_g2s(sB + w * C::IMG_BYTES, p.wimg + (size_t)w * (C::IMG_BYTES / 4), WLOAD, wbar);
  }
  pdl_launch();                                    // only after this CTA owns its TMEM columns
  pdl_wait();
  const int scale_slot = TWO ? C::NIMG * (B_BYTES / 4) : WIMG_SCALE_SLOT;
  if (tid >= EPI_WARP0 * 32 && tid < EPI_WARP0 * 32 + 32) {
    // y = lrelu(scale * (acc * 2^-s + bias) + shift) = lrelu(acc * alpha + beta)
    const int c = tid - EPI_WARP0 * 32;
    const snb_conv_epilogue& e = p.e;
    const float bias = e.bias ? e.bias[c] : 0.f, sc = e.scale ? e.scale[c] : 1.f, sh = e.scale ? e.shift[c] : 0.f;
    sPar[c] = sc * __ldg(p.wimg + scale_slot);
    sPar[32 + c] = fmaf(sc, bias, sh);
  }

  if (warp == 0) {
    // =============================================================== producer: one TMA tile load per raw window
    if (lane == 0) {
      uint32_t ac = 0;
      long long w_r = 0; const long long t0 = clock64();
      const uint32_t bytes = (uint32_t)RW * (MODE == MODE_C4 ? 16u : 128u);
      WS_FOR_STRIPS(sid) {
        const Strip s = decode_strip<D3>(p, sid);
        if (s.ntiles == 0) continue;
        for (int u = 0; u < s.ntiles + 2; ++u) {
#pragma unroll
          for (int win = 0; win < NWIN; ++win) {
            const uint32_t sa = ac % NR;
            WSWAIT(w_r, tc::mbar_wait(&rempty[sa], ((ac / NR) & 1) ^ 1));
            mbar_expect_tx(&rfull[sa], bytes);
            if (D3) tma_load_4d(base + sa * C::RAW_BYTES, &tmap, &rfull[sa], 0, s.cb * 128 - 1 + (win - 1) * p.W, s.z0 + u - 1, s.b);
            else if (MODE == MODE_P4) tma_load_4d(base + sa * C::RAW_BYTES, win == 0 ? &tmap : (win == 1 ? &tmap_p1 : (win == 2 ? &tmap_p2 : &tmap_p3)),
                                                  &rfull[sa], 0, s.cb * 128 - 1, s.z0 + u - 1, s.b);
            else    tma_load_4d(base + sa * C::RAW_BYTES, &tmap, &rfull[sa], 0, s.cb * 128 - p.dil, s.z0 + (u - 1) * p.dil, s.b);   // (C4: dil = 1, 16-B rows)
            ++ac;
          }
        }
      }
      if (p.dbg) { long long* dd = p.dbg + blockIdx.x * 16; dd[0] = w_r; dd[1] = clock64() - t0; }
    }
    __syncwarp();
  } else if (warp == 1) {
    // =============================================================== MMA issuer (converged warp, elected lane), window-major
    const long long t_w0 = p.dbg ? clock64() : 0;
    tc::mbar_wait_spin(wbar, 0);                   // resident weight images
    if (p.dbg && lane == 0) { long long* dd = p.dbg + blockIdx.x * 16; dd[8] = t_w0 - t_entry; dd[9] = clock64() - t_w0; }
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t sb_u32 = __shfl_sync(0xffffffffu, base_u32, 0) + NR * C::RAW_BYTES + 2 * C::NSTG * STG_BYTES;
    uint32_t tile_base = 0;                                        // (32-bit on purpose: these feed % and / on every tile)
    uint32_t win_count = 0;
    long long t_full = 0, t_tempty = 0; const long long t_mbegin = clock64();
    WS_FOR_STRIPS(sid) {
      const Strip s = decode_strip<D3>(p, sid);
      if (s.ntiles == 0) continue;
      for (int u = 0; u < s.ntiles + 2; ++u) {
        // active tiles of this walk step: j = u - kz in [0, ntiles); ascending tile index = descending kz = ascending weight rows
        const int jlo = max(u - 2, 0), jhi = min(u, s.ntiles - 1);          // (jhi >= jlo always: u <= ntiles + 1)
        const bool has_new = u < s.ntiles;                                   // tile u is touched for the first time in this step
        const int rowblk0 = 2 - (u - jlo);                                   // weight row block of tile jlo (kz = u - jlo)
        // MMA groups of this walk step, computed once: a group = (ring block of its first tile, weight row block, instruction
        // descriptor for N = 32 x #tiles).  FOLD: contiguous ring blocks form one group (two where the ring wraps); else one group
        // per tile.  `old` groups exclude the new tile u (first product of a new tile, see issue_fresh).
        const int pos_lo = (int)((tile_base + (uint32_t)jlo) % RING);
        const int n_all = jhi - jlo + 1, n_old = has_new ? n_all - 1 : n_all;
        uint32_t g_d[3], g_b[3], g_i[3]; int ng;
        uint32_t go_d[2], go_b[2], go_i[2];
        if (FOLD) {
          const int l0 = min(n_all, RING - pos_lo), l1 = n_all - l0;
          g_d[0] = pos_lo * 32; g_b[0] = rowblk0 * 4096; g_i[0] = idesc_n(l0);
          g_d[1] = 0; g_b[1] = (rowblk0 + l0) * 4096; g_i[1] = idesc_n(l1 > 0 ? l1 : 1);
          g_d[2] = 0; g_b[2] = 0; g_i[2] = 0;
          ng = l1 > 0 ? 2 : 1;
          const int m0 = min(n_old, RING - pos_lo), m1 = n_old - m0;
          go_d[0] = pos_lo * 32; go_b[0] = rowblk0 * 4096; go_i[0] = m0 > 0 ? idesc_n(m0) : 0u;
          go_d[1] = 0; go_b[1] = (rowblk0 + m0) * 4096; go_i[1] = m1 > 0 ? idesc_n(m1) : 0u;
        } else {
#pragma unroll
          for (int t = 0; t < 3; ++t) { g_d[t] = (uint32_t)((pos_lo + t) % RING) * 32; g_b[t] = (uint32_t)(rowblk0 + t) * 4096; g_i[t] = idesc_n(1); }
          ng = n_all;
          go_d[0] = g_d[0]; go_b[0] = g_b[0]; go_i[0] = n_old > 0 ? idesc_n(1) : 0u;
          go_d[1] = g_d[1]; go_b[1] = g_b[1]; go_i[1] = n_old > 1 ? idesc_n(1) : 0u;
        }
        const uint32_t new_d = ((tile_base + (uint32_t)u) % RING) * 32;         // ring block of the new tile (weight row block 2: kz = 0)
        if (has_new) {        // the epilogue must have drained the ring block of the new tile
          const uint32_t tc_new = tile_base + (uint32_t)u;
          WSWAIT(t_tempty, mbar_wait_warp(&tempty[tc_new % RING], (uint32_t)(((tc_new / RING) & 1) ^ 1)));
          tc_fence_after();
        }
        const uint32_t d1 = tmem_u + C::D1_BASE, d2 = tmem_u + (TWO ? C::D2_BASE : C::D1_BASE);
#pragma unroll
        for (int win = 0; win < NWIN; ++win, ++win_count) {
          const uint32_t aslot = win_count % NA;
          WSWAIT(t_full, mbar_wait_warp(&afull[aslot], (win_count / NA) & 1));
          tc_fence_after();
          const uint32_t ta = tmem_u + C::A_BASE + aslot * 96;
          const bool fresh_step = has_new && win == 0;          // the new tile's accumulators have not been written yet
          const uint32_t img0 = sb_u32 + C::img_base(win) * C::IMG_BYTES;  // image (win, kw = 0)
          const int nkw = C::nkw(win);                          // a constant per unrolled window
          if (elect_one()) {
            if (fresh_step) {
              // first product(s) of a new tile: the old tiles accumulate, the new one starts with accumulate = 0
              if (go_i[0]) mma_f16_i(d1 + go_d[0], ta, make_desc(img0 + go_b[0]), go_i[0], 1);
              if (go_i[1]) mma_f16_i(d1 + go_d[1], ta, make_desc(img0 + go_b[1]), go_i[1], 1);
              mma_f16_i(d1 + new_d, ta, make_desc(img0 + 2 * 4096), idesc_n(1), 0);             // D1 = xh . wh
              if (TWO && !SINGLE) {
                if (go_i[0]) mma_f16_i(d2 + go_d[0], ta + 16, make_desc(img0 + go_b[0]), go_i[0], 1);
                if (go_i[1]) mma_f16_i(d2 + go_d[1], ta + 16, make_desc(img0 + go_b[1]), go_i[1], 1);
                mma_f16_i(d2 + new_d, ta + 16, make_desc(img0 + 2 * 4096), idesc_n(1), 0);      // D2 = xl' . wh
              }
              constexpr int NKW0 = C::nkw(0);                   // (window 0 has three kw taps; C4: one)
              if (ng == 1) issue_window<MODE, 1, true, NKW0, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
              else if (ng == 2) issue_window<MODE, 2, true, NKW0, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
              else issue_window<MODE, 3, true, NKW0, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
            } else if (MODE == MODE_C4) {
              if (ng == 1) issue_window<MODE, 1, false, 1, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
              else if (ng == 2) issue_window<MODE, 2, false, 1, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
              else issue_window<MODE, 3, false, 1, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
            } else if (nkw == 3) {
              if (ng == 1) issue_window<MODE, 1, false, 3, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
              else if (ng == 2) issue_window<MODE, 2, false, 3, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
              else issue_window<MODE, 3, false, 3, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
            } else {                                            // P4, odd-column phase (never the first window of a step)
              if (ng == 1) issue_window<MODE, 1, false, 2, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
              else if (ng == 2) issue_window<MODE, 2, false, 2, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
              else issue_window<MODE, 3, false, 2, SINGLE>(d1, d2, g_d, ta, img0, g_b, g_i);
            }
            if (win == NWIN - 1 && u >= 2) mma_commit_raw(&tfull[(tile_base + (uint32_t)(u - 2)) % RING]);   // tile u-2 has all its kz taps
            mma_commit_raw(&aempty[aslot]);
          }
          __syncwarp();
        }
      }
      tile_base += (uint32_t)s.ntiles;
    }
    if (p.dbg && lane == 0) { long long* dd = p.dbg + blockIdx.x * 16; dd[2] = t_full; dd[3] = t_tempty; dd[4] = clock64() - t_mbegin; }
    __syncwarp();
  } else if (warp < EPI_WARP0) {
    // =============================================================== converters: 2 groups of 4 warps, alternating windows (TMEM lane
    // quadrant = warp % 4, thread = output position m).  For kw = 0,1,2: raw row m + kw*dil -> (xh | xl') -> A slot [kw].
    // (Converting every row once into a packed smem copy was measured: 800 shared-memory wavefronts per window instead of 384.)
    const int quad = warp & 3;
    const uint32_t grp = (uint32_t)(warp - CONV_WARP0) >> 2;
    const int m = quad * 32 + lane;
    const uint32_t tlane = tmem_base + ((uint32_t)(quad * 32) << 16);
    long long w_rf = 0, w_ae = 0, w_rs = 0; const long long t0 = clock64();
    uint32_t cnt = 0;                                              // windows so far (all strips)
    uint32_t tile_base = 0;                                        // (32-bit on purpose: these feed % and / on every tile)
    WS_FOR_STRIPS(sid) {
      const Strip s = decode_strip<D3>(p, sid);
      if (s.ntiles == 0) continue;
      int wcol = 0;
      if (D3) wcol = (s.cb * 128 + m) % p.W;                       // image column of output position m (same for every slice)
      for (int u = 0; u < s.ntiles + 2; ++u) {
#pragma unroll
        for (int win = 0; win < NWIN; ++win, ++cnt) {
          if ((cnt & 1) != grp) continue;
          const uint32_t sr = cnt % NR, aslot = cnt % NA;
          WSWAIT(w_rf, tc::mbar_wait(&rfull[sr], (cnt / NR) & 1));
          const unsigned char* rawp = base + sr * C::RAW_BYTES;
          const uint32_t ta = tlane + C::A_BASE + aslot * 96;
          // 2-D: this window is the centre row (kz = 1) of tile j = u - 1: its un-shifted pixels are that tile's residual
          const bool centre = MODE == MODE_2D && p.res_mode == 1 && u >= 1 && u <= s.ntiles;
          const int nkw = C::nkw(win);
          const uint32_t tcount = tile_base + (uint32_t)(u - 1);   // (only used for 1 <= u <= ntiles)
          bool a_free = false;
          if (MODE == MODE_C4) {
            // four-channel rows: pixels m, m+1, m+2 are 48 contiguous bytes = the 12 used K values (k = kw*4 + ch) of ONE K = 16 slice
            const unsigned char* rp = rawp + m * 16;
            const float4 q0 = *reinterpret_cast<const float4*>(rp), q1 = *reinterpret_cast<const float4*>(rp + 16),
                         q2 = *reinterpret_cast<const float4*>(rp + 32);
            const float xv[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
            uint32_t hl[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) hl[i] = 0u;
#pragma unroll
            for (int j = 0; j < 6; ++j) {
              const uint32_t h = pack_f16x2(xv[2 * j], xv[2 * j + 1]);
              const float2 f = unpack_f16x2(h);
              hl[j] = h;
              hl[16 + j] = pack_f16x2((xv[2 * j] - f.x) * 2048.f, (xv[2 * j + 1] - f.y) * 2048.f);
            }
            {
              const uint32_t dep = hl[0] ^ hl[2] ^ hl[4];                  // one word of each of the three loads
              __syncwarp();
              if (lane == 0) mbar_arrive_after(&rempty[sr], dep);
            }
            WSWAIT(w_ae, tc::mbar_wait(&aempty[aslot], ((cnt / NA) & 1) ^ 1));
            tc_fence_after();
            tmem_st32(ta, hl);
            a_free = true;
          } else if (C::ONCE) {
            // 3-D: nine (kh,kw) operand copies per walk step made the converters — not the tensor pipe — the bound of this kernel
            // (all converters idled: 59 -> 35 us per KITTI layer; the MMA warp waited for operands a third of the time).  So every
            // raw row is split once, IN PLACE (the 128-B fp32 row becomes the 128-B [xh | xl'] row, same swizzle), and the three
            // kw-shifted copies are plain 128-B reads: a third of the conversion arithmetic for 256 more smem wavefronts per window.
            unsigned char* rw = base + sr * C::RAW_BYTES;
            {
              unsigned char* rp = rw + m * 128;
              float4 v[8];
#pragma unroll
              for (int c = 0; c < 8; ++c) v[c] = *reinterpret_cast<const float4*>(rp + ((c ^ (m & 7)) << 4));
              if (SINGLE) {                                   // the xh half only (chunks 0..3); chunks 4..7 are never read
                uint32_t h[16];
                hi_f16(v, h);
#pragma unroll
                for (int c = 0; c < 4; ++c)
                  *reinterpret_cast<uint4*>(rp + ((c ^ (m & 7)) << 4)) = make_uint4(h[4 * c], h[4 * c + 1], h[4 * c + 2], h[4 * c + 3]);
              } else {
                uint32_t hl[32];
                split_f16(v, hl);
#pragma unroll
                for (int c = 0; c < 8; ++c)
                  *reinterpret_cast<uint4*>(rp + ((c ^ (m & 7)) << 4)) = make_uint4(hl[4 * c], hl[4 * c + 1], hl[4 * c + 2], hl[4 * c + 3]);
              }
            }
            if (quad == 3 && lane < 16) {                     // the two halo rows 128, 129: one 16-B input chunk per lane
              const int row = 128 + (lane >> 3), c = lane & 7;
              unsigned char* rp = rw + row * 128;
              const float4 x = *reinterpret_cast<const float4*>(rp + ((c ^ (row & 7)) << 4));
              const uint32_t h0 = pack_f16x2(x.x, x.y), h1 = pack_f16x2(x.z, x.w);
              uint32_t l0 = 0u, l1 = 0u;
              if (!SINGLE) {
                const float2 f0 = unpack_f16x2(h0), f1 = unpack_f16x2(h1);
                l0 = pack_f16x2((x.x - f0.x) * 2048.f, (x.y - f0.y) * 2048.f);
                l1 = pack_f16x2((x.z - f1.x) * 2048.f, (x.w - f1.y) * 2048.f);
              }
              __syncwarp(0x0000ffffu);                        // in place: every lane has read its chunk before any lane writes
              *reinterpret_cast<uint2*>(rp + (((c >> 1) ^ (row & 7)) << 4) + (c & 1) * 8) = make_uint2(h0, h1);
              if (!SINGLE) *reinterpret_cast<uint2*>(rp + (((4 + (c >> 1)) ^ (row & 7)) << 4) + (c & 1) * 8) = make_uint2(l0, l1);
            }
            fence_async_smem();                               // these generic-proxy writes precede the TMA's next write of the slot
            group_bar(7 + (int)grp);                          // the split rows of all four warps are visible
            WSWAIT(w_ae, tc::mbar_wait(&aempty[aslot], ((cnt / NA) & 1) ^ 1));
            tc_fence_after();
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
              if (kw >= nkw) break;
              const int row = m + kw;
              const unsigned char* rp = rw + row * 128;
              if (SINGLE) {                                   // xh half of the split row -> xh half of A slot [kw]
                uint32_t h[16];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                  const uint4 q = *reinterpret_cast<const uint4*>(rp + ((c ^ (row & 7)) << 4));
                  h[4 * c] = q.x; h[4 * c + 1] = q.y; h[4 * c + 2] = q.z; h[4 * c + 3] = q.w;
                }
                if (kw == nkw - 1) {
                  const uint32_t dep = h[0] ^ h[4] ^ h[8] ^ h[12];
                  __syncwarp();
                  if (lane == 0) mbar_arrive_after(&rempty[sr], dep);
                }
                if ((kw == 0 && wcol == 0) || (kw == 2 && wcol == p.W - 1)) {
#pragma unroll
                  for (int i = 0; i < 16; ++i) h[i] = 0u;
                }
                tmem_st16(ta + kw * 32, h);
                continue;
              }
              uint32_t hl[32];
#pragma unroll
              for (int c = 0; c < 8; ++c) {
                const uint4 q = *reinterpret_cast<const uint4*>(rp + ((c ^ (row & 7)) << 4));
                hl[4 * c] = q.x; hl[4 * c + 1] = q.y; hl[4 * c + 2] = q.z; hl[4 * c + 3] = q.w;
              }
              if (kw == nkw - 1) {                            // last read of the window: release it once the loads have returned
                const uint32_t dep = hl[0] ^ hl[4] ^ hl[8] ^ hl[12] ^ hl[16] ^ hl[20] ^ hl[24] ^ hl[28];
                __syncwarp();
                if (lane == 0) mbar_arrive_after(&rempty[sr], dep);
              }
              if (D3 && ((kw == 0 && wcol == 0) || (kw == 2 && wcol == p.W - 1))) {
                // un-padded flat index: this tap wrapped into the neighbouring image row -> it is zero padding
#pragma unroll
                for (int i = 0; i < 32; ++i) hl[i] = 0u;
              }
              tmem_st32(ta + kw * 32, hl);
            }
            a_free = true;
          } else
#pragma unroll
          for (int kw = 0; kw < 3; ++kw) {
            if (kw >= nkw) break;
            const int row = m + kw * p.dil;
            const unsigned char* rp = rawp + row * 128;
            float4 v[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) v[c] = *reinterpret_cast<const float4*>(rp + ((c ^ (row & 7)) << 4));
            uint32_t hl[32];
            if (SINGLE) hi_f16(v, reinterpret_cast<uint32_t (&)[16]>(hl));     // xh only: hl[0..15]
            else split_f16(v, hl);
            if (kw == nkw - 1) {                             // last read of the raw window: release it once the loads have returned
              const uint32_t dep = SINGLE ? hl[0] ^ hl[2] ^ hl[4] ^ hl[6] ^ hl[8] ^ hl[10] ^ hl[12] ^ hl[14]
                                          : hl[0] ^ hl[5] ^ hl[10] ^ hl[15] ^ hl[3] ^ hl[6] ^ hl[9] ^ hl[12];     // one word of each of the 8 loads
              __syncwarp();
              if (lane == 0) mbar_arrive_after(&rempty[sr], dep);
            }
            if (D3 && ((kw == 0 && wcol == 0) || (kw == 2 && wcol == p.W - 1))) {
              // un-padded flat index: this tap wrapped into the neighbouring image row -> it is zero padding
#pragma unroll
              for (int i = 0; i < 32; ++i) hl[i] = 0u;
            }
            if (!a_free) {
              WSWAIT(w_ae, tc::mbar_wait(&aempty[aslot], ((cnt / NA) & 1) ^ 1));
              tc_fence_after();
              a_free = true;
            }
            if (SINGLE) tmem_st16(ta + kw * 32, reinterpret_cast<const uint32_t (&)[16]>(hl));
            else tmem_st32(ta + kw * 32, hl);
            if (MODE == MODE_2D && kw == 1 && centre) {
              const int rslot = (int)(tcount % NRES);
              WSWAIT(w_rs, tc::mbar_wait(&rsempty[rslot], (uint32_t)(((tcount / NRES) & 1) ^ 1)));
              tc_fence_after();
              uint32_t raw[32];
#pragma unroll
              for (int c = 0; c < 8; ++c) {
                raw[4 * c] = __float_as_uint(v[c].x); raw[4 * c + 1] = __float_as_uint(v[c].y);
                raw[4 * c + 2] = __float_as_uint(v[c].z); raw[4 * c + 3] = __float_as_uint(v[c].w);
              }
              tmem_st32(tlane + C::RES_BASE + rslot * 32, raw);
            }
          }
          tmem_wait_st();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&afull[aslot]);
        }
      }
      tile_base += (uint32_t)s.ntiles;
    }
    if (p.dbg && warp == CONV_WARP0 && lane == 0) { long long* dd = p.dbg + blockIdx.x * 16; dd[11] = w_rf; dd[12] = w_ae; dd[13] = clock64() - t0; dd[14] = w_rs; }
  } else {
    // =============================================================== epilogue: 2 groups of 4 warps, alternating tiles (TMEM lane
    // quadrant = warp % 4, thread = position).
    const int egrp = (warp - EPI_WARP0) >> 2;
    const int ew = (warp - EPI_WARP0) & 3;
    const int quad = warp & 3;
    const int m = quad * 32 + lane;
    const int et = (tid - EPI_WARP0 * 32) & 127;
    const int chunk = et & 7, rg = et >> 3;          // coalesced pass: rows rg + 16*i, 16-B chunk `chunk`
    const uint32_t tlane = tmem_base + ((uint32_t)(quad * 32) << 16);
    const snb_conv_epilogue& e = p.e;
    const bool has_stats = !SINGLE && e.stats != nullptr;
    const float slope = e.lrelu ? SNB_LRELU_SLOPE : 1.f;
    float* red = sRed + egrp * 256;
    // Output path: the staged tile (SWIZZLE_128B image of 128 positions x 32 ch) leaves through ONE TMA tile store (positions
    // past the row / slice are clipped by the tensor map) — no read-back pass.  res_mode 2 (a residual that is not the input:
    // data gradients of the residual blocks): its tile is TMA-LOADED into the staging buffer while the tile's MMAs still run, in
    // the very layout the store uses, and every thread adds its own row in place (a coalesced read-add-store pass over global
    // memory did this before and doubled the kernel: 88 against 45 us per full-resolution data gradient).  Train-mode statistics
    // are a read-only column pass over the staged tile.
    constexpr bool tma_out = true;
    uint32_t ntile_g = 0;                                     // tiles this group has staged so far
    const int bar_id = 4 + egrp;
    asm volatile("bar.sync 6, 256;\n" ::: "memory");          // sPar (written by the first epilogue warp) is visible
    uint32_t tcount = 0;
    long long t_tfull = 0, t_px = 0, t_out = 0, t_bar = 0, t_ld = 0, t_bar2 = 0; const long long t_ebegin = clock64();
    WS_FOR_STRIPS(sid) {
      const Strip s = decode_strip<D3>(p, sid);
      const int x0 = s.cb * 128;                               // first pixel (2-D) / flat position (3-D) of the tile
      for (int j = 0; j < s.ntiles; ++j, ++tcount) {
        if ((int)(tcount & 1) != egrp) continue;
        const int slot = (int)(tcount % RING);
        const uint32_t accphase = (uint32_t)((tcount / RING) & 1);
        const int rslot = (int)(tcount % NRES);
        const int z = D3 ? s.z0 + j : s.z0 + j * p.dil;        // slice / image row of this tile
        const int lim = D3 ? HW : p.W;                         // positions x0 + r >= lim do not exist
        const size_t rowbase = D3 ? ((size_t)s.b * p.D + z) * HW : ((size_t)s.b * p.H + z) * p.W;
        float* stg = reinterpret_cast<float*>(sStg + (egrp * C::NSTG + (ntile_g % C::NSTG)) * STG_BYTES);
        if (tma_out && ntile_g >= (uint32_t)C::NSTG) {  // the TMA store that read this buffer NSTG tiles ago must have drained it
          if (et == 0) {
            if (C::NSTG == 2) asm volatile("cp.async.bulk.wait_group.read 1;\n" ::: "memory");
            else              asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory");
          }
          group_bar(bar_id);
        }
        uint64_t* rbar = &resfull[egrp * 2 + (ntile_g % C::NSTG)];
        const uint32_t rpar = (ntile_g / C::NSTG) & 1;
        if (RES2 && et == 0) {                          // residual tile -> staging buffer (zero fill past the row / slice)
          mbar_expect_tx(rbar, STG_BYTES);
          tma_load_4d(stg, &tmap_res, rbar, 0, x0, z, s.b);
        }
        ++ntile_g;
        WSWAIT(t_tfull, tc::mbar_wait(&tfull[slot], accphase));
        tc_fence_after();
        const long long tB = p.dbg ? clock64() : 0;
        {
          float acc[32], res[32];
          if (TWO && !SINGLE) {
            tmem_ld32x2(tlane + C::D1_BASE + slot * 32, tlane + C::D2_BASE + slot * 32, acc, res);
#pragma unroll
            for (int i = 0; i < 32; ++i) acc[i] = fmaf(res[i], 1.f / 2048.f, acc[i]);             // D1 + 2^-11 D2
          } else if (p.res_mode == 1) {
            tmem_ld32x2(tlane + C::D1_BASE + slot * 32, tlane + C::RES_BASE + rslot * 32, acc, res);
          } else {
            tmem_ld32(tlane + C::D1_BASE + slot * 32, acc);
          }
          if (p.dbg) t_ld += clock64() - tB;
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { mbar_arrive(&tempty[slot]); if (!TWO && p.res_mode == 1) mbar_arrive(&rsempty[rslot]); }
          float* row = stg + m * 32;
          if (RES2) tc::mbar_wait(rbar, rpar);
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const float4 a4 = *reinterpret_cast<const float4*>(sPar + 4 * c);
            const float4 b4 = *reinterpret_cast<const float4*>(sPar + 32 + 4 * c);
            float4 o;
            o.x = fmaf(acc[4 * c], a4.x, b4.x); o.y = fmaf(acc[4 * c + 1], a4.y, b4.y);
            o.z = fmaf(acc[4 * c + 2], a4.z, b4.z); o.w = fmaf(acc[4 * c + 3], a4.w, b4.w);
            o.x = o.x > 0.f ? o.x : o.x * slope; o.y = o.y > 0.f ? o.y : o.y * slope;
            o.z = o.z > 0.f ? o.z : o.z * slope; o.w = o.w > 0.f ? o.w : o.w * slope;
            if (!TWO && p.res_mode == 1) { o.x += res[4 * c]; o.y += res[4 * c + 1]; o.z += res[4 * c + 2]; o.w += res[4 * c + 3]; }
            if (RES2) {
              const float4 rr = *reinterpret_cast<const float4*>(row + ((c ^ (m & 7)) << 2));
              o.x += rr.x; o.y += rr.y; o.z += rr.z; o.w += rr.w;
            }
            *reinterpret_cast<float4*>(row + ((c ^ (m & 7)) << 2)) = o;
          }
        }
        if (p.dbg) t_px += clock64() - tB;
        if (tma_out) fence_async_smem();              // generic-proxy writes of the tile -> visible to the TMA (async proxy)
        WSWAIT(t_bar, group_bar(bar_id));             // tile staged
        const long long tC = p.dbg ? clock64() : 0;
        if (tma_out && et == 0) {
          asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];\n"
                       :: "l"(reinterpret_cast<uint64_t>(&tmap_out)), "r"(smem_u32(stg)), "r"(0), "r"(x0), "r"(z), "r"(s.b) : "memory");
          asm volatile("cp.async.bulk.commit_group;\n" ::: "memory");
        }
        float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
        if (!tma_out || has_stats)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = rg + 16 * i;
          const int xx = x0 + r;
          float4 o = *reinterpret_cast<const float4*>(stg + r * 32 + ((chunk ^ (r & 7)) << 2));
          if (xx < lim) {
            const size_t off = (rowbase + xx) * 32 + chunk * 4;
            if (has_stats) {
              s1[0] += o.x; s1[1] += o.y; s1[2] += o.z; s1[3] += o.w;
              s2[0] = fmaf(o.x, o.x, s2[0]); s2[1] = fmaf(o.y, o.y, s2[1]); s2[2] = fmaf(o.z, o.z, s2[2]); s2[3] = fmaf(o.w, o.w, s2[3]);
            }
            if (!tma_out) __stcg(reinterpret_cast<float4*>(p.y + off), o);
          }
        }
        if (has_stats) {      // one stats row per tile: 2-D [(b*H + h)*ncb + cb], 3-D [(b*D + d)*ncb + cb], each [2][32]
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            s1[c] += __shfl_xor_sync(0xffffffffu, s1[c], 8); s1[c] += __shfl_xor_sync(0xffffffffu, s1[c], 16);
            s2[c] += __shfl_xor_sync(0xffffffffu, s2[c], 8); s2[c] += __shfl_xor_sync(0xffffffffu, s2[c], 16);
          }
          if (lane < 8) {
#pragma unroll
            for (int c = 0; c < 4; ++c) { red[ew * 64 + lane * 4 + c] = s1[c]; red[ew * 64 + 32 + lane * 4 + c] = s2[c]; }
          }
          group_bar(bar_id);
          if (et < 64) {
            float a = 0.f;
#pragma unroll
            for (int wq = 0; wq < 4; ++wq) a += red[wq * 64 + et];
            const size_t trow = D3 ? ((size_t)s.b * p.D + z) * p.ncb + s.cb : ((size_t)s.b * p.H + z) * p.ncb + s.cb;
            e.stats[trow * 64 + et] = a;
          }
        }
        if (p.dbg) t_out += clock64() - tC;
        if (!tma_out || has_stats) WSWAIT(t_bar2, group_bar(bar_id));       // staging tile / stats scratch may be rewritten
      }
    }
    if (tma_out && et == 0) asm volatile("cp.async.bulk.wait_group 0;\n" ::: "memory");    // all stores complete before the CTA exits
    if (p.dbg && et == 0 && egrp == 0) { long long* d = p.dbg + blockIdx.x * 16; d[5] = t_tfull; d[6] = clock64() - t_ebegin; d[7] = t_bar; d[10] = t_out; d[15] = clock64() - t_entry; }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" :: "r"(tmem_base) : "memory");
  }
}

}  // namespace wsk

// ---- host side
static int ws_setup(const snb_conv_geom* g, wsk::Params& p, const char* who) {
  SNB_REQUIRE(g != nullptr, "%s: null geometry", who);
  SNB_REQUIRE(g->transposed == 0 && g->stride == 1 && g->KH == 3 && g->KW == 3 && (g->KD == 1 || g->KD == 3), "%s: needs a stride-1 3x3(x3) conv", who);
  SNB_REQUIRE(g->OD == g->D && g->OH == g->H && g->OW == g->W && g->ph == g->dil && g->pw == g->dil &&
              g->pd == (g->KD == 3 ? 1 : 0), "%s: needs 'same' padding", who);
  const bool d3 = g->KD == 3;
  SNB_REQUIRE(g->dil >= 1 && g->dil <= (d3 ? 1 : 16), "%s: dilation out of range", who);
  SNB_REQUIRE(d3 || g->D == 1, "%s: a 2-D conv has D = 1", who);
  p.B = g->B; p.D = g->D; p.H = g->H; p.W = g->W; p.dil = g->dil;
  p.ncb = d3 ? snb_ceil_div((long long)g->H * g->W, 128) : snb_ceil_div(g->W, 128);
  p.cmax = d3 ? g->D : snb_ceil_div(g->H, g->dil);
  // Strips: every chain of cmax tiles along the walk axis is cut into nsa strips of La tiles plus one strip of the remaining Lb
  // tiles; a strip of L tiles costs L + 2 walk steps.  (La, nsa) minimises the steps of the busiest CTA under the snake dealing of
  // strip_at() — e.g. the KITTI cost volume (58 chains of 24 slices): 2 x 10 + 4 -> 12 steps on 148 CTAs, where equal halves
  // (2 x 12) cost 14 steps on 116 CTAs.  The result is cached per (chains, cmax).
  int dev = 0, sms = 148;
  SNB_CUDA(cudaGetDevice(&dev));
  SNB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const long long nchains = (long long)g->B * p.ncb * (d3 ? 1 : g->dil);
  SNB_REQUIRE(nchains * p.cmax < (1ll << 30), "%s: too many strips", who);
  struct Plan { long long nchains; int cmax, sms, La, nsa, Lb; };
  static std::mutex mu;
  static std::vector<Plan> cache;
  Plan plan{nchains, p.cmax, sms, 0, 0, 0};
  bool hit = false;
  {
    std::lock_guard<std::mutex> lk(mu);
    for (const Plan& c : cache) if (c.nchains == nchains && c.cmax == p.cmax && c.sms == sms) { plan = c; hit = true; break; }
  }
  if (!hit) {
    long long best = -1;
    std::vector<long long> load;
    for (int La = 1; La <= p.cmax; ++La) {
      const int nsa = p.cmax / La, Lb = p.cmax - nsa * La;
      if ((La < 2 || (Lb > 0 && Lb < 2 && La > 2)) && p.cmax >= 4) continue;      // strips of one tile cost three steps: not worth looking at
      const long long nlong = nchains * nsa, ns = nlong + (Lb > 0 ? nchains : 0);
      long long cost;
      if (ns > 16ll * sms) {
        cost = ((nlong + sms - 1) / sms) * (La + 2) + (Lb > 0 ? ((nchains + sms - 1) / sms) * (Lb + 2) : 0);   // many strips: an upper bound will do
      } else {
        const int G = (int)(ns < sms ? ns : sms);
        load.assign(G, 0);
        for (long long sid = 0; sid < ns; ++sid) {
          const long long k = sid / G; const int pos = (int)(sid % G);
          load[(k & 1) ? G - 1 - pos : pos] += (sid < nlong ? La : Lb) + 2;
        }
        cost = 0;
        for (long long v : load) cost = v > cost ? v : cost;
      }
      if (best < 0 || cost < best) { best = cost; plan.La = La; plan.nsa = nsa; plan.Lb = Lb; }
    }
    std::lock_guard<std::mutex> lk(mu);
    if (cache.size() > 256) cache.clear();
    cache.push_back(plan);
  }
  p.La = plan.La; p.nsa = plan.nsa; p.Lb = plan.Lb;
  p.nchains = (int)nchains; p.nlong = (int)(nchains * p.nsa);
  const long long ns = (long long)p.nlong + (p.Lb > 0 ? nchains : 0);
  SNB_REQUIRE(ns < (1ll << 30), "%s: too many strips", who);
  p.nstrips = (int)ns;
  return 0;
}

extern "C" int snb_conv_c32_ws_num_tiles(const snb_conv_geom* g) {
  wsk::Params p;
  if (ws_setup(g, p, "snb_conv_c32_ws_num_tiles")) return -1;
  return g->KD == 3 ? p.B * p.D * p.ncb : p.B * p.H * p.ncb;          // one stats row per output tile
}

extern "C" int snb_conv_weights_ws_floats(int kd) {      // kd = 5: the ten-image set of the 5x5 stride-2 layer (MODE_P4)
  return kd == 5 ? 10 * (tc::B_BYTES / 4) + 4 : (kd == 3 ? 9 * (tc::B_BYTES / 4) + 4 : 3 * tc::WIMG_FLOATS_PER_WINDOW);
}

// p4: 0 = plain conv; 1 = MODE_P4 over a split input x = phases [4][B][OH][OW][32]; 2 = MODE_P4 over the un-split input
// x [B][in_h][in_w][32] through strided tensor maps (phase (a,b) = x[2i+a][2j+b], zero fill past the odd edge).
// single: the single-product variant of MODE_2D / MODE_3D (snb_conv_c32_ws_f16).
static int ws_launch(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                     long long* dbg, void* stream, int p4 = 0, int in_h = 0, int in_w = 0, bool c4 = false, bool single = false) {
  wsk::Params p;
  if (int rc = ws_setup(g, p, "snb_conv_c32_ws")) return rc;
  SNB_REQUIRE(x && wimg && y && e, "snb_conv_c32_ws: null pointer");
  SNB_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0, "snb_conv_c32_ws: x / y must be 16-byte aligned");
  SNB_REQUIRE(!e->scale || e->shift, "snb_conv_c32_ws: scale without shift");
  SNB_REQUIRE(!e->stats || (!e->scale && !e->lrelu && !e->residual), "snb_conv_c32_ws: statistics are taken of the plain conv + bias output");
  const bool d3 = g->KD == 3;
  SNB_REQUIRE(!p4 || (!d3 && g->dil == 1), "snb_conv5x5s2_c32_ws: bad geometry");
  SNB_REQUIRE(!c4 || (!d3 && !p4 && g->dil == 1 && !e->residual), "snb_conv_c4_ws: bad geometry");
  p.wimg = wimg; p.y = y; p.e = *e; p.dbg = dbg;
  p.res_mode = e->residual == nullptr ? 0 : ((e->residual == x && !d3 && !p4) ? 1 : 2);
  snb_encode_tiled_fn enc = snb_get_encode_tiled();
  SNB_REQUIRE(enc != nullptr, "snb_conv_c32_ws: cuTensorMapEncodeTiled is not available from the driver");
  CUtensorMap tmap, tmap_out, tmap_res;
  cuuint64_t dims[4], strides[3];
  if (d3) {
    const cuuint64_t HW = (cuuint64_t)g->H * g->W;
    dims[0] = 32; dims[1] = HW; dims[2] = (cuuint64_t)g->D; dims[3] = (cuuint64_t)g->B;
    strides[0] = 128; strides[1] = HW * 128; strides[2] = HW * 128 * (cuuint64_t)g->D;
  } else {
    dims[0] = 32; dims[1] = (cuuint64_t)g->W; dims[2] = (cuuint64_t)g->H; dims[3] = (cuuint64_t)g->B;
    strides[0] = 128; strides[1] = (cuuint64_t)g->W * 128; strides[2] = (cuuint64_t)g->W * g->H * 128;
  }
  const cuuint32_t box[4] = {32, (cuuint32_t)(128 + 2 * g->dil), 1, 1};
  const cuuint32_t box_out[4] = {32, 128, 1, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUtensorMap tmap_ph[4];
  CUresult cr = CUDA_SUCCESS;
  for (int k = 0; k < (p4 ? 4 : 1) && cr == CUDA_SUCCESS; ++k) {
    const float* base_k = x;
    cuuint64_t dk[4] = {dims[0], dims[1], dims[2], dims[3]}, sk[3] = {strides[0], strides[1], strides[2]};
    if (p4 == 1) {
      base_k = x + (size_t)k * g->B * g->H * g->W * 32;
    } else if (p4 == 2) {
      const int a = k >> 1, b = k & 1;
      base_k = x + ((size_t)a * in_w + b) * 32;
      dk[1] = (cuuint64_t)((in_w - b + 1) / 2); dk[2] = (cuuint64_t)((in_h - a + 1) / 2);
      sk[0] = 2 * 128; sk[1] = (cuuint64_t)in_w * 2 * 128; sk[2] = (cuuint64_t)in_w * in_h * 128;
    }
    cuuint32_t box_k[4] = {box[0], box[1], box[2], box[3]};
    CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B;
    if (c4) {                       // [B][H][W][4] fp32: a position row is 16 B, rows contiguous in smem, no swizzle
      dk[0] = 4; sk[0] = 16; sk[1] = (cuuint64_t)g->W * 16; sk[2] = (cuuint64_t)g->W * g->H * 16;
      box_k[0] = 4; swz = CU_TENSOR_MAP_SWIZZLE_NONE;
    }
    cr = enc(&tmap_ph[k], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base_k), dk, sk, box_k, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  }
  SNB_REQUIRE(cr == CUDA_SUCCESS, "snb_conv_c32_ws: cuTensorMapEncodeTiled failed (%d)", (int)cr);
  if (!p4) tmap_ph[1] = tmap_ph[2] = tmap_ph[3] = tmap_ph[0];
  tmap = tmap_ph[0];
  cr = enc(&tmap_out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, y, dims, strides, box_out, estr,
           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SNB_REQUIRE(cr == CUDA_SUCCESS, "snb_conv_c32_ws: cuTensorMapEncodeTiled (output) failed (%d)", (int)cr);
  tmap_res = tmap_out;
  if (p.res_mode == 2) {
    SNB_REQUIRE((reinterpret_cast<uintptr_t>(e->residual) & 15) == 0, "snb_conv_c32_ws: residual must be 16-byte aligned");
    cr = enc(&tmap_res, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(e->residual), dims, strides, box_out, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    SNB_REQUIRE(cr == CUDA_SUCCESS, "snb_conv_c32_ws: cuTensorMapEncodeTiled (residual) failed (%d)", (int)cr);
  }
  int dev = 0, sms = 148;
  SNB_CUDA(cudaGetDevice(&dev));
  SNB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int grid = p.nstrips < sms ? p.nstrips : sms;
#define WS_GO(MODEV, FOLDV, RESV, SINGLEV) do { \
    SNB_CUDA(cudaFuncSetAttribute(wsk::conv_c32_ws_kernel<MODEV, FOLDV, RESV, SINGLEV>, cudaFuncAttributeMaxDynamicSharedMemorySize, wsk::Cfg<MODEV>::SMEM_BYTES)); \
    snb_launch(wsk::conv_c32_ws_kernel<MODEV, FOLDV, RESV, SINGLEV>, grid, wsk::NTHREADS_WS, wsk::Cfg<MODEV>::SMEM_BYTES, stream, tmap, tmap_out, tmap_res, tmap_ph[1], tmap_ph[2], tmap_ph[3], p); } while (0)
  const bool res2 = p.res_mode == 2;
  if (single) {
    if (d3) { if (res2) WS_GO(wsk::MODE_3D, true, true, true); else WS_GO(wsk::MODE_3D, true, false, true); }
    else    { if (res2) WS_GO(wsk::MODE_2D, true, true, true); else WS_GO(wsk::MODE_2D, true, false, true); }
  }
  else if (c4) WS_GO(wsk::MODE_C4, true, false, false);
  else if (p4) { if (res2) WS_GO(wsk::MODE_P4, true, true, false); else WS_GO(wsk::MODE_P4, true, false, false); }
  else if (d3) { if (res2) WS_GO(wsk::MODE_3D, true, true, false); else WS_GO(wsk::MODE_3D, true, false, false); }
  else    { if (res2) WS_GO(wsk::MODE_2D, true, true, false); else WS_GO(wsk::MODE_2D, true, false, false); }
#undef WS_GO
  SNB_LAUNCH_CHECK("conv_c32_ws_kernel");
  return 0;
}

extern "C" int snb_conv_c32_ws(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                               void* stream) {
  return ws_launch(x, wimg, y, g, e, nullptr, stream);
}

// The single-product variant: same contract and weight image as snb_conv_c32_ws, out = 2^-s (xh . wh); inference only (no `stats`).
extern "C" int snb_conv_c32_ws_f16(const float* x, const float* wimg, float* y, const snb_conv_geom* g, const snb_conv_epilogue* e,
                                   void* stream) {
  SNB_REQUIRE(e != nullptr, "snb_conv_c32_ws_f16: null epilogue");
  SNB_REQUIRE(e->stats == nullptr, "snb_conv_c32_ws_f16: `stats` must be NULL (train-mode BatchNorm statistics stay on snb_conv_c32_ws)");
  return ws_launch(x, wimg, y, g, e, nullptr, stream, 0, 0, 0, false, true);
}

extern "C" int snb_conv_c32_ws_profile(const float* x, const float* wimg, float* y, const snb_conv_geom* g,
                                       const snb_conv_epilogue* e, long long* counters, void* stream) {
  SNB_REQUIRE(counters != nullptr, "snb_conv_c32_ws_profile: null counters");
  return ws_launch(x, wimg, y, g, e, counters, stream);
}

// 5x5 stride-2 pad-2 32->32 convolution (downsample[1:], stereo_net.py:64-70) over the polyphase images of its input:
// phases [4][B][OH][OW][32] (phase a*2+b holds x[2i+a][2j+b], zero where that is outside x), y [B][OH][OW][32].
extern "C" int snb_conv5x5s2_c32_ws(const float* phases, const float* wimg, float* y, int B, int OH, int OW,
                                    const snb_conv_epilogue* e, void* stream) {
  snb_conv_geom g;
  g.B = B; g.D = 1; g.H = OH; g.W = OW; g.OD = 1; g.OH = OH; g.OW = OW; g.KD = 1; g.KH = 3; g.KW = 3;
  g.stride = 1; g.dil = 1; g.pd = 0; g.ph = 1; g.pw = 1; g.transposed = 0;
  SNB_REQUIRE(e && !e->residual, "snb_conv5x5s2_c32_ws: no residual input");
  return ws_launch(phases, wimg, y, &g, e, nullptr, stream, 1);
}

// The same layer straight from the un-split input x [B][H][W][32] (H, W >= 2): the four polyphase images are strided TMA views of x,
// y [B][ceil(H/2)][ceil(W/2)][32].
extern "C" int snb_conv5x5s2_c32_ws_x(const float* x, const float* wimg, float* y, int B, int H, int W,
                                      const snb_conv_epilogue* e, void* stream) {
  SNB_REQUIRE(H >= 2 && W >= 2, "snb_conv5x5s2_c32_ws_x: needs H, W >= 2");
  snb_conv_geom g;
  const int OH = (H + 1) / 2, OW = (W + 1) / 2;
  g.B = B; g.D = 1; g.H = OH; g.W = OW; g.OD = 1; g.OH = OH; g.OW = OW; g.KD = 1; g.KH = 3; g.KW = 3;
  g.stride = 1; g.dil = 1; g.pd = 0; g.ph = 1; g.pw = 1; g.transposed = 0;
  SNB_REQUIRE(e && !e->residual, "snb_conv5x5s2_c32_ws_x: no residual input");
  return ws_launch(x, wimg, y, &g, e, nullptr, stream, 2, H, W);
}

// 3x3 'same' conv of a four-channel channels-last image x4 [B][H][W][4] -> y [B][H][W][32] (the refinement's input layer, the
// image packed by snb_refine_pack_input).  wimg: snb_prep_conv_weights_tc(kd = 1, SNB_CONV_WS) of the [32][32][3][3] tensor
// W'[co][kw*4 + ch][kh][0] = w[co][ch][kh][kw] (zero elsewhere); only its first image is read.  Epilogue as snb_conv_c32_ws
// (bias, folded BN, LeakyReLU, train-mode statistics); no residual.
extern "C" int snb_conv_c4_ws(const float* x4, const float* wimg, float* y, int B, int H, int W,
                              const snb_conv_epilogue* e, void* stream) {
  snb_conv_geom g;
  g.B = B; g.D = 1; g.H = H; g.W = W; g.OD = 1; g.OH = H; g.OW = W; g.KD = 1; g.KH = 3; g.KW = 3;
  g.stride = 1; g.dil = 1; g.pd = 0; g.ph = 1; g.pw = 1; g.transposed = 0;
  SNB_REQUIRE(e != nullptr, "snb_conv_c4_ws: null epilogue");
  return ws_launch(x4, wimg, y, &g, e, nullptr, stream, 0, 0, 0, true);
}
