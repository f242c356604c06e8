// Fused photometric (Monodepth) loss of the adaptation step, forward AND gradient w.r.t. the predicted disparity in one
// pass — SURVEY.md §8 row f1.  Replaces ~150 PyTorch elementwise / pooling / indexing kernels per step:
//   LinearWarping.forward(right_to_left=True)   adaptive_stereo/models/linear_warping.py:18-57
//   SSIM, L1, edge-aware smoothness, monodepth  adaptive_stereo/utils/loss_functions.py:41-138
//   masked mean                                 adapt.py:78-86
//
//   I^ = grid_sample(R, (col - d, row), bilinear, border, align_corners=False)   (the reference's -0.5 px quirk included)
//   mask = normalised sample coordinate within [-1, 1]
//   loss = mean_mask[ 0.85 * mean_c SSIM_c(L, I^) + 0.15 * mean_c |L - I^| + w_s * smooth(d / (mean(d) + 1e-7), L) ]
//
// Three launches:  (1) per-batch partial sums of d;  (2) one CTA per 16x64 tile (+2 halo): warp, 3x3 moments, SSIM, L1,
// smoothness, loss partials AND the un-normalised gradient (SSIM's pooling is differentiated analytically: dSSIM/dI^' is
// affine in (L', I^') with per-centre coefficients, gathered over the 3x3 neighbourhood);  (3) finalise: deterministic
// reduction of the partials, loss = sum / count, ddisp = (g - T / ((m + eps)^2 HW)) / count  (T: the coupling of every pixel
// through the mean-normalised disparity).
#include "common.cuh"

namespace {

constexpr int TH = 16, TW = 64;                 // output tile
constexpr int R2H = TH + 4, R2W = TW + 4;       // + halo 2: warped image / left image / disparity
constexpr int R1H = TH + 2, R1W = TW + 2;       // + halo 1: SSIM centres
constexpr float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
constexpr int NSUMBLK = 64;                     // partial sums of d per batch

__global__ void __launch_bounds__(256)
disp_partial_sum_kernel(const float* __restrict__ d, float* __restrict__ part, int HW) {
  pdl_launch(); pdl_wait();
  __shared__ double red[256];
  const int b = blockIdx.y;
  const float* p = d + (size_t)b * HW;
  double s = 0.0;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < HW; i += NSUMBLK * 256) s += (double)p[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int off = 128; off > 0; off >>= 1) {
    if (threadIdx.x < off) red[threadIdx.x] += red[threadIdx.x + off];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[b * NSUMBLK + blockIdx.x] = (float)red[0];
}

__device__ __forceinline__ float mean_disp(const float* __restrict__ part, int b, int HW) {
  double s = 0.0;
  for (int i = 0; i < NSUMBLK; ++i) s += (double)part[b * NSUMBLK + i];
  return (float)(s / (double)HW);
}

// sample coordinate of linear_warping.py:41-57 + grid_sample(align_corners=False, border)
struct Warp { int x0, x1, y0, y1; float wx, wy, gmul; bool valid; };

__device__ __forceinline__ Warp warp_coord(int row, int col, float d, int H, int W) {
  Warp w;
  const float gx = (2.f * ((float)col - d)) / (float)W - 1.f;
  const float gy = (2.f * (float)row) / (float)H - 1.f;
  w.valid = gx >= -1.f && gx <= 1.f && gy >= -1.f && gy <= 1.f;
  float ix = ((gx + 1.f) * (float)W - 1.f) * 0.5f;
  float iy = ((gy + 1.f) * (float)H - 1.f) * 0.5f;
  w.gmul = 1.f;                                   // clip_coordinates_set_grad: zero gradient where the coordinate is clamped
  if (ix <= 0.f) { ix = 0.f; w.gmul = 0.f; } else if (ix >= (float)(W - 1)) { ix = (float)(W - 1); w.gmul = 0.f; }
  if (iy <= 0.f) iy = 0.f; else if (iy >= (float)(H - 1)) iy = (float)(H - 1);
  const float fx = floorf(ix), fy = floorf(iy);
  w.x0 = (int)fx; w.y0 = (int)fy; w.x1 = w.x0 + 1; w.y1 = w.y0 + 1;
  w.wx = ix - fx; w.wy = iy - fy;
  return w;
}

__global__ void __launch_bounds__(256)
photo_loss_tile_kernel(const float* __restrict__ left, const float* __restrict__ right, const float* __restrict__ disp,
                       const float* __restrict__ dsum_part, float* __restrict__ g_out, float* __restrict__ part,
                       int H, int W, float smooth_w) {
  pdl_launch(); pdl_wait();
  extern __shared__ float sm[];
  float* sL = sm;                              // [3][R2H*R2W]   left image (0 outside the image = avg_pool zero padding)
  float* sI = sL + 3 * R2H * R2W;              // [3][R2H*R2W]   warped right image
  float* sD = sI + 3 * R2H * R2W;              // [R2H*R2W]      disparity
  float* sDI = sD + R2H * R2W;                 // [3][TH*TW]     dI^/dd of the tile pixels
  float* sK = sDI + 3 * TH * TW;               // [9][R1H*R1W]   w_p * (K0, K1, K2) per channel at the SSIM centres
  float* sM = sK + 9 * R1H * R1W;              // [R2H*R2W]      valid mask (0/1)
  __shared__ double red[3][8];

  const int t = threadIdx.x;
  const int b = blockIdx.z;
  const int y0 = blockIdx.y * TH, x0 = blockIdx.x * TW;
  const int HW = H * W;
  const float* Lb = left + (size_t)b * 3 * HW;
  const float* Rb = right + (size_t)b * 3 * HW;
  const float* Db = disp + (size_t)b * HW;
  const float m_eps = mean_disp(dsum_part, b, HW) + 1e-7f;

  // ---- 1. region + halo 2: disparity, mask, left image, warped right image
  for (int i = t; i < R2H * R2W; i += 256) {
    const int ry = i / R2W, rx = i - ry * R2W;
    const int y = y0 + ry - 2, x = x0 + rx - 2;
    float d = 0.f, mk = 0.f, l0 = 0.f, l1 = 0.f, l2 = 0.f, i0 = 0.f, i1 = 0.f, i2 = 0.f;
    if ((unsigned)y < (unsigned)H && (unsigned)x < (unsigned)W) {
      d = Db[y * W + x];
      const Warp w = warp_coord(y, x, d, H, W);
      mk = w.valid ? 1.f : 0.f;
      const int o = y * W + x;
      l0 = Lb[o]; l1 = Lb[HW + o]; l2 = Lb[2 * HW + o];
      const int xa = w.x0, xb = min(w.x1, W - 1), ya = w.y0, yb = min(w.y1, H - 1);
      const float wxb = (w.x1 <= W - 1) ? w.wx : 0.f, wyb = (w.y1 <= H - 1) ? w.wy : 0.f;       // out-of-bounds corners weigh 0
      const float w00 = (1.f - w.wx) * (1.f - w.wy), w01 = wxb * (1.f - w.wy), w10 = (1.f - w.wx) * wyb, w11 = wxb * wyb;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float* Rc = Rb + (size_t)c * HW;
        const float r00 = Rc[ya * W + xa], r01 = Rc[ya * W + xb], r10 = Rc[yb * W + xa], r11 = Rc[yb * W + xb];
        const float v = r00 * w00 + r01 * w01 + r10 * w10 + r11 * w11;
        if (c == 0) i0 = v; else if (c == 1) i1 = v; else i2 = v;
        const int ty = ry - 2, tx = rx - 2;
        if ((unsigned)ty < (unsigned)TH && (unsigned)tx < (unsigned)TW) {
          // d ix / dd = -1 (where not clamped):  dI^/dd = -gmul * [(1-wy)(r01 - r00) + wy (r11 - r10)] with OOB corners dropped
          const float gx = (w.x1 <= W - 1) ? ((1.f - w.wy) * (r01 - r00) + wyb * (r11 - r10)) : 0.f;
          sDI[c * TH * TW + ty * TW + tx] = -w.gmul * gx;
        }
      }
    }
    sD[i] = d; sM[i] = mk;
    sL[i] = l0; sL[R2H * R2W + i] = l1; sL[2 * R2H * R2W + i] = l2;
    sI[i] = i0; sI[R2H * R2W + i] = i1; sI[2 * R2H * R2W + i] = i2;
  }
  __syncthreads();

  // ---- 2. SSIM centres (tile + halo 1): 3x3 moments, value (tile pixels only) and gradient coefficients
  double loss_acc = 0.0, cnt_acc = 0.0, t_acc = 0.0;
  for (int i = t; i < R1H * R1W; i += 256) {
    const int ry = i / R1W, rx = i - ry * R1W;            // R1 coords; R2 coords = +1
    const int y = y0 + ry - 1, x = x0 + rx - 1;
    const bool inimg = (unsigned)y < (unsigned)H && (unsigned)x < (unsigned)W;
    const int c2 = (ry + 1) * R2W + (rx + 1);
    const float mk = inimg ? sM[c2] : 0.f;
    const bool intile = ry >= 1 && ry <= TH && rx >= 1 && rx <= TW;
    float ssim_sum = 0.f, l1_sum = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float* Lc = sL + c * R2H * R2W; const float* Ic = sI + c * R2H * R2W;
      float sx = 0.f, sy = 0.f, sxx = 0.f, syy = 0.f, sxy = 0.f;
#pragma unroll
      for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
          const float l = Lc[c2 + dy * R2W + dx], v = Ic[c2 + dy * R2W + dx];
          sx += l; sy += v; sxx = fmaf(l, l, sxx); syy = fmaf(v, v, syy); sxy = fmaf(l, v, sxy);
        }
      const float mux = sx * (1.f / 9.f), muy = sy * (1.f / 9.f);
      const float sgx = sxx * (1.f / 9.f) - mux * mux, sgy = syy * (1.f / 9.f) - muy * muy, sgxy = sxy * (1.f / 9.f) - mux * muy;
      const float a = 2.f * mux * muy + C1, bb = 2.f * sgxy + C2;
      const float cc = mux * mux + muy * muy + C1, e = sgx + sgy + C2;
      const float n = a * bb, dn = cc * e;
      const float raw = (1.f - n / dn) * 0.5f;
      const float val = fminf(fmaxf(raw, 0.f), 1.f);
      const float wgt = (inimg && raw >= 0.f && raw <= 1.f) ? mk * (0.85f / 3.f) : 0.f;
      const float inv = 1.f / dn;
      sK[(3 * c + 0) * R1H * R1W + i] = wgt * (-(1.f / 9.f)) * (mux * (bb - a) * inv - n * muy * (e - cc) * inv * inv);
      sK[(3 * c + 1) * R1H * R1W + i] = wgt * (-a * inv * (1.f / 9.f));
      sK[(3 * c + 2) * R1H * R1W + i] = wgt * (n * cc * inv * inv * (1.f / 9.f));
      ssim_sum += val;
      l1_sum += fabsf(Lc[c2] - Ic[c2]);
    }
    if (intile && inimg) {
      loss_acc += (double)(mk * (0.85f * ssim_sum * (1.f / 3.f) + 0.15f * l1_sum * (1.f / 3.f)));
      cnt_acc += (double)mk;
    }
  }
  __syncthreads();

  // ---- 3. tile pixels: gradient through SSIM/L1/warp, smoothness value and gradient
  const float inv_m = 1.f / m_eps;
  for (int i = t; i < TH * TW; i += 256) {
    const int ty = i / TW, tx = i - ty * TW;
    const int y = y0 + ty, x = x0 + tx;
    if (y >= H || x >= W) continue;
    const int c2 = (ty + 2) * R2W + (tx + 2), c1 = (ty + 1) * R1W + (tx + 1);
    const float mk = sM[c2];
    float g = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float k0 = 0.f, k1 = 0.f, k2 = 0.f;
#pragma unroll
      for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
          const int q = c1 + dy * R1W + dx;
          k0 += sK[(3 * c + 0) * R1H * R1W + q]; k1 += sK[(3 * c + 1) * R1H * R1W + q]; k2 += sK[(3 * c + 2) * R1H * R1W + q];
        }
      const float l = sL[c * R2H * R2W + c2], v = sI[c * R2H * R2W + c2];
      float gi = k0 + k1 * l + k2 * v;
      const float df = v - l;
      gi += mk * (0.15f / 3.f) * (df > 0.f ? 1.f : (df < 0.f ? -1.f : 0.f));
      g = fmaf(gi, sDI[c * TH * TW + i], g);
    }
    // edge-aware smoothness on dn = d / (mean + eps)   (loss_functions.py:64-75,106-138).  Each difference of dn is taken as
    // (d_a - d_b) * inv_m: its sign is exact and it is 0 exactly where d_a == d_b, as in the reference.  (d_a * inv_m -
    // d_b * inv_m contracts to an FMA that leaves the rounding error of d_a * inv_m, of either sign, for equal disparities.)
    const float d0 = sD[c2];
    float sval = 0.f, h = 0.f;
    auto edge = [&](int q2a, int q2b) {           // exp(-mean_c |L(a) - L(b)|)
      const float e0 = fabsf(sL[q2a] - sL[q2b]), e1 = fabsf(sL[R2H * R2W + q2a] - sL[R2H * R2W + q2b]),
                  e2 = fabsf(sL[2 * R2H * R2W + q2a] - sL[2 * R2H * R2W + q2b]);
      return __expf(-(e0 + e1 + e2) * (1.f / 3.f));
    };
    auto sgn = [](float v) { return v > 0.f ? 1.f : (v < 0.f ? -1.f : 0.f); };
    if (x + 1 < W) { const float df = (d0 - sD[c2 + 1]) * inv_m; const float ex = edge(c2, c2 + 1); sval += fabsf(df) * ex; h += mk * sgn(df) * ex; }
    if (y + 1 < H) { const float df = (d0 - sD[c2 + R2W]) * inv_m; const float ey = edge(c2, c2 + R2W); sval += fabsf(df) * ey; h += mk * sgn(df) * ey; }
    if (x >= 1) { const float df = (sD[c2 - 1] - d0) * inv_m; h -= sM[c2 - 1] * sgn(df) * edge(c2 - 1, c2); }
    if (y >= 1) { const float df = (sD[c2 - R2W] - d0) * inv_m; h -= sM[c2 - R2W] * sgn(df) * edge(c2 - R2W, c2); }
    loss_acc += (double)(mk * smooth_w * sval);
    t_acc += (double)(smooth_w * h * sD[c2]);
    g_out[(size_t)b * HW + y * W + x] = g + smooth_w * h * inv_m;
  }

  // ---- 4. block partials: [loss, count, T]
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    loss_acc += __shfl_xor_sync(0xffffffffu, loss_acc, o);
    cnt_acc += __shfl_xor_sync(0xffffffffu, cnt_acc, o);
    t_acc += __shfl_xor_sync(0xffffffffu, t_acc, o);
  }
  if ((t & 31) == 0) { red[0][t >> 5] = loss_acc; red[1][t >> 5] = cnt_acc; red[2][t >> 5] = t_acc; }
  __syncthreads();
  if (t < 3) {
    double s = 0.0;
    for (int i = 0; i < 8; ++i) s += red[t][i];
    const int blk = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    part[blk * 4 + t] = (float)s;
  }
}

// loss = sum / count;  ddisp = (g - T_b / ((m_b + eps)^2 HW)) / count (0 when count is 0).  Every block re-reduces the (few
// hundred) partials in the same fixed order, so the result is deterministic and needs no extra launch.
__global__ void __launch_bounds__(256)
photo_loss_finalize_kernel(const float* __restrict__ part, const float* __restrict__ dsum_part, float* __restrict__ g,
                           float* __restrict__ loss_out, int B, int HW, int blocks_per_batch) {
  pdl_launch(); pdl_wait();
  __shared__ double sh[3];
  __shared__ double red[256];
  const int b = blockIdx.y, t = threadIdx.x;
  const int nblk = B * blocks_per_batch;
  for (int q = 0; q < 3; ++q) {
    double s = 0.0;
    const int lo = (q == 2) ? b * blocks_per_batch : 0, hi = (q == 2) ? (b + 1) * blocks_per_batch : nblk;
    for (int i = lo + t; i < hi; i += 256) s += (double)part[i * 4 + q];
    red[t] = s;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
      if (t < off) red[t] += red[t + off];
      __syncthreads();
    }
    if (t == 0) sh[q] = red[0];
    __syncthreads();
  }
  const double cnt = sh[1];
  // an empty mask: the reference's total[mask].mean() is NaN with an all-zero gradient, so the loss stays 0/0 and the
  // gradient scale is 0 (every g and the coupling are 0 there; 1/0 would turn them into NaN)
  const float inv_cnt = cnt > 0.0 ? (float)(1.0 / cnt) : 0.f;
  const float m_eps = mean_disp(dsum_part, b, HW) + 1e-7f;
  const float coupling = (float)(sh[2] / ((double)m_eps * (double)m_eps * (double)HW));
  if (blockIdx.x == 0 && b == 0 && t == 0) loss_out[0] = (float)(sh[0] / cnt);
  if (blockIdx.x == 0) {                       // masked mean over sample b alone -> loss_out[1 + b] (OVS validation, adapt.py:122-142)
    for (int q = 0; q < 2; ++q) {
      double s = 0.0;
      for (int i = b * blocks_per_batch + t; i < (b + 1) * blocks_per_batch; i += 256) s += (double)part[i * 4 + q];
      red[t] = s;
      __syncthreads();
      for (int off = 128; off > 0; off >>= 1) {
        if (t < off) red[t] += red[t + off];
        __syncthreads();
      }
      if (t == 0) sh[q] = red[0];
      __syncthreads();
    }
    if (t == 0) loss_out[1 + b] = (float)(sh[0] / sh[1]);
  }
  float* gb = g + (size_t)b * HW;
  for (int i = blockIdx.x * 256 + t; i < HW; i += gridDim.x * 256) gb[i] = (gb[i] - coupling) * inv_cnt;
}

}  // namespace

extern "C" int snb_photo_loss_workspace_floats(int B, int H, int W) {
  const int tiles = snb_ceil_div(W, TW) * snb_ceil_div(H, TH);
  return B * NSUMBLK + B * tiles * 4;
}

extern "C" int snb_photo_loss(const float* left, const float* right, const float* disp, float* loss_out, float* ddisp,
                              float* workspace, int B, int H, int W, float smooth_w, void* stream) {
  SNB_REQUIRE(left && right && disp && loss_out && ddisp && workspace && B > 0 && H > 1 && W > 1, "snb_photo_loss: bad args");
  cudaStream_t st = (cudaStream_t)stream;
  const int HW = H * W;
  float* dsum = workspace;
  float* part = workspace + B * NSUMBLK;
  snb_launch(disp_partial_sum_kernel, dim3(NSUMBLK, B), 256, 0, st, disp, dsum, HW);
  SNB_LAUNCH_CHECK("disp_partial_sum_kernel");
  const dim3 grid(snb_ceil_div(W, TW), snb_ceil_div(H, TH), B);
  const int smem = (3 * R2H * R2W * 2 + R2H * R2W * 2 + 3 * TH * TW + 9 * R1H * R1W) * 4;
  SNB_CUDA(cudaFuncSetAttribute(photo_loss_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  snb_launch(photo_loss_tile_kernel, grid, 256, smem, st, left, right, disp, dsum, ddisp, part, H, W, smooth_w);
  SNB_LAUNCH_CHECK("photo_loss_tile_kernel");
  snb_launch(photo_loss_finalize_kernel, dim3(148, B), 256, 0, st, part, dsum, ddisp, loss_out, B, HW, (int)(grid.x * grid.y));
  SNB_LAUNCH_CHECK("photo_loss_finalize_kernel");
  return 0;
}
