// Online adaptation behind the C-ABI (adapt.py:304-396): snb_stereonet_adapt_forward runs the train-mode forward of both images,
// the photometric loss and the feature-contrast score; snb_stereonet_adapt_update runs the backward from the activations the
// forward saved, packs every gradient into the flat bucket of optim.FusedAdamClip and applies clip + Adam.  The _replay variants
// add the experience-replay pass of adapt.py:339-349 (a second train-mode pass on a stored sample, its Khamis loss weighted into
// the total) and differentiate both passes.  All issue the launch sequence of the Python step AdaptStepper(..., FusedAdamClip,
// two_streams=False) with gradients enabled (autograd/functions.py forward + backward) through the same launchers, so both sides
// agree bit for bit; tests/test_gpu_native_adapt.py and tests/test_gpu_native_adapt_replay.py hold them to it.
//
// Four small kernels are new here: the gradient pack (layout moves + the sum of the per-pass, per-side gradients in autograd's
// order into the bucket, one launch per 64 tensors), the scaling of the replay loss gradient with the total loss, the fixed-order
// mean of the feature-contrast map, and the writer of Adam's chunk table.  Every table travels as a kernel parameter: no
// allocation, no synchronisation, no host-to-device copy.
#include <cmath>
#include <mutex>
#include <unordered_map>
#include <vector>
#include "model.cuh"

using namespace snb_model;

namespace {

// ------------------------------------------------------------------------------------------------ kernels
// dst[r * cols + c] = ((src[0] + src[1]) + src[2]) + src[3] at [r * rs + c * cs], summed left to right up to the first NULL source;
// src[0] == NULL writes zeros.  The host puts the sources in the order autograd accumulates them (see accumulation_rank).
constexpr int PACK_SRC = 4;
struct PackItem { const float* src[PACK_SRC]; float* dst; int rows, cols, rs, cs; };
constexpr int PACK_MAX = 64;
struct PackTable { PackItem it[PACK_MAX]; int n; };
static_assert(sizeof(PackTable) <= 4096, "kernel parameter block");

__global__ void __launch_bounds__(256) grad_pack_kernel(const __grid_constant__ PackTable t) {
  pdl_launch(); pdl_wait();
  const PackItem& e = t.it[blockIdx.y];
  const int n = e.rows * e.cols;
  for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) {
    const int r = i / e.cols, c = i - r * e.cols;
    const long long s = (long long)r * e.rs + (long long)c * e.cs;
    float v = e.src[0] ? e.src[0][s] : 0.f;
#pragma unroll
    for (int j = 1; j < PACK_SRC; ++j)
      if (e.src[j]) v = __fadd_rn(v, e.src[j][s]);
    e.dst[i] = v;
  }
}

// The replay term's share of the loss and its gradient (adapt.py:343-345 as AdaptStepper.step forms it): the Khamis gradient
// times autograd's incoming gradient fl(1 * er_weight), in place; total = fl(loss[0] + fl(er_weight * khamis)), unfused.
__global__ void __launch_bounds__(256) replay_scale_kernel(float* __restrict__ dpred, long long n, float er_weight,
                                                           const float* __restrict__ loss, float* __restrict__ loss_replay) {
  pdl_launch(); pdl_wait();
  const float gout = __fmul_rn(1.f, er_weight);
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
    dpred[i] = __fmul_rn(dpred[i], gout);
  if (blockIdx.x == 0 && threadIdx.x == 0) loss_replay[1] = __fadd_rn(loss[0], __fmul_rn(er_weight, loss_replay[0]));
}

// out[0] = mean of x[0..n): per-thread strided sums, then a fixed tree, all in double.
__global__ void __launch_bounds__(256) mean_kernel(const float* __restrict__ x, long long n, float* __restrict__ out) {
  pdl_launch(); pdl_wait();
  __shared__ double red[256];
  double s = 0.0;
  for (long long i = threadIdx.x; i < n; i += 256) s += (double)x[i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) { if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o]; __syncthreads(); }
  if (threadIdx.x == 0) out[0] = (float)(red[0] / (double)n);
}

// Adam's chunk table ([nchunks][3] int64 = {parameter address of the chunk, flat offset, count <= 1024}) as FusedAdamClip builds it.
struct ChunkItem { const float* p; long long off; int n, row0; };
constexpr int CHUNK_MAX = 128;
struct ChunkTable { ChunkItem it[CHUNK_MAX]; int n; };
static_assert(sizeof(ChunkTable) <= 4096, "kernel parameter block");

__global__ void chunk_table_kernel(const __grid_constant__ ChunkTable t, long long* __restrict__ table) {
  pdl_launch(); pdl_wait();
  const ChunkItem& e = t.it[blockIdx.x];
  for (int c = threadIdx.x; c * 1024 < e.n; c += blockDim.x) {
    long long* r = table + 3 * (long long)(e.row0 + c);
    r[0] = (long long)reinterpret_cast<uintptr_t>(e.p + (size_t)c * 1024);
    r[1] = e.off + (long long)c * 1024;
    r[2] = e.n - c * 1024 < 1024 ? e.n - c * 1024 : 1024;
  }
}

// ------------------------------------------------------------------------------------------------ state
constexpr int N_BN = 17;                   // BatchNorm layers the step trains, module order
constexpr float BN_MOMENTUM = 0.1f, BN_EPS = 1e-5f, SMOOTH_W = 1e-3f;

struct StateLayout {
  std::vector<Tensor> t;
  std::vector<long long> slot;             // per tensor: element offset in the bucket, -1 for the running statistics
  std::vector<long long> img_f, img_b;     // per tensor: byte offsets of the forward / data-gradient weight images, -1 if none
  long long img_b_stride = 0;              // between the four phase images of a 5x5 stride-2 layer
  long long n_total = 0, n_clip = 0;
  long long grad, m, v, step, adam_ws, table, wflip, total;
  int nchunks = 0, nused = 0;
};

StateLayout state_layout(int k) {
  StateLayout L;
  L.t = model_tensors(k);
  const int n = (int)L.t.size(), s0 = stereo_first(k);
  L.slot.assign(n, -1); L.img_f.assign(n, -1); L.img_b.assign(n, -1);
  long long off = 0;
  for (int pass = 0; pass < 2; ++pass)     // FusedAdamClip's order: stereo_net, then feature_net; parameters only
    for (int i = pass == 0 ? s0 : 0; i < (pass == 0 ? n : s0); ++i) {
      if (L.t[i].role == R_NONE) continue;
      L.slot[i] = off;
      off += L.t[i].numel;
      L.nchunks += (L.t[i].numel + 1023) / 1024;
      ++L.nused;
      if (pass == 0) L.n_clip = off;
    }
  L.n_total = off;
  long long b = 0;
  auto take = [&](long long bytes) { const long long o = b; b += align_up(bytes); return o; };
  L.grad = take(L.n_total * 4); L.m = take(L.n_total * 4); L.v = take(L.n_total * 4); L.step = take(4);
  L.adam_ws = take(snb_adam_clip_workspace_bytes());
  L.table = take(L.nchunks * 24ll);
  const long long ws1 = snb_conv_weights_ws_floats(1) * 4ll;
  L.img_b_stride = align_up(ws1);
  for (int i = 0; i < n; ++i) {
    switch (L.t[i].role) {
      case R_WS2: L.img_f[i] = take(ws1); L.img_b[i] = take(ws1); break;
      case R_WS3: L.img_f[i] = take(snb_conv_weights_ws_floats(3) * 4ll); L.img_b[i] = take(snb_conv_weights_ws_floats(3) * 4ll); break;
      case R_P4:
        L.img_f[i] = take(snb_conv_weights_ws_floats(5) * 4ll);
        L.img_b[i] = take(ws1);
        for (int a = 1; a < 4; ++a) take(ws1);
        break;
      default: break;
    }
  }
  L.wflip = take(32 * 9 * 4);
  L.total = b;
  return L;
}

// ------------------------------------------------------------------------------------------------ workspace
// Bump allocator over the caller's workspace.  With base 0 ("dry") the same code only measures: snb_stereonet_adapt_workspace_bytes
// runs the forward and the update that way, so the size it reports is by construction the high-water mark of the real calls.
struct Arena {
  uintptr_t base;
  long long off = 0, peak = 0;
  float* take(long long floats) {
    const long long o = off;
    off += align_up(floats * 4);
    peak = off > peak ? off : peak;
    return reinterpret_cast<float*>(base + o);
  }
  long long mark() const { return off; }
  void reset(long long m) { off = m; }
};

// What the forward leaves for the update (both carve it first, in the same order).
struct Saved {
  float* images;                           // copy of the input pair [2][B][3][H][W]
  float *act[2][16], *z[2][6], *y[2][6], *bn[2][6], *feat[2];    // feature passes: downsample outputs, BasicBlocks, conv_alone
  float *cv, *z3[4], *y3[4], *bn3[4], *cost, *pred, *fcs;       // stereo head
  float *up, *zr[7], *yr[7], *bnr[7], *disp, *ddisp;            // refinement (layer 0: the 4->32 input conv), loss gradient
};

Saved carve_saved(const Dims& d, Arena& ar) {
  Saved s;
  const long long B = d.B, HW = (long long)d.H * d.W, hw = (long long)d.h * d.w, cv = B * d.D * hw * 32;
  s.images = ar.take(2 * B * 3 * HW);
  for (int side = 0; side < 2; ++side) {
    for (int i = 0; i < d.k; ++i) s.act[side][i] = ar.take(B * d.Hs[i + 1] * d.Ws[i + 1] * 32);
    for (int j = 0; j < 6; ++j) { s.z[side][j] = ar.take(B * hw * 32); s.y[side][j] = ar.take(B * hw * 32); s.bn[side][j] = ar.take(128); }
    s.feat[side] = ar.take(B * hw * 32);
  }
  s.cv = ar.take(cv);
  for (int j = 0; j < 4; ++j) { s.z3[j] = ar.take(cv); s.y3[j] = ar.take(cv); s.bn3[j] = ar.take(128); }
  s.cost = ar.take(B * d.D * hw); s.pred = ar.take(B * hw); s.fcs = ar.take(B * hw);
  s.up = ar.take(B * HW);
  for (int j = 0; j < 7; ++j) { s.zr[j] = ar.take(B * HW * 32); s.yr[j] = ar.take(B * HW * 32); s.bnr[j] = ar.take(128); }
  s.disp = ar.take(B * HW); s.ddisp = ar.take(B * HW);
  return s;
}

constexpr int DILS[6] = {1, 2, 4, 8, 1, 1};

// Every launch goes through RUN: skipped when only measuring.
#define RUN(call) do { if (!dry) { if (int rc_ = (call)) return rc_; } } while (0)

// The experience-replay pass of a forward (adapt.py:339-349): a stored sample of its own batch RB (rb == 0: no replay pass) at the
// stream frame's H and W, with ground truth gt [RB][H][W] (gt <= 0: invalid); loss [2] receives {khamis term, total loss}.
struct Replay {
  int rb = 0;
  const float* images = nullptr;
  const float* gt = nullptr;
  float er_weight = 0.f;
  float* loss = nullptr;
};

Dims replay_dims(const Dims& d, int rb) {
  Dims r = d;
  r.B = rb;
  return r;
}

// The forward's workspace: the stream pass's Saved block, then the replay pass's (if any), then scratch.
int forward_impl(float* const* params, long long* const* bn_counters, const Dims& d, const float* images, const Replay& rp, char* state,
                 uintptr_t workspace, float* loss, float* disp, float* fcs, float* fcs_mean, void* stream, long long* bytes) {
  const bool dry = workspace == 0;
  const StateLayout L = state_layout(d.k);
  Arena ar{workspace};
  const Saved sv = carve_saved(d, ar);
  const Dims dr = replay_dims(d, rp.rb);
  const Saved svr = rp.rb ? carve_saved(dr, ar) : Saved{};
  auto P = [&](int i) -> const float* { return dry ? nullptr : params[i]; };
  auto IMGF = [&](int i) -> const float* { return dry ? nullptr : reinterpret_cast<const float*>(state + L.img_f[i]); };
  auto counter = [&](int j) { return bn_counters ? bn_counters[j] : nullptr; };

  // ---- WeightPrepBatch.refresh(): forward and data-gradient images of every 32->32 conv, one launch pair
  if (!dry) {
    std::vector<snb_prep_item> items;
    auto item = [&](int i, long long off, int cfg) {
      items.push_back(snb_prep_item{P(i), {nullptr, nullptr, nullptr}, reinterpret_cast<float*>(state + off), cfg, 0});
    };
    for (int i = 0; i < (int)L.t.size(); ++i) {
      switch (L.t[i].role) {
        case R_WS2: item(i, L.img_f[i], 3 | SNB_CONV_WS << 8); item(i, L.img_b[i], 3 | (1 | SNB_CONV_WS) << 8); break;
        case R_WS3: item(i, L.img_f[i], 9 | SNB_CONV_WS << 8); item(i, L.img_b[i], 9 | (1 | SNB_CONV_WS) << 8); break;
        case R_P4:
          item(i, L.img_f[i], 10 | SNB_CONV_WS << 8 | 2 << 16);
          for (int a = 0; a < 4; ++a)
            item(i, L.img_b[i] + a * L.img_b_stride, 3 | (1 | SNB_CONV_WS) << 8 | 1 << 16 | (a >> 1) << 24 | (a & 1) << 28);
          break;
        case R_C4: item(i, L.wflip, 6 << 16); break;
        default: break;
      }
    }
    RUN(snb_prep_param_launch(items.data(), (int)items.size(), stream));
  }

  // conv (+ bias, BN partial sums) -> train-mode BN (running statistics updated, counter += 1) -> [x +] LeakyReLU (ConvBnLrelu)
  auto conv_bn = [&](const float* x, float* z, float* y, float* bnv, const snb_conv_geom& g, bool residual, int ti,
                     long long* nbt) -> int {
    const long long m = ar.mark(), npos = (long long)g.B * g.D * g.H * g.W;
    const int nt = snb_conv_c32_ws_num_tiles(&g);
    float* stats = ar.take((long long)nt * 64);
    float* scratch = ar.take(64 * 64);
    snb_conv_epilogue e = {P(ti + 1), nullptr, nullptr, nullptr, stats, 0};
    RUN(snb_conv_c32_ws(x, IMGF(ti), z, &g, &e, stream));
    RUN(snb_bn_finalize_ws(stats, nt, npos, P(ti + 2), P(ti + 3), params[ti + 4], params[ti + 5], nbt, BN_MOMENTUM, BN_EPS,
                           bnv, bnv + 32, bnv + 64, bnv + 96, scratch, stream));
    RUN(snb_bn_apply(z, bnv, bnv + 32, residual ? x : nullptr, y, npos, 1, stream));
    ar.reset(m);
    return 0;
  };

  // One grad-enabled train-mode pass of the pair `images` ([2][d.B][3][H][W]) into `sv`: AdaptStepper.predict, ending in sv.disp.
  auto pass = [&](const Dims& d, const Saved& sv, const float* images) -> int {
    const int k = d.k, B = d.B, H = d.H, W = d.W, h = d.h, w = d.w, D = d.D, s0 = stereo_first(k);
    const long long HW = (long long)H * W;
    if (!dry) SNB_CUDA(cudaMemcpyAsync(sv.images, images, sizeof(float) * 2 * B * 3 * HW, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));

    // ---- feature extractor, left pass then right pass (adapt.py:72; batch-B train-mode BN statistics each)
    const snb_conv_geom gf = geom3x3(B, 1, h, w, 1, false);
    for (int side = 0; side < 2; ++side) {
      const float* img = sv.images + (size_t)side * B * 3 * HW;
      RUN(snb_conv5x5s2_c3(img, P(0), P(1), sv.act[side][0], B, H, W, stream));
      for (int i = 1; i < k; ++i) {                                 // fused.conv5x5s2_c32
        snb_conv_epilogue e = {P(2 * i + 1), nullptr, nullptr, nullptr, nullptr, 0};
        const float* wi = IMGF(2 * i);
        if (!split_layer(d, i)) {
          RUN(snb_conv5x5s2_c32_ws_x(sv.act[side][i - 1], wi, sv.act[side][i], B, d.Hs[i], d.Ws[i], &e, stream));
        } else {
          const long long m = ar.mark();
          float* ph = ar.take(4ll * B * d.Hs[i + 1] * d.Ws[i + 1] * 32);
          RUN(snb_phase_split(sv.act[side][i - 1], ph, B, d.Hs[i], d.Ws[i], stream));
          RUN(snb_conv5x5s2_c32_ws(ph, wi, sv.act[side][i], B, d.Hs[i + 1], d.Ws[i + 1], &e, stream));
          ar.reset(m);
        }
      }
      for (int j = 0; j < 6; ++j) {
        const float* x = j == 0 ? sv.act[side][k - 1] : sv.y[side][j - 1];
        if (int rc = conv_bn(x, sv.z[side][j], sv.y[side][j], sv.bn[side][j], gf, true, 2 * k + 6 * j, counter(j))) return rc;
      }
      snb_conv_epilogue e = {P(2 * k + 37), nullptr, nullptr, nullptr, nullptr, 0};   // conv_alone
      RUN(snb_conv_c32_ws(sv.y[side][5], IMGF(2 * k + 36), sv.feat[side], &gf, &e, stream));
    }

    // ---- stereo head (StereoNet.forward with grad: CostVolume, ConvBnLrelu x 4, Conv3dOutSoftargmin)
    RUN(snb_cost_volume_fwd(sv.feat[0], sv.feat[1], sv.cv, B, D, h, w, stream));
    const snb_conv_geom g3 = geom3x3(B, D, h, w, 1, true);
    for (int j = 0; j < 4; ++j)
      if (int rc = conv_bn(j == 0 ? sv.cv : sv.y3[j - 1], sv.z3[j], sv.y3[j], sv.bn3[j], g3, false, s0 + 6 * j, counter(6 + j))) return rc;
    RUN(snb_conv3d_out_softargmin(sv.y3[3], P(s0 + 24), P(s0 + 25), sv.cost, sv.pred, D > 2 ? sv.fcs : nullptr, B, D, h, w, stream));

    // ---- refinement (RefineHead, six dilated ConvBnLrelu, RefineTail); the coarse output's separate Upsample feeds nothing here
    const int r0 = s0 + 26;
    const float* left = sv.images;
    const float mul = (float)((double)W / (double)w);
    {
      const long long m = ar.mark();
      const int nt = snb_refine_in_conv_num_tiles(B, H, W);
      float* stats = ar.take((long long)nt * 64);
      float* scratch = ar.take(64 * 64);
      snb_conv_epilogue e = {P(r0 + 1), nullptr, nullptr, nullptr, stats, 0};
      RUN(snb_refine_in_conv(sv.pred, left, P(r0), sv.up, sv.zr[0], B, h, w, H, W, mul, &e, stream));
      RUN(snb_bn_finalize_ws(stats, nt, B * HW, P(r0 + 2), P(r0 + 3), params[r0 + 4], params[r0 + 5], counter(10), BN_MOMENTUM, BN_EPS,
                             sv.bnr[0], sv.bnr[0] + 32, sv.bnr[0] + 64, sv.bnr[0] + 96, scratch, stream));
      RUN(snb_bn_apply(sv.zr[0], sv.bnr[0], sv.bnr[0] + 32, nullptr, sv.yr[0], B * HW, 1, stream));
      ar.reset(m);
    }
    for (int j = 0; j < 6; ++j)
      if (int rc = conv_bn(sv.yr[j], sv.zr[j + 1], sv.yr[j + 1], sv.bnr[j + 1], geom3x3(B, 1, H, W, DILS[j], false), true,
                           r0 + 6 + 6 * j, counter(11 + j))) return rc;
    const int t0 = r0 + 42;
    {
      const long long m = ar.mark();
      float* taps = ar.take((long long)B * 9 * HW);
      RUN(snb_conv_c32_taps(sv.yr[6], P(t0), taps, B, H * W, 9, stream));
      RUN(snb_tapsum_refine_out(taps, P(t0 + 1), sv.up, sv.disp, B, H, W, 1, stream));
      ar.reset(m);
    }
    return 0;
  };

  // ---- the stream pass, its photometric loss (adapt.py:78-86) and gradient
  if (int rc = pass(d, sv, images)) return rc;
  const int B = d.B, H = d.H, W = d.W, h = d.h, w = d.w;
  const long long HW = (long long)H * W;
  {
    const long long m = ar.mark();
    float* lws = ar.take(snb_photo_loss_workspace_floats(B, H, W));
    RUN(snb_photo_loss(sv.images, sv.images + (size_t)B * 3 * HW, sv.disp, loss, sv.ddisp, lws, B, H, W, SMOOTH_W, stream));
    ar.reset(m);
  }
  // ---- the replay pass (its BatchNorm updates after the stream pass's, as in the reference), the Khamis loss and its gradient
  if (rp.rb) {
    if (int rc = pass(dr, svr, rp.images)) return rc;
    const long long n = (long long)rp.rb * HW, m = ar.mark();
    float* kws = ar.take(snb_khamis_loss_workspace_floats(n));
    RUN(snb_khamis_loss(svr.disp, rp.gt, rp.loss, svr.ddisp, kws, n, stream));
    ar.reset(m);
    if (!dry) {
      const int nb = snb_ceil_div(n, 1024);
      snb_launch(replay_scale_kernel, nb < 592 ? nb : 592, 256, 0, stream, svr.ddisp, n, rp.er_weight, (const float*)loss, rp.loss);
      SNB_LAUNCH_CHECK("replay_scale_kernel");
    }
  }
  if (!dry && disp) SNB_CUDA(cudaMemcpyAsync(disp, sv.disp, sizeof(float) * B * HW, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (!dry && fcs) SNB_CUDA(cudaMemcpyAsync(fcs, sv.fcs, sizeof(float) * B * h * w, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (fcs_mean) {
    snb_launch(mean_kernel, 1, 256, 0, stream, (const float*)sv.fcs, (long long)B * h * w, fcs_mean);
    SNB_LAUNCH_CHECK("mean_kernel");
  }
  if (bytes) *bytes = ar.peak;
  return 0;
}

// The order in which autograd adds up the gradient contributions of a parameter that several passes use.  Its engine sums them into
// one buffer as the producing nodes run, and it runs the ready node with the highest sequence number first: the replay pass's graph,
// recorded after the stream pass's, is differentiated first, and within a pass the right feature pass (recorded after the left)
// before the left one.  A feature-net parameter thus gets ((replay R + replay L) + stream R) + stream L, a stereo-net parameter
// replay + stream.  pass: 0 stream, 1 replay; side: 0 left, 1 right; the pack sums the sources in increasing rank.
int accumulation_rank(int pass, int side, int npass) { return (npass - 1 - pass) * 2 + (1 - side); }

// The update's workspace: the forward's Saved blocks, then the gradients of every pass (kept until they are packed into the
// bucket), then scratch, released phase by phase (refinement, stereo head, each feature pass) and pass by pass.  The high-water mark
// is the refinement phase: four full-resolution buffers (dres and three 32-channel gradients, ~180 MB at KITTI) on top of the Saved
// blocks; the forward needs less.  `dr`: the replay pass's dims, or NULL.  `bytes` / `grad_bytes` (measuring run): total size and
// the size of the gradient region.
int update_impl(float* const* params, const Dims& d, const Dims* dr, char* state, uintptr_t workspace, float max_norm, double lr,
                double beta1, double beta2, double eps, void* stream, long long* bytes, long long* grad_bytes) {
  const bool dry = workspace == 0;
  const StateLayout L = state_layout(d.k);
  Arena ar{workspace};
  const Saved sv = carve_saved(d, ar);
  const Saved svr = dr ? carve_saved(*dr, ar) : Saved{};
  long long gsize = 0;
  if (!dry) {
    long long total = 0;
    if (int rc = update_impl(nullptr, d, dr, nullptr, 0, 0.f, 0.0, 0.0, 0.0, 0.0, nullptr, &total, &gsize)) return rc;
  }
  Arena ga{dry ? 0 : workspace + ar.off};                         // gradients
  ar.off += gsize;
  auto P = [&](int i) -> const float* { return dry ? nullptr : params[i]; };
  auto IMGB = [&](int i) -> const float* { return dry ? nullptr : reinterpret_cast<const float*>(state + L.img_b[i]); };

  // Where each tensor's gradient ended up (per pass, and per side of the feature extractor, in accumulation_rank order) and how it
  // maps onto PyTorch's layout.
  struct Src { const float* p[PACK_SRC]; int rows, cols, rs, cs; };
  std::vector<Src> src(L.t.size(), Src{{nullptr, nullptr, nullptr, nullptr}, 0, 0, 0, 0});
  const int npass = dr ? 2 : 1;

  // The backward of one pass from its Saved block, starting at the loss gradient the forward left in sv.ddisp.
  auto pass_bwd = [&](const Dims& d, const Saved& sv, int pass) -> int {
    const int k = d.k, B = d.B, H = d.H, W = d.W, h = d.h, w = d.w, D = d.D, s0 = stereo_first(k);
    const long long HW = (long long)H * W, hw = (long long)h * w;
    const long long m_pass = ar.mark();
    auto set = [&](int i, int side, const float* p, int rows, int cols, int rs, int cs) {
      src[i].p[accumulation_rank(pass, side, npass)] = p; src[i].rows = rows; src[i].cols = cols; src[i].rs = rs; src[i].cs = cs;
    };
    auto set_id = [&](int i, int side, const float* p) { set(i, side, p, 1, L.t[i].numel, 0, 1); };

    auto reduce = [&](const float* part, int n, int len, float* out) { return snb_reduce_partials(part, n, len, out, 1.f, stream); };
    // ops.channel_sum: bias gradient of a plain convolution
    auto channel_sum = [&](const float* dy, long long npos, float* out) -> int {
      const int nb = snb_bwd_num_blocks(npos);
      const long long m = ar.mark();
      float* part = ar.take((long long)nb * 32);
      RUN(snb_channel_sum(dy, part, npos, stream));
      RUN(reduce(part, nb, 32, out));
      ar.reset(m);
      return 0;
    };
    // ops.bn_lrelu_bwd (train-mode statistics): dz, sums = {dbeta [32], dgamma [32]}, dbias
    auto bn_bwd = [&](const float* z, const float* dy, const float* bnv, long long npos, float* dz, float* sums, float* dbias) -> int {
      const int nb = snb_bwd_num_blocks(npos);
      const long long m = ar.mark();
      float* part = ar.take((long long)nb * 64);
      float* dzpart = ar.take((long long)nb * 32);
      RUN(snb_bn_lrelu_bwd_reduce(z, dy, bnv, bnv + 32, bnv + 64, bnv + 96, part, npos, 1, stream));
      RUN(reduce(part, nb, 64, sums));
      RUN(snb_bn_lrelu_bwd_apply(z, dy, bnv, bnv + 32, bnv + 64, bnv + 96, sums, npos, 1, 1, dz, dzpart, stream));
      RUN(reduce(dzpart, nb, 32, dbias));
      ar.reset(m);
      return 0;
    };
    // ConvBnLrelu.backward: dx = conv(dz, data-gradient image) [+ dy], weight gradient on the tensor cores
    auto conv_bn_bwd = [&](const float* x, const float* z, const float* bnv, const float* dy, float* dz, float* dx,
                           const snb_conv_geom& g, bool residual, int ti, int side) -> int {
      const long long npos = (long long)g.B * g.D * g.H * g.W;
      const int taps = g.KD * 9;
      float* sums = ga.take(64);
      float* dbias = ga.take(32);
      float* dw = ga.take(taps * 1024);
      if (int rc = bn_bwd(z, dy, bnv, npos, dz, sums, dbias)) return rc;
      snb_conv_epilogue e = {nullptr, nullptr, nullptr, residual ? dy : nullptr, nullptr, 0};
      RUN(snb_conv_c32_ws(dz, IMGB(ti), dx, &g, &e, stream));
      const long long m = ar.mark();
      const int n = snb_conv_c32_wgrad_tc_num_partials(&g);
      float* part = ar.take((long long)n * taps * 1024);
      RUN(snb_conv_c32_wgrad_tc(x, dz, part, &g, 3, stream));
      RUN(snb_reduce_wgrad_partials(part, n, taps, dw, stream));
      ar.reset(m);
      set_id(ti, side, dw); set_id(ti + 1, side, dbias); set_id(ti + 2, side, sums + 32); set_id(ti + 3, side, sums);
      return 0;
    };
    // Backward of a 32->1 conv (conv_c32_taps_bwd): dx, and the reduced [taps][32] weight gradient followed by the bias gradient
    auto taps_bwd = [&](const float* x, int ti, const float* g, float* dx, int Dd, int Hh, int Ww, int ntaps) -> int {
      const long long npos = (long long)B * Dd * Hh * Ww;
      const int nblk = (int)((npos + 127) / 128), len = ntaps * 32 + 1;
      float* red = ga.take(len);
      const long long m = ar.mark();
      float* part = ar.take((long long)nblk * len);
      RUN(snb_conv_c32_taps_bwd(x, P(ti), g, dx, part, B, Dd, Hh, Ww, ntaps, stream));
      RUN(reduce(part, nblk, len, red));
      ar.reset(m);
      set(ti, 0, red, 32, ntaps, 1, 32);                            // dw[c][t] = red[t * 32 + c]
      set(ti + 1, 0, red + ntaps * 32, 1, 1, 0, 1);
      return 0;
    };

    // ---- refinement: RefineTail, six dilated blocks, RefineHead (the loss gradient: the stream pass's ddisp * 1.0 = ddisp, the
    // replay pass's already scaled by the forward)
    const int r0 = s0 + 26, t0 = r0 + 42;
    const float mul = (float)((double)W / (double)w);
    float* dpred = ar.take(B * hw);                                 // read by the stereo head's backward
    const long long m_refine = ar.mark();
    float* dres = ar.take(B * HW);
    float *ra = ar.take(B * HW * 32), *rb = ar.take(B * HW * 32), *rz = ar.take(B * HW * 32);
    RUN(snb_relu_bwd(sv.disp, sv.ddisp, dres, B * HW, stream));
    if (int rc = taps_bwd(sv.yr[6], t0, dres, ra, 1, H, W, 9)) return rc;
    float *cur = ra, *nxt = rb;
    for (int j = 5; j >= 0; --j) {
      if (int rc = conv_bn_bwd(sv.yr[j], sv.zr[j + 1], sv.bnr[j + 1], cur, rz, nxt, geom3x3(B, 1, H, W, DILS[j], false), true,
                               r0 + 6 + 6 * j, 0)) return rc;
      float* t_ = cur; cur = nxt; nxt = t_;
    }
    {
      float* sums = ga.take(64);
      float* dbias = ga.take(32);
      float* dw = ga.take(36 * 32);
      if (int rc = bn_bwd(sv.zr[0], cur, sv.bnr[0], B * HW, rz, sums, dbias)) return rc;
      const long long m = ar.mark();
      const int n = snb_refine_in_conv_num_tiles(B, H, W);
      float* part = ar.take((long long)n * 36 * 32);
      RUN(snb_refine_in_wgrad(sv.pred, sv.images, rz, part, B, h, w, H, W, mul, stream));
      RUN(reduce(part, n, 36 * 32, dw));
      ar.reset(m);
      set(r0, 0, dw, 32, 36, 1, 32);                                // [ci][kh][kw][co] -> [co][ci][kh][kw]
      set_id(r0 + 1, 0, dbias); set_id(r0 + 2, 0, sums + 32); set_id(r0 + 3, 0, sums);
      float* taps = ar.take((long long)B * 9 * HW);
      float* dup = ar.take(B * HW);
      RUN(snb_conv_c32_taps(rz, reinterpret_cast<const float*>(state + L.wflip), taps, B, H * W, 9, stream));
      RUN(snb_tapsum_refine_out(taps, nullptr, dres, dup, B, H, W, 0, stream));
      RUN(snb_upsample_bilinear_bwd(dup, dpred, B, h, w, H, W, mul, stream));
    }
    ar.reset(m_refine);

    // ---- stereo head.  autograd hands Conv3dOutSoftargmin a materialised zero gradient for the unused cost output; adding those
    // zeros turns -0 into +0, so they are passed too.
    const long long cvn = B * D * hw * 32;
    float* dfeat[2] = {ar.take(B * hw * 32), ar.take(B * hw * 32)};  // read by the feature passes' backward
    const long long m_head = ar.mark();
    float* zero = ar.take(B * D * hw);
    float* dcost = ar.take(B * D * hw);
    float *ca = ar.take(cvn), *cb = ar.take(cvn), *cz = ar.take(cvn);
    if (!dry) SNB_CUDA(cudaMemsetAsync(zero, 0, sizeof(float) * B * D * hw, (cudaStream_t)stream));
    RUN(snb_softargmin_bwd(sv.cost, sv.pred, dpred, zero, dcost, B, D, h, w, stream));
    if (int rc = taps_bwd(sv.y3[3], s0 + 24, dcost, ca, D, h, w, 27)) return rc;
    cur = ca; nxt = cb;
    const snb_conv_geom g3 = geom3x3(B, D, h, w, 1, true);
    for (int j = 3; j >= 0; --j) {
      if (int rc = conv_bn_bwd(j == 0 ? sv.cv : sv.y3[j - 1], sv.z3[j], sv.bn3[j], cur, cz, nxt, g3, false, s0 + 6 * j, 0)) return rc;
      float* t_ = cur; cur = nxt; nxt = t_;
    }
    RUN(snb_cost_volume_bwd(cur, dfeat[0], dfeat[1], B, D, h, w, stream));
    ar.reset(m_head);

    // ---- feature extractor, each pass (conv_alone, BasicBlocks, downsample[k-1..1], downsample[0])
    const snb_conv_geom gf = geom3x3(B, 1, h, w, 1, false);
    for (int side = 0; side < 2; ++side) {
      const long long m_side = ar.mark();
      float *fa = ar.take(B * hw * 32), *fb = ar.take(B * hw * 32), *fz = ar.take(B * hw * 32);
      const float* dy = dfeat[side];
      {
        const int ci = 2 * k + 36;
        float* dw = ga.take(9 * 1024);
        float* db = ga.take(32);
        snb_conv_epilogue e = {nullptr, nullptr, nullptr, nullptr, nullptr, 0};
        RUN(snb_conv_c32_ws(dy, IMGB(ci), fa, &gf, &e, stream));
        const long long m = ar.mark();
        const int n = snb_conv_c32_wgrad_tc_num_partials(&gf);
        float* part = ar.take((long long)n * 9 * 1024);
        RUN(snb_conv_c32_wgrad_tc(sv.y[side][5], dy, part, &gf, 3, stream));
        RUN(snb_reduce_wgrad_partials(part, n, 9, dw, stream));
        ar.reset(m);
        if (int rc = channel_sum(dy, B * hw, db)) return rc;
        set_id(ci, side, dw); set_id(ci + 1, side, db);
      }
      float *fc = fa, *fn = fb;
      for (int j = 5; j >= 0; --j) {
        const float* x = j == 0 ? sv.act[side][k - 1] : sv.y[side][j - 1];
        if (int rc = conv_bn_bwd(x, sv.z[side][j], sv.bn[side][j], fc, fz, fn, gf, true, 2 * k + 6 * j, side)) return rc;
        float* t_ = fc; fc = fn; fn = t_;
      }
      const float* g = fc;
      for (int i = k - 1; i >= 1; --i) {                           // ConvC32.backward, 5x5 stride 2
        const int Hi = d.Hs[i], Wi = d.Ws[i], Ho = d.Hs[i + 1], Wo = d.Ws[i + 1];
        float* dx = ar.take((long long)B * Hi * Wi * 32);
        float* dw = ga.take(25 * 1024);
        float* db = ga.take(32);
        long long m = ar.mark();
        const long long phn = (long long)B * Ho * Wo * 32;
        float* ph = ar.take(4 * phn);
        const snb_conv_geom gp = geom3x3(B, 1, Ho, Wo, 1, false);
        for (int a = 0; a < 4; ++a) {
          snb_conv_epilogue e = {nullptr, nullptr, nullptr, nullptr, nullptr, 0};
          RUN(snb_conv_c32_ws(g, IMGB(2 * i) + a * (L.img_b_stride / 4), ph + a * phn, &gp, &e, stream));
        }
        RUN(snb_phase_merge(ph, dx, B, Hi, Wi, stream));
        ar.reset(m);
        snb_conv_geom g5;
        g5.B = B; g5.D = 1; g5.H = Hi; g5.W = Wi; g5.OD = 1; g5.OH = Ho; g5.OW = Wo;
        g5.KD = 1; g5.KH = 5; g5.KW = 5; g5.stride = 2; g5.dil = 1; g5.pd = 0; g5.ph = 2; g5.pw = 2; g5.transposed = 0;
        m = ar.mark();
        const int n = snb_conv_c32_wgrad_num_partials(&g5);
        float* part = ar.take((long long)n * 25 * 1024);
        RUN(snb_conv_c32_wgrad(sv.act[side][i - 1], g, part, &g5, stream));
        RUN(snb_reduce_wgrad_partials(part, n, 25, dw, stream));
        ar.reset(m);
        if (int rc = channel_sum(g, (long long)B * Ho * Wo, db)) return rc;
        set_id(2 * i, side, dw); set_id(2 * i + 1, side, db);
        g = dx;
      }
      {                                                             // Conv5x5s2First.backward
        float* dw = ga.take(75 * 32);
        float* db = ga.take(32);
        const long long m = ar.mark();
        const int n = snb_conv5x5s2_c3_num_tiles(B, H, W);
        float* part = ar.take((long long)n * 75 * 32);
        RUN(snb_conv5x5s2_c3_wgrad(sv.images + (size_t)side * B * 3 * HW, g, part, B, H, W, stream));
        RUN(reduce(part, n, 75 * 32, dw));
        ar.reset(m);
        if (int rc = channel_sum(g, (long long)B * d.Hs[1] * d.Ws[1], db)) return rc;
        set(0, side, dw, 32, 75, 1, 32);                            // [ci][kh][kw][co] -> [co][ci][kh][kw]
        set_id(1, side, db);
      }
      ar.reset(m_side);
    }
    ar.reset(m_pass);
    return 0;
  };

  if (int rc = pass_bwd(d, sv, 0)) return rc;
  if (dr)
    if (int rc = pass_bwd(*dr, svr, 1)) return rc;
  if (dry) {
    if (bytes) *bytes = ar.peak + ga.peak;
    if (grad_bytes) *grad_bytes = ga.peak;
    return 0;
  }

  // ---- the bucket (FusedAdamClip.pack: every pass's gradients summed as autograd accumulates them), then clip + Adam
  float* grad = reinterpret_cast<float*>(state + L.grad);
  std::vector<PackItem> items;
  for (size_t i = 0; i < L.t.size(); ++i) {
    if (L.slot[i] < 0) continue;
    const Src& s = src[i];
    PackItem it{{nullptr, nullptr, nullptr, nullptr}, grad + L.slot[i], 1, L.t[i].numel, 0, 1};
    int n = 0;
    for (int r = 0; r < PACK_SRC; ++r)                            // increasing rank, without the passes / sides that gave nothing
      if (s.p[r]) it.src[n++] = s.p[r];
    if (n) { it.rows = s.rows; it.cols = s.cols; it.rs = s.rs; it.cs = s.cs; }
    items.push_back(it);
  }
  for (size_t base = 0; base < items.size(); base += PACK_MAX) {
    PackTable t;
    t.n = (int)(items.size() - base < (size_t)PACK_MAX ? items.size() - base : PACK_MAX);
    int mx = 1;
    for (int i = 0; i < t.n; ++i) {
      t.it[i] = items[base + i];
      mx = t.it[i].rows * t.it[i].cols > mx ? t.it[i].rows * t.it[i].cols : mx;
    }
    snb_launch(grad_pack_kernel, dim3(snb_ceil_div(mx, 2048), t.n), 256, 0, stream, t);
    SNB_LAUNCH_CHECK("grad_pack_kernel");
  }
  return snb_adam_clip_step(reinterpret_cast<const long long*>(state + L.table), L.nchunks, grad, reinterpret_cast<float*>(state + L.m),
                            reinterpret_cast<float*>(state + L.v), reinterpret_cast<float*>(state + L.step), L.n_total, L.n_clip,
                            max_norm, 1.f, lr, beta1, beta2, eps, state + L.adam_ws, stream);
}

#undef RUN

// What the last forward on each workspace was called with, so that its update can reject other arguments before launching
// anything (an update with a larger shape than its forward's would write past a workspace sized for the forward).  Host-side and
// keyed by the workspace address: it holds under CUDA-graph capture too, where each call runs on the host once.
struct ForwardRecord {
  int k, s, maxdisp, B, H, W;
  int RB;                                  // batch of the replay pass, 0: snb_stereonet_adapt_forward (no replay pass)
  const void* state;
  std::vector<const float*> params;
};
std::mutex g_forwards_mutex;
std::unordered_map<uintptr_t, ForwardRecord> g_forwards;

void record_forward(const void* workspace, ForwardRecord r) {
  std::lock_guard<std::mutex> lock(g_forwards_mutex);
  g_forwards[reinterpret_cast<uintptr_t>(workspace)] = std::move(r);
}

// RB: the update's replay batch, 0 for snb_stereonet_adapt_update.  A replay update needs a replay forward of the same RB and a
// plain update a plain forward: the other pairings would read saved activations that are not there, or leave half of them unused.
int check_against_forward(const char* who, float* const* params, const Dims& d, int maxdisp, int RB, const void* state,
                          const void* workspace) {
  std::lock_guard<std::mutex> lock(g_forwards_mutex);
  const auto it = g_forwards.find(reinterpret_cast<uintptr_t>(workspace));
  SNB_REQUIRE(it != g_forwards.end(), "%s: no snb_stereonet_adapt_forward or _forward_replay has run on this `workspace`", who);
  const ForwardRecord& r = it->second;
  SNB_REQUIRE(RB != 0 || r.RB == 0, "%s: the forward on this workspace ran a `replay` pass (RB = %d); its update is "
              "snb_stereonet_adapt_update_replay", who, r.RB);
  SNB_REQUIRE(RB == 0 || r.RB != 0, "%s: `RB` is %d but the forward on this workspace ran no replay pass (snb_stereonet_adapt_forward)",
              who, RB);
  SNB_REQUIRE(RB == r.RB, "%s: `RB` is %d but the forward on this workspace ran with %d", who, RB, r.RB);
  const char* names[6] = {"k", "input_scale", "maxdisp", "B", "H", "W"};
  const int got[6] = {d.k, d.s, maxdisp, d.B, d.H, d.W}, want[6] = {r.k, r.s, r.maxdisp, r.B, r.H, r.W};
  for (int i = 0; i < 6; ++i)
    SNB_REQUIRE(got[i] == want[i], "%s: `%s` is %d but the forward on this workspace ran with %d", who, names[i], got[i], want[i]);
  SNB_REQUIRE(state == r.state, "%s: `state` is not the one the forward on this workspace used", who);
  for (size_t i = 0; i < r.params.size(); ++i)
    SNB_REQUIRE(params[i] == r.params[i], "%s: `params[%d]` is not the tensor the forward on this workspace read", who, (int)i);
  return 0;
}

int check_params(const char* who, float* const* params, int k) {
  SNB_REQUIRE(params != nullptr, "%s: null `params`", who);
  const int n = 2 * k + 108;
  for (int i = 0; i < n; ++i)
    SNB_REQUIRE(params[i] != nullptr && aligned(params[i], 16), "%s: `params[%d]` must be a non-null 16-byte aligned pointer", who, i);
  return 0;
}

}  // namespace

extern "C" long long snb_stereonet_adapt_state_bytes(int k) {
  SNB_REQUIRE(k >= 1 && k <= 16, "snb_stereonet_adapt_state_bytes: k must be in [1, 16] (got %d)", k);
  return state_layout(k).total;
}

extern "C" int snb_stereonet_adapt_state_piece(int k, int what, long long* offset, long long* bytes) {
  const char* who = "snb_stereonet_adapt_state_piece";
  SNB_REQUIRE(k >= 1 && k <= 16, "%s: k must be in [1, 16] (got %d)", who, k);
  SNB_REQUIRE(offset && bytes, "%s: null `offset` / `bytes`", who);
  SNB_REQUIRE(what >= 0 && what <= 3, "%s: `what` must be 0 (flat_grad), 1 (exp_avg), 2 (exp_avg_sq) or 3 (step) (got %d)", who, what);
  const StateLayout L = state_layout(k);
  const long long offs[4] = {L.grad, L.m, L.v, L.step};
  *offset = offs[what];
  *bytes = what == 3 ? 4 : L.n_total * 4;
  return 0;
}

extern "C" int snb_stereonet_adapt_grad_slot(int k, int index, long long* offset, long long* count) {
  const char* who = "snb_stereonet_adapt_grad_slot";
  SNB_REQUIRE(k >= 1 && k <= 16, "%s: k must be in [1, 16] (got %d)", who, k);
  SNB_REQUIRE(offset && count, "%s: null `offset` / `count`", who);
  const StateLayout L = state_layout(k);
  SNB_REQUIRE(index >= 0 && index < (int)L.t.size(), "%s: index %d outside [0, %d)", who, index, (int)L.t.size());
  *offset = L.slot[index] < 0 ? 0 : L.slot[index];
  *count = L.slot[index] < 0 ? 0 : L.t[index].numel;
  return 0;
}

extern "C" int snb_stereonet_adapt_init(float* const* params, int k, void* state, void* stream) {
  const char* who = "snb_stereonet_adapt_init";
  SNB_REQUIRE(k >= 1 && k <= 16, "%s: k must be in [1, 16] (got %d)", who, k);
  if (int rc = check_params(who, params, k)) return rc;
  SNB_REQUIRE(state != nullptr && aligned(state, ALIGN), "%s: `state` must be a non-null 256-byte aligned pointer", who);
  const StateLayout L = state_layout(k);
  char* st = static_cast<char*>(state);
  SNB_CUDA(cudaMemsetAsync(st, 0, L.table, (cudaStream_t)stream));        // bucket, moments, step, Adam scratch
  ChunkTable t;
  t.n = 0;
  int row = 0;
  for (int pass = 0; pass < 2; ++pass)
    for (int i = 0; i < (int)L.t.size(); ++i) {
      if (L.slot[i] < 0 || (pass == 0) != (i >= stereo_first(k))) continue;
      t.it[t.n++] = ChunkItem{params[i], L.slot[i], L.t[i].numel, row};
      row += (L.t[i].numel + 1023) / 1024;
    }
  snb_launch(chunk_table_kernel, t.n, 32, 0, stream, t, reinterpret_cast<long long*>(st + L.table));
  SNB_LAUNCH_CHECK("chunk_table_kernel");
  return 0;
}

namespace {

// Both calls' allocation sequence, measured without launching anything (RB = 0: no replay pass).
long long workspace_bytes(const char* who, int k, int input_scale, int maxdisp, int B, int H, int W, int RB) {
  Dims d;
  if (check_dims(who, k, input_scale, maxdisp, B, H, W, d)) return -1;
  const Dims dr = replay_dims(d, RB);
  Replay rp;
  rp.rb = RB;
  long long f = 0, u = 0;
  float dummy = 0.f;
  if (forward_impl(nullptr, nullptr, d, nullptr, rp, nullptr, 0, &dummy, nullptr, nullptr, nullptr, nullptr, &f)) return -1;
  if (update_impl(nullptr, d, RB ? &dr : nullptr, nullptr, 0, 0.f, 0.0, 0.0, 0.0, 0.0, nullptr, &u, nullptr)) return -1;
  return f > u ? f : u;
}

}  // namespace

extern "C" long long snb_stereonet_adapt_workspace_bytes(int k, int input_scale, int maxdisp, int B, int H, int W) {
  return workspace_bytes("snb_stereonet_adapt_workspace_bytes", k, input_scale, maxdisp, B, H, W, 0);
}

extern "C" long long snb_stereonet_adapt_replay_workspace_bytes(int k, int input_scale, int maxdisp, int B, int H, int W, int RB) {
  const char* who = "snb_stereonet_adapt_replay_workspace_bytes";
  if (RB < 1) {
    snb_fail("%s: `RB` must be >= 1 (got %d)", who, RB);
    return -1;
  }
  return workspace_bytes(who, k, input_scale, maxdisp, B, H, W, RB);
}

namespace {

// The argument checks both forwards share (before any launch), and the record their update checks against.
int check_forward(const char* who, float* const* params, long long* const* bn_counters, int k, int input_scale, int maxdisp,
                  const float* images, int B, int H, int W, void* state, void* workspace, float* loss, float* disp, float* fcs,
                  float* fcs_mean, Dims& d) {
  if (int rc = check_dims(who, k, input_scale, maxdisp, B, H, W, d)) return rc;
  if (int rc = check_params(who, params, k)) return rc;
  if (bn_counters)
    for (int j = 0; j < N_BN; ++j) SNB_REQUIRE(bn_counters[j] != nullptr, "%s: `bn_counters[%d]` is null", who, j);
  SNB_REQUIRE(state != nullptr && aligned(state, ALIGN), "%s: `state` must be a non-null 256-byte aligned pointer", who);
  SNB_REQUIRE(workspace != nullptr && aligned(workspace, ALIGN), "%s: `workspace` must be a non-null 256-byte aligned pointer", who);
  SNB_REQUIRE(images != nullptr && aligned(images, 16), "%s: `images` must be a non-null 16-byte aligned pointer", who);
  SNB_REQUIRE(loss != nullptr && aligned(loss, 4), "%s: `loss` must be a non-null 4-byte aligned pointer", who);
  SNB_REQUIRE(aligned(disp, 16), "%s: `disp` must be 16-byte aligned", who);
  SNB_REQUIRE(aligned(fcs, 16), "%s: `fcs` must be 16-byte aligned", who);
  SNB_REQUIRE(aligned(fcs_mean, 4), "%s: `fcs_mean` must be 4-byte aligned", who);
  SNB_REQUIRE((!fcs && !fcs_mean) || d.D > 2, "%s: `fcs` / `fcs_mean` need more than 2 coarse disparity levels (maxdisp %d gives %d)",
              who, maxdisp, d.D);
  return 0;
}

int check_update(const char* who, float* const* params, int k, int input_scale, int maxdisp, int B, int H, int W, int RB, void* state,
                 void* workspace, double lr, double beta1, double beta2, double eps, Dims& d) {
  if (int rc = check_dims(who, k, input_scale, maxdisp, B, H, W, d)) return rc;
  if (int rc = check_params(who, params, k)) return rc;
  SNB_REQUIRE(state != nullptr && aligned(state, ALIGN), "%s: `state` must be a non-null 256-byte aligned pointer", who);
  SNB_REQUIRE(workspace != nullptr && aligned(workspace, ALIGN), "%s: `workspace` must be a non-null 256-byte aligned pointer", who);
  SNB_REQUIRE(lr >= 0.0 && beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.0,
              "%s: `beta1` and `beta2` must be in [0, 1), `lr` and `eps` >= 0 (got %g, %g, %g, %g)", who, beta1, beta2, lr, eps);
  return check_against_forward(who, params, d, maxdisp, RB, state, workspace);
}

}  // namespace

extern "C" int snb_stereonet_adapt_forward(float* const* params, long long* const* bn_counters, int k, int input_scale, int maxdisp,
                                           const float* images, int B, int H, int W, void* state, void* workspace, float* loss,
                                           float* disp, float* fcs, float* fcs_mean, void* stream) {
  Dims d;
  if (int rc = check_forward("snb_stereonet_adapt_forward", params, bn_counters, k, input_scale, maxdisp, images, B, H, W, state,
                             workspace, loss, disp, fcs, fcs_mean, d)) return rc;
  record_forward(workspace,
                 ForwardRecord{k, input_scale, maxdisp, B, H, W, 0, state, std::vector<const float*>(params, params + 2 * k + 108)});
  return forward_impl(params, bn_counters, d, images, Replay{}, static_cast<char*>(state), reinterpret_cast<uintptr_t>(workspace), loss,
                      disp, fcs, fcs_mean, stream, nullptr);
}

extern "C" int snb_stereonet_adapt_forward_replay(float* const* params, long long* const* bn_counters, int k, int input_scale,
                                                  int maxdisp, const float* images, int B, int H, int W, const float* replay_images,
                                                  const float* replay_gt, int RB, float er_weight, void* state, void* workspace,
                                                  float* loss, float* loss_replay, float* disp, float* fcs, float* fcs_mean,
                                                  void* stream) {
  const char* who = "snb_stereonet_adapt_forward_replay";
  Dims d;
  if (int rc = check_forward(who, params, bn_counters, k, input_scale, maxdisp, images, B, H, W, state, workspace, loss, disp, fcs,
                             fcs_mean, d)) return rc;
  SNB_REQUIRE(RB >= 1, "%s: `RB` must be >= 1 (got %d)", who, RB);
  SNB_REQUIRE(replay_images != nullptr && aligned(replay_images, 16), "%s: `replay_images` must be a non-null 16-byte aligned pointer",
              who);
  SNB_REQUIRE(replay_gt != nullptr && aligned(replay_gt, 4), "%s: `replay_gt` must be a non-null 4-byte aligned pointer", who);
  SNB_REQUIRE(std::isfinite(er_weight) && er_weight >= 0.f, "%s: `er_weight` must be finite and >= 0 (got %g)", who, (double)er_weight);
  SNB_REQUIRE(loss_replay != nullptr && aligned(loss_replay, 4), "%s: `loss_replay` must be a non-null 4-byte aligned pointer", who);
  record_forward(workspace,
                 ForwardRecord{k, input_scale, maxdisp, B, H, W, RB, state, std::vector<const float*>(params, params + 2 * k + 108)});
  Replay rp;
  rp.rb = RB; rp.images = replay_images; rp.gt = replay_gt; rp.er_weight = er_weight; rp.loss = loss_replay;
  return forward_impl(params, bn_counters, d, images, rp, static_cast<char*>(state), reinterpret_cast<uintptr_t>(workspace), loss, disp,
                      fcs, fcs_mean, stream, nullptr);
}

extern "C" int snb_stereonet_adapt_update(float* const* params, int k, int input_scale, int maxdisp, int B, int H, int W, void* state,
                                          void* workspace, float max_norm, double lr, double beta1, double beta2, double eps,
                                          void* stream) {
  Dims d;
  if (int rc = check_update("snb_stereonet_adapt_update", params, k, input_scale, maxdisp, B, H, W, 0, state, workspace, lr, beta1, beta2,
                            eps, d)) return rc;
  return update_impl(params, d, nullptr, static_cast<char*>(state), reinterpret_cast<uintptr_t>(workspace), max_norm, lr, beta1, beta2,
                     eps, stream, nullptr, nullptr);
}

extern "C" int snb_stereonet_adapt_update_replay(float* const* params, int k, int input_scale, int maxdisp, int B, int H, int W, int RB,
                                                 void* state, void* workspace, float max_norm, double lr, double beta1, double beta2,
                                                 double eps, void* stream) {
  const char* who = "snb_stereonet_adapt_update_replay";
  SNB_REQUIRE(RB >= 1, "%s: `RB` must be >= 1 (got %d)", who, RB);
  Dims d;
  if (int rc = check_update(who, params, k, input_scale, maxdisp, B, H, W, RB, state, workspace, lr, beta1, beta2, eps, d)) return rc;
  const Dims dr = replay_dims(d, RB);
  return update_impl(params, d, &dr, static_cast<char*>(state), reinterpret_cast<uintptr_t>(workspace), max_norm, lr, beta1, beta2, eps,
                     stream, nullptr, nullptr);
}
