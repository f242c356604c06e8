// Whole-model StereoNet inference (eval mode) behind the C-ABI: snb_stereonet_prepare derives every read-only tensor of the forward
// from the reference's parameters in one launch pair, snb_stereonet_forward issues the launch sequence of the Python eval path
// (runtime.StereoEngine._forward with the "ws" back end: models/stereo_net.py + autograd/fused.py) by calling the same launchers.
// Both sides are written to agree bit for bit; tests/test_gpu_native.py holds them to it.
//
// Host code only: every kernel it launches lives in the other translation units.  No allocation, no synchronisation, no state.
#include <vector>
#include "model.cuh"

using namespace snb_model;

namespace {

long long weights_total(const std::vector<Tensor>& t) { return t.back().off + align_up(t.back().bytes); }

// Workspace pieces, offsets in bytes.
struct Carve {
  long long fa, fb, fc, ca, cb, taps, pred, x4, up, ra, rb, total;
};

Carve carve(const Dims& d) {
  const long long N2 = 2ll * d.B, B = d.B, HW = (long long)d.H * d.W, hw = (long long)d.h * d.w;
  long long feat = N2 * d.Hs[1] * d.Ws[1] * 32, split = 0;                 // phases of downsample[0] take the same room
  for (int i = 1; i < d.k; ++i)
    if (split_layer(d, i)) {
      const long long s = 4 * N2 * ((d.Hs[i] + 1) / 2) * ((d.Ws[i] + 1) / 2) * 32;
      split = s > split ? s : split;
    }
  const long long cost = B * d.D * hw * 32;
  const long long taps = B * d.D * 27 * hw > B * 9 * HW ? B * d.D * 27 * hw : B * 9 * HW;
  Carve c;
  long long off = 0;
  auto take = [&](long long floats) { const long long o = off; off += align_up(floats * 4); return o; };
  c.fa = take(feat); c.fb = take(feat); c.fc = take(split);
  c.ca = take(cost); c.cb = take(cost);
  c.taps = take(taps); c.pred = take(B * hw);
  c.x4 = take(B * HW * 4); c.up = take(B * HW);
  c.ra = take(B * HW * 32); c.rb = take(B * HW * 32);
  c.total = off;
  return c;
}

}  // namespace

extern "C" int snb_stereonet_num_params(int k) {
  SNB_REQUIRE(k >= 1 && k <= 16, "snb_stereonet_num_params: k must be in [1, 16] (got %d)", k);
  return (int)model_tensors(k).size();
}

extern "C" long long snb_stereonet_weights_bytes(int k) {
  SNB_REQUIRE(k >= 1 && k <= 16, "snb_stereonet_weights_bytes: k must be in [1, 16] (got %d)", k);
  return weights_total(model_tensors(k));
}

extern "C" int snb_stereonet_weights_piece(int k, int index, long long* offset, long long* bytes) {
  SNB_REQUIRE(k >= 1 && k <= 16, "snb_stereonet_weights_piece: k must be in [1, 16] (got %d)", k);
  SNB_REQUIRE(offset && bytes, "snb_stereonet_weights_piece: null `offset` / `bytes`");
  const std::vector<Tensor> t = model_tensors(k);
  SNB_REQUIRE(index >= 0 && index < (int)t.size(), "snb_stereonet_weights_piece: index %d outside [0, %d)", index, (int)t.size());
  *offset = t[index].off;
  *bytes = t[index].bytes;
  return 0;
}

extern "C" int snb_stereonet_prepare(const float* const* params, int k, void* weights, void* stream) {
  SNB_REQUIRE(k >= 1 && k <= 16, "snb_stereonet_prepare: k must be in [1, 16] (got %d)", k);
  SNB_REQUIRE(params != nullptr, "snb_stereonet_prepare: null `params`");
  SNB_REQUIRE(weights != nullptr && aligned(weights, ALIGN), "snb_stereonet_prepare: `weights` must be a non-null 256-byte aligned pointer");
  const std::vector<Tensor> t = model_tensors(k);
  for (size_t i = 0; i < t.size(); ++i)
    SNB_REQUIRE(params[i] != nullptr, "snb_stereonet_prepare: `params[%d]` is null", (int)i);
  char* base = static_cast<char*>(weights);
  std::vector<snb_prep_item> items;
  for (size_t i = 0; i < t.size(); ++i) {
    const Tensor& e = t[i];
    snb_prep_item it = {params[i], {nullptr, nullptr, nullptr}, reinterpret_cast<float*>(base + e.off), 0, 0};
    switch (e.role) {
      case R_RAW: it.cfg = 5 << 16; it.count = e.numel; break;
      case R_WS2: it.cfg = 3 | SNB_CONV_WS << 8; break;
      case R_WS3: it.cfg = 9 | SNB_CONV_WS << 8; break;
      case R_P4: it.cfg = 10 | SNB_CONV_WS << 8 | 2 << 16; break;
      case R_C4: it.cfg = 3 | SNB_CONV_WS << 8 | 3 << 16; break;
      case R_BN_W:
        it.cfg = 4 << 16;
        it.aux[0] = params[i + 1]; it.aux[1] = params[i + 2]; it.aux[2] = params[i + 3];     // bias, running_mean, running_var
        break;
      case R_BN_B: case R_NONE: continue;
    }
    items.push_back(it);
  }
  return snb_prep_param_launch(items.data(), (int)items.size(), stream);
}

extern "C" long long snb_stereonet_workspace_bytes(int k, int input_scale, int maxdisp, int B, int H, int W) {
  Dims d;
  if (check_dims("snb_stereonet_workspace_bytes", k, input_scale, maxdisp, B, H, W, d)) return -1;
  return carve(d).total;
}

// Which 32->32 walk-kernel layers the reduced-precision forward runs on the single-product variant (snb_conv_c32_ws_f16).
constexpr int F16_2D = 1, F16_3D = 2;
constexpr int F16_LAYERS = F16_2D | F16_3D;

// The forward of both exported entry points: `single` = 0 (snb_stereonet_forward) or F16_LAYERS (snb_stereonet_forward_f16).
static int stereonet_forward(int single, const char* who, const void* weights, int k, int input_scale, int maxdisp,
                             const float* images, int B, int H, int W, void* workspace, float* disp, float* coarse, float* cost,
                             float* fcs, void* stream) {
  Dims d;
  if (int rc = check_dims(who, k, input_scale, maxdisp, B, H, W, d)) return rc;
  SNB_REQUIRE(weights != nullptr && aligned(weights, ALIGN), "%s: `weights` must be a non-null 256-byte aligned pointer", who);
  SNB_REQUIRE(workspace != nullptr && aligned(workspace, ALIGN), "%s: `workspace` must be a non-null 256-byte aligned pointer", who);
  SNB_REQUIRE(images != nullptr && aligned(images, 16), "%s: `images` must be a non-null 16-byte aligned pointer", who);
  SNB_REQUIRE(disp != nullptr && aligned(disp, 16), "%s: `disp` must be a non-null 16-byte aligned pointer", who);
  SNB_REQUIRE(aligned(coarse, 16), "%s: `coarse` must be 16-byte aligned", who);
  SNB_REQUIRE(aligned(cost, 16), "%s: `cost` must be 16-byte aligned", who);
  SNB_REQUIRE(aligned(fcs, 16), "%s: `fcs` must be 16-byte aligned", who);
  SNB_REQUIRE(!fcs || cost, "%s: `fcs` is computed from `cost`, which is null", who);
  SNB_REQUIRE(!fcs || d.D > 2, "%s: `fcs` needs more than 2 coarse disparity levels (maxdisp %d gives %d)", who, maxdisp, d.D);

  const std::vector<Tensor> t = model_tensors(k);
  const char* wb = static_cast<const char*>(weights);
  size_t ti = 0;                                                   // cursor over the tensors, in the order the forward reads them
  auto next = [&]() { return reinterpret_cast<const float*>(wb + t[ti++].off); };
  const Carve c = carve(d);
  char* ws = static_cast<char*>(workspace);
  auto buf = [&](long long off) { return reinterpret_cast<float*>(ws + off); };
  float *fa = buf(c.fa), *fb = buf(c.fb), *fc = buf(c.fc);
  const int N2 = 2 * B;

  // ---- feature extractor on the 2B batch [left; right] (StereoEngine._forward, FeatureExtractorNetwork.forward)
  const float* w0 = next(); const float* b0 = next();
  float* x = fa;
  if (d.phases0) {                                                 // fused.downsample_pair, even intermediate size
    if (int rc = snb_conv5x5s2_c3_phases(images, w0, b0, fa, N2, H, W, stream)) return rc;
    const float* w1 = next(); const float* b1 = next();
    snb_conv_epilogue e = {b1, nullptr, nullptr, nullptr, nullptr, 0};
    if (int rc = snb_conv5x5s2_c32_ws(fa, w1, fb, N2, d.Hs[2], d.Ws[2], &e, stream)) return rc;
    x = fb;
  } else {
    if (int rc = snb_conv5x5s2_c3(images, w0, b0, fa, N2, H, W, stream)) return rc;
  }
  for (int i = d.phases0 ? 2 : 1; i < k; ++i) {                    // fused.conv_plain -> conv5x5s2_c32
    const float* wi = next(); const float* bi = next();
    float* y = x == fa ? fb : fa;
    snb_conv_epilogue e = {bi, nullptr, nullptr, nullptr, nullptr, 0};
    if (!split_layer(d, i)) {
      if (int rc = snb_conv5x5s2_c32_ws_x(x, wi, y, N2, d.Hs[i], d.Ws[i], &e, stream)) return rc;
    } else {
      if (int rc = snb_phase_split(x, fc, N2, d.Hs[i], d.Ws[i], stream)) return rc;
      if (int rc = snb_conv5x5s2_c32_ws(fc, wi, y, N2, d.Hs[i + 1], d.Ws[i + 1], &e, stream)) return rc;
    }
    x = y;
  }
  const int h = d.h, w = d.w;
  auto conv_ws = [&](int kind) { return (single & kind) ? snb_conv_c32_ws_f16 : snb_conv_c32_ws; };
  auto conv_bn_lrelu = [&](float* in, float* out, const snb_conv_geom& g, bool residual) {
    const float* wi = next(); const float* bi = next(); const float* sc = next(); const float* sh = next();
    ti += 2;                                                       // running statistics: folded into sc / sh
    snb_conv_epilogue e = {bi, sc, sh, residual ? in : nullptr, nullptr, 1};
    return conv_ws(g.KD == 3 ? F16_3D : F16_2D)(in, wi, out, &g, &e, stream);
  };
  const snb_conv_geom gf = geom3x3(N2, 1, h, w, 1, false);
  for (int i = 0; i < 6; ++i) {                                    // BasicBlock: x + LeakyReLU(BN(conv1(x)))
    float* y = x == fa ? fb : fa;
    if (int rc = conv_bn_lrelu(x, y, gf, true)) return rc;
    x = y;
  }
  {                                                                // conv_alone
    const float* wi = next(); const float* bi = next();
    float* y = x == fa ? fb : fa;
    snb_conv_epilogue e = {bi, nullptr, nullptr, nullptr, nullptr, 0};
    if (int rc = conv_ws(F16_2D)(x, wi, y, &gf, &e, stream)) return rc;
    x = y;
  }
  const float* left = x;
  const float* right = x + (size_t)B * h * w * 32;

  // ---- stereo head (StereoNet.forward)
  float *ca = buf(c.ca), *cb = buf(c.cb);
  if (int rc = snb_cost_volume_fwd(left, right, ca, B, d.D, h, w, stream)) return rc;
  const snb_conv_geom g3 = geom3x3(B, d.D, h, w, 1, true);
  float* v = ca;
  for (int i = 0; i < 4; ++i) {
    float* y = v == ca ? cb : ca;
    if (int rc = conv_bn_lrelu(v, y, g3, false)) return rc;
    v = y;
  }
  float* taps = buf(c.taps);
  float* pred = buf(c.pred);
  {                                                                // conv3d_alone + softmax + DisparityRegression
    const float* w3 = next(); const float* b3 = next();
    if (int rc = snb_conv_c32_taps(v, w3, taps, (long long)B * d.D, h * w, 27, stream)) return rc;
    if (int rc = snb_tapsum_softargmin(taps, b3, cost, pred, B, d.D, h, w, stream)) return rc;
  }

  // ---- refinement (EdgeAwareRefinement.forward_with_up); the coarse output is the refinement's own upsampled input when the
  // factor W / w is 2^k, otherwise a separate upsample (stereo_net.py:201-202)
  const bool shared_up = W == w * (1 << k);
  float* up = (shared_up && coarse) ? coarse : buf(c.up);
  if (!shared_up && coarse)
    if (int rc = snb_upsample_bilinear(pred, coarse, B, h, w, H, W, (float)(1 << k), stream)) return rc;
  float* x4 = buf(c.x4);
  float *ra = buf(c.ra), *rb = buf(c.rb);
  if (int rc = snb_refine_pack_input(pred, images, x4, up, B, h, w, H, W, (float)((double)W / (double)w), stream)) return rc;
  {
    const float* wi = next(); const float* bi = next(); const float* sc = next(); const float* sh = next();
    ti += 2;
    snb_conv_epilogue e = {bi, sc, sh, nullptr, nullptr, 1};
    if (int rc = snb_conv_c4_ws(x4, wi, ra, B, H, W, &e, stream)) return rc;
  }
  float* r = ra;
  const int dils[6] = {1, 2, 4, 8, 1, 1};
  for (int i = 0; i < 6; ++i) {
    float* y = r == ra ? rb : ra;
    if (int rc = conv_bn_lrelu(r, y, geom3x3(B, 1, H, W, dils[i], false), true)) return rc;
    r = y;
  }
  {                                                                // conv2d_out + ReLU(up + residual)
    const float* wo = next(); const float* bo = next();
    if (int rc = snb_conv_c32_taps(r, wo, taps, B, H * W, 9, stream)) return rc;
    if (int rc = snb_tapsum_refine_out(taps, bo, up, disp, B, H, W, 1, stream)) return rc;
  }
  if (fcs)
    if (int rc = snb_feature_contrast(cost, fcs, B, d.D, h, w, stream)) return rc;
  return 0;
}

extern "C" int snb_stereonet_forward(const void* weights, int k, int input_scale, int maxdisp, const float* images, int B, int H, int W,
                                     void* workspace, float* disp, float* coarse, float* cost, float* fcs, void* stream) {
  return stereonet_forward(0, "snb_stereonet_forward", weights, k, input_scale, maxdisp, images, B, H, W, workspace, disp, coarse,
                           cost, fcs, stream);
}

extern "C" int snb_stereonet_forward_f16(const void* weights, int k, int input_scale, int maxdisp, const float* images, int B, int H,
                                         int W, void* workspace, float* disp, float* coarse, float* cost, float* fcs, void* stream) {
  return stereonet_forward(F16_LAYERS, "snb_stereonet_forward_f16", weights, k, input_scale, maxdisp, images, B, H, W, workspace, disp,
                           coarse, cost, fcs, stream);
}
