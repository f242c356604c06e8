// Host-side description of the whole model shared by the inference (model.cu) and adaptation (adapt.cu) entry points: the
// parameter list in the reference's state_dict order, the shape bookkeeping of the forward, and small argument helpers.
#pragma once
#include <vector>
#include "common.cuh"

namespace snb_model {

// What one tensor of the parameter list leaves in the prepared-weights buffer.
enum Role {
  R_RAW,      // copied as is (biases, downsample[0], the 32->1 layers' taps)
  R_WS2,      // "ws" image of a 3x3 32->32 conv (snb_conv_weights_ws_floats(1))
  R_WS3,      // "ws" image of a 3x3x3 32->32 conv (snb_conv_weights_ws_floats(3))
  R_P4,       // ten-image set of a 5x5 stride-2 32->32 conv (snb_conv_weights_ws_floats(5))
  R_C4,       // image of the refinement's 4->32 input conv (same size as R_WS2)
  R_BN_W,     // BatchNorm weight: folded scale [32]
  R_BN_B,     // BatchNorm bias: folded shift [32] (written by the fold of the preceding R_BN_W)
  R_NONE,     // running statistics: read by the fold, nothing of their own
};

struct Tensor { Role role; int numel; long long off, bytes; };

constexpr long long ALIGN = 256;
inline long long align_up(long long v) { return (v + ALIGN - 1) / ALIGN * ALIGN; }

// The tensors of the eval forward in the reference's state_dict order (feature_net, then stereo_net), BasicBlock.conv2.* and
// num_batches_tracked left out; with their pieces of the prepared-weights buffer.
inline std::vector<Tensor> model_tensors(int k) {
  std::vector<Tensor> t;
  auto add = [&](Role r, int numel) { t.push_back(Tensor{r, numel, 0, 0}); };
  auto convbn = [&](Role r, int numel) {
    add(r, numel); add(R_RAW, 32);
    add(R_BN_W, 32); add(R_BN_B, 32); add(R_NONE, 32); add(R_NONE, 32);
  };
  add(R_RAW, 32 * 3 * 25); add(R_RAW, 32);                                // downsample.0
  for (int i = 1; i < k; ++i) { add(R_P4, 32 * 32 * 25); add(R_RAW, 32); }  // downsample.i
  for (int i = 0; i < 6; ++i) convbn(R_WS2, 32 * 32 * 9);                   // residual_blocks.i.conv1.0
  add(R_WS2, 32 * 32 * 9); add(R_RAW, 32);                                 // conv_alone
  for (int i = 0; i < 4; ++i) convbn(R_WS3, 32 * 32 * 27);                  // filter.i.0
  add(R_RAW, 27 * 32); add(R_RAW, 1);                                      // conv3d_alone
  convbn(R_C4, 32 * 4 * 9);                                                // edge_aware_refinements.0.conv2d_feature.0
  for (int i = 0; i < 6; ++i) convbn(R_WS2, 32 * 32 * 9);                   // .residual_astrous_blocks.i.conv1.0
  add(R_RAW, 9 * 32); add(R_RAW, 1);                                       // .conv2d_out
  long long off = 0;
  for (Tensor& e : t) {
    long long floats = 0;
    switch (e.role) {
      case R_RAW: floats = e.numel; break;
      case R_WS2: case R_C4: floats = snb_conv_weights_ws_floats(1); break;
      case R_WS3: floats = snb_conv_weights_ws_floats(3); break;
      case R_P4: floats = snb_conv_weights_ws_floats(5); break;
      case R_BN_W: case R_BN_B: floats = 32; break;
      case R_NONE: floats = 0; break;
    }
    e.off = off;
    e.bytes = floats * 4;
    off += align_up(e.bytes);               // R_BN_B lands 256 bytes after its R_BN_W: the fold writes shift at scale + 64 floats
  }
  return t;
}

// Index of the first stereo_net tensor in model_tensors(k): downsample 2k, six BasicBlocks of six tensors, conv_alone 2.
inline int stereo_first(int k) { return 2 * k + 38; }

// Sizes of the forward's intermediates.
struct Dims {
  int B, H, W, k, s, D;           // D = coarse disparity levels
  int Hs[32], Ws[32];             // resolution after i downsampling layers
  int h, w;
  bool phases0;                   // downsample[0] writes the polyphase images downsample[1] reads
};

inline bool split_layer(const Dims& d, int i) { return d.Hs[i] < 2 || d.Ws[i] < 2; }   // downsample[i] input too small for strided views

inline int check_dims(const char* who, int k, int input_scale, int maxdisp, int B, int H, int W, Dims& d) {
  SNB_REQUIRE(k >= 1 && k <= 16, "%s: k must be in [1, 16] (got %d)", who, k);
  SNB_REQUIRE(input_scale >= 0 && input_scale + k <= 30, "%s: input_scale must be >= 0 with input_scale + k <= 30 (got %d)", who,
              input_scale);
  SNB_REQUIRE(B > 0 && H > 0 && W > 0, "%s: B, H, W must be positive (got %d, %d, %d)", who, B, H, W);
  SNB_REQUIRE(maxdisp >= 0, "%s: maxdisp must be >= 0 (got %d)", who, maxdisp);
  const long long D = ((long long)maxdisp + 1) >> (input_scale + k);          // stereo_net.py:169
  SNB_REQUIRE(D >= 1 && D <= 32, "%s: maxdisp %d gives %lld coarse disparity levels at scale %d; 1 to 32 are supported", who,
              maxdisp, D, input_scale + k);
  d.B = B; d.H = H; d.W = W; d.k = k; d.s = input_scale; d.D = (int)D;
  d.Hs[0] = H; d.Ws[0] = W;
  for (int i = 0; i < k; ++i) { d.Hs[i + 1] = (d.Hs[i] - 1) / 2 + 1; d.Ws[i + 1] = (d.Ws[i] - 1) / 2 + 1; }
  d.h = d.Hs[k]; d.w = d.Ws[k];
  d.phases0 = k >= 2 && d.Hs[1] % 2 == 0 && d.Ws[1] % 2 == 0;             // fused.downsample_pair
  return 0;
}

inline snb_conv_geom geom3x3(int B, int D, int H, int W, int dil, bool three_d) {     // ops.geom(..., 3, dil=dil): stride-1 'same'
  snb_conv_geom g;
  g.B = B; g.D = D; g.H = H; g.W = W; g.OD = D; g.OH = H; g.OW = W;
  g.KD = three_d ? 3 : 1; g.KH = 3; g.KW = 3; g.stride = 1; g.dil = dil;
  g.pd = three_d ? 1 : 0; g.ph = dil; g.pw = dil; g.transposed = 0;
  return g;
}

inline bool aligned(const void* p, uintptr_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

}  // namespace snb_model
