// Online adaptation of StereoNet from C++ through include/snb200.h, single pass or with experience replay: no Python, no torch.
//
//   stereonet_adapt WEIGHTS IMAGES B H W FRAMES OUT [LR [REPLAY_IMAGES REPLAY_GT RB N]]
//
// WEIGHTS  a file written by stereonet_b200.native.export_weights (format in that module's docstring)
// IMAGES   raw float32 [FRAMES][2][B][3][H][W] (per frame: left batch, then right batch), NCHW
// OUT      receives the adapted parameters and running statistics in the WEIGHTS format (stereonet_infer reads it)
// LR       Adam's learning rate (default 5e-5, adapt.py's); clipping at 1.0 on stereo_net as adapt.py:391-392
// REPLAY_IMAGES, REPLAY_GT  raw float32 [N][2][RB][3][H][W] and [N][RB][H][W] (gt <= 0: invalid): N stored samples with ground
//          truth; frame f replays sample f % N (adapt.py's train_val_dataset[step % N]) with weight 0.05 (the ER mode)
//
// Uploads the parameters, captures snb_stereonet_adapt_forward and snb_stereonet_adapt_update (with replay: their _replay variants)
// as two CUDA graphs, and replays both for every frame (each frame updates: the host-side policy of adapt.py, which may skip an
// update, is left out).  Prints each frame's photometric loss (with replay also the Khamis term and the total).
// Build: python adaptive-stereo-icra-2021_b200/build.py --example
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cuda_runtime.h>

#include "snb200.h"

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
  fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); return 1; } } while (0)
#define SNB(call) do { if ((call) != 0) { fprintf(stderr, "%s: %s\n", #call, snb_last_error()); return 1; } } while (0)

static bool read_file(const char* path, std::vector<char>& out) {
  FILE* f = fopen(path, "rb");
  if (!f) return false;
  fseek(f, 0, SEEK_END);
  const long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  out.resize(n > 0 ? (size_t)n : 0);
  const bool ok = n >= 0 && fread(out.data(), 1, out.size(), f) == out.size();
  fclose(f);
  return ok;
}

static void* device_alloc(size_t bytes) {        // cudaMalloc returns 256-byte aligned memory
  void* p = nullptr;
  return cudaMalloc(&p, bytes ? bytes : 1) == cudaSuccess ? p : nullptr;
}

int main(int argc, char** argv) {
  if (argc < 8 || (argc > 9 && argc != 13)) {
    fprintf(stderr, "usage: %s WEIGHTS IMAGES B H W FRAMES OUT [LR [REPLAY_IMAGES REPLAY_GT RB N]]\n", argv[0]);
    return 2;
  }
  const int B = atoi(argv[3]), H = atoi(argv[4]), W = atoi(argv[5]), frames = atoi(argv[6]);
  const double lr = argc > 8 ? atof(argv[8]) : 5e-5;
  const bool replay = argc == 13;
  const int RB = replay ? atoi(argv[11]) : 0, nrep = replay ? atoi(argv[12]) : 0;
  const float er_weight = 0.05f;

  // ---- weights file: magic, {k, input_scale, maxdisp, n}, then n x {numel, data}
  std::vector<char> wf;
  if (!read_file(argv[1], wf) || wf.size() < 24 || memcmp(wf.data(), "SNBSTW01", 8) != 0) {
    fprintf(stderr, "%s: not a weights file\n", argv[1]);
    return 1;
  }
  int32_t hdr[4];
  memcpy(hdr, wf.data() + 8, sizeof(hdr));
  const int k = hdr[0], input_scale = hdr[1], maxdisp = hdr[2], n = hdr[3];
  if (n != snb_stereonet_num_params(k)) {
    fprintf(stderr, "%s: %d tensors, the library expects %d for k = %d\n", argv[1], n, snb_stereonet_num_params(k), k);
    return 1;
  }
  std::vector<size_t> offs, counts;                 // parameters packed into one device buffer, each 256-byte aligned
  size_t pos = 24, dev_bytes = 0;
  for (int i = 0; i < n; ++i) {
    int32_t numel;
    if (pos + 4 > wf.size()) { fprintf(stderr, "%s: truncated\n", argv[1]); return 1; }
    memcpy(&numel, wf.data() + pos, 4);
    pos += 4;
    if (numel < 0 || pos + (size_t)numel * 4 > wf.size()) { fprintf(stderr, "%s: truncated\n", argv[1]); return 1; }
    offs.push_back(pos);
    counts.push_back((size_t)numel);
    pos += (size_t)numel * 4;
    dev_bytes += ((size_t)numel * 4 + 255) / 256 * 256;
  }

  std::vector<char> img;
  const size_t frame_bytes = (size_t)2 * B * 3 * H * W * sizeof(float);
  if (frames < 1 || !read_file(argv[2], img) || img.size() != frame_bytes * frames) {
    fprintf(stderr, "%s: expected %zu bytes of float32 [%d][2][%d][3][%d][%d]\n", argv[2], frame_bytes * (frames > 0 ? frames : 0),
            frames, B, H, W);
    return 1;
  }
  std::vector<char> rimg, rgt;
  const size_t rimg_bytes = (size_t)2 * RB * 3 * H * W * sizeof(float), rgt_bytes = (size_t)RB * H * W * sizeof(float);
  if (replay && (RB < 1 || nrep < 1 || !read_file(argv[9], rimg) || rimg.size() != rimg_bytes * nrep || !read_file(argv[10], rgt) ||
                 rgt.size() != rgt_bytes * nrep)) {
    fprintf(stderr, "%s, %s: expected %zu and %zu bytes of float32 [%d][2][%d][3][%d][%d] and [%d][%d][%d][%d]\n", argv[9], argv[10],
            rimg_bytes * (nrep > 0 ? nrep : 0), rgt_bytes * (nrep > 0 ? nrep : 0), nrep, RB, H, W, nrep, RB, H, W);
    return 1;
  }

  cudaStream_t stream;
  CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  char* dparams = static_cast<char*>(device_alloc(dev_bytes));
  if (!dparams) { fprintf(stderr, "cudaMalloc failed\n"); return 1; }
  std::vector<float*> params(n);
  size_t dpos = 0;
  for (int i = 0; i < n; ++i) {
    params[i] = reinterpret_cast<float*>(dparams + dpos);
    CK(cudaMemcpyAsync(dparams + dpos, wf.data() + offs[i], counts[i] * 4, cudaMemcpyHostToDevice, stream));
    dpos += (counts[i] * 4 + 255) / 256 * 256;
  }

  const long long sbytes = snb_stereonet_adapt_state_bytes(k);
  const long long wsbytes = replay ? snb_stereonet_adapt_replay_workspace_bytes(k, input_scale, maxdisp, B, H, W, RB)
                                   : snb_stereonet_adapt_workspace_bytes(k, input_scale, maxdisp, B, H, W);
  if (sbytes < 0 || wsbytes < 0) { fprintf(stderr, "%s\n", snb_last_error()); return 1; }
  void* state = device_alloc((size_t)sbytes);
  void* workspace = device_alloc((size_t)wsbytes);
  float* dimg = static_cast<float*>(device_alloc(frame_bytes));
  float* loss = static_cast<float*>(device_alloc((size_t)(1 + B) * sizeof(float)));
  float* drimg = replay ? static_cast<float*>(device_alloc(rimg_bytes)) : nullptr;          // static replay buffers of the graphs
  float* dgt = replay ? static_cast<float*>(device_alloc(rgt_bytes)) : nullptr;
  float* loss_replay = replay ? static_cast<float*>(device_alloc(2 * sizeof(float))) : nullptr;
  if (!state || !workspace || !dimg || !loss || (replay && (!drimg || !dgt || !loss_replay))) {
    fprintf(stderr, "cudaMalloc failed\n");
    return 1;
  }
  SNB(snb_stereonet_adapt_init(params.data(), k, state, stream));
  CK(cudaStreamSynchronize(stream));

  cudaGraph_t graph[2];
  cudaGraphExec_t exec[2];
  for (int gi = 0; gi < 2; ++gi) {
    CK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    int rc;
    if (!replay)
      rc = gi == 0
          ? snb_stereonet_adapt_forward(params.data(), nullptr, k, input_scale, maxdisp, dimg, B, H, W, state, workspace, loss, nullptr,
                                        nullptr, nullptr, stream)
          : snb_stereonet_adapt_update(params.data(), k, input_scale, maxdisp, B, H, W, state, workspace, 1.0f, lr, 0.9, 0.999, 1e-8,
                                       stream);
    else
      rc = gi == 0
          ? snb_stereonet_adapt_forward_replay(params.data(), nullptr, k, input_scale, maxdisp, dimg, B, H, W, drimg, dgt, RB, er_weight,
                                               state, workspace, loss, loss_replay, nullptr, nullptr, nullptr, stream)
          : snb_stereonet_adapt_update_replay(params.data(), k, input_scale, maxdisp, B, H, W, RB, state, workspace, 1.0f, lr, 0.9, 0.999,
                                              1e-8, stream);
    CK(cudaStreamEndCapture(stream, &graph[gi]));
    if (rc != 0) {
      static const char* names[2][2] = {{"snb_stereonet_adapt_forward", "snb_stereonet_adapt_update"},
                                        {"snb_stereonet_adapt_forward_replay", "snb_stereonet_adapt_update_replay"}};
      fprintf(stderr, "%s: %s\n", names[replay][gi], snb_last_error());
      return 1;
    }
    CK(cudaGraphInstantiate(&exec[gi], graph[gi], 0));
  }

  float host_loss = 0.f, host_replay[2] = {0.f, 0.f};
  for (int f = 0; f < frames; ++f) {
    CK(cudaMemcpyAsync(dimg, img.data() + frame_bytes * f, frame_bytes, cudaMemcpyHostToDevice, stream));
    if (replay) {
      CK(cudaMemcpyAsync(drimg, rimg.data() + rimg_bytes * (f % nrep), rimg_bytes, cudaMemcpyHostToDevice, stream));
      CK(cudaMemcpyAsync(dgt, rgt.data() + rgt_bytes * (f % nrep), rgt_bytes, cudaMemcpyHostToDevice, stream));
    }
    CK(cudaGraphLaunch(exec[0], stream));
    CK(cudaGraphLaunch(exec[1], stream));
    CK(cudaMemcpyAsync(&host_loss, loss, sizeof(float), cudaMemcpyDeviceToHost, stream));
    if (replay) CK(cudaMemcpyAsync(host_replay, loss_replay, 2 * sizeof(float), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    if (replay)
      printf("stereonet_adapt: frame %d loss %.7f khamis %.7f total %.7f\n", f, host_loss, host_replay[0], host_replay[1]);
    else
      printf("stereonet_adapt: frame %d loss %.7f\n", f, host_loss);
  }

  // ---- the adapted tensors, in the input's format
  FILE* out = fopen(argv[7], "wb");
  if (!out) { fprintf(stderr, "%s: cannot write\n", argv[7]); return 1; }
  bool ok = fwrite(wf.data(), 1, 24, out) == 24;
  std::vector<float> buf;
  for (int i = 0; i < n && ok; ++i) {
    const int32_t numel = (int32_t)counts[i];
    buf.resize(counts[i]);
    CK(cudaMemcpy(buf.data(), params[i], counts[i] * 4, cudaMemcpyDeviceToHost));
    ok = fwrite(&numel, 4, 1, out) == 1 && fwrite(buf.data(), 4, counts[i], out) == counts[i];
  }
  if (fclose(out) != 0 || !ok) { fprintf(stderr, "%s: write failed\n", argv[7]); return 1; }

  for (int gi = 0; gi < 2; ++gi) {
    CK(cudaGraphExecDestroy(exec[gi]));
    CK(cudaGraphDestroy(graph[gi]));
  }
  CK(cudaFree(dparams));
  CK(cudaFree(state));
  CK(cudaFree(workspace));
  CK(cudaFree(dimg));
  CK(cudaFree(loss));
  if (replay) {
    CK(cudaFree(drimg));
    CK(cudaFree(dgt));
    CK(cudaFree(loss_replay));
  }
  CK(cudaStreamDestroy(stream));
  return 0;
}
