// Single-pass online adaptation of StereoNet from C++ through include/snb200.h: no Python, no torch.
//
//   stereonet_adapt WEIGHTS IMAGES B H W FRAMES OUT [LR]
//
// WEIGHTS  a file written by stereonet_b200.native.export_weights (format in that module's docstring)
// IMAGES   raw float32 [FRAMES][2][B][3][H][W] (per frame: left batch, then right batch), NCHW
// OUT      receives the adapted parameters and running statistics in the WEIGHTS format (stereonet_infer reads it)
// LR       Adam's learning rate (default 5e-5, adapt.py's); clipping at 1.0 on stereo_net as adapt.py:391-392
//
// Uploads the parameters, captures snb_stereonet_adapt_forward and snb_stereonet_adapt_update as two CUDA graphs, and replays both
// for every frame (each frame updates: the host-side policy of adapt.py, which may skip an update, is left out).  Prints each
// frame's photometric loss.  Build: python adaptive-stereo-icra-2021_b200/build.py --example
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
  if (argc < 8) {
    fprintf(stderr, "usage: %s WEIGHTS IMAGES B H W FRAMES OUT [LR]\n", argv[0]);
    return 2;
  }
  const int B = atoi(argv[3]), H = atoi(argv[4]), W = atoi(argv[5]), frames = atoi(argv[6]);
  const double lr = argc > 8 ? atof(argv[8]) : 5e-5;

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
  const long long wsbytes = snb_stereonet_adapt_workspace_bytes(k, input_scale, maxdisp, B, H, W);
  if (sbytes < 0 || wsbytes < 0) { fprintf(stderr, "%s\n", snb_last_error()); return 1; }
  void* state = device_alloc((size_t)sbytes);
  void* workspace = device_alloc((size_t)wsbytes);
  float* dimg = static_cast<float*>(device_alloc(frame_bytes));
  float* loss = static_cast<float*>(device_alloc((size_t)(1 + B) * sizeof(float)));
  if (!state || !workspace || !dimg || !loss) { fprintf(stderr, "cudaMalloc failed\n"); return 1; }
  SNB(snb_stereonet_adapt_init(params.data(), k, state, stream));
  CK(cudaStreamSynchronize(stream));

  cudaGraph_t graph[2];
  cudaGraphExec_t exec[2];
  for (int gi = 0; gi < 2; ++gi) {
    CK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    const int rc = gi == 0
        ? snb_stereonet_adapt_forward(params.data(), nullptr, k, input_scale, maxdisp, dimg, B, H, W, state, workspace, loss, nullptr,
                                      nullptr, nullptr, stream)
        : snb_stereonet_adapt_update(params.data(), k, input_scale, maxdisp, B, H, W, state, workspace, 1.0f, lr, 0.9, 0.999, 1e-8,
                                     stream);
    CK(cudaStreamEndCapture(stream, &graph[gi]));
    if (rc != 0) { fprintf(stderr, "%s: %s\n", gi == 0 ? "snb_stereonet_adapt_forward" : "snb_stereonet_adapt_update", snb_last_error()); return 1; }
    CK(cudaGraphInstantiate(&exec[gi], graph[gi], 0));
  }

  float host_loss = 0.f;
  for (int f = 0; f < frames; ++f) {
    CK(cudaMemcpyAsync(dimg, img.data() + frame_bytes * f, frame_bytes, cudaMemcpyHostToDevice, stream));
    CK(cudaGraphLaunch(exec[0], stream));
    CK(cudaGraphLaunch(exec[1], stream));
    CK(cudaMemcpyAsync(&host_loss, loss, sizeof(float), cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
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
  CK(cudaStreamDestroy(stream));
  return 0;
}
