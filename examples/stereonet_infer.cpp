// Whole-model StereoNet inference from C++ through include/snb200.h: no Python, no torch.
//
//   stereonet_infer WEIGHTS IMAGES B H W OUT [ITERS [f16]]
//
// WEIGHTS  a file written by stereonet_b200.native.export_weights (format in that module's docstring)
// IMAGES   raw float32 [2][B][3][H][W] (left batch, then right batch), NCHW
// OUT      receives the full-resolution disparity, raw float32 [B][H][W]
// ITERS    graph replays to time (default 100)
// f16      run the opt-in reduced-precision forward snb_stereonet_forward_f16 instead (results reported apart from fp32 parity)
//
// Uploads the parameters, runs snb_stereonet_prepare, captures one snb_stereonet_forward into a CUDA graph, replays it ITERS
// times and reports the mean time per frame from CUDA events.  Build: python adaptive-stereo-icra-2021_b200/build.py --example
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
  if (argc < 7) {
    fprintf(stderr, "usage: %s WEIGHTS IMAGES B H W OUT [ITERS [f16]]\n", argv[0]);
    return 2;
  }
  const int B = atoi(argv[3]), H = atoi(argv[4]), W = atoi(argv[5]);
  const int iters = argc > 7 ? atoi(argv[7]) : 100;
  const bool f16 = argc > 8 && strcmp(argv[8], "f16") == 0;
  if (argc > 8 && !f16) { fprintf(stderr, "%s: the only precision option is f16\n", argv[8]); return 2; }
  auto forward = f16 ? snb_stereonet_forward_f16 : snb_stereonet_forward;
  const char* fwd_name = f16 ? "snb_stereonet_forward_f16" : "snb_stereonet_forward";

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
  const size_t img_bytes = (size_t)2 * B * 3 * H * W * sizeof(float);
  if (!read_file(argv[2], img) || img.size() != img_bytes) {
    fprintf(stderr, "%s: expected %zu bytes of float32 [2][%d][3][%d][%d]\n", argv[2], img_bytes, B, H, W);
    return 1;
  }

  cudaStream_t stream;
  CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  char* dparams = static_cast<char*>(device_alloc(dev_bytes));
  if (!dparams) { fprintf(stderr, "cudaMalloc failed\n"); return 1; }
  std::vector<const float*> params(n);
  size_t dpos = 0;
  for (int i = 0; i < n; ++i) {
    params[i] = reinterpret_cast<const float*>(dparams + dpos);
    CK(cudaMemcpyAsync(dparams + dpos, wf.data() + offs[i], counts[i] * 4, cudaMemcpyHostToDevice, stream));
    dpos += (counts[i] * 4 + 255) / 256 * 256;
  }

  const long long wbytes = snb_stereonet_weights_bytes(k);
  const long long wsbytes = snb_stereonet_workspace_bytes(k, input_scale, maxdisp, B, H, W);
  if (wbytes < 0 || wsbytes < 0) { fprintf(stderr, "%s\n", snb_last_error()); return 1; }
  void* weights = device_alloc((size_t)wbytes);
  void* workspace = device_alloc((size_t)wsbytes);
  float* dimg = static_cast<float*>(device_alloc(img_bytes));
  float* disp = static_cast<float*>(device_alloc((size_t)B * H * W * sizeof(float)));
  if (!weights || !workspace || !dimg || !disp) { fprintf(stderr, "cudaMalloc failed\n"); return 1; }
  CK(cudaMemcpyAsync(dimg, img.data(), img_bytes, cudaMemcpyHostToDevice, stream));

  SNB(snb_stereonet_prepare(params.data(), k, weights, stream));
  CK(cudaStreamSynchronize(stream));
  CK(cudaFree(dparams));                            // `weights` is self-contained

  cudaGraph_t graph;
  cudaGraphExec_t exec;
  CK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
  const int rc = forward(weights, k, input_scale, maxdisp, dimg, B, H, W, workspace, disp, nullptr, nullptr, nullptr, stream);
  CK(cudaStreamEndCapture(stream, &graph));
  if (rc != 0) { fprintf(stderr, "%s: %s\n", fwd_name, snb_last_error()); return 1; }
  CK(cudaGraphInstantiate(&exec, graph, 0));

  CK(cudaGraphLaunch(exec, stream));                // warm-up
  cudaEvent_t t0, t1;
  CK(cudaEventCreate(&t0));
  CK(cudaEventCreate(&t1));
  CK(cudaEventRecord(t0, stream));
  for (int i = 0; i < iters; ++i) CK(cudaGraphLaunch(exec, stream));
  CK(cudaEventRecord(t1, stream));
  CK(cudaEventSynchronize(t1));
  float ms = 0.f;
  CK(cudaEventElapsedTime(&ms, t0, t1));
  printf("stereonet_infer: k=%d input_scale=%d maxdisp=%d B=%d %dx%d%s: %.3f ms per frame (mean of %d graph replays)\n",
         k, input_scale, maxdisp, B, H, W, f16 ? " f16" : "", iters > 0 ? ms / iters : 0.f, iters);

  std::vector<float> out((size_t)B * H * W);
  CK(cudaMemcpyAsync(out.data(), disp, out.size() * sizeof(float), cudaMemcpyDeviceToHost, stream));
  CK(cudaStreamSynchronize(stream));
  FILE* f = fopen(argv[6], "wb");
  if (!f || fwrite(out.data(), sizeof(float), out.size(), f) != out.size()) { fprintf(stderr, "%s: write failed\n", argv[6]); return 1; }
  fclose(f);

  CK(cudaGraphExecDestroy(exec));
  CK(cudaGraphDestroy(graph));
  CK(cudaEventDestroy(t0));
  CK(cudaEventDestroy(t1));
  CK(cudaFree(weights));
  CK(cudaFree(workspace));
  CK(cudaFree(dimg));
  CK(cudaFree(disp));
  CK(cudaStreamDestroy(stream));
  return 0;
}
