// Shared-model data-parallel online adaptation of StereoNet from C++ through include/snb200.h and NCCL: no Python, no torch.
//
//   stereonet_adapt_dp G WEIGHTS IMAGES B H W FRAMES OUT [LR [REPLAY_IMAGES REPLAY_GT RB N]]
//
// G        number of GPUs (devices 0 .. G-1); one process drives them all (ncclCommInitAll)
// WEIGHTS  a file written by stereonet_b200.native.export_weights (format in that module's docstring)
// IMAGES   raw float32 [F][G][2][B][3][H][W] for some F >= 1 (per frame and rank: left batch, then right batch), NCHW; step f
//          adapts rank r on frame f % F of its own stream (with G = 1 and F = FRAMES: stereonet_adapt's IMAGES file)
// FRAMES   number of steps
// OUT      receives rank 0's adapted parameters and running statistics in the WEIGHTS format (stereonet_infer reads it)
// LR       Adam's learning rate (default 5e-5, adapt.py's); clipping at 1.0 on stereo_net as adapt.py:391-392
// REPLAY_IMAGES, REPLAY_GT  raw float32 [N][2][RB][3][H][W] and [N][RB][H][W] (gt <= 0: invalid): N stored samples with ground
//          truth; at step f rank r replays sample (f + r) % N with weight 0.05 (the ER mode)
//
// Every rank holds a replica of the model.  Per step each rank replays one captured CUDA graph (snb_stereonet_adapt_forward and
// snb_stereonet_adapt_backward, or their _replay variants), then one eager ncclAllReduce(SUM) per rank, grouped, runs over the
// state's dp_flat piece ([gradient bucket | BatchNorm running statistics]), then each rank replays a second graph,
// snb_stereonet_adapt_apply(world = G).  The collective stays outside the graphs: captured, it hung a two-GPU run (DESIGN.md
// section 5).  At the end the replicas' parameters, running statistics and Adam state must be byte-identical; the program prints
// each step's losses and the time per step from device events (the steps after the first, which loads the graphs).
// Build: python adaptive-stereo-icra-2021_b200/build.py --example (needs NCCL, found through the nvidia.nccl Python package)
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <cuda_runtime.h>
#include <nccl.h>

#include "snb200.h"

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
  fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); return 1; } } while (0)
#define NC(call) do { ncclResult_t e_ = (call); if (e_ != ncclSuccess) { \
  fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #call, ncclGetErrorString(e_)); return 1; } } while (0)
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

// Page-locked copy of `src`, so that the per-step uploads are asynchronous.
static char* pinned_copy(const std::vector<char>& src) {
  void* p = nullptr;
  if (cudaMallocHost(&p, src.size() ? src.size() : 1) != cudaSuccess) return nullptr;
  memcpy(p, src.data(), src.size());
  return static_cast<char*>(p);
}

struct Replica {
  cudaStream_t stream;
  char* dparams;
  std::vector<float*> params;
  void *state, *workspace;
  float *img, *loss, *rimg, *gt, *loss_replay;
  float* dp_flat;
  cudaGraph_t graph[2];
  cudaGraphExec_t exec[2];
  cudaEvent_t start, stop;
};

int main(int argc, char** argv) {
  if (argc < 9 || (argc > 10 && argc != 14)) {
    fprintf(stderr, "usage: %s G WEIGHTS IMAGES B H W FRAMES OUT [LR [REPLAY_IMAGES REPLAY_GT RB N]]\n", argv[0]);
    return 2;
  }
  const int G = atoi(argv[1]);
  const int B = atoi(argv[4]), H = atoi(argv[5]), W = atoi(argv[6]), frames = atoi(argv[7]);
  const double lr = argc > 9 ? atof(argv[9]) : 5e-5;
  const bool replay = argc == 14;
  const int RB = replay ? atoi(argv[12]) : 0, nrep = replay ? atoi(argv[13]) : 0;
  const float er_weight = 0.05f;
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (G < 1 || G > ndev) {
    fprintf(stderr, "G = %d, but %d devices are visible\n", G, ndev);
    return 1;
  }

  // ---- weights file: magic, {k, input_scale, maxdisp, n}, then n x {numel, data}
  std::vector<char> wf;
  if (!read_file(argv[2], wf) || wf.size() < 24 || memcmp(wf.data(), "SNBSTW01", 8) != 0) {
    fprintf(stderr, "%s: not a weights file\n", argv[2]);
    return 1;
  }
  int32_t hdr[4];
  memcpy(hdr, wf.data() + 8, sizeof(hdr));
  const int k = hdr[0], input_scale = hdr[1], maxdisp = hdr[2], n = hdr[3];
  if (n != snb_stereonet_num_params(k)) {
    fprintf(stderr, "%s: %d tensors, the library expects %d for k = %d\n", argv[2], n, snb_stereonet_num_params(k), k);
    return 1;
  }
  std::vector<size_t> offs, counts;                 // parameters packed into one device buffer per replica, each 256-byte aligned
  size_t pos = 24, dev_bytes = 0;
  for (int i = 0; i < n; ++i) {
    int32_t numel;
    if (pos + 4 > wf.size()) { fprintf(stderr, "%s: truncated\n", argv[2]); return 1; }
    memcpy(&numel, wf.data() + pos, 4);
    pos += 4;
    if (numel < 0 || pos + (size_t)numel * 4 > wf.size()) { fprintf(stderr, "%s: truncated\n", argv[2]); return 1; }
    offs.push_back(pos);
    counts.push_back((size_t)numel);
    pos += (size_t)numel * 4;
    dev_bytes += ((size_t)numel * 4 + 255) / 256 * 256;
  }

  std::vector<char> img_file;
  const size_t frame_bytes = (size_t)2 * B * 3 * H * W * sizeof(float);
  if (frames < 1 || !read_file(argv[3], img_file) || img_file.empty() || img_file.size() % (frame_bytes * G) != 0) {
    fprintf(stderr, "%s: expected a whole number (>= 1) of %zu-byte frames of float32 [%d][2][%d][3][%d][%d]\n", argv[3],
            frame_bytes * G, G, B, H, W);
    return 1;
  }
  const size_t nfile = img_file.size() / (frame_bytes * G);
  std::vector<char> rimg_file, rgt_file;
  const size_t rimg_bytes = (size_t)2 * RB * 3 * H * W * sizeof(float), rgt_bytes = (size_t)RB * H * W * sizeof(float);
  if (replay && (RB < 1 || nrep < 1 || !read_file(argv[10], rimg_file) || rimg_file.size() != rimg_bytes * nrep ||
                 !read_file(argv[11], rgt_file) || rgt_file.size() != rgt_bytes * nrep)) {
    fprintf(stderr, "%s, %s: expected %zu and %zu bytes of float32 [%d][2][%d][3][%d][%d] and [%d][%d][%d][%d]\n", argv[10], argv[11],
            rimg_bytes * (nrep > 0 ? nrep : 0), rgt_bytes * (nrep > 0 ? nrep : 0), nrep, RB, H, W, nrep, RB, H, W);
    return 1;
  }
  char* img = pinned_copy(img_file);
  char* rimg = replay ? pinned_copy(rimg_file) : nullptr;
  char* rgt = replay ? pinned_copy(rgt_file) : nullptr;
  if (!img || (replay && (!rimg || !rgt))) { fprintf(stderr, "cudaMallocHost failed\n"); return 1; }

  const long long sbytes = snb_stereonet_adapt_state_bytes(k);
  const long long wsbytes = replay ? snb_stereonet_adapt_replay_workspace_bytes(k, input_scale, maxdisp, B, H, W, RB)
                                   : snb_stereonet_adapt_workspace_bytes(k, input_scale, maxdisp, B, H, W);
  long long dp_off = 0, dp_bytes = 0;
  if (sbytes < 0 || wsbytes < 0 || snb_stereonet_adapt_state_piece(k, 5, &dp_off, &dp_bytes) != 0) {
    fprintf(stderr, "%s\n", snb_last_error());
    return 1;
  }
  const size_t dp_count = (size_t)dp_bytes / sizeof(float);

  // ---- one replica per device: parameters, state, workspace, static graph inputs, and the two captured graphs
  std::vector<Replica> rep(G);
  for (int r = 0; r < G; ++r) {
    Replica& R = rep[r];
    CK(cudaSetDevice(r));
    CK(cudaStreamCreateWithFlags(&R.stream, cudaStreamNonBlocking));
    R.dparams = static_cast<char*>(device_alloc(dev_bytes));
    R.state = device_alloc((size_t)sbytes);
    R.workspace = device_alloc((size_t)wsbytes);
    R.img = static_cast<float*>(device_alloc(frame_bytes));
    R.loss = static_cast<float*>(device_alloc((size_t)(1 + B) * sizeof(float)));
    R.rimg = replay ? static_cast<float*>(device_alloc(rimg_bytes)) : nullptr;
    R.gt = replay ? static_cast<float*>(device_alloc(rgt_bytes)) : nullptr;
    R.loss_replay = replay ? static_cast<float*>(device_alloc(2 * sizeof(float))) : nullptr;
    if (!R.dparams || !R.state || !R.workspace || !R.img || !R.loss || (replay && (!R.rimg || !R.gt || !R.loss_replay))) {
      fprintf(stderr, "cudaMalloc failed on device %d\n", r);
      return 1;
    }
    R.dp_flat = reinterpret_cast<float*>(static_cast<char*>(R.state) + dp_off);
    R.params.resize(n);
    size_t dpos = 0;
    for (int i = 0; i < n; ++i) {
      R.params[i] = reinterpret_cast<float*>(R.dparams + dpos);
      CK(cudaMemcpyAsync(R.dparams + dpos, wf.data() + offs[i], counts[i] * 4, cudaMemcpyHostToDevice, R.stream));
      dpos += (counts[i] * 4 + 255) / 256 * 256;
    }
    SNB(snb_stereonet_adapt_init(R.params.data(), k, R.state, R.stream));
    CK(cudaStreamSynchronize(R.stream));
    for (int gi = 0; gi < 2; ++gi) {
      CK(cudaStreamBeginCapture(R.stream, cudaStreamCaptureModeThreadLocal));
      int rc = 0;
      const char* what = "";
      if (gi == 0 && !replay) {
        what = "snb_stereonet_adapt_forward / _backward";
        rc = snb_stereonet_adapt_forward(R.params.data(), nullptr, k, input_scale, maxdisp, R.img, B, H, W, R.state, R.workspace, R.loss,
                                         nullptr, nullptr, nullptr, R.stream);
        if (!rc) rc = snb_stereonet_adapt_backward(R.params.data(), k, input_scale, maxdisp, B, H, W, R.state, R.workspace, R.stream);
      } else if (gi == 0) {
        what = "snb_stereonet_adapt_forward_replay / _backward_replay";
        rc = snb_stereonet_adapt_forward_replay(R.params.data(), nullptr, k, input_scale, maxdisp, R.img, B, H, W, R.rimg, R.gt, RB,
                                                er_weight, R.state, R.workspace, R.loss, R.loss_replay, nullptr, nullptr, nullptr,
                                                R.stream);
        if (!rc)
          rc = snb_stereonet_adapt_backward_replay(R.params.data(), k, input_scale, maxdisp, B, H, W, RB, R.state, R.workspace,
                                                   R.stream);
      } else {
        what = "snb_stereonet_adapt_apply";
        rc = snb_stereonet_adapt_apply(R.params.data(), k, R.state, G, 1.0f, lr, 0.9, 0.999, 1e-8, R.stream);
      }
      CK(cudaStreamEndCapture(R.stream, &R.graph[gi]));
      if (rc != 0) {
        fprintf(stderr, "%s: %s\n", what, snb_last_error());
        return 1;
      }
      CK(cudaGraphInstantiate(&R.exec[gi], R.graph[gi], 0));
    }
    CK(cudaEventCreate(&R.start));
    CK(cudaEventCreate(&R.stop));
  }

  std::vector<ncclComm_t> comms(G);
  std::vector<int> devs(G);
  for (int r = 0; r < G; ++r) devs[r] = r;
  NC(ncclCommInitAll(comms.data(), G, devs.data()));

  // per step and rank: {loss, khamis, total}, copied back without a synchronisation and printed at the end
  float* host_loss = nullptr;
  CK(cudaMallocHost(reinterpret_cast<void**>(&host_loss), sizeof(float) * 3 * G * frames));
  for (int f = 0; f < frames; ++f) {
    for (int r = 0; r < G; ++r) {
      Replica& R = rep[r];
      CK(cudaSetDevice(r));
      if (f == 1 || (f == 0 && frames == 1)) CK(cudaEventRecord(R.start, R.stream));
      CK(cudaMemcpyAsync(R.img, img + frame_bytes * ((f % nfile) * G + r), frame_bytes, cudaMemcpyHostToDevice, R.stream));
      if (replay) {
        const int s = (f + r) % nrep;
        CK(cudaMemcpyAsync(R.rimg, rimg + rimg_bytes * s, rimg_bytes, cudaMemcpyHostToDevice, R.stream));
        CK(cudaMemcpyAsync(R.gt, rgt + rgt_bytes * s, rgt_bytes, cudaMemcpyHostToDevice, R.stream));
      }
      CK(cudaGraphLaunch(R.exec[0], R.stream));
    }
    NC(ncclGroupStart());
    for (int r = 0; r < G; ++r)
      NC(ncclAllReduce(rep[r].dp_flat, rep[r].dp_flat, dp_count, ncclFloat, ncclSum, comms[r], rep[r].stream));
    NC(ncclGroupEnd());
    for (int r = 0; r < G; ++r) {
      Replica& R = rep[r];
      CK(cudaSetDevice(r));
      CK(cudaGraphLaunch(R.exec[1], R.stream));
      float* h = host_loss + 3 * ((size_t)f * G + r);
      CK(cudaMemcpyAsync(h, R.loss, sizeof(float), cudaMemcpyDeviceToHost, R.stream));
      if (replay) CK(cudaMemcpyAsync(h + 1, R.loss_replay, 2 * sizeof(float), cudaMemcpyDeviceToHost, R.stream));
      if (f == frames - 1) CK(cudaEventRecord(R.stop, R.stream));
    }
  }
  float us = 0.f;
  for (int r = 0; r < G; ++r) {
    CK(cudaSetDevice(r));
    CK(cudaStreamSynchronize(rep[r].stream));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, rep[r].start, rep[r].stop));
    us = ms * 1e3f > us ? ms * 1e3f : us;
  }
  for (int f = 0; f < frames; ++f)
    for (int r = 0; r < G; ++r) {
      const float* h = host_loss + 3 * ((size_t)f * G + r);
      if (replay)
        printf("stereonet_adapt_dp: frame %d rank %d loss %.7f khamis %.7f total %.7f\n", f, r, h[0], h[1], h[2]);
      else
        printf("stereonet_adapt_dp: frame %d rank %d loss %.7f\n", f, r, h[0]);
    }
  const int timed = frames > 1 ? frames - 1 : 1;
  printf("stereonet_adapt_dp: %d GPUs, %d timed steps, %.1f us per step\n", G, timed, us / timed);

  // ---- the replicas must be byte-identical: parameters (running statistics included) and Adam's moments and step
  std::vector<std::vector<char>> snap(G);
  for (int r = 0; r < G; ++r) {
    CK(cudaSetDevice(r));
    snap[r].resize(dev_bytes + (size_t)sbytes);
    CK(cudaMemcpy(snap[r].data(), rep[r].dparams, dev_bytes, cudaMemcpyDeviceToHost));
    for (int what = 1; what <= 3; ++what) {
      long long o = 0, b = 0;
      SNB(snb_stereonet_adapt_state_piece(k, what, &o, &b));
      CK(cudaMemcpy(snap[r].data() + dev_bytes + o, static_cast<char*>(rep[r].state) + o, (size_t)b, cudaMemcpyDeviceToHost));
    }
  }
  bool identical = true;
  for (int r = 1; r < G; ++r) identical = identical && snap[r] == snap[0];
  if (!identical) {
    fprintf(stderr, "stereonet_adapt_dp: the replicas differ\n");
    return 1;
  }
  printf("stereonet_adapt_dp: %d replicas identical\n", G);

  // ---- rank 0's adapted tensors, in the input's format
  FILE* out = fopen(argv[8], "wb");
  if (!out) { fprintf(stderr, "%s: cannot write\n", argv[8]); return 1; }
  bool ok = fwrite(wf.data(), 1, 24, out) == 24;
  size_t dpos = 0;
  for (int i = 0; i < n && ok; ++i) {
    const int32_t numel = (int32_t)counts[i];
    ok = fwrite(&numel, 4, 1, out) == 1 && fwrite(snap[0].data() + dpos, 4, counts[i], out) == counts[i];
    dpos += (counts[i] * 4 + 255) / 256 * 256;
  }
  if (fclose(out) != 0 || !ok) { fprintf(stderr, "%s: write failed\n", argv[8]); return 1; }

  for (int r = 0; r < G; ++r) NC(ncclCommDestroy(comms[r]));
  for (int r = 0; r < G; ++r) {
    Replica& R = rep[r];
    CK(cudaSetDevice(r));
    for (int gi = 0; gi < 2; ++gi) {
      CK(cudaGraphExecDestroy(R.exec[gi]));
      CK(cudaGraphDestroy(R.graph[gi]));
    }
    CK(cudaEventDestroy(R.start));
    CK(cudaEventDestroy(R.stop));
    CK(cudaFree(R.dparams));
    CK(cudaFree(R.state));
    CK(cudaFree(R.workspace));
    CK(cudaFree(R.img));
    CK(cudaFree(R.loss));
    if (replay) {
      CK(cudaFree(R.rimg));
      CK(cudaFree(R.gt));
      CK(cudaFree(R.loss_replay));
    }
    CK(cudaStreamDestroy(R.stream));
  }
  CK(cudaFreeHost(host_loss));
  CK(cudaFreeHost(img));
  if (replay) {
    CK(cudaFreeHost(rimg));
    CK(cudaFreeHost(rgt));
  }
  return 0;
}
