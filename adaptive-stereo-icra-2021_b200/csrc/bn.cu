// Train-mode BatchNorm pieces (batch statistics while adapting, adapt.py:313-314; nn.BatchNorm2d/3d defaults,
// stereo_net.py:17,29: eps 1e-5, momentum 0.1, biased variance to normalise, unbiased for the running update).
// Forward: conv epilogues emit per-tile (sum, sumsq) partials -> snb_bn_finalize reduces them in double precision and
// emits per-channel scale/shift -> snb_bn_apply does y = [residual +] LeakyReLU(z*scale + shift).
#include "common.cuh"

namespace {

template <typename T>      // T: float (the conv epilogues' partial rows) or double (the pre-reduced chunk sums)
__global__ void __launch_bounds__(1024)
bn_finalize_kernel(const T* __restrict__ stats, int ntiles, double count, const float* __restrict__ gamma,
                   const float* __restrict__ beta, float* running_mean, float* running_var, long long* num_batches_tracked, float momentum, float eps,
                   float* scale, float* shift, float* mean_out, float* invstd_out) {
  pdl_launch(); pdl_wait();
  __shared__ double red[16][64];
  const int c = threadIdx.x & 63, part = threadIdx.x >> 6;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;          // 4 independent chains: the loop is bound by the fp64 add latency
  int i = part;
  for (; i + 48 < ntiles; i += 64) {
    a0 += (double)stats[(size_t)i * 64 + c];        a1 += (double)stats[(size_t)(i + 16) * 64 + c];
    a2 += (double)stats[(size_t)(i + 32) * 64 + c]; a3 += (double)stats[(size_t)(i + 48) * 64 + c];
  }
  for (; i < ntiles; i += 16) a0 += (double)stats[(size_t)i * 64 + c];
  red[part][c] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  if (threadIdx.x < 32) {
    double s1 = 0.0, s2 = 0.0;
    for (int i = 0; i < 16; ++i) { s1 += red[i][threadIdx.x]; s2 += red[i][32 + threadIdx.x]; }
    const double mean = s1 / count;
    double var = s2 / count - mean * mean;
    if (var < 0.0) var = 0.0;
    const double invstd = 1.0 / sqrt(var + (double)eps);
    const int ch = threadIdx.x;
    if (running_mean) {
      const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
      running_mean[ch] = (float)((1.0 - momentum) * (double)running_mean[ch] + momentum * mean);
      running_var[ch] = (float)((1.0 - momentum) * (double)running_var[ch] + momentum * unbiased);
      if (ch == 0 && num_batches_tracked != nullptr) *num_batches_tracked += 1;      // nn.BatchNorm's int64 counter, same launch
    }
    const float sc = gamma[ch] * (float)invstd;
    scale[ch] = sc;
    shift[ch] = beta[ch] - (float)mean * sc;
    if (mean_out) mean_out[ch] = (float)mean;
    if (invstd_out) invstd_out[ch] = (float)invstd;
  }
}

// Running-statistics update of ONE train-mode BatchNorm call, applied later than its bn_finalize (which was launched without the
// running buffers): lets two passes through the same layers run on two streams (left / right image, adapt.py:72) and still
// update running_mean / running_var / num_batches_tracked in the reference's order.  var = 1 / invstd^2 - eps.
__global__ void bn_running_update_kernel(const float* __restrict__ mean, const float* __restrict__ invstd, double count, float eps,
                                         float momentum, float* running_mean, float* running_var, long long* num_batches_tracked) {
  pdl_launch(); pdl_wait();
  const int ch = threadIdx.x;
  const double is = (double)invstd[ch];
  double var = 1.0 / (is * is) - (double)eps;
  if (var < 0.0) var = 0.0;
  const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
  running_mean[ch] = (float)((1.0 - momentum) * (double)running_mean[ch] + momentum * (double)mean[ch]);
  running_var[ch] = (float)((1.0 - momentum) * (double)running_var[ch] + momentum * unbiased);
  if (ch == 0 && num_batches_tracked != nullptr) *num_batches_tracked += 1;
}

// Stage 1 of the two-stage statistics reduction: block b sums rows [b*chunk, (b+1)*chunk) of stats [ntiles][64] into
// scratch[b][64] (fp64 accumulation, fixed order, kept in fp64: var = E[z^2] - mean^2 cancels, and rounding the chunk sums to
// fp32 cost 5.3e-5 against 1.3e-5 relative in invstd at mean/std = 100 over 3760 tile rows, measured on a B200).  A single CTA walking ~1 MB of partials (one row per image row x column
// block at full resolution) is bound by one SM's load bandwidth: 12-23 us per layer, 23 layers per adaptation step.
__global__ void __launch_bounds__(256)
bn_stats_prereduce_kernel(const float* __restrict__ stats, int ntiles, int chunk, double* __restrict__ scratch) {
  pdl_launch(); pdl_wait();
  __shared__ double red[4][64];
  const int c = threadIdx.x & 63, part = threadIdx.x >> 6;
  const int lo = blockIdx.x * chunk, hi = min(lo + chunk, ntiles);
  double a = 0.0;
  for (int i = lo + part; i < hi; i += 4) a += (double)stats[(size_t)i * 64 + c];
  red[part][c] = a;
  __syncthreads();
  if (part == 0) scratch[(size_t)blockIdx.x * 64 + c] = (red[0][c] + red[1][c]) + (red[2][c] + red[3][c]);
}

__global__ void __launch_bounds__(256)
bn_apply_kernel(const float4* __restrict__ z, const float* __restrict__ scale, const float* __restrict__ shift,
                const float4* __restrict__ residual, float4* __restrict__ y, long long n4, int do_lrelu) {
  pdl_launch(); pdl_wait();
  __shared__ float4 sSc[8], sSh[8];
  if (threadIdx.x < 8) {
    sSc[threadIdx.x] = reinterpret_cast<const float4*>(scale)[threadIdx.x];
    sSh[threadIdx.x] = reinterpret_cast<const float4*>(shift)[threadIdx.x];
  }
  __syncthreads();
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    const float4 sc = sSc[i & 7], sh = sSh[i & 7];
    float4 v = z[i];
    v.x = fmaf(v.x, sc.x, sh.x); v.y = fmaf(v.y, sc.y, sh.y); v.z = fmaf(v.z, sc.z, sh.z); v.w = fmaf(v.w, sc.w, sh.w);
    if (do_lrelu) { v.x = lrelu(v.x); v.y = lrelu(v.y); v.z = lrelu(v.z); v.w = lrelu(v.w); }
    if (residual) { const float4 r = residual[i]; v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w; }
    y[i] = v;
  }
}

}  // namespace

template <typename T>
static int bn_finalize_impl(const T* stats, int ntiles, long long count, const float* gamma, const float* beta,
                            float* running_mean, float* running_var, long long* num_batches_tracked, float momentum, float eps,
                            float* scale, float* shift, float* mean, float* invstd, void* stream) {
  SNB_REQUIRE(stats && gamma && beta && scale && shift && ntiles > 0 && count > 0, "snb_bn_finalize: bad args");
  SNB_REQUIRE((running_mean == nullptr) == (running_var == nullptr), "snb_bn_finalize: running stats must come in pairs");
  snb_launch(bn_finalize_kernel<T>, 1, 1024, 0, stream, stats, ntiles, (double)count, gamma, beta, running_mean, running_var,
             num_batches_tracked, momentum, eps, scale, shift, mean, invstd);
  SNB_LAUNCH_CHECK("bn_finalize_kernel");
  return 0;
}

extern "C" int snb_bn_finalize(const float* stats, int ntiles, long long count, const float* gamma, const float* beta,
                               float* running_mean, float* running_var, float momentum, float eps,
                               float* scale, float* shift, float* mean, float* invstd, void* stream) {
  return bn_finalize_impl(stats, ntiles, count, gamma, beta, running_mean, running_var, nullptr, momentum, eps, scale, shift, mean, invstd, stream);
}

extern "C" int snb_bn_finalize_ws(const float* stats, int ntiles, long long count, const float* gamma, const float* beta,
                                  float* running_mean, float* running_var, long long* num_batches_tracked, float momentum, float eps,
                                  float* scale, float* shift, float* mean, float* invstd, double* scratch, void* stream) {
  SNB_REQUIRE(scratch != nullptr, "snb_bn_finalize_ws: null scratch");
  if (ntiles <= 256)
    return bn_finalize_impl(stats, ntiles, count, gamma, beta, running_mean, running_var, num_batches_tracked, momentum, eps, scale, shift, mean, invstd, stream);
  SNB_REQUIRE(stats && gamma && beta && scale && shift && count > 0, "snb_bn_finalize_ws: bad args");
  const int nblk = 64, chunk = (ntiles + nblk - 1) / nblk;
  snb_launch(bn_stats_prereduce_kernel, nblk, 256, 0, stream, stats, ntiles, chunk, scratch);
  SNB_LAUNCH_CHECK("bn_stats_prereduce_kernel");
  return bn_finalize_impl(scratch, nblk, count, gamma, beta, running_mean, running_var, num_batches_tracked, momentum, eps, scale, shift, mean, invstd, stream);
}

extern "C" int snb_bn_running_update(const float* mean, const float* invstd, long long count, float* running_mean, float* running_var,
                                     long long* num_batches_tracked, float momentum, float eps, void* stream) {
  SNB_REQUIRE(mean && invstd && running_mean && running_var && count > 0, "snb_bn_running_update: bad args");
  snb_launch(bn_running_update_kernel, 1, 32, 0, stream, mean, invstd, (double)count, eps, momentum, running_mean, running_var,
             num_batches_tracked);
  SNB_LAUNCH_CHECK("bn_running_update_kernel");
  return 0;
}

extern "C" int snb_bn_apply(const float* z, const float* scale, const float* shift, const float* residual, float* y,
                            long long npos, int lrelu_flag, void* stream) {
  SNB_REQUIRE(z && scale && shift && y && npos > 0, "snb_bn_apply: bad args");
  const long long n4 = npos * 8;
  long long blocks = (n4 + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  snb_launch(bn_apply_kernel, (int)blocks, 256, 0, stream, (const float4*)z, scale, shift, (const float4*)residual,
                                                                (float4*)y, n4, lrelu_flag);
  SNB_LAUNCH_CHECK("bn_apply_kernel");
  return 0;
}
