// normalize_features (src/feature_extraction.py:157-181): z-score over axis 0.
//
// np.mean / np.std over axis 0 sum in one of two orders, chosen by the array's layout (checked
// against NumPy 2.3.5).  When another axis is the iterator's inner loop (C order, row- or
// column-strided C views) they add the rows one after another.  When axis 0 is the inner loop
// (1-D, (n, 1), Fortran order, transposed views) every column is a 1-D pairwise sum.  The fit is
// one thread per column doing the same: rows in order, or with `pairwise` set NumPy's pairwise
// tree.  The caller picks the mode from its array's strides before copying it to C order
// (batch._axis0_is_inner), so the result is bit-identical to the reference, which matters
// because these statistics feed the KNN distances.
#include "kernels.cuh"
#include "misc.cuh"

namespace dsp {

namespace {

__global__ void zscore_fit_kernel(const double* __restrict__ x, int64_t n, int d, int pairwise,
                                  double* __restrict__ mean, double* __restrict__ std) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= d) return;
  double mu, var;
  if (pairwise) {
    auto t = [&](int64_t i) { return x[i * d + j]; };
    mu = np_pairwise_sum(t, n) / (double)n;
    auto t2 = [&](int64_t i) { const double v = x[i * d + j] - mu; return v * v; };
    var = np_pairwise_sum(t2, n) / (double)n;
  } else {
    double s = 0.0;
    for (int64_t i = 0; i < n; ++i) s += x[i * d + j];
    mu = s / (double)n;
    double s2 = 0.0;
    for (int64_t i = 0; i < n; ++i) { const double v = x[i * d + j] - mu; s2 += v * v; }
    var = s2 / (double)n;
  }
  mean[j] = mu;
  std[j] = sqrt(var);
}

// std == 0 -> 1 (feature_extraction.py:177); done once so the returned std matches the reference.
__global__ void zscore_fix_std_kernel(double* std, int d) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < d && std[j] == 0.0) std[j] = 1.0;
}

__global__ void zscore_apply_kernel(const double* __restrict__ x, int64_t total, int d,
                                    const double* __restrict__ mean, const double* __restrict__ std,
                                    double* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int j = (int)(i % d);
    out[i] = (x[i] - mean[j]) / std[j];
  }
}

// the same on float32 statistics straight out of the fused front end (widened exactly, then the reference's arithmetic)
__global__ void zscore_apply_f32_kernel(const float* __restrict__ x, int64_t total, int d,
                                        const double* __restrict__ mean, const double* __restrict__ std,
                                        double* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int j = (int)(i % d);
    const double s = std[j] == 0.0 ? 1.0 : std[j];
    out[i] = ((double)x[i] - mean[j]) / s;
  }
}

__global__ void f32_to_f64_kernel(const float* __restrict__ in, int64_t n, double* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (double)in[i];
}

}  // namespace

cudaError_t zscore_fit(const double* x, int64_t n, int d, int pairwise, double* mean, double* std,
                       cudaStream_t st) {
  zscore_fit_kernel<<<(d + 63) / 64, 64, 0, st>>>(x, n, d, pairwise, mean, std);
  return cudaGetLastError();
}

cudaError_t zscore_apply(const double* x, int64_t n, int d, const double* mean, double* std, double* out,
                         cudaStream_t st) {
  zscore_fix_std_kernel<<<(d + 63) / 64, 64, 0, st>>>(std, d);
  const int64_t total = n * d;
  if (total > 0) {
    const int grid = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
    zscore_apply_kernel<<<grid, 256, 0, st>>>(x, total, d, mean, std, out);
  }
  return cudaGetLastError();
}

cudaError_t zscore_apply_f32(const float* x, int64_t n, int d, const double* mean, const double* std, double* out,
                             cudaStream_t st) {
  const int64_t total = n * d;
  if (total > 0) {
    const int grid = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
    zscore_apply_f32_kernel<<<grid, 256, 0, st>>>(x, total, d, mean, std, out);
  }
  return cudaGetLastError();
}

cudaError_t widen_f32(const float* in, int64_t n, double* out, cudaStream_t st) {
  if (n > 0) {
    const int grid = (int)((n + 255) / 256 < 4096 ? (n + 255) / 256 : 4096);
    f32_to_f64_kernel<<<grid, 256, 0, st>>>(in, n, out);
  }
  return cudaGetLastError();
}

}  // namespace dsp
