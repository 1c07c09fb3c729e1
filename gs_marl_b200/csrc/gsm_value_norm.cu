// gsm_value_norm.cu — the critics' value normaliser (SPEC.md §15): the lineage's ValueNorm
// (utils/popart.py, SOURCES.txt:34), one per critic head, updated once per minibatch in the order the update
// trains on them.  Its own translation unit so that no env, actor or learner kernel is compiled differently.
//
// The returns do not change during an update, so one call does a whole epoch's normaliser work after the
// epoch's permutation is drawn: value_moments_kernel gathers R[rows[i]] over the epoch's
// n_mini_batch x mb permuted rows and writes per-block fp64 partial sums of R_h and R_h^2.  A minibatch owns
// blocks_per_mb(mb) blocks and no block straddles two minibatches, so the partition depends on
// (mb, n_mini_batch) only.  value_fold_kernel (one block) folds each minibatch's partials in a fixed tree
// order and runs the EMA over b = 0 .. n_mini_batch - 1, writing the affine each minibatch's backward reads.
// No atomics, no host sync: bit-identical across calls, streams and devices, capturable in a CUDA graph.
#include <cuda_runtime.h>

#include <climits>
#include <cstdint>

#include "../../include/gsmarl_b200.h"

namespace gsm_vn {

constexpr int F = 4;                       // partial sums per block: R_0, R_0^2, R_1, R_1^2
constexpr int THREADS = 256;
constexpr int ROWS_PER_BLOCK = THREADS * 8;
constexpr int MAX_BLOCKS_PER_MB = 512;     // a constant, NOT the device's SM count (determinism)
constexpr int FOLD_CHUNKS = 64;            // value_fold_kernel: F x FOLD_CHUNKS threads

inline int64_t blocks_per_mb(int64_t mb) {
  const int64_t b = (mb + ROWS_PER_BLOCK - 1) / ROWS_PER_BLOCK;
  return b < MAX_BLOCKS_PER_MB ? b : MAX_BLOCKS_PER_MB;
}

// block = (minibatch b, part k): rows [k chunk, (k + 1) chunk) of the minibatch, thread t takes every
// THREADS-th of them; the thread sums, then a warp shuffle tree, then the warps in ascending order
__global__ void __launch_bounds__(THREADS) value_moments_kernel(const float* __restrict__ ret,
                                                                const int64_t* __restrict__ rows, int64_t mb,
                                                                int parts, double* __restrict__ ws) {
  __shared__ double s[THREADS / 32][F];
  const int64_t b = blockIdx.x / parts;
  const int k = (int)(blockIdx.x - b * parts);
  const int64_t chunk = (mb + parts - 1) / parts;
  const int64_t lo = k * chunk, hi = lo + chunk < mb ? lo + chunk : mb;
  const int64_t* __restrict__ r = rows + b * mb;
  double v[F] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 4
  for (int64_t i = lo + threadIdx.x; i < hi; i += THREADS) {
    const int64_t src = r[i];
    const double x0 = ret[2 * src], x1 = ret[2 * src + 1];
    v[0] += x0; v[1] += x0 * x0; v[2] += x1; v[3] += x1 * x1;   // squares of fp32 values: exact in fp64
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int f = 0; f < F; f++) {
#pragma unroll
    for (int off = 16; off; off >>= 1) v[f] += __shfl_down_sync(0xffffffffu, v[f], off);
    if (lane == 0) s[w][f] = v[f];
  }
  __syncthreads();
  if (threadIdx.x < F) {
    double t = s[0][threadIdx.x];
    for (int q = 1; q < THREADS / 32; q++) t += s[q][threadIdx.x];
    ws[(int64_t)blockIdx.x * F + threadIdx.x] = t;
  }
}

// (mu, sigma) of one head's state (m, s, d), fp64 with one rounding per operation, rounded to fp32
__device__ void affine_of(const double* st, double eps, double var_floor, float* out) {
  const double d = fmax(st[2], eps);
  const double mu = __ddiv_rn(st[0], d);
  const double var = fmax(__dsub_rn(__ddiv_rn(st[1], d), __dmul_rn(mu, mu)), var_floor);
  out[0] = (float)mu;
  out[1] = (float)__dsqrt_rn(var);
}

// thread (chunk c, field f) sums partials c, c + FOLD_CHUNKS, ... of the minibatch; the chunk sums are halved
// pairwise in a fixed tree; thread 0 runs the EMA (explicit roundings: no contraction into fma)
__global__ void __launch_bounds__(F * FOLD_CHUNKS) value_fold_kernel(const double* __restrict__ ws, int parts,
                                                                     int64_t n_mini_batch, int64_t mb,
                                                                     double* __restrict__ state,
                                                                     float* __restrict__ affine, double beta,
                                                                     double eps, double var_floor) {
  __shared__ double s[FOLD_CHUNKS][F];
  const int f = threadIdx.x % F, c = threadIdx.x / F;
  double st[2][3];
  if (threadIdx.x == 0) {
#pragma unroll
    for (int h = 0; h < 2; h++)
      for (int q = 0; q < 3; q++) st[h][q] = state[3 * h + q];
  }
  const double omb = 1.0 - beta, n = (double)mb;
  for (int64_t b = 0; b < n_mini_batch; b++) {
    double acc = 0.0;
    for (int g = c; g < parts; g += FOLD_CHUNKS) acc += ws[(b * parts + g) * F + f];
    s[c][f] = acc;
    __syncthreads();
#pragma unroll
    for (int h = FOLD_CHUNKS / 2; h; h >>= 1) {
      if (c < h) s[c][f] += s[c + h][f];
      __syncthreads();
    }
    if (threadIdx.x == 0) {
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const double mean = __ddiv_rn(s[0][2 * h], n), mean_sq = __ddiv_rn(s[0][2 * h + 1], n);
        st[h][0] = __dadd_rn(__dmul_rn(beta, st[h][0]), __dmul_rn(omb, mean));
        st[h][1] = __dadd_rn(__dmul_rn(beta, st[h][1]), __dmul_rn(omb, mean_sq));
        st[h][2] = __dadd_rn(__dmul_rn(beta, st[h][2]), omb);
        affine_of(st[h], eps, var_floor, affine + (b * 2 + h) * 2);
      }
    }
    __syncthreads();                       // thread 0 has read s[0] before the next minibatch overwrites it
  }
  if (threadIdx.x == 0) {
#pragma unroll
    for (int h = 0; h < 2; h++) {
      for (int q = 0; q < 3; q++) state[3 * h + q] = st[h][q];
      affine_of(st[h], eps, var_floor, affine + (n_mini_batch * 2 + h) * 2);
    }
  }
}

struct DevGuard {
  int prev = -1;
  bool ok = true;
  explicit DevGuard(int d) {
    cudaGetDevice(&prev);
    if (d != prev) ok = cudaSetDevice(d) == cudaSuccess;
  }
  ~DevGuard() { int cur; cudaGetDevice(&cur); if (cur != prev && prev >= 0) cudaSetDevice(prev); }
};

// the grid (n_mini_batch x parts blocks) fits a launch and the row count fits int64
bool bad_shape(int64_t mb, int64_t n_mini_batch) {
  if (mb < 1 || n_mini_batch < 1) return true;
  return n_mini_batch > INT_MAX / blocks_per_mb(mb) || mb > INT64_MAX / n_mini_batch;
}

}  // namespace gsm_vn

extern "C" {

int64_t gsm_value_norm_update_workspace(int64_t mb, int64_t n_mini_batch) {
  if (gsm_vn::bad_shape(mb, n_mini_batch)) return GSM_ERR_INVALID_ARG;
  return n_mini_batch * gsm_vn::blocks_per_mb(mb) * gsm_vn::F * (int64_t)sizeof(double);
}

int gsm_value_norm_update(const gsm_value_norm_io* io, void* workspace, size_t workspace_bytes, int device,
                          void* stream) {
  if (!io) return GSM_ERR_INVALID_ARG;
  if (io->struct_size != sizeof(gsm_value_norm_io)) return GSM_ERR_ABI;
  if (!io->state || !io->affine || !io->returns || !io->rows) return GSM_ERR_INVALID_ARG;
  if (gsm_vn::bad_shape(io->mb, io->n_mini_batch)) return GSM_ERR_INVALID_ARG;
  if (!(io->beta >= 0.0 && io->beta < 1.0) || !(io->epsilon > 0.0) || !(io->var_floor > 0.0))
    return GSM_ERR_INVALID_ARG;
  const int64_t need = gsm_value_norm_update_workspace(io->mb, io->n_mini_batch);
  if (!workspace || workspace_bytes < (size_t)need) return GSM_ERR_INVALID_ARG;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return GSM_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= ndev) return GSM_ERR_INVALID_ARG;
  gsm_vn::DevGuard guard(device);
  if (!guard.ok) return GSM_ERR_CUDA;
  const cudaStream_t st = (cudaStream_t)stream;
  const int parts = (int)gsm_vn::blocks_per_mb(io->mb);
  double* ws = static_cast<double*>(workspace);
  gsm_vn::value_moments_kernel<<<(unsigned)(io->n_mini_batch * parts), gsm_vn::THREADS, 0, st>>>(
      io->returns, io->rows, io->mb, parts, ws);
  gsm_vn::value_fold_kernel<<<1, gsm_vn::F * gsm_vn::FOLD_CHUNKS, 0, st>>>(
      ws, parts, io->n_mini_batch, io->mb, io->state, io->affine, io->beta, io->epsilon, io->var_floor);
  return cudaGetLastError() == cudaSuccess ? GSM_OK : GSM_ERR_CUDA;
}

}  // extern "C"
