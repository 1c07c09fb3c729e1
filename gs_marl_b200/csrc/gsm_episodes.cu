// gsm_episodes.cu — episode return, cost and length across rollouts, per agent and per team
// (SPEC.md §13): the runner's episode logging over the rollout buffer's reward / cost / done slots
// (runner/mpe_runner.py, utils/graph_separated_buffer.py; SOURCES.txt:28,33).  Its own translation unit
// so that no env or actor kernel is compiled differently.
//
// episode_stats_kernel: one thread per row (one agent of one env), a block holds whole envs
// (rows_per_block = a multiple of N).  Per row the fp64 carry (R, C, n) walks the T slots in ascending t.
// The slots are loaded in groups of U with independent loads, so a thread's loop costs ceil(T / U) memory
// latencies, not T.  Every row parks its (R, C) after each slot of the group in shared memory; where the
// agent-0 row of some env of the block has done set inside the group (one __syncthreads_or per group), the
// env's first thread sums the parked values in ascending agent order.  Per-thread partials are summed per
// block in a fixed tree order into the workspace; episode_totals_kernel adds the G block partials in a fixed
// order.  G = min(tiles, EP_MAX_BLOCKS) depends on (n_rows, N) only, so `totals` is bit-identical across
// calls, streams and devices.  No floating-point atomics, no host sync: two launches, capturable in a CUDA
// graph.
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/gsmarl_b200.h"

namespace gsm_ep {

constexpr int F = GSM_EPISODE_STAT_FIELDS;
constexpr int EP_MAX_BLOCKS = 148 * 8;   // a constant, NOT the device's SM count (determinism)
constexpr int RED_CHUNKS = 32;           // episode_totals_kernel: F x RED_CHUNKS threads

struct EpParams {
  const void* reward; const void* cost; const uint8_t* done;
  double* carry_r; double* carry_c; int32_t* carry_n;
  double* last_r; double* last_c; int32_t* last_n;
  int32_t* episodes; double* team_last_r; double* team_last_c;
  double* ws;
  int64_t n_rows, slot_rows, n_tiles;
  int T, N, rows_per_block;
  double agent_limit, team_limit;
};

// rows per block: as many whole envs as fit 256 threads (N <= 256), else one env
inline int rows_per_block(int N) { return N <= 256 ? (256 / N) * N : N; }
inline int64_t n_tiles(int64_t n_rows, int N) {
  const int rpb = rows_per_block(N);
  return (n_rows + rpb - 1) / rpb;
}
inline int64_t n_blocks(int64_t n_rows, int N) {
  const int64_t t = n_tiles(n_rows, N);
  return t < EP_MAX_BLOCKS ? t : EP_MAX_BLOCKS;
}

struct Acc {   // one thread's partial totals of its row's agent episodes
  int count = 0, safe = 0, over = 0;
  double len = 0, r = 0, r2 = 0, c = 0, c2 = 0;
};

// blockDim.x = MAXT-bounded multiple of 32 >= rows_per_block; threads past rows_per_block only join the
// barriers and the reduction
template <class Real, int MAXT>
__global__ void __launch_bounds__(MAXT) episode_stats_kernel(const __grid_constant__ EpParams p) {
  // slots per load group (3 U registers of prefetch); the 1024-thread instance must fit 64 registers
  constexpr int U = MAXT > 256 ? 2 : (sizeof(Real) == 4 ? 8 : 4);
  constexpr int ENVS = MAXT > 256 ? 1 : 256;        // envs per block: N > 256 means one
  constexpr int H = F / 2;                           // fields per kind of episode
  __shared__ double s_r[U][MAXT], s_c[U][MAXT];       // every row's (R, C) after each slot of the group
  __shared__ double s_team[H][ENVS];                 // team partials; only the env's first thread touches its column
  double (*s_red)[F] = reinterpret_cast<double (*)[F]>(&s_r[0][0]);   // the block reduction reuses s_r
  static_assert((MAXT / 32) * F <= U * MAXT, "s_red fits in s_r");
  const Real* __restrict__ rw = static_cast<const Real*>(p.reward);
  const Real* __restrict__ cw = static_cast<const Real*>(p.cost);
  const int tid = threadIdx.x;
  const bool in_tile = tid < p.rows_per_block;
  const bool leader = in_tile && tid % p.N == 0;
  const int env_in_block = tid / p.N;
  for (int k = tid; k < H * ENVS; k += blockDim.x) (&s_team[0][0])[k] = 0.0;
  Acc a;
  for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
    const int64_t row = tile * p.rows_per_block + tid;
    const bool live = in_tile && row < p.n_rows;     // n_rows % N == 0: an env is wholly live or not
    double R = 0.0, Cs = 0.0;
    int n = 0, eps = 0;
    if (live) { R = p.carry_r[row]; Cs = p.carry_c[row]; n = p.carry_n[row]; }
    for (int t0 = 0; t0 < p.T; t0 += U) {
      Real r[U], c[U];
      uint32_t d[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        r[u] = Real(0); c[u] = Real(0); d[u] = 0;
        if (live && t0 + u < p.T) {
          const int64_t o = (int64_t)(t0 + u) * p.slot_rows + row;
          r[u] = rw[o]; c[u] = cw[o]; d[u] = p.done[o];
        }
      }
      int n_at[U];                                    // the row's length at each slot (agent 0's is the team's)
      uint32_t ends = 0;                              // slots of the group where this row's episode ends
#pragma unroll
      for (int u = 0; u < U; u++) {
        if (t0 + u >= p.T) break;                     // uniform across the block
        R += (double)r[u]; Cs += (double)c[u]; n++;
        s_r[u][tid] = R; s_c[u][tid] = Cs; n_at[u] = n;
        if (d[u]) {
          a.count++; a.len += n; a.r += R; a.r2 += R * R; a.c += Cs; a.c2 += Cs * Cs;
          a.safe += Cs == 0.0; a.over += Cs > p.agent_limit;
          if (p.last_r) p.last_r[row] = R;
          if (p.last_c) p.last_c[row] = Cs;
          if (p.last_n) p.last_n[row] = n;
          R = 0.0; Cs = 0.0; n = 0;
          ends |= 1u << u;
        }
      }
      if (__syncthreads_or(leader && ends)) {         // some env of the block ends inside this group
        if (leader && ends) {
#pragma unroll
          for (int u = 0; u < U; u++) {
            if (!(ends >> u & 1u)) continue;
            double tr = 0.0, tc = 0.0;
            for (int j = 0; j < p.N; j++) { tr += s_r[u][tid + j]; tc += s_c[u][tid + j]; }
            tr /= p.N;
            double* t = &s_team[0][env_in_block];
            t[0 * ENVS] += 1.0; t[1 * ENVS] += tr; t[2 * ENVS] += tr * tr; t[3 * ENVS] += tc;
            t[4 * ENVS] += tc * tc; t[5 * ENVS] += n_at[u]; t[6 * ENVS] += tc == 0.0;
            t[7 * ENVS] += tc > p.team_limit;
            eps++;
            const int64_t env = row / p.N;        // a later completion overwrites: the last one stays
            if (p.team_last_r) p.team_last_r[env] = tr;
            if (p.team_last_c) p.team_last_c[env] = tc;
          }
        }
        __syncthreads();                              // the reads above before the next group's parking
      }
    }
    if (live) {
      p.carry_r[row] = R; p.carry_c[row] = Cs; p.carry_n[row] = n;
      if (leader) p.episodes[row / p.N] = eps;
    }
  }
  // block partials in a fixed order: warp shuffle tree, then the warps' sums in ascending order; thread k
  // brings the team partials of the block's env k
  __syncthreads();
  const bool tk = tid < p.rows_per_block / p.N;
  double v[F] = {(double)a.count, a.r, a.r2, a.c, a.c2, a.len, (double)a.safe, (double)a.over};
#pragma unroll
  for (int f = 0; f < H; f++) v[H + f] = tk ? s_team[f][tid] : 0.0;
  const int lane = tid & 31, w = tid >> 5;
#pragma unroll
  for (int f = 0; f < F; f++) {
#pragma unroll
    for (int off = 16; off; off >>= 1) v[f] += __shfl_down_sync(0xffffffffu, v[f], off);
    if (lane == 0) s_red[w][f] = v[f];
  }
  __syncthreads();
  if (tid < F) {
    double s = s_red[0][tid];
    for (int q = 1; q < (int)(blockDim.x >> 5); q++) s += s_red[q][tid];
    p.ws[(int64_t)blockIdx.x * F + tid] = s;
  }
}

// totals[f] = sum of the G block partials: thread (chunk c, field f) sums partials c, c + 32, ...; the 32
// chunk sums are then halved pairwise in a fixed tree.  Consecutive threads read consecutive doubles.
__global__ void __launch_bounds__(F * RED_CHUNKS) episode_totals_kernel(const double* __restrict__ ws, int G,
                                                                        double* __restrict__ totals) {
  __shared__ double s[RED_CHUNKS][F];
  const int f = threadIdx.x % F, c = threadIdx.x / F;
  double acc = 0.0;
#pragma unroll 4
  for (int g = c; g < G; g += RED_CHUNKS) acc += ws[(int64_t)g * F + f];
  s[c][f] = acc;
  __syncthreads();
#pragma unroll
  for (int h = RED_CHUNKS / 2; h; h >>= 1) {
    if (c < h) s[c][f] += s[c + h][f];
    __syncthreads();
  }
  if (c == 0) totals[f] = s[0][f];
}

template <class Real>
int launch(const EpParams& p0, double* totals, cudaStream_t st) {
  EpParams p = p0;
  const int G = (int)n_blocks(p.n_rows, p.N);
  p.rows_per_block = rows_per_block(p.N);
  p.n_tiles = n_tiles(p.n_rows, p.N);
  const unsigned block = (unsigned)((p.rows_per_block + 31) / 32 * 32);
  if (block <= 256) episode_stats_kernel<Real, 256><<<G, block, 0, st>>>(p);
  else episode_stats_kernel<Real, 1024><<<G, block, 0, st>>>(p);
  episode_totals_kernel<<<1, F * RED_CHUNKS, 0, st>>>(p.ws, G, totals);
  return (int)cudaGetLastError();
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

bool bad_shape(int64_t n_rows, int32_t N) {
  return n_rows < 0 || N < 1 || N > 1024 || n_rows % N != 0;
}

}  // namespace gsm_ep

extern "C" {

int64_t gsm_episode_stats_workspace(int64_t n_rows, int32_t agents_per_env) {
  if (gsm_ep::bad_shape(n_rows, agents_per_env)) return GSM_ERR_INVALID_ARG;
  return gsm_ep::n_blocks(n_rows, agents_per_env) * gsm_ep::F * (int64_t)sizeof(double);
}

int gsm_episode_stats(const gsm_episode_io* io, void* workspace, size_t workspace_bytes, int device,
                      void* stream) {
  if (!io) return GSM_ERR_INVALID_ARG;
  if (io->struct_size != sizeof(gsm_episode_io)) return GSM_ERR_ABI;
  if (!io->reward || !io->cost || !io->done || !io->carry_return || !io->carry_cost || !io->carry_length ||
      !io->totals || !io->episodes)
    return GSM_ERR_INVALID_ARG;
  if (io->n_steps < 1 || gsm_ep::bad_shape(io->n_rows, io->agents_per_env) || io->slot_rows < io->n_rows)
    return GSM_ERR_INVALID_ARG;
  if (io->dtype != GSM_F32 && io->dtype != GSM_F64) return GSM_ERR_INVALID_ARG;
  const int64_t need = gsm_episode_stats_workspace(io->n_rows, io->agents_per_env);
  if (need > 0 && (!workspace || workspace_bytes < (size_t)need)) return GSM_ERR_INVALID_ARG;
  if (io->n_rows == 0) return GSM_OK;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return GSM_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= ndev) return GSM_ERR_INVALID_ARG;
  gsm_ep::DevGuard guard(device);
  if (!guard.ok) return GSM_ERR_CUDA;
  gsm_ep::EpParams p{};
  p.reward = io->reward; p.cost = io->cost; p.done = io->done;
  p.carry_r = io->carry_return; p.carry_c = io->carry_cost; p.carry_n = io->carry_length;
  p.last_r = io->last_return; p.last_c = io->last_cost; p.last_n = io->last_length;
  p.episodes = io->episodes; p.team_last_r = io->team_last_return; p.team_last_c = io->team_last_cost;
  p.ws = static_cast<double*>(workspace);
  p.n_rows = io->n_rows; p.slot_rows = io->slot_rows;
  p.T = io->n_steps; p.N = io->agents_per_env;
  p.agent_limit = io->agent_cost_limit; p.team_limit = io->team_cost_limit;
  const cudaStream_t st = (cudaStream_t)stream;
  const int e = io->dtype == GSM_F32 ? gsm_ep::launch<float>(p, io->totals, st)
                                     : gsm_ep::launch<double>(p, io->totals, st);
  return e ? GSM_ERR_CUDA : GSM_OK;
}

}  // extern "C"
