// gsm_policy.cu — SURVEY.md §8 row f3: the graph-attention actor's forward pass over the padded
// neighbour rows the env kernels write, plus action sampling, as ONE kernel, and the collect
// loop (row f1) as a C-level launch sequence of {actor, env step} pairs.
//
// Reference side (withheld): the GNN encoder of gsmarl/algorithms/* over torch-geometric
// (requirements.txt:119) called from runner/mpe_runner.py's collect (SOURCES.txt:28).  The
// architecture is therefore DECLARED (SPEC.md §10), not GS-MARL's: shared parameters over agents,
//   e   = relu(W_e obs + b_e)                               [H]
//   m_r = relu(W_n feat_r + b_n),  r < cnt                  [H] per valid neighbour row
//   a_r = softmax_r(w_a . m_r + b_a)                        masked to the cnt valid rows
//   z   = W_h [e ; sum_r a_r m_r] + b_h                     [n_actions] logits
//   action = argmax_k (z_k + Gumbel_k),  Gumbel from Philox4x32-10 keyed like the env resets.
// For continuous-action worlds the same embedding feeds a diagonal Gaussian head (SPEC.md §10b / §12b,
// HeadKind below): action = W_mu h + b_mu + exp(log_std) eps, eps by Box-Muller on the same Philox stream.
//
// Design for sm_100a (details in front of graph_actor_kernel below): a block owns 128 agents; the
// ego branch runs as packed FFMA2 over agent pairs, the block's VALID neighbour rows are flattened
// into one list of work items processed two per thread as packed FFMA2 (no divergence on the
// per-agent row count), and a per-agent online softmax folds the parked row results.  The weights
// ride in the kernel PARAMETER space (9.5 KB, __grid_constant__): the 64-wide hidden loops are fully
// unrolled, every weight has an immediate constant-bank offset, ptxas fetches four at a time with
// LDCU.128 into uniform registers and the FFMA2s take them as the broadcast uniform-scalar operand —
// no weight ever goes through a load/store unit.  The head is linear, so W_h's neighbour half is
// applied to every row's m_r on the fly (hr = W_h[:, H:] m_r): nothing of size H is ever stored.
// Only the cnt valid rows are visited; the padded rows the env kernel zero-fills are never read.
// Bound: fp32 issue / FMA pipe (54 % of the measured 72 TFLOP/s FFMA peak at 786k rows), not HBM
// (220 B per agent in, 8 B out).  History of the rejected forms (thread per agent, hidden-unit pair
// packing, shared-memory weights with rolled loops): profiles/README.md, profiles/rejected/.
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstring>
#include <type_traits>

#include "../../include/gsmarl_b200.h"

namespace gsm {

constexpr int H = GSM_POLICY_HIDDEN;

struct PolicyParams {                 // kernel-parameter image of gsm_policy_weights
  float ego_w[H][GSM_OBS_DIM];
  float ego_b[H];
  float nbr_w[H][GSM_NBR_FEAT_DIM];
  float nbr_b[H];
  float att_w[H];
  // rows 0..NA-1: action logits; rows NA, NA+1: the two critics (reward value, cost value)
  float head_w[GSM_POLICY_MAX_ACTIONS + GSM_POLICY_VALUE_HEADS][2 * H];
  float head_b[GSM_POLICY_MAX_ACTIONS + GSM_POLICY_VALUE_HEADS];
  float att_b;
};

// Head kinds (SPEC.md §10 / §10b).  The embedding h = [e; sum_r a_r m_r] and everything that computes
// it are shared; the kind selects the weights' image, the action type and the epilogue.
//   HEAD_CAT:   NA logits, categorical sample (Gumbel-max), int32 action.
//   HEAD_GAUSS: NA = GSM_POLICY_GAUSS_DIM means, diagonal Gaussian with a state-independent log_std,
//               float action [2] = mean + exp(log_std) eps (Box-Muller), no clamping.
enum HeadKind { HEAD_CAT = 0, HEAD_GAUSS = 1 };
constexpr int GD = GSM_POLICY_GAUSS_DIM;

struct GaussParams {                  // kernel-parameter image of gsm_policy_gauss_weights
  float ego_w[H][GSM_OBS_DIM];
  float ego_b[H];
  float nbr_w[H][GSM_NBR_FEAT_DIM];
  float nbr_b[H];
  float att_w[H];
  // rows 0..GD-1: the means; rows GD, GD+1: the two critics
  float head_w[GD + GSM_POLICY_VALUE_HEADS][2 * H];
  float head_b[GD + GSM_POLICY_VALUE_HEADS];
  float att_b;
  float log_std[GD];
};

template <int KIND> struct Head;
template <> struct Head<HEAD_CAT> { using Params = PolicyParams; using Act = int32_t; };
template <> struct Head<HEAD_GAUSS> { using Params = GaussParams; using Act = float; };

template <int KIND> struct ActorIO {
  const float* obs; const float* nbr_feat; const int32_t* nbr_cnt;
  typename Head<KIND>::Act* actions;   // [n_rows] (categorical) or [n_rows][GD] (Gaussian)
  float* logp;
  float* dist;                         // [n_rows][NA]: the logits or the means; NULL = skip
  float* values;
  int64_t n_rows; uint64_t row_offset, seed, step;
  int K, greedy;
};
using PolicyIO = ActorIO<HEAD_CAT>;
using GaussIO = ActorIO<HEAD_GAUSS>;

__device__ __forceinline__ void philox_p(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                         uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
    const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = h1 ^ c1 ^ k0, n2 = h0 ^ c3 ^ k1;
    c0 = n0; c1 = l1; c2 = n2; c3 = l0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// the categorical sampler's map of a Philox word to (0, 1), below
__device__ __forceinline__ float unit_open(uint32_t x) {
  return (float)(x >> 9) * 1.1920928955078125e-7f + 5.9604644775390625e-8f;
}

// SPEC.md §10b: log N(a; mu, exp(log_std)^2) summed over the two dimensions, with
// delta_d = (a_d - mu_d) exp(-log_std_d) returned for the backward.  The actor and the learner call
// this ONE function on the STORED action, and every rounding is explicit (no contraction that could
// differ between the call sites), so what collect wrote and what evaluate returns are bit-identical.
// A non-finite action gives NaN: a - a is 0 for every finite a and NaN otherwise.
__device__ __forceinline__ float gauss_logp(float a0, float a1, float mu0, float mu1, float ls0, float ls1,
                                            float& d0, float& d1) {
  constexpr float LOG_2PI = 1.8378770664093453f;
  d0 = __fmul_rn(__fsub_rn(a0, mu0), expf(-ls0));
  d1 = __fmul_rn(__fsub_rn(a1, mu1), expf(-ls1));
  const float t0 = __fsub_rn(__fmul_rn(-0.5f, __fmul_rn(d0, d0)), ls0);
  const float t1 = __fsub_rn(__fmul_rn(-0.5f, __fmul_rn(d1, d1)), ls1);
  const float fin = __fadd_rn(__fsub_rn(a0, a0), __fsub_rn(a1, a1));
  return __fadd_rn(__fsub_rn(__fadd_rn(t0, t1), LOG_2PI), fin);
}

// entropy of the diagonal Gaussian: sum_d log_std_d + 1/2 (1 + log 2 pi)
__device__ __forceinline__ float gauss_entropy(float ls0, float ls1) {
  constexpr float HALF_LOG_2PIE = 1.4189385332046727f;
  return __fadd_rn(__fadd_rn(ls0, HALF_LOG_2PIE), __fadd_rn(ls1, HALF_LOG_2PIE));
}

// NV = 0: actor only; NV = GSM_POLICY_VALUE_HEADS: the critics ride along as NV more rows of the head
// (+2 FFMA per hidden unit and row), for collect loops that store value predictions.
//
// Work decomposition ("flattened rows").  A block owns 128 consecutive agents.  Phase 1: the ego
// branch, agents (t, t + 64) packed into the two halves of float2 registers on warps 0-1.  Phase 2:
// the block's valid neighbour rows — sum(cnt) of them, found through an exclusive prefix of cnt —
// are one flat list of independent work items; a thread takes items q and q + 128 (agent by binary
// search in the prefix, 7 steps), again packed in float2 halves, computes their attention scores and
// head contributions and parks 1 + NZ floats per row in shared memory.  Phase 3: thread a folds its
// own agent's rows, in row order, into the online softmax.  Every lane of every warp carries a real
// row in phase 2 whatever the per-agent counts are (30 of 32 lanes active; the thread-per-agent
// version had 20.8, and 28.1 after a per-block counting sort by cnt).  Row items are processed in
// chunks of CH so that shared memory does not depend on K.
//
// Arithmetic: Blackwell's packed fp32 FMA (FFMA2, `fma.rn.f32x2`) with the weight as the BROADCAST
// uniform scalar operand (`FFMA2 R, R.F32x2, UR.F32, R.F32x2`) — profiles/fma_peak.cu measures that
// form at the full 127 FMA/clk/SM for half the issue slots of scalar FFMA, while a constant PAIR
// operand (packing two hidden units instead of two rows) runs at 32.  Feature loads are scalar on
// purpose: a 64-bit load pins (x, y) of one row to an aligned register pair and ptxas then
// re-assembles every (row 0, row 1) operand pair with two MOVs per FFMA2.
__device__ __forceinline__ float2 bc(float w) { return make_float2(w, w); }

//
// KIND (HeadKind) changes only the epilogue after the z rows are complete: NA logits or NA = GD means.
template <int NA, int NV, int KIND>
__global__ void __launch_bounds__(128)
graph_actor_kernel(const __grid_constant__ typename Head<KIND>::Params w, const __grid_constant__ ActorIO<KIND> io) {
  constexpr int NZ = NA + NV, AG = 128, RS = NZ + 1, CH = RS <= 10 ? 1024 : 512;   // static smem <= 48 KB
  __shared__ int s_pre[AG + 1];
  __shared__ int s_wtot[4];
  __shared__ float s_row[CH * RS];
  __shared__ float s_z[AG * NZ];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t base = (int64_t)blockIdx.x * AG;
  const int64_t i = base + tid;
  const bool valid = i < io.n_rows;
  int cnt = 0;
  if (valid) { cnt = io.nbr_cnt[i]; cnt = cnt < 0 ? 0 : (cnt > io.K ? io.K : cnt); }
  {  // exclusive prefix of cnt over the block
    int x = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(~0u, x, d); if (lane >= d) x += y; }
    if (lane == 31) s_wtot[warp] = x;
    __syncthreads();
    int off = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) off += k < warp ? s_wtot[k] : 0;
    s_pre[tid] = off + x - cnt;
    if (tid == AG - 1) s_pre[AG] = off + x;
  }

  // phase 1: ego branch, agents (t, t + 64) packed into one thread of warps 0-1 (FFMA2, as below);
  // warps 2-3 go straight to the barrier and leave their issue slots to other blocks
  if (tid < AG / 2 && valid) {
    const int64_t iB = i + AG / 2 < io.n_rows ? i + AG / 2 : i;
    const float* oA = io.obs + i * GSM_OBS_DIM;
    const float* oB = io.obs + iB * GSM_OBS_DIM;
    const float2 d0 = make_float2(oA[0], oB[0]), d1 = make_float2(oA[1], oB[1]), d2 = make_float2(oA[2], oB[2]),
                 d3 = make_float2(oA[3], oB[3]), d4 = make_float2(oA[4], oB[4]), d5 = make_float2(oA[5], oB[5]);
    float2 z2[NZ];
#pragma unroll
    for (int a = 0; a < NZ; a++) z2[a] = bc(w.head_b[a]);
#pragma unroll
    for (int j = 0; j < H; j++) {
      float2 e = bc(w.ego_b[j]);
      e = __ffma2_rn(bc(w.ego_w[j][0]), d0, e); e = __ffma2_rn(bc(w.ego_w[j][1]), d1, e);
      e = __ffma2_rn(bc(w.ego_w[j][2]), d2, e); e = __ffma2_rn(bc(w.ego_w[j][3]), d3, e);
      e = __ffma2_rn(bc(w.ego_w[j][4]), d4, e); e = __ffma2_rn(bc(w.ego_w[j][5]), d5, e);
      e.x = fmaxf(e.x, 0.f); e.y = fmaxf(e.y, 0.f);
#pragma unroll
      for (int a = 0; a < NZ; a++) z2[a] = __ffma2_rn(bc(w.head_w[a][j]), e, z2[a]);
    }
#pragma unroll
    for (int a = 0; a < NZ; a++) { s_z[tid * NZ + a] = z2[a].x; s_z[(tid + AG / 2) * NZ + a] = z2[a].y; }
  }
  __syncthreads();                      // s_pre complete
  const int total = s_pre[AG];
  const int my0 = s_pre[tid], my1 = my0 + cnt;
  float z[NZ];
#pragma unroll
  for (int a = 0; a < NZ; a++) z[a] = s_z[tid * NZ + a];       // garbage for !valid threads, never used

  // online softmax state of MY agent over its rows, in row order
  float mx = -__int_as_float(0x7f800000), s = 0.f, acc[NZ];
#pragma unroll
  for (int a = 0; a < NZ; a++) acc[a] = 0.f;
  const float* ffeat = io.nbr_feat + base * (int64_t)io.K * GSM_NBR_FEAT_DIM;

  for (int c0 = 0; c0 < total; c0 += CH) {          // block-uniform trip count
    const int cend = total < c0 + CH ? total : c0 + CH;
    // phase 2: TWO neighbour rows per thread (items q and q + AG), packed into the halves of float2
    // registers for Blackwell's packed fp32 FMA (FFMA2, `fma.rn.f32x2`) with the weight as the
    // broadcast uniform scalar operand — full FMA rate at half the issue slots of scalar FFMA
    // (profiles/fma_peak.cu).  Items are homogeneous, so the pairing costs no divergence; an odd
    // tail duplicates its row into the second half and stores it once.
    for (int q = c0 + tid; q < cend; q += 2 * AG) {
      const int q1 = q + AG < cend ? q + AG : q;
      int lo0 = 0, hi0 = AG, lo1 = 0, hi1 = AG;     // largest a with s_pre[a] <= q
#pragma unroll
      for (int it = 0; it < 7; it++) {
        const int m0 = (lo0 + hi0) >> 1, m1 = (lo1 + hi1) >> 1;
        if (s_pre[m0] <= q) lo0 = m0; else hi0 = m0;
        if (s_pre[m1] <= q1) lo1 = m1; else hi1 = m1;
      }
      // scalar loads on purpose: a 64-bit load pins (x, y) of ONE row to an aligned register pair and
      // ptxas then re-assembles every (row 0, row 1) operand pair with two MOVs per FFMA2
      const float* g0 = ffeat + ((int64_t)lo0 * io.K + (q - s_pre[lo0])) * GSM_NBR_FEAT_DIM;
      const float* g1 = ffeat + ((int64_t)lo1 * io.K + (q1 - s_pre[lo1])) * GSM_NBR_FEAT_DIM;
      const float2 d0 = make_float2(g0[0], g1[0]), d1 = make_float2(g0[1], g1[1]), d2 = make_float2(g0[2], g1[2]),
                   d3 = make_float2(g0[3], g1[3]), d4 = make_float2(g0[4], g1[4]), d5 = make_float2(g0[5], g1[5]);
      float2 t2 = bc(w.att_b), hr[NZ];
#pragma unroll
      for (int a = 0; a < NZ; a++) hr[a] = make_float2(0.f, 0.f);
#pragma unroll
      for (int j = 0; j < H; j++) {
        float2 m = bc(w.nbr_b[j]);
        m = __ffma2_rn(bc(w.nbr_w[j][0]), d0, m); m = __ffma2_rn(bc(w.nbr_w[j][1]), d1, m);
        m = __ffma2_rn(bc(w.nbr_w[j][2]), d2, m); m = __ffma2_rn(bc(w.nbr_w[j][3]), d3, m);
        m = __ffma2_rn(bc(w.nbr_w[j][4]), d4, m); m = __ffma2_rn(bc(w.nbr_w[j][5]), d5, m);
        m.x = fmaxf(m.x, 0.f); m.y = fmaxf(m.y, 0.f);
        t2 = __ffma2_rn(bc(w.att_w[j]), m, t2);
#pragma unroll
        for (int a = 0; a < NZ; a++) hr[a] = __ffma2_rn(bc(w.head_w[a][H + j]), m, hr[a]);
      }
      float* o0 = s_row + (q - c0) * RS;
      o0[0] = t2.x;
#pragma unroll
      for (int a = 0; a < NZ; a++) o0[1 + a] = hr[a].x;
      if (q1 != q) {
        float* o1 = s_row + (q1 - c0) * RS;
        o1[0] = t2.y;
#pragma unroll
        for (int a = 0; a < NZ; a++) o1[1 + a] = hr[a].y;
      }
    }
    __syncthreads();
    {  // phase 3: fold my agent's rows of this chunk
      const int lo = my0 > c0 ? my0 : c0, hi = my1 < cend ? my1 : cend;
      for (int q = lo; q < hi; q++) {
        const float* o = s_row + (q - c0) * RS;
        const float t = o[0];
        const float nm = fmaxf(mx, t);
        const float sc = expf(mx - nm), pw = expf(t - nm);   // first row: exp(-inf) = 0
        s = fmaf(s, sc, pw);
#pragma unroll
        for (int a = 0; a < NZ; a++) acc[a] = fmaf(acc[a], sc, pw * o[1 + a]);
        mx = nm;
      }
    }
    __syncthreads();                    // before the next chunk overwrites s_row
  }
  if (!valid) return;
  if (cnt > 0) {
    const float inv = 1.f / s;
#pragma unroll
    for (int a = 0; a < NZ; a++) z[a] = fmaf(acc[a], inv, z[a]);
  }
  if (NV > 0) {
#pragma unroll
    for (int v = 0; v < NV; v++) io.values[i * NV + v] = z[NA + v];
  }

  if (io.dist) {
#pragma unroll
    for (int a = 0; a < NA; a++) io.dist[i * NA + a] = z[a];
  }

  if constexpr (KIND == HEAD_GAUSS) {
    static_assert(NA == GD, "the Gaussian head has GD means");
    // sample: Box-Muller on words 0, 1 of one Philox block, counter (row lo, row hi, step, 0x80000000)
    float a0 = z[0], a1 = z[1];
    if (!io.greedy) {
      const uint64_t g = io.row_offset + (uint64_t)i;
      uint32_t r[4];
      philox_p((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)io.step, 0x80000000u,
               (uint32_t)io.seed, (uint32_t)(io.seed >> 32), r);
      const float rho = sqrtf(-2.f * logf(unit_open(r[0])));
      float sn, cs;
      sincospif(2.f * unit_open(r[1]), &sn, &cs);      // 2 u is exact
      a0 = fmaf(expf(w.log_std[0]), rho * cs, z[0]);
      a1 = fmaf(expf(w.log_std[1]), rho * sn, z[1]);
    }
    io.actions[i * GD] = a0;
    io.actions[i * GD + 1] = a1;
    if (io.logp) {
      float d0, d1;
      io.logp[i] = gauss_logp(a0, a1, z[0], z[1], w.log_std[0], w.log_std[1], d0, d1);
    }
    return;                             // (the categorical epilogue below is unreachable here)
  }

  // sample: Gumbel-max, one Philox block per 4 actions; counter (row lo, row hi, step, block)
  int best = 0;
  float zb = z[0];                      // logit of the chosen action
  if (io.greedy) {
#pragma unroll
    for (int a = 1; a < NA; a++) if (z[a] > zb) { zb = z[a]; best = a; }
  } else {
    const uint64_t g = io.row_offset + (uint64_t)i;
    float bv = 0.f;
#pragma unroll
    for (int b = 0; b < (NA + 3) / 4; b++) {
      uint32_t r[4];
      philox_p((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)io.step, 0x80000000u | (uint32_t)b,
               (uint32_t)io.seed, (uint32_t)(io.seed >> 32), r);
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const int a = 4 * b + q;
        if (a < NA) {
          // 23 random bits + half a step: every value k * 2^-23 + 2^-24 is exact in fp32 and lies in (0, 1)
          const float u = (float)(r[q] >> 9) * 1.1920928955078125e-7f + 5.9604644775390625e-8f;
          const float v = z[a] - logf(-logf(u));
          if (a == 0 || v > bv) { bv = v; best = a; zb = z[a]; }
        }
      }
    }
  }
  io.actions[i] = best;
  if (io.logp) {
    float zm = z[0];
#pragma unroll
    for (int a = 1; a < NA; a++) zm = fmaxf(zm, z[a]);
    float se = 0.f;
#pragma unroll
    for (int a = 0; a < NA; a++) se += expf(z[a] - zm);
    io.logp[i] = zb - zm - logf(se);
  }
}

// ---- buffer.compute_returns / compute_cost_returns (utils/graph_separated_buffer.py, SOURCES.txt:33;
// withheld — the on-policy lineage's GAE recursion, [DECL] SPEC.md §11): one thread per (row, head),
// backward scan over the T slots; consecutive threads touch consecutive addresses in every slot.
struct GaeParams {
  const float* reward; const float* cost; const float* values; const uint8_t* done;
  float* returns; float* adv;
  int64_t n_rows, slot_rows;
  int T;
  float gamma, lam;
};
__global__ void __launch_bounds__(256) gae_kernel(const __grid_constant__ GaeParams p) {
  constexpr int V = GSM_POLICY_VALUE_HEADS;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= p.n_rows * V) return;
  const int64_t row = g / V;
  const int head = (int)(g - row * V);
  const float* rw = head == 0 ? p.reward : p.cost;
  float gae = 0.f;
  float v_next = p.values[((int64_t)p.T * p.slot_rows + row) * V + head];
  for (int t = p.T - 1; t >= 0; t--) {
    const int64_t o = (int64_t)t * p.slot_rows + row;
    const float mask = p.done[o] ? 0.f : 1.f;      // done at step t: slot t+1 starts a new episode
    const float v = p.values[o * V + head];
    const float delta = rw[o] + p.gamma * v_next * mask - v;
    gae = delta + p.gamma * p.lam * mask * gae;
    if (p.adv) p.adv[o * V + head] = gae;
    p.returns[o * V + head] = gae + v;
    v_next = v;
  }
}

// ---- learner pass (SPEC.md §12): evaluate_actions forward and backward -------------------------
// The lineage's evaluate_actions (SOURCES.txt:8, withheld) over the declared actor: per row the
// log-prob of a GIVEN action, the entropy of softmax(z) and the two critics, and the gradient of
//   L = sum_i d_logp[i] logp[i] + d_entropy[i] entropy[i] + d_values[i] . values[i]
// with respect to the parameter vector (torch parameters_to_vector order, a DEVICE vector that an
// optimiser changes every step: it cannot travel in the parameter space like gsm_policy_weights, so
// every block copies it to shared memory).
//
// Forward (policy_eval_kernel): thread per row, the operation order of graph_actor_kernel — the same
// fmaf chains over j (FFMA2 halves are independent fma.rn, so scalar fmaf rounds identically), the
// rows folded in row order through the same online softmax — so logp and values are bit-identical
// to what gsm_policy_act / gsm_collect wrote.  One row per thread instead of the actor's flattened
// row items: simpler, divergent on nbr_cnt, and the learner pass is not the collect loop's hot path.
//
// Backward (policy_backward_kernel), with h = [e; g], g = sum_r a_r m_r, Z = [z; v], W = [W_h; W_v]:
//   dz = d_logp (onehot(a) - p) - d_entropy p o (log p + entropy),  dZ = [dz; d_values]
//   dh = W^T dZ;  dW += dZ h^T;  de = dh[:H] o [e > 0];  dg = dh[H:]
//   m_r . dg = dZ . hr_r with hr_r = W[:, H:] m_r, so ds_r = a_r (dZ . hr_r - dZ . (sum_r a_r hr_r))
//   needs no H-vector; dm_r = a_r dg + ds_r w_a;  du_r = dm_r o [u_r > 0]
//   dW_n += du_r f_r^T;  db_n += du_r;  dw_a += ds_r m_r;  db_a += ds_r;  dW_e += de obs^T;  db_e += de.
// A block owns AG = 64 rows per tile.  Phase A, thread per row: the forward (first pass over the
// rows), dZ, then a second pass over the rows recomputing (t_r, hr_r) to get a_r and ds_r, parked in
// shared memory (8 B per valid row) — nothing of size H per neighbour row is stored anywhere.
// Phase B, thread per HIDDEN UNIT j: loops over the tile's rows in order, recomputes e_j and u_rj from
// obs and f_r (broadcast reads) and accumulates every gradient entry of unit j in registers
// (dW_e[j], db_e[j], dW_n[j], db_n[j], dw_a[j], W[:, j], W[:, H + j]); the NZ + 1 bias sums ride on
// threads 0..NZ-1 and H-1.  Each thread owns distinct entries, so there is no atomic: a block walks
// tiles blockIdx, blockIdx + G, ... in order and writes ONE partial vector to the workspace;
// policy_grad_reduce_kernel sums the G partials in a fixed order.  G = min(tiles, BWD_MAX_BLOCKS)
// depends on n_rows only, so grad is bit-identical across calls, streams and B200s.
constexpr int V2 = GSM_POLICY_VALUE_HEADS;
constexpr int BWD_AG = 64;                 // rows per tile = threads per backward block (= H)
constexpr int BWD_MAX_BLOCKS = 148 * 6;    // one wave at 6 blocks/SM (168 registers); a constant, NOT the device's SM count
static_assert(BWD_AG == H, "phase B maps one thread to one hidden unit");

template <int NA, int KIND> struct PV {     // offsets into the parameter vector
  // the Gaussian's log_std [NA] sits between the head and the critics (parameters_to_vector order)
  static constexpr int EW = 0, EB = EW + H * GSM_OBS_DIM, NW = EB + H, NB = NW + H * GSM_NBR_FEAT_DIM,
                       AW = NB + H, AB = AW + H, HW = AB + 1, HB = HW + NA * 2 * H, LS = HB + NA,
                       VW = LS + (KIND == HEAD_GAUSS ? NA : 0), VB = VW + V2 * 2 * H, N = VB + V2;
  static __host__ __device__ constexpr int row(int a) { return a < NA ? HW + a * 2 * H : VW + (a - NA) * 2 * H; }
  static __host__ __device__ constexpr int bias(int a) { return a < NA ? HB + a : VB + (a - NA); }
};
static_assert(PV<5, HEAD_CAT>::N == GSM_POLICY_N_PARAMS(5) && PV<5, HEAD_CAT>::N == 1864 &&
              PV<9, HEAD_CAT>::N == 2380, "vector size");
static_assert(PV<GD, HEAD_GAUSS>::N == GSM_POLICY_GAUSS_N_PARAMS && GSM_POLICY_GAUSS_N_PARAMS == 1479, "vector size");

template <int KIND> struct EvalArgs {
  const float* params; const float* obs; const float* nbr_feat; const int32_t* nbr_cnt;
  const typename Head<KIND>::Act* actions;   // [src_rows] or [src_rows][GD]
  const int64_t* rows;
  float* logp; float* entropy; float* values;                 // forward outputs
  const float* d_logp; const float* d_entropy; const float* d_values;   // backward inputs
  float* ws;                                                  // backward: [gridDim.x][N] partials
  int64_t n_rows, n_tiles;
  int K;
};

// e-branch of graph_actor_kernel: z[a] = b[a] + sum_j W[a][j] relu(W_e obs + b_e)_j, same chains
template <int NA, int KIND>
__device__ __forceinline__ void ego_logits(const float* W, const float* o, float (&z)[NA + V2]) {
  using P = PV<NA, KIND>;
  const float o0 = o[0], o1 = o[1], o2 = o[2], o3 = o[3], o4 = o[4], o5 = o[5];
#pragma unroll
  for (int a = 0; a < NA + V2; a++) z[a] = W[P::bias(a)];
#pragma unroll
  for (int j = 0; j < H; j++) {
    const float* we = W + P::EW + j * GSM_OBS_DIM;
    float e = W[P::EB + j];
    e = fmaf(we[0], o0, e); e = fmaf(we[1], o1, e); e = fmaf(we[2], o2, e);
    e = fmaf(we[3], o3, e); e = fmaf(we[4], o4, e); e = fmaf(we[5], o5, e);
    e = fmaxf(e, 0.f);
#pragma unroll
    for (int a = 0; a < NA + V2; a++) z[a] = fmaf(W[P::row(a) + j], e, z[a]);
  }
}

// one valid neighbour row: returns the attention score t_r, hr[a] = W[a][H:] . m_r (phase 2 chains)
template <int NA, int KIND>
__device__ __forceinline__ float nbr_row(const float* W, const float* f, float (&hr)[NA + V2]) {
  using P = PV<NA, KIND>;
  // an offset the compiler cannot see through: without it the ~1200 shared-memory weight loads are
  // hoisted out of the caller's row loop as loop invariants and spilled to local memory
  int off = 0;
  asm volatile("" : "+r"(off));
  W += off;
  const float f0 = f[0], f1 = f[1], f2 = f[2], f3 = f[3], f4 = f[4], f5 = f[5];
  float t = W[P::AB];
#pragma unroll
  for (int a = 0; a < NA + V2; a++) hr[a] = 0.f;
#pragma unroll
  for (int j = 0; j < H; j++) {
    const float* wn = W + P::NW + j * GSM_NBR_FEAT_DIM;
    float m = W[P::NB + j];
    m = fmaf(wn[0], f0, m); m = fmaf(wn[1], f1, m); m = fmaf(wn[2], f2, m);
    m = fmaf(wn[3], f3, m); m = fmaf(wn[4], f4, m); m = fmaf(wn[5], f5, m);
    m = fmaxf(m, 0.f);
    t = fmaf(W[P::AW + j], m, t);
#pragma unroll
    for (int a = 0; a < NA + V2; a++) hr[a] = fmaf(W[P::row(a) + H + j], m, hr[a]);
  }
  return t;
}

// The forward of one row in graph_actor_kernel's order.  Out: z = [logits; values]; mx, s: the
// softmax max and sum over the valid rows; acc[a] * (1 / s) = sum_r a_r hr_r[a] (cnt > 0).
template <int NA, int KIND>
__device__ __forceinline__ void row_forward(const float* W, const float* o, const float* f, int cnt,
                                            float (&z)[NA + V2], float (&acc)[NA + V2], float& mx, float& s) {
  ego_logits<NA, KIND>(W, o, z);
  mx = -__int_as_float(0x7f800000); s = 0.f;
#pragma unroll
  for (int a = 0; a < NA + V2; a++) acc[a] = 0.f;
  for (int r = 0; r < cnt; r++) {
    float hr[NA + V2];
    const float t = nbr_row<NA, KIND>(W, f + r * GSM_NBR_FEAT_DIM, hr);
    const float nm = fmaxf(mx, t);
    const float sc = expf(mx - nm), pw = expf(t - nm);     // first row: exp(-inf) = 0
    s = fmaf(s, sc, pw);
#pragma unroll
    for (int a = 0; a < NA + V2; a++) acc[a] = fmaf(acc[a], sc, pw * hr[a]);
    mx = nm;
  }
  if (cnt > 0) {
    const float inv = 1.f / s;
#pragma unroll
    for (int a = 0; a < NA + V2; a++) z[a] = fmaf(acc[a], inv, z[a]);
  }
}

// logp of action `act` exactly as graph_actor_kernel computes it (NaN for act outside [0, NA));
// zm, se: max and sum of exp(z - zm) over the logits.
template <int NA>
__device__ __forceinline__ float row_logp(const float (&z)[NA + V2], int act, float& zm, float& se) {
  zm = z[0];
#pragma unroll
  for (int a = 1; a < NA; a++) zm = fmaxf(zm, z[a]);
  se = 0.f;
#pragma unroll
  for (int a = 0; a < NA; a++) se += expf(z[a] - zm);
  float za = __int_as_float(0x7fc00000);
#pragma unroll
  for (int a = 0; a < NA; a++) if (act == a) za = z[a];
  return za - zm - logf(se);
}

__device__ __forceinline__ int clamp_cnt(int c, int K) { return c < 0 ? 0 : (c > K ? K : c); }

template <int NA, int KIND>
__global__ void __launch_bounds__(128) policy_eval_kernel(const __grid_constant__ EvalArgs<KIND> p) {
  using P = PV<NA, KIND>;
  constexpr int NP = P::N;
  __shared__ float s_w[NP];
  for (int k = threadIdx.x; k < NP; k += blockDim.x) s_w[k] = p.params[k];
  __syncthreads();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.n_rows) return;
  const int64_t src = p.rows ? p.rows[i] : i;
  const int cnt = clamp_cnt(p.nbr_cnt[src], p.K);
  float z[NA + V2], acc[NA + V2], mx, s;
  row_forward<NA, KIND>(s_w, p.obs + src * GSM_OBS_DIM, p.nbr_feat + src * p.K * GSM_NBR_FEAT_DIM, cnt, z, acc, mx, s);
  if (p.values) {
#pragma unroll
    for (int v = 0; v < V2; v++) p.values[i * V2 + v] = z[NA + v];
  }
  if constexpr (KIND == HEAD_GAUSS) {
    const float ls0 = s_w[P::LS], ls1 = s_w[P::LS + 1];
    float d0, d1;
    const float lp = gauss_logp(p.actions[src * GD], p.actions[src * GD + 1], z[0], z[1], ls0, ls1, d0, d1);
    if (p.logp) p.logp[i] = lp;
    if (p.entropy) p.entropy[i] = gauss_entropy(ls0, ls1);
  } else {
    float zm, se;
    const float lp = row_logp<NA>(z, p.actions[src], zm, se);
    if (p.logp) p.logp[i] = lp;
    if (p.entropy) {                     // log(se) - sum_k p_k (z_k - zm) = logsumexp(z) - sum_k p_k z_k
      const float inv = 1.f / se;
      float pz = 0.f;
#pragma unroll
      for (int a = 0; a < NA; a++) pz = fmaf(expf(z[a] - zm) * inv, z[a] - zm, pz);
      p.entropy[i] = logf(se) - pz;
    }
  }
}

template <int NA, int KIND> struct BwdSmem {
  float w[PV<NA, KIND>::N];
  float obs[BWD_AG][GSM_OBS_DIM];
  float dz[BWD_AG][NA + V2];
  float dsum[BWD_AG];                  // sum_r ds_r of the row (db_a)
  int cnt[BWD_AG];
  long long src[BWD_AG];
};
// the Gaussian adds each row's two dlog_std terms (summed by threads NZ, NZ + 1 in phase B); the
// categorical layout stays as it is
template <int NA> struct BwdSmemGauss : BwdSmem<NA, HEAD_GAUSS> {
  float dls[BWD_AG][GD];
};
template <int NA, int KIND>
using BwdSmemOf = std::conditional_t<KIND == HEAD_GAUSS, BwdSmemGauss<NA>, BwdSmem<NA, KIND>>;

// ---- fused PPO loss (SPEC.md §14): the loss seeds computed in phase A from the row's own logp, entropy
// and values, per-row statistics parked in shared memory and summed per block in row order ----------
constexpr int PPO_ROW_STATS = 7;      // L_pi, L_V reward, L_V cost, entropy, rho, clipped, approx KL
constexpr int PPO_WS_STATS = 8;       // workspace floats per block behind its gradient partial

template <int KIND> struct PpoArgs : EvalArgs<KIND> {
  const float* old_logp; const float* old_values; const float* returns; const float* adv;   // source rows
  const float* adv_moments; const float* lagrange;                                          // device scalars
  float clip, value_clip, value_coef, entropy_coef, inv_n;
};
template <class Base> struct PpoSmem : Base {
  float st[BWD_AG][PPO_ROW_STATS];     // the tile's per-row statistics
  float stacc[PPO_ROW_STATS];          // the block's sums over its tiles (thread k owns entry k)
};

// SPEC.md §14 for one row: the seeds d_logp, d_entropy, d_values of the §12 chain and the row's statistics.
// A comparison with a NaN operand is false, so a NaN log-prob (an action outside the head's range)
// reaches d_logp and poisons the gradient, as in gsm_policy_backward.
template <int KIND>
__device__ __forceinline__ void ppo_seeds(const PpoArgs<KIND>& p, int64_t src, float lp, float ent, const float* v,
                                          float& dlp, float& dent, float (&dv)[V2], float* st) {
  const float* mom = p.adv_moments;
  const float a0 = (p.adv[src * V2] - mom[0]) / (mom[1] + 1e-5f);
  const float a1 = (p.adv[src * V2 + 1] - mom[2]) / (mom[3] + 1e-5f);
  const float A = a0 - p.lagrange[0] * a1;
  const float olp = p.old_logp[src];
  const float rho = expf(lp - olp);
  const float s1 = rho * A, s2 = fminf(fmaxf(rho, 1.f - p.clip), 1.f + p.clip) * A;
  dlp = s2 < s1 ? 0.f : -s1 * p.inv_n;
  st[0] = -(s2 < s1 ? s2 : s1);
#pragma unroll
  for (int h = 0; h < V2; h++) {
    const float ov = p.old_values[src * V2 + h], R = p.returns[src * V2 + h];
    const float dov = v[h] - ov;
    const float vc = ov + fminf(fmaxf(dov, -p.value_clip), p.value_clip);
    const float e1 = v[h] - R, e2 = vc - R, q1 = e1 * e1, q2 = e2 * e2;
    // the clipped branch carries the gradient where the clip is not active (vc = v up to rounding)
    const bool inside = fabsf(dov) <= p.value_clip;
    dv[h] = q1 < q2 ? (inside ? p.value_coef * e2 * p.inv_n : 0.f) : p.value_coef * e1 * p.inv_n;
    st[1 + h] = 0.5f * (q1 < q2 ? q2 : q1);
  }
  dent = -p.entropy_coef * p.inv_n;
  st[3] = ent; st[4] = rho; st[5] = fabsf(rho - 1.f) > p.clip ? 1.f : 0.f; st[6] = olp - lp;
}

#define GSM_BWD_KERNEL policy_backward_kernel
#define GSM_BWD_ARGS EvalArgs
#define GSM_BWD_LOSS false
#include "gsm_policy_backward.inl"
#undef GSM_BWD_KERNEL
#undef GSM_BWD_ARGS
#undef GSM_BWD_LOSS
#define GSM_BWD_KERNEL ppo_backward_kernel
#define GSM_BWD_ARGS PpoArgs
#define GSM_BWD_LOSS true
#include "gsm_policy_backward.inl"
#undef GSM_BWD_KERNEL
#undef GSM_BWD_ARGS
#undef GSM_BWD_LOSS

// grad[k] = sum of the G partials in a fixed order: warp w sums partials w, w + 8, ... (lane = k),
// then warp 0 adds the 8 warp sums in order.
__global__ void __launch_bounds__(256) policy_grad_reduce_kernel(const float* __restrict__ ws, int G, int NP,
                                                                 float* __restrict__ grad) {
  __shared__ float s[8][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int k = blockIdx.x * 32 + lane;
  float acc = 0.f;
  if (k < NP) {
#pragma unroll 4
    for (int g = w; g < G; g += 8) acc += ws[(int64_t)g * NP + k];
  }
  s[w][lane] = acc;
  __syncthreads();
  if (w == 0 && k < NP) {
    float t = s[0][lane];
#pragma unroll
    for (int q = 1; q < 8; q++) t += s[q][lane];
    grad[k] = t;
  }
}

// ppo_backward_kernel's partials: blocks 0 .. ceil(NP / 32) - 1 reduce the gradient exactly as
// policy_grad_reduce_kernel does (partials of stride NP + PPO_WS_STATS); the last block reduces the
// statistics in the same order, then lanes 0..6 write their means over the n rows and lane 0 adds
// L = L_pi + c_v (L_V reward + L_V cost) - c_e entropy.  Counts (the clip fraction) are exact in fp32
// below 2^24 rows.
__global__ void __launch_bounds__(256) ppo_reduce_kernel(const float* __restrict__ ws, int G, int NP,
                                                         float* __restrict__ grad, float* __restrict__ stats,
                                                         float n, float value_coef, float entropy_coef) {
  __shared__ float s[8][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int ngrad = (NP + 31) / 32;
  const bool is_stats = (int)blockIdx.x == ngrad;
  const int k = is_stats ? NP + lane : blockIdx.x * 32 + lane;
  const bool live = is_stats ? lane < PPO_ROW_STATS : k < NP;
  const int64_t stride = NP + PPO_WS_STATS;
  float acc = 0.f;
  if (live) {
#pragma unroll 4
    for (int g = w; g < G; g += 8) acc += ws[(int64_t)g * stride + k];
  }
  s[w][lane] = acc;
  __syncthreads();
  if (w != 0) return;
  float t = s[0][lane];
#pragma unroll
  for (int q = 1; q < 8; q++) t += s[q][lane];
  if (!is_stats) {
    if (live) grad[k] = t;
    return;
  }
  const float mean = t / n;
  const float lpi = __shfl_sync(~0u, mean, 0), lv0 = __shfl_sync(~0u, mean, 1), lv1 = __shfl_sync(~0u, mean, 2),
              ent = __shfl_sync(~0u, mean, 3);
  if (live) stats[lane] = mean;
  if (lane == 0) stats[PPO_ROW_STATS] = lpi + value_coef * (lv0 + lv1) - entropy_coef * ent;
}

// ---- Adam step (SPEC.md §14): torch.nn.utils.clip_grad_norm_ then torch.optim.Adam (no weight decay,
// no amsgrad) over the whole parameter vector in ONE block: the norm as a fixed-order fp64 sum (thread
// partials in index order, a shuffle tree, the warp sums in order), the clip, the update.  A non-finite
// norm skips the step (p, m, v and the step counter unchanged); the norm is written either way.
struct AdamArgs {
  float* params; const float* grad; float* m; float* v; int32_t* step; float* grad_norm;
  int64_t n;
  float lr, beta1, beta2, eps, max_norm;
};
constexpr int ADAM_THREADS = 1024;

__global__ void __launch_bounds__(ADAM_THREADS) adam_step_kernel(const __grid_constant__ AdamArgs a) {
  __shared__ double s_part[ADAM_THREADS / 32];
  __shared__ float s_norm;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double ss = 0.0;
  for (int64_t k = tid; k < a.n; k += ADAM_THREADS) { const double g = a.grad[k]; ss = fma(g, g, ss); }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) ss += __shfl_xor_sync(~0u, ss, d);
  if (lane == 0) s_part[warp] = ss;
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int q = 0; q < ADAM_THREADS / 32; q++) t += s_part[q];
    const float norm = (float)sqrt(t);
    s_norm = norm;
    *a.grad_norm = norm;
  }
  __syncthreads();
  const float norm = s_norm;
  if (!isfinite(norm)) return;                       // block-uniform
  const float coef = fminf(a.max_norm / (norm + 1e-6f), 1.f);
  const int32_t t = *a.step + 1;
  const double bc1 = 1.0 - pow((double)a.beta1, (double)t), bc2 = 1.0 - pow((double)a.beta2, (double)t);
  const float step_size = (float)((double)a.lr / bc1), bc2_sqrt = (float)sqrt(bc2);
  const float b1 = a.beta1, b2 = a.beta2;
  for (int64_t k = tid; k < a.n; k += ADAM_THREADS) {
    const float g = a.grad[k] * coef;
    const float m = b1 * a.m[k] + (1.f - b1) * g;
    const float v = b2 * a.v[k] + (1.f - b2) * (g * g);
    a.m[k] = m;
    a.v[k] = v;
    a.params[k] -= step_size * (m / (sqrtf(v) / bc2_sqrt + a.eps));
  }
  __syncthreads();                                   // every thread has read *step
  if (tid == 0) *a.step = t;
}

static int64_t bwd_blocks(int64_t n_rows) {
  const int64_t tiles = (n_rows + BWD_AG - 1) / BWD_AG;
  return tiles < BWD_MAX_BLOCKS ? tiles : BWD_MAX_BLOCKS;
}

static int n_params(int n_actions) { return n_actions == 5 ? PV<5, HEAD_CAT>::N : PV<9, HEAD_CAT>::N; }

static int launch_evaluate(const EvalArgs<HEAD_CAT>& a, int n_actions, cudaStream_t st) {
  const unsigned grid = (unsigned)((a.n_rows + 127) / 128);
  if (n_actions == 5) policy_eval_kernel<5, HEAD_CAT><<<grid, 128, 0, st>>>(a);
  else policy_eval_kernel<9, HEAD_CAT><<<grid, 128, 0, st>>>(a);
  return (int)cudaGetLastError();
}

static int launch_evaluate_gauss(const EvalArgs<HEAD_GAUSS>& a, cudaStream_t st) {
  policy_eval_kernel<GD, HEAD_GAUSS><<<(unsigned)((a.n_rows + 127) / 128), 128, 0, st>>>(a);
  return (int)cudaGetLastError();
}

template <int NA, int KIND>
static int launch_backward_na(EvalArgs<KIND> a, float* grad, cudaStream_t st) {
  const int64_t G = bwd_blocks(a.n_rows);
  a.n_tiles = (a.n_rows + BWD_AG - 1) / BWD_AG;
  const size_t dyn = 2 * sizeof(float) * BWD_AG * (size_t)a.K;
  if (sizeof(BwdSmemOf<NA, KIND>) + dyn > 48 * 1024) {      // large max_nbrs: opt in to more shared memory
    const cudaError_t e = cudaFuncSetAttribute(policy_backward_kernel<NA, KIND>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) {            // max_nbrs beyond the block's shared memory: report it here and clear
      cudaGetLastError();              // it, or the next launch's cudaGetLastError() would report it again
      return (int)e;
    }
  }
  policy_backward_kernel<NA, KIND><<<(unsigned)G, BWD_AG, dyn, st>>>(a);
  policy_grad_reduce_kernel<<<(PV<NA, KIND>::N + 31) / 32, 256, 0, st>>>(a.ws, (int)G, PV<NA, KIND>::N, grad);
  return (int)cudaGetLastError();
}

template <int NA, int KIND>
static int launch_ppo_na(PpoArgs<KIND> a, float* grad, float* stats, cudaStream_t st) {
  const int64_t G = bwd_blocks(a.n_rows);
  a.n_tiles = (a.n_rows + BWD_AG - 1) / BWD_AG;
  a.inv_n = 1.f / (float)a.n_rows;
  const size_t dyn = 2 * sizeof(float) * BWD_AG * (size_t)a.K;
  if (sizeof(PpoSmem<BwdSmemOf<NA, KIND>>) + dyn > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(ppo_backward_kernel<NA, KIND>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) { cudaGetLastError(); return (int)e; }
  }
  ppo_backward_kernel<NA, KIND><<<(unsigned)G, BWD_AG, dyn, st>>>(a);
  constexpr int NP = PV<NA, KIND>::N;
  ppo_reduce_kernel<<<(NP + 31) / 32 + 1, 256, 0, st>>>(a.ws, (int)G, NP, grad, stats, (float)a.n_rows,
                                                         a.value_coef, a.entropy_coef);
  return (int)cudaGetLastError();
}

static int launch_actor(const PolicyParams& w, const PolicyIO& io, int n_actions, cudaStream_t st) {
  if (io.n_rows == 0) return 0;
  const int block = 128;            // = AG, the agents a block owns
  const int64_t grid = (io.n_rows + block - 1) / block;
  constexpr int V = GSM_POLICY_VALUE_HEADS;
  const unsigned gd = (unsigned)grid;
  if (n_actions == 5 && !io.values) graph_actor_kernel<5, 0, HEAD_CAT><<<gd, block, 0, st>>>(w, io);
  else if (n_actions == 5) graph_actor_kernel<5, V, HEAD_CAT><<<gd, block, 0, st>>>(w, io);
  else if (n_actions == 9 && !io.values) graph_actor_kernel<9, 0, HEAD_CAT><<<gd, block, 0, st>>>(w, io);
  else if (n_actions == 9) graph_actor_kernel<9, V, HEAD_CAT><<<gd, block, 0, st>>>(w, io);
  else return -1;
  return (int)cudaGetLastError();
}

static int launch_actor_gauss(const GaussParams& w, const GaussIO& io, cudaStream_t st) {
  if (io.n_rows == 0) return 0;
  const unsigned gd = (unsigned)((io.n_rows + 127) / 128);
  if (!io.values) graph_actor_kernel<GD, 0, HEAD_GAUSS><<<gd, 128, 0, st>>>(w, io);
  else graph_actor_kernel<GD, GSM_POLICY_VALUE_HEADS, HEAD_GAUSS><<<gd, 128, 0, st>>>(w, io);
  return (int)cudaGetLastError();
}

}  // namespace gsm

// ---- C ABI ------------------------------------------------------------------------------------
namespace {
thread_local char g_policy_err[256] = "";
int pfail(int status, const char* msg) {
  std::strncpy(g_policy_err, msg, sizeof(g_policy_err) - 1);
  return status;
}
int pack(const gsm_policy_weights* w, gsm::PolicyParams* p) {
  if (!w) return pfail(GSM_ERR_INVALID_ARG, "gsm_policy: weights is NULL");
  if (w->struct_size != sizeof(gsm_policy_weights)) return pfail(GSM_ERR_ABI, "gsm_policy: weights.struct_size mismatch");
  if (w->n_actions != 5 && w->n_actions != 9)
    return pfail(GSM_ERR_UNSUPPORTED, "gsm_policy: compiled actor instances exist for n_actions 5 and 9 only");
  static_assert(sizeof(p->ego_w) == sizeof(w->ego_w), "layout");
  std::memcpy(p->ego_w, w->ego_w, sizeof(p->ego_w));   std::memcpy(p->ego_b, w->ego_b, sizeof(p->ego_b));
  std::memcpy(p->nbr_w, w->nbr_w, sizeof(p->nbr_w));   std::memcpy(p->nbr_b, w->nbr_b, sizeof(p->nbr_b));
  std::memcpy(p->att_w, w->att_w, sizeof(p->att_w));   p->att_b = w->att_b;
  std::memset(p->head_w, 0, sizeof(p->head_w)); std::memset(p->head_b, 0, sizeof(p->head_b));
  std::memcpy(p->head_w, w->head_w, sizeof(float) * 2 * GSM_POLICY_HIDDEN * w->n_actions);
  std::memcpy(p->head_b, w->head_b, sizeof(float) * w->n_actions);
  std::memcpy(p->head_w[w->n_actions], w->value_w, sizeof(w->value_w));   // critics right behind the logits' rows
  std::memcpy(&p->head_b[w->n_actions], w->value_b, sizeof(w->value_b));
  return GSM_OK;
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
// 0 <= device < device count, as gsm_create checks; GSM_OK or the error status to return.
int check_device(int device, const char* who) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return pfail(GSM_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  }
  if (device < 0 || device >= ndev) {
    static thread_local char msg[96];
    snprintf(msg, sizeof(msg), "%s: device index out of range", who);
    return pfail(GSM_ERR_INVALID_ARG, msg);
  }
  return GSM_OK;
}
int pfailf(int status, const char* who, const char* msg) {
  snprintf(g_policy_err, sizeof(g_policy_err), "%s: %s", who, msg);
  return status;
}
// The checks the evaluate and backward entry points of both heads share; none touches the device.
template <class IO> int check_eval_io_t(const IO* io, const char* who) {
  if (!io) return pfailf(GSM_ERR_INVALID_ARG, who, "io is NULL");
  if (io->struct_size != sizeof(IO)) return pfailf(GSM_ERR_ABI, who, "io.struct_size mismatch");
  if constexpr (std::is_same_v<IO, gsm_policy_eval_io>) {
    if (io->n_actions != 5 && io->n_actions != 9)
      return pfailf(GSM_ERR_UNSUPPORTED, who, "compiled learner instances exist for n_actions 5 and 9 only");
  } else {
    if (io->action_dim != GSM_POLICY_GAUSS_DIM)
      return pfailf(GSM_ERR_UNSUPPORTED, who, "the Gaussian learner instance has action_dim 2 only");
  }
  if (!io->params || !io->obs || !io->nbr_feat || !io->nbr_cnt || !io->actions)
    return pfailf(GSM_ERR_INVALID_ARG, who, "params, obs, nbr_feat, nbr_cnt and actions are required");
  if (io->n_rows < 0 || io->max_nbrs < 1) return pfailf(GSM_ERR_INVALID_ARG, who, "bad n_rows / max_nbrs");
  if (io->n_rows > ((int64_t)1 << 31) * 128 - 128) return pfailf(GSM_ERR_INVALID_ARG, who, "n_rows too large");
  return GSM_OK;
}
int check_eval_io(const gsm_policy_eval_io* io, const char* who) { return check_eval_io_t(io, who); }
template <int KIND, class IO> gsm::EvalArgs<KIND> eval_args(const IO* io) {
  gsm::EvalArgs<KIND> a{};
  a.params = io->params; a.obs = io->obs; a.nbr_feat = io->nbr_feat; a.nbr_cnt = io->nbr_cnt;
  a.actions = io->actions; a.rows = io->rows;
  a.n_rows = io->n_rows; a.K = io->max_nbrs;
  return a;
}
int pack_gauss(const gsm_policy_gauss_weights* w, gsm::GaussParams* p) {
  if (!w) return pfail(GSM_ERR_INVALID_ARG, "gsm_policy_gauss: weights is NULL");
  if (w->struct_size != sizeof(gsm_policy_gauss_weights))
    return pfail(GSM_ERR_ABI, "gsm_policy_gauss: weights.struct_size mismatch");
  static_assert(sizeof(p->ego_w) == sizeof(w->ego_w) && sizeof(p->log_std) == sizeof(w->log_std), "layout");
  std::memcpy(p->ego_w, w->ego_w, sizeof(p->ego_w));   std::memcpy(p->ego_b, w->ego_b, sizeof(p->ego_b));
  std::memcpy(p->nbr_w, w->nbr_w, sizeof(p->nbr_w));   std::memcpy(p->nbr_b, w->nbr_b, sizeof(p->nbr_b));
  std::memcpy(p->att_w, w->att_w, sizeof(p->att_w));   p->att_b = w->att_b;
  std::memcpy(p->head_w, w->mean_w, sizeof(w->mean_w));                        // means, then the critics
  std::memcpy(p->head_w[GSM_POLICY_GAUSS_DIM], w->value_w, sizeof(w->value_w));
  std::memcpy(p->head_b, w->mean_b, sizeof(w->mean_b));
  std::memcpy(&p->head_b[GSM_POLICY_GAUSS_DIM], w->value_b, sizeof(w->value_b));
  std::memcpy(p->log_std, w->log_std, sizeof(p->log_std));
  return GSM_OK;
}
int check_loss_io(const gsm_ppo_loss_io* l, const char* who) {
  if (!l) return pfailf(GSM_ERR_INVALID_ARG, who, "loss is NULL");
  if (l->struct_size != sizeof(gsm_ppo_loss_io)) return pfailf(GSM_ERR_ABI, who, "loss.struct_size mismatch");
  if (!l->old_logp || !l->old_values || !l->returns || !l->advantages || !l->adv_moments || !l->lagrange || !l->stats)
    return pfailf(GSM_ERR_INVALID_ARG, who,
                  "old_logp, old_values, returns, advantages, adv_moments, lagrange and stats are required");
  if (!(l->clip > 0.f) || !(l->value_clip > 0.f)) return pfailf(GSM_ERR_INVALID_ARG, who, "clip and value_clip must be > 0");
  if (!(l->value_coef >= 0.f) || !(l->entropy_coef >= 0.f))
    return pfailf(GSM_ERR_INVALID_ARG, who, "value_coef and entropy_coef must be >= 0");
  return GSM_OK;
}
template <int KIND> void set_loss(gsm::PpoArgs<KIND>& a, const gsm_ppo_loss_io* l) {
  a.old_logp = l->old_logp; a.old_values = l->old_values; a.returns = l->returns; a.adv = l->advantages;
  a.adv_moments = l->adv_moments; a.lagrange = l->lagrange;
  a.clip = l->clip; a.value_clip = l->value_clip; a.value_coef = l->value_coef; a.entropy_coef = l->entropy_coef;
}
// the argument checks and the launch of both heads; need: the workspace bytes for io->n_rows
template <int KIND, class IO, class Launch>
int ppo_backward_t(const IO* io, const gsm_ppo_loss_io* loss, float* grad, void* workspace, size_t workspace_bytes,
                   int device, void* stream, const char* who, int64_t (*need_fn)(const IO*), Launch launch) {
  if (const int st = check_eval_io_t(io, who)) return st;
  if (const int st = check_loss_io(loss, who)) return st;
  if (!grad) return pfailf(GSM_ERR_INVALID_ARG, who, "grad is required");
  const int64_t need = need_fn(io);
  if (need > 0 && (!workspace || workspace_bytes < (size_t)need))
    return pfailf(GSM_ERR_INVALID_ARG, who, "workspace smaller than the ppo backward workspace for n_rows");
  if (io->n_rows == 0) return GSM_OK;
  if (const int ds = check_device(device, who)) return ds;
  DevGuard guard(device);
  if (!guard.ok) return pfailf(GSM_ERR_CUDA, who, "cudaSetDevice failed");
  gsm::PpoArgs<KIND> a{};
  static_cast<gsm::EvalArgs<KIND>&>(a) = eval_args<KIND>(io);
  set_loss(a, loss);
  a.ws = (float*)workspace;
  const int e = launch(a, grad, loss->stats, (cudaStream_t)stream);
  if (e) return pfail(GSM_ERR_CUDA, cudaGetErrorString((cudaError_t)e));
  return GSM_OK;
}
}  // namespace

extern "C" {

int gsm_policy_evaluate(const gsm_policy_eval_io* io, int device, void* stream) {
  if (const int st = check_eval_io(io, "gsm_policy_evaluate")) return st;
  if (io->n_rows == 0) return GSM_OK;
  if (const int ds = check_device(device, "gsm_policy_evaluate")) return ds;
  DevGuard guard(device);
  if (!guard.ok) return pfail(GSM_ERR_CUDA, "gsm_policy_evaluate: cudaSetDevice failed");
  gsm::EvalArgs<gsm::HEAD_CAT> a = eval_args<gsm::HEAD_CAT>(io);
  a.logp = io->logp; a.entropy = io->entropy; a.values = io->values;
  const int e = gsm::launch_evaluate(a, io->n_actions, (cudaStream_t)stream);
  if (e) return pfail(GSM_ERR_CUDA, cudaGetErrorString((cudaError_t)e));
  return GSM_OK;
}

int64_t gsm_policy_backward_workspace(int64_t n_rows, int32_t n_actions) {
  if (n_actions != 5 && n_actions != 9)
    return pfailf(GSM_ERR_UNSUPPORTED, "gsm_policy_backward_workspace", "n_actions must be 5 or 9");
  if (n_rows < 0) return pfailf(GSM_ERR_INVALID_ARG, "gsm_policy_backward_workspace", "n_rows < 0");
  return gsm::bwd_blocks(n_rows) * gsm::n_params(n_actions) * (int64_t)sizeof(float);
}

int gsm_policy_backward(const gsm_policy_eval_io* io, const float* d_logp, const float* d_entropy,
                        const float* d_values, float* grad, void* workspace, size_t workspace_bytes,
                        int device, void* stream) {
  const char* who = "gsm_policy_backward";
  if (const int st = check_eval_io(io, who)) return st;
  if (!grad) return pfailf(GSM_ERR_INVALID_ARG, who, "grad is required");
  const int64_t need = gsm_policy_backward_workspace(io->n_rows, io->n_actions);
  if (need > 0 && (!workspace || workspace_bytes < (size_t)need))
    return pfailf(GSM_ERR_INVALID_ARG, who, "workspace smaller than gsm_policy_backward_workspace(n_rows, n_actions)");
  if (io->n_rows == 0) return GSM_OK;
  if (const int ds = check_device(device, who)) return ds;
  DevGuard guard(device);
  if (!guard.ok) return pfail(GSM_ERR_CUDA, "gsm_policy_backward: cudaSetDevice failed");
  gsm::EvalArgs<gsm::HEAD_CAT> a = eval_args<gsm::HEAD_CAT>(io);
  a.d_logp = d_logp; a.d_entropy = d_entropy; a.d_values = d_values;
  a.ws = (float*)workspace;
  const int e = io->n_actions == 5 ? gsm::launch_backward_na<5, gsm::HEAD_CAT>(a, grad, (cudaStream_t)stream)
                                   : gsm::launch_backward_na<9, gsm::HEAD_CAT>(a, grad, (cudaStream_t)stream);
  if (e) return pfail(GSM_ERR_CUDA, cudaGetErrorString((cudaError_t)e));
  return GSM_OK;
}

const char* gsm_policy_last_error(void) { return g_policy_err; }

int gsm_policy_act(const gsm_policy_weights* w, const gsm_policy_io* io, int device, void* stream) {
  gsm::PolicyParams p;
  int st = pack(w, &p);
  if (st) return st;
  if (!io || !io->obs || !io->nbr_feat || !io->nbr_cnt || !io->actions)
    return pfail(GSM_ERR_INVALID_ARG, "gsm_policy_act: obs, nbr_feat, nbr_cnt and actions are required");
  if (io->n_rows < 0 || io->max_nbrs < 1) return pfail(GSM_ERR_INVALID_ARG, "gsm_policy_act: bad n_rows / max_nbrs");
  if (io->n_rows > ((int64_t)1 << 31) * 128 - 128) return pfail(GSM_ERR_INVALID_ARG, "gsm_policy_act: n_rows too large");
  if (const int ds = check_device(device, "gsm_policy_act")) return ds;
  DevGuard guard(device);
  if (!guard.ok) return pfail(GSM_ERR_CUDA, "gsm_policy_act: cudaSetDevice failed");
  gsm::PolicyIO k;
  k.obs = io->obs; k.nbr_feat = io->nbr_feat; k.nbr_cnt = io->nbr_cnt;
  k.actions = io->actions; k.logp = io->logp; k.dist = io->logits; k.values = io->values;
  k.n_rows = io->n_rows; k.row_offset = io->row_offset; k.seed = io->seed; k.step = io->step;
  k.K = io->max_nbrs; k.greedy = io->greedy;
  const int e = gsm::launch_actor(p, k, w->n_actions, (cudaStream_t)stream);
  if (e) return pfail(GSM_ERR_CUDA, cudaGetErrorString((cudaError_t)e));
  return GSM_OK;
}

int gsm_policy_act_gauss(const gsm_policy_gauss_weights* w, const gsm_policy_gauss_io* io, int device,
                         void* stream) {
  gsm::GaussParams p;
  int st = pack_gauss(w, &p);
  if (st) return st;
  if (!io || !io->obs || !io->nbr_feat || !io->nbr_cnt || !io->actions)
    return pfail(GSM_ERR_INVALID_ARG, "gsm_policy_act_gauss: obs, nbr_feat, nbr_cnt and actions are required");
  if (io->n_rows < 0 || io->max_nbrs < 1) return pfail(GSM_ERR_INVALID_ARG, "gsm_policy_act_gauss: bad n_rows / max_nbrs");
  if (io->n_rows > ((int64_t)1 << 31) * 128 - 128) return pfail(GSM_ERR_INVALID_ARG, "gsm_policy_act_gauss: n_rows too large");
  if (const int ds = check_device(device, "gsm_policy_act_gauss")) return ds;
  DevGuard guard(device);
  if (!guard.ok) return pfail(GSM_ERR_CUDA, "gsm_policy_act_gauss: cudaSetDevice failed");
  gsm::GaussIO k;
  k.obs = io->obs; k.nbr_feat = io->nbr_feat; k.nbr_cnt = io->nbr_cnt;
  k.actions = io->actions; k.logp = io->logp; k.dist = io->mean; k.values = io->values;
  k.n_rows = io->n_rows; k.row_offset = io->row_offset; k.seed = io->seed; k.step = io->step;
  k.K = io->max_nbrs; k.greedy = io->greedy;
  const int e = gsm::launch_actor_gauss(p, k, (cudaStream_t)stream);
  if (e) return pfail(GSM_ERR_CUDA, cudaGetErrorString((cudaError_t)e));
  return GSM_OK;
}

int gsm_policy_evaluate_gauss(const gsm_policy_gauss_eval_io* io, int device, void* stream) {
  const char* who = "gsm_policy_evaluate_gauss";
  if (const int st = check_eval_io_t(io, who)) return st;
  if (io->n_rows == 0) return GSM_OK;
  if (const int ds = check_device(device, who)) return ds;
  DevGuard guard(device);
  if (!guard.ok) return pfail(GSM_ERR_CUDA, "gsm_policy_evaluate_gauss: cudaSetDevice failed");
  gsm::EvalArgs<gsm::HEAD_GAUSS> a = eval_args<gsm::HEAD_GAUSS>(io);
  a.logp = io->logp; a.entropy = io->entropy; a.values = io->values;
  const int e = gsm::launch_evaluate_gauss(a, (cudaStream_t)stream);
  if (e) return pfail(GSM_ERR_CUDA, cudaGetErrorString((cudaError_t)e));
  return GSM_OK;
}

int64_t gsm_policy_backward_workspace_gauss(int64_t n_rows) {
  if (n_rows < 0) return pfailf(GSM_ERR_INVALID_ARG, "gsm_policy_backward_workspace_gauss", "n_rows < 0");
  return gsm::bwd_blocks(n_rows) * GSM_POLICY_GAUSS_N_PARAMS * (int64_t)sizeof(float);
}

int gsm_policy_backward_gauss(const gsm_policy_gauss_eval_io* io, const float* d_logp, const float* d_entropy,
                              const float* d_values, float* grad, void* workspace, size_t workspace_bytes,
                              int device, void* stream) {
  const char* who = "gsm_policy_backward_gauss";
  if (const int st = check_eval_io_t(io, who)) return st;
  if (!grad) return pfailf(GSM_ERR_INVALID_ARG, who, "grad is required");
  const int64_t need = gsm_policy_backward_workspace_gauss(io->n_rows);
  if (need > 0 && (!workspace || workspace_bytes < (size_t)need))
    return pfailf(GSM_ERR_INVALID_ARG, who, "workspace smaller than gsm_policy_backward_workspace_gauss(n_rows)");
  if (io->n_rows == 0) return GSM_OK;
  if (const int ds = check_device(device, who)) return ds;
  DevGuard guard(device);
  if (!guard.ok) return pfail(GSM_ERR_CUDA, "gsm_policy_backward_gauss: cudaSetDevice failed");
  gsm::EvalArgs<gsm::HEAD_GAUSS> a = eval_args<gsm::HEAD_GAUSS>(io);
  a.d_logp = d_logp; a.d_entropy = d_entropy; a.d_values = d_values;
  a.ws = (float*)workspace;
  const int e = gsm::launch_backward_na<gsm::GD, gsm::HEAD_GAUSS>(a, grad, (cudaStream_t)stream);
  if (e) return pfail(GSM_ERR_CUDA, cudaGetErrorString((cudaError_t)e));
  return GSM_OK;
}

int64_t gsm_ppo_backward_workspace(int64_t n_rows, int32_t n_actions) {
  if (n_actions != 5 && n_actions != 9)
    return pfailf(GSM_ERR_UNSUPPORTED, "gsm_ppo_backward_workspace", "n_actions must be 5 or 9");
  if (n_rows < 0) return pfailf(GSM_ERR_INVALID_ARG, "gsm_ppo_backward_workspace", "n_rows < 0");
  return gsm::bwd_blocks(n_rows) * (gsm::n_params(n_actions) + gsm::PPO_WS_STATS) * (int64_t)sizeof(float);
}

int64_t gsm_ppo_backward_workspace_gauss(int64_t n_rows) {
  if (n_rows < 0) return pfailf(GSM_ERR_INVALID_ARG, "gsm_ppo_backward_workspace_gauss", "n_rows < 0");
  return gsm::bwd_blocks(n_rows) * (GSM_POLICY_GAUSS_N_PARAMS + gsm::PPO_WS_STATS) * (int64_t)sizeof(float);
}

int gsm_ppo_backward(const gsm_policy_eval_io* io, const gsm_ppo_loss_io* loss, float* grad, void* workspace,
                     size_t workspace_bytes, int device, void* stream) {
  return ppo_backward_t<gsm::HEAD_CAT>(
      io, loss, grad, workspace, workspace_bytes, device, stream, "gsm_ppo_backward",
      +[](const gsm_policy_eval_io* q) { return gsm_ppo_backward_workspace(q->n_rows, q->n_actions); },
      [&](const gsm::PpoArgs<gsm::HEAD_CAT>& a, float* g, float* st, cudaStream_t s) {
        return io->n_actions == 5 ? gsm::launch_ppo_na<5, gsm::HEAD_CAT>(a, g, st, s)
                                  : gsm::launch_ppo_na<9, gsm::HEAD_CAT>(a, g, st, s);
      });
}

int gsm_ppo_backward_gauss(const gsm_policy_gauss_eval_io* io, const gsm_ppo_loss_io* loss, float* grad,
                           void* workspace, size_t workspace_bytes, int device, void* stream) {
  return ppo_backward_t<gsm::HEAD_GAUSS>(
      io, loss, grad, workspace, workspace_bytes, device, stream, "gsm_ppo_backward_gauss",
      +[](const gsm_policy_gauss_eval_io* q) { return gsm_ppo_backward_workspace_gauss(q->n_rows); },
      [](const gsm::PpoArgs<gsm::HEAD_GAUSS>& a, float* g, float* st, cudaStream_t s) {
        return gsm::launch_ppo_na<gsm::GD, gsm::HEAD_GAUSS>(a, g, st, s);
      });
}

int gsm_adam_step(float* params, const float* grad, float* m, float* v, int32_t* step, int64_t n, float lr,
                  float beta1, float beta2, float eps, float max_grad_norm, float* grad_norm, int device,
                  void* stream) {
  const char* who = "gsm_adam_step";
  if (!params || !grad || !m || !v || !step || !grad_norm)
    return pfailf(GSM_ERR_INVALID_ARG, who, "params, grad, m, v, step and grad_norm are required");
  if (n < 1) return pfailf(GSM_ERR_INVALID_ARG, who, "n < 1");
  if (!(beta1 >= 0.f && beta1 < 1.f) || !(beta2 >= 0.f && beta2 < 1.f))
    return pfailf(GSM_ERR_INVALID_ARG, who, "beta1 and beta2 must lie in [0, 1)");
  if (!(lr >= 0.f) || !(eps >= 0.f) || !(max_grad_norm > 0.f))
    return pfailf(GSM_ERR_INVALID_ARG, who, "lr and eps must be >= 0 and max_grad_norm > 0");
  if (const int ds = check_device(device, who)) return ds;
  DevGuard guard(device);
  if (!guard.ok) return pfailf(GSM_ERR_CUDA, who, "cudaSetDevice failed");
  const gsm::AdamArgs a{params, grad, m, v, step, grad_norm, n, lr, beta1, beta2, eps, max_grad_norm};
  gsm::adam_step_kernel<<<1, gsm::ADAM_THREADS, 0, (cudaStream_t)stream>>>(a);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(GSM_ERR_CUDA, cudaGetErrorString(e));
  return GSM_OK;
}

int gsm_gae(const float* reward, const float* cost, const float* values, const uint8_t* done, int32_t n_steps,
            int64_t n_rows, int64_t slot_rows, float gamma, float lam, float* returns, float* advantages,
            int device, void* stream) {
  if (!reward || !cost || !values || !done || !returns)
    return pfail(GSM_ERR_INVALID_ARG, "gsm_gae: reward, cost, values, done and returns are required");
  if (n_steps < 1 || n_rows < 0 || slot_rows < n_rows) return pfail(GSM_ERR_INVALID_ARG, "gsm_gae: bad sizes");
  if (const int ds = check_device(device, "gsm_gae")) return ds;
  if (n_rows == 0) return GSM_OK;
  DevGuard guard(device);
  if (!guard.ok) return pfail(GSM_ERR_CUDA, "gsm_gae: cudaSetDevice failed");
  gsm::GaeParams p{reward, cost, values, done, returns, advantages, n_rows, slot_rows, n_steps, gamma, lam};
  const int64_t threads = n_rows * GSM_POLICY_VALUE_HEADS;
  gsm::gae_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(GSM_ERR_CUDA, cudaGetErrorString(e));
  return GSM_OK;
}

}  // extern "C"
