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

// The kernel-parameter image both heads share: the embedding and NH head rows.
template <int NH> struct EmbedParams {
  float ego_w[H][GSM_OBS_DIM];
  float ego_b[H];
  float nbr_w[H][GSM_NBR_FEAT_DIM];
  float nbr_b[H];
  float att_w[H];
  // rows 0..NA-1: the head (logits or means); rows NA, NA+1: the two critics (reward value, cost value)
  float head_w[NH][2 * H];
  float head_b[NH];
  float att_b;
};
// kernel-parameter image of gsm_policy_weights
using PolicyParams = EmbedParams<GSM_POLICY_MAX_ACTIONS + GSM_POLICY_VALUE_HEADS>;

// Head kinds (SPEC.md §10 / §10b).  The embedding h = [e; sum_r a_r m_r] and everything that computes
// it are shared; the kind selects the weights' image, the action type and the epilogue.
//   HEAD_CAT:   NA logits, categorical sample (Gumbel-max), int32 action.
//   HEAD_GAUSS: NA = GSM_POLICY_GAUSS_DIM means, diagonal Gaussian with a state-independent log_std,
//               float action [2] = mean + exp(log_std) eps (Box-Muller), no clamping.
enum HeadKind { HEAD_CAT = 0, HEAD_GAUSS = 1 };
constexpr int GD = GSM_POLICY_GAUSS_DIM;

// kernel-parameter image of gsm_policy_gauss_weights: log_std right behind the shared part
struct GaussParams : EmbedParams<GD + GSM_POLICY_VALUE_HEADS> {
  float log_std[GD];
};
static_assert(sizeof(GaussParams) == sizeof(EmbedParams<GD + GSM_POLICY_VALUE_HEADS>) + sizeof(float) * GD, "layout");

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

// a Philox word to (0, 1): 23 random bits + half a step, every value k * 2^-23 + 2^-24 is exact in fp32
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
          const float v = z[a] - logf(-logf(unit_open(r[q])));
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
// NORM (SPEC.md §15, gsm_gae_normalized): the critics' values are normalised; every V_h[t] is denormalised
// as fmaf(V, sigma_h, mu_h) with the [2][2] affine (mu_h, sigma_h) before the recursion.
struct GaeNormParams : GaeParams {
  const float* affine;
};
template <bool NORM> using GaeArgs = std::conditional_t<NORM, GaeNormParams, GaeParams>;
template <bool NORM>
__global__ void __launch_bounds__(256) gae_kernel(const __grid_constant__ GaeArgs<NORM> p) {
  constexpr int V = GSM_POLICY_VALUE_HEADS;
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= p.n_rows * V) return;
  const int64_t row = g / V;
  const int head = (int)(g - row * V);
  const float* rw = head == 0 ? p.reward : p.cost;
  float mu = 0.f, sd = 1.f;
  if constexpr (NORM) { mu = p.affine[2 * head]; sd = p.affine[2 * head + 1]; }
  float gae = 0.f;
  float v_next = p.values[((int64_t)p.T * p.slot_rows + row) * V + head];
  if constexpr (NORM) v_next = fmaf(v_next, sd, mu);
  for (int t = p.T - 1; t >= 0; t--) {
    const int64_t o = (int64_t)t * p.slot_rows + row;
    const float mask = p.done[o] ? 0.f : 1.f;      // done at step t: slot t+1 starts a new episode
    float v = p.values[o * V + head];
    if constexpr (NORM) v = fmaf(v, sd, mu);
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
// Backward (backward_kernel), with h = [e; g], g = sum_r a_r m_r, Z = [z; v], W = [W_h; W_v]:
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
// SPEC.md §15 (gsm_ppo_backward_normalized): the minibatch's value-normaliser affine [2][2] (mu_h, sigma_h)
template <int KIND> struct PpoNormArgs : PpoArgs<KIND> {
  const float* value_affine;
};
template <class Base> struct PpoSmem : Base {
  float st[BWD_AG][PPO_ROW_STATS];     // the tile's per-row statistics
  float stacc[PPO_ROW_STATS];          // the block's sums over its tiles (thread k owns entry k)
};

// backward_kernel's LOSS modes: the seeds are inputs (gsm_policy_backward); the §14 loss computes them
// (gsm_ppo_backward); the §14 loss on normalised value targets, R_h -> (R_h - mu_h) / sigma_h (§15,
// gsm_ppo_backward_normalized)
constexpr int LOSS_NONE = 0, LOSS_PPO = 1, LOSS_PPO_VNORM = 2;
template <int KIND, int LOSS>
using BwdArgs = std::conditional_t<LOSS == LOSS_NONE, EvalArgs<KIND>,
                                   std::conditional_t<LOSS == LOSS_PPO, PpoArgs<KIND>, PpoNormArgs<KIND>>>;

// SPEC.md §14 for one row: the seeds d_logp, d_entropy, d_values of the §12 chain and the row's statistics.
// A comparison with a NaN operand is false, so a NaN log-prob (an action outside the head's range)
// reaches d_logp and poisons the gradient, as in gsm_policy_backward.
template <int KIND, int LOSS>
__device__ __forceinline__ void ppo_seeds(const BwdArgs<KIND, LOSS>& p, int64_t src, float lp, float ent,
                                          const float* v, float& dlp, float& dent, float (&dv)[V2], float* st) {
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
    const float ov = p.old_values[src * V2 + h];
    float R = p.returns[src * V2 + h];
    if constexpr (LOSS == LOSS_PPO_VNORM) R = (R - p.value_affine[2 * h]) / p.value_affine[2 * h + 1];
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

// The backward kernel.  LOSS_NONE (gsm_policy_backward): the seeds d_logp, d_entropy, d_values are
// inputs.  LOSS_PPO (gsm_ppo_backward): phase A computes them from the PPO-Lagrangian loss (ppo_seeds,
// SPEC.md §14) and the block also sums the loss statistics; LOSS_PPO_VNORM normalises the value targets
// first.  The loss modes add code only under `if constexpr`, so the LOSS_NONE instances carry none of it.  (A __forceinline__ device function
// shared by two thin kernels would not do: the inliner changes the optimisation pipeline and the SASS of
// every instance.)
template <int NA, int KIND, int LOSS>
using BwdSmemT = std::conditional_t<LOSS != LOSS_NONE, PpoSmem<BwdSmemOf<NA, KIND>>, BwdSmemOf<NA, KIND>>;

// The normalised <9, CAT> instance names a minimum of one block per SM: left to its own occupancy target,
// ptxas caps it at 168 registers and spills one value.  A bound of 0 is no bound: every other instance
// compiles as it does without one (the bound on <5, CAT> and <2, GAUSS> would raise their registers and cost
// occupancy).
template <int NA, int KIND, int LOSS>
__global__ void __launch_bounds__(BWD_AG, LOSS == LOSS_PPO_VNORM && NA == 9 ? 1 : 0)
    backward_kernel(const __grid_constant__ BwdArgs<KIND, LOSS> p) {
  using P = PV<NA, KIND>;
  constexpr bool PPO = LOSS != LOSS_NONE;
  constexpr int NZ = NA + V2, NP = P::N, WS = NP + (PPO ? PPO_WS_STATS : 0);
  __shared__ BwdSmemT<NA, KIND, LOSS> sm;
  extern __shared__ float s_rows[];    // [BWD_AG][K][2]: (a_r, ds_r) of the valid rows; a float2 array
                                       // would round every kernel's static shared memory in this file up to 16 B
  const int tid = threadIdx.x;
  for (int k = tid; k < NP; k += BWD_AG) sm.w[k] = p.params[k];
  const float* W = sm.w;
  // phase-B accumulators of hidden unit j = tid, live across the tiles
  float gwe[GSM_OBS_DIM], gwn[GSM_NBR_FEAT_DIM], ghe[NZ], ghg[NZ];
  float gbe = 0.f, gbn = 0.f, gwa = 0.f, gsc = 0.f;   // gsc: bias sum of dZ[tid] (tid < NZ) or db_a (tid = H-1)
#pragma unroll
  for (int k = 0; k < GSM_OBS_DIM; k++) { gwe[k] = 0.f; gwn[k] = 0.f; }
#pragma unroll
  for (int a = 0; a < NZ; a++) { ghe[a] = 0.f; ghg[a] = 0.f; }
  if constexpr (PPO) { if (tid < PPO_ROW_STATS) sm.stacc[tid] = 0.f; }
  __syncthreads();

  for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {   // block-uniform
    const int64_t base = tile * BWD_AG;
    const int nag = p.n_rows - base < BWD_AG ? (int)(p.n_rows - base) : BWD_AG;
    // ---- phase A: thread = row ----
    if (tid < nag) {
      const int64_t i = base + tid;
      const int64_t src = p.rows ? p.rows[i] : i;
      const int cnt = clamp_cnt(p.nbr_cnt[src], p.K);
      const float* o = p.obs + src * GSM_OBS_DIM;
      const float* f = p.nbr_feat + src * p.K * GSM_NBR_FEAT_DIM;
      float z[NZ], acc[NZ], mx, s;
      row_forward<NA, KIND>(W, o, f, cnt, z, acc, mx, s);
      // The categorical dz stays at this scope for BOTH kinds, on purpose: guarded by
      // `if constexpr (KIND == HEAD_CAT)` (or nested in an if-constexpr / else) it changes the register
      // allocation and SASS of the categorical instances, which must stay as they were.  For the
      // Gaussian it is dead code: act is the constant 0, every dz[a < NA] it writes is rewritten by the
      // Gaussian block below and nothing else reads its values, so the compiler removes it (same
      // registers as the nested form).  Only dlp and dent are shared with the Gaussian block.
      float zm, se;
      const int act = KIND == HEAD_CAT ? (int)p.actions[src] : 0;
      const float lp = row_logp<NA>(z, act, zm, se);
      float dlp = 0.f, dent = 0.f, dvl[V2];
      if constexpr (!PPO) { dlp = p.d_logp ? p.d_logp[i] : 0.f; dent = p.d_entropy ? p.d_entropy[i] : 0.f; }
      const float lse = zm + logf(se), inv_se = 1.f / se;
      float pr[NA], ent = 0.f;
#pragma unroll
      for (int a = 0; a < NA; a++) { pr[a] = expf(z[a] - zm) * inv_se; ent = fmaf(pr[a], z[a] - zm, ent); }
      ent = logf(se) - ent;
      // the categorical loss: lp and ent are evaluate's (same row_logp, same entropy chain)
      if constexpr (PPO && KIND == HEAD_CAT) ppo_seeds<KIND, LOSS>(p, src, lp, ent, z + NA, dlp, dent, dvl, sm.st[tid]);
      // an action outside [0, NA) has no one-hot: its NaN logp poisons the gradient it feeds
      const float bad = (dlp != 0.f && lp != lp) ? __int_as_float(0x7fc00000) : 0.f;
      float dz[NZ];
#pragma unroll
      for (int a = 0; a < NA; a++)
        dz[a] = dlp * ((act == a ? 1.f : 0.f) - pr[a] + bad) - dent * pr[a] * ((z[a] - lse) + ent);
      if constexpr (KIND == HEAD_GAUSS) {
        // SPEC.md §12b: dmu_d = d_logp delta_d exp(-log_std_d);
        // dlog_std_d = d_logp (delta_d^2 - 1) + d_entropy.  A non-finite action (NaN logp) gives a NaN
        // gradient exactly where d_logp != 0; where d_logp == 0 the action does not enter it.
        const float ls0 = W[P::LS], ls1 = W[P::LS + 1];
        float d0, d1;
        const float glp = gauss_logp(p.actions[src * GD], p.actions[src * GD + 1], z[0], z[1], ls0, ls1, d0, d1);
        if constexpr (PPO) ppo_seeds<KIND, LOSS>(p, src, glp, gauss_entropy(ls0, ls1), z + NA, dlp, dent, dvl, sm.st[tid]);
        const bool use = dlp != 0.f;
        const float gbad = (use && glp != glp) ? __int_as_float(0x7fc00000) : 0.f;
        dz[0] = use ? dlp * d0 * expf(-ls0) + gbad : 0.f;
        dz[1] = use ? dlp * d1 * expf(-ls1) + gbad : 0.f;
        sm.dls[tid][0] = (use ? dlp * fmaf(d0, d0, -1.f) + gbad : 0.f) + dent;
        sm.dls[tid][1] = (use ? dlp * fmaf(d1, d1, -1.f) + gbad : 0.f) + dent;
      }
#pragma unroll
      for (int v = 0; v < V2; v++) {
        if constexpr (PPO) dz[NA + v] = dvl[v];
        else dz[NA + v] = p.d_values ? p.d_values[i * V2 + v] : 0.f;
      }
      float dsum = 0.f;
      if (cnt > 0) {
        const float inv = 1.f / s;
        float gdg = 0.f;                 // g . dg = dZ . sum_r a_r hr_r
#pragma unroll
        for (int a = 0; a < NZ; a++) gdg = fmaf(dz[a], acc[a] * inv, gdg);
        float* pr_rows = s_rows + 2 * tid * p.K;
        for (int r = 0; r < cnt; r++) {  // second pass: the same t_r, hr_r as the first
          float hr[NZ];
          const float t = nbr_row<NA, KIND>(W, f + r * GSM_NBR_FEAT_DIM, hr);
          const float ar = expf(t - mx) * inv;
          float q = 0.f;
#pragma unroll
          for (int a = 0; a < NZ; a++) q = fmaf(dz[a], hr[a], q);
          const float ds = ar * (q - gdg);
          pr_rows[2 * r] = ar; pr_rows[2 * r + 1] = ds;
          dsum += ds;
        }
      }
#pragma unroll
      for (int k = 0; k < GSM_OBS_DIM; k++) sm.obs[tid][k] = o[k];
#pragma unroll
      for (int a = 0; a < NZ; a++) sm.dz[tid][a] = dz[a];
      sm.dsum[tid] = dsum;
      sm.cnt[tid] = cnt;
      sm.src[tid] = src;
    }
    __syncthreads();
    // ---- phase B: thread = hidden unit j ----
    {
      const int j = tid;
      float we[GSM_OBS_DIM], wn[GSM_NBR_FEAT_DIM], wh[NZ], wg[NZ];
#pragma unroll
      for (int k = 0; k < GSM_OBS_DIM; k++) { we[k] = W[P::EW + j * GSM_OBS_DIM + k]; wn[k] = W[P::NW + j * GSM_NBR_FEAT_DIM + k]; }
#pragma unroll
      for (int a = 0; a < NZ; a++) { wh[a] = W[P::row(a) + j]; wg[a] = W[P::row(a) + H + j]; }
      const float be = W[P::EB + j], bn = W[P::NB + j], wa = W[P::AW + j];
      for (int ag = 0; ag < nag; ag++) {
        float dZ[NZ];
#pragma unroll
        for (int a = 0; a < NZ; a++) dZ[a] = sm.dz[ag][a];
        float u = be;
#pragma unroll
        for (int k = 0; k < GSM_OBS_DIM; k++) u = fmaf(we[k], sm.obs[ag][k], u);
        const float e = fmaxf(u, 0.f);
        float dh = 0.f;
#pragma unroll
        for (int a = 0; a < NZ; a++) { dh = fmaf(wh[a], dZ[a], dh); ghe[a] = fmaf(dZ[a], e, ghe[a]); }
        const float de = u > 0.f ? dh : 0.f;            // ReLU'(0) = 0, as in torch
#pragma unroll
        for (int k = 0; k < GSM_OBS_DIM; k++) gwe[k] = fmaf(de, sm.obs[ag][k], gwe[k]);
        gbe += de;
        const int c = sm.cnt[ag];                        // block-uniform: no divergence
        if (c > 0) {
          float dg = 0.f, g = 0.f;
#pragma unroll
          for (int a = 0; a < NZ; a++) dg = fmaf(wg[a], dZ[a], dg);
          const float* f = p.nbr_feat + sm.src[ag] * p.K * GSM_NBR_FEAT_DIM;
          const float* rr = s_rows + 2 * ag * p.K;
          for (int r = 0; r < c; r++) {
            float fr[GSM_NBR_FEAT_DIM];
#pragma unroll
            for (int k = 0; k < GSM_NBR_FEAT_DIM; k++) fr[k] = __ldg(f + r * GSM_NBR_FEAT_DIM + k);
            float um = bn;
#pragma unroll
            for (int k = 0; k < GSM_NBR_FEAT_DIM; k++) um = fmaf(wn[k], fr[k], um);
            const float m = fmaxf(um, 0.f);
            const float ar = rr[2 * r], ds = rr[2 * r + 1];
            g = fmaf(ar, m, g);
            const float du = um > 0.f ? fmaf(ar, dg, ds * wa) : 0.f;
#pragma unroll
            for (int k = 0; k < GSM_NBR_FEAT_DIM; k++) gwn[k] = fmaf(du, fr[k], gwn[k]);
            gbn += du;
            gwa = fmaf(ds, m, gwa);
          }
#pragma unroll
          for (int a = 0; a < NZ; a++) ghg[a] = fmaf(dZ[a], g, ghg[a]);
        }
        if (j < NZ) gsc += sm.dz[ag][j];
        else if (j == H - 1) gsc += sm.dsum[ag];
        else if constexpr (KIND == HEAD_GAUSS) { if (j < NZ + GD) gsc += sm.dls[ag][j - NZ]; }
      }
    }
    if constexpr (PPO) {                 // the tile's statistics, in row order
      if (tid < PPO_ROW_STATS) {
        float acc = sm.stacc[tid];
        for (int ag = 0; ag < nag; ag++) acc += sm.st[ag][tid];
        sm.stacc[tid] = acc;
      }
    }
    __syncthreads();                     // before the next tile overwrites the row state
  }
  // ---- this block's partial gradient, in vector order (then its statistics) ----
  float* out = p.ws + (int64_t)blockIdx.x * WS;
  const int j = tid;
#pragma unroll
  for (int k = 0; k < GSM_OBS_DIM; k++) {
    out[P::EW + j * GSM_OBS_DIM + k] = gwe[k];
    out[P::NW + j * GSM_NBR_FEAT_DIM + k] = gwn[k];
  }
  out[P::EB + j] = gbe; out[P::NB + j] = gbn; out[P::AW + j] = gwa;
#pragma unroll
  for (int a = 0; a < NZ; a++) { out[P::row(a) + j] = ghe[a]; out[P::row(a) + H + j] = ghg[a]; }
  if (j < NZ) out[j < NA ? P::HB + j : P::VB + (j - NA)] = gsc;
  else if (j == H - 1) out[P::AB] = gsc;
  else if constexpr (KIND == HEAD_GAUSS) { if (j < NZ + GD) out[P::LS + (j - NZ)] = gsc; }
  if constexpr (PPO) { if (j < PPO_WS_STATS) out[NP + j] = j < PPO_ROW_STATS ? sm.stacc[j] : 0.f; }
}

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

// the loss modes' backward_kernel partials: blocks 0 .. ceil(NP / 32) - 1 reduce the gradient exactly as
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

// f(std::integral_constant<int, NA>()) for the compiled instance of a head: NA = n_actions (5 or 9, checked
// by the caller) for the categorical head, GD for the Gaussian
template <int KIND, class F> static auto for_na(int n_actions, F f) {
  if constexpr (KIND == HEAD_GAUSS) return f(std::integral_constant<int, GD>());
  else return n_actions == 5 ? f(std::integral_constant<int, 5>()) : f(std::integral_constant<int, 9>());
}

template <int KIND>
static int launch_actor(const typename Head<KIND>::Params& w, const ActorIO<KIND>& io, int n_actions, cudaStream_t st) {
  if (io.n_rows == 0) return 0;
  const unsigned grid = (unsigned)((io.n_rows + 127) / 128);   // 128 = AG, the agents a block owns
  for_na<KIND>(n_actions, [&](auto na) {
    constexpr int NA = decltype(na)::value;
    if (io.values) graph_actor_kernel<NA, GSM_POLICY_VALUE_HEADS, KIND><<<grid, 128, 0, st>>>(w, io);
    else graph_actor_kernel<NA, 0, KIND><<<grid, 128, 0, st>>>(w, io);
  });
  return (int)cudaGetLastError();
}

template <int KIND> static int launch_evaluate(const EvalArgs<KIND>& a, int n_actions, cudaStream_t st) {
  const unsigned grid = (unsigned)((a.n_rows + 127) / 128);
  for_na<KIND>(n_actions, [&](auto na) { policy_eval_kernel<decltype(na)::value, KIND><<<grid, 128, 0, st>>>(a); });
  return (int)cudaGetLastError();
}

// the backward kernel, then the reduction of its G partials: the gradient (and, with the loss, the statistics)
template <int NA, int KIND, int LOSS>
static int launch_backward(BwdArgs<KIND, LOSS> a, float* grad, float* stats, cudaStream_t st) {
  constexpr int NP = PV<NA, KIND>::N;
  const int64_t G = bwd_blocks(a.n_rows);
  a.n_tiles = (a.n_rows + BWD_AG - 1) / BWD_AG;
  if constexpr (LOSS != LOSS_NONE) a.inv_n = 1.f / (float)a.n_rows;
  const size_t dyn = 2 * sizeof(float) * BWD_AG * (size_t)a.K;
  if (sizeof(BwdSmemT<NA, KIND, LOSS>) + dyn > 48 * 1024) {      // large max_nbrs: opt in to more shared memory
    const cudaError_t e = cudaFuncSetAttribute(backward_kernel<NA, KIND, LOSS>,
                                               cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
    if (e != cudaSuccess) {            // max_nbrs beyond the block's shared memory: report it here and clear
      cudaGetLastError();              // it, or the next launch's cudaGetLastError() would report it again
      return (int)e;
    }
  }
  backward_kernel<NA, KIND, LOSS><<<(unsigned)G, BWD_AG, dyn, st>>>(a);
  if constexpr (LOSS != LOSS_NONE)
    ppo_reduce_kernel<<<(NP + 31) / 32 + 1, 256, 0, st>>>(a.ws, (int)G, NP, grad, stats, (float)a.n_rows,
                                                           a.value_coef, a.entropy_coef);
  else
    policy_grad_reduce_kernel<<<(NP + 31) / 32, 256, 0, st>>>(a.ws, (int)G, NP, grad);
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
int pfailf(int status, const char* who, const char* msg) {
  snprintf(g_policy_err, sizeof(g_policy_err), "%s: %s", who, msg);
  return status;
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
// check_device, then launch() (a cudaError_t) with `device` current; GSM_OK or the error status to return.
template <class Launch> int on_device(int device, const char* who, Launch launch) {
  if (const int ds = check_device(device, who)) return ds;
  DevGuard guard(device);
  if (!guard.ok) return pfailf(GSM_ERR_CUDA, who, "cudaSetDevice failed");
  const int e = launch();
  if (e) return pfail(GSM_ERR_CUDA, cudaGetErrorString((cudaError_t)e));
  return GSM_OK;
}

// the embedding and the critics, which follow the head's na rows
template <class W, class P> void pack_embedding(const W* w, P* p, int na) {
  static_assert(sizeof(p->ego_w) == sizeof(w->ego_w), "layout");
  std::memcpy(p->ego_w, w->ego_w, sizeof(p->ego_w));   std::memcpy(p->ego_b, w->ego_b, sizeof(p->ego_b));
  std::memcpy(p->nbr_w, w->nbr_w, sizeof(p->nbr_w));   std::memcpy(p->nbr_b, w->nbr_b, sizeof(p->nbr_b));
  std::memcpy(p->att_w, w->att_w, sizeof(p->att_w));   p->att_b = w->att_b;
  std::memcpy(p->head_w[na], w->value_w, sizeof(w->value_w));
  std::memcpy(&p->head_b[na], w->value_b, sizeof(w->value_b));
}
int pack(const gsm_policy_weights* w, gsm::PolicyParams* p) {
  if (!w) return pfail(GSM_ERR_INVALID_ARG, "gsm_policy: weights is NULL");
  if (w->struct_size != sizeof(gsm_policy_weights)) return pfail(GSM_ERR_ABI, "gsm_policy: weights.struct_size mismatch");
  if (w->n_actions != 5 && w->n_actions != 9)
    return pfail(GSM_ERR_UNSUPPORTED, "gsm_policy: compiled actor instances exist for n_actions 5 and 9 only");
  std::memset(p->head_w, 0, sizeof(p->head_w)); std::memset(p->head_b, 0, sizeof(p->head_b));
  pack_embedding(w, p, w->n_actions);
  std::memcpy(p->head_w, w->head_w, sizeof(float) * 2 * GSM_POLICY_HIDDEN * w->n_actions);
  std::memcpy(p->head_b, w->head_b, sizeof(float) * w->n_actions);
  return GSM_OK;
}
int pack(const gsm_policy_gauss_weights* w, gsm::GaussParams* p) {
  if (!w) return pfail(GSM_ERR_INVALID_ARG, "gsm_policy_gauss: weights is NULL");
  if (w->struct_size != sizeof(gsm_policy_gauss_weights))
    return pfail(GSM_ERR_ABI, "gsm_policy_gauss: weights.struct_size mismatch");
  static_assert(sizeof(p->log_std) == sizeof(w->log_std), "layout");
  pack_embedding(w, p, gsm::GD);
  std::memcpy(p->head_w, w->mean_w, sizeof(w->mean_w));
  std::memcpy(p->head_b, w->mean_b, sizeof(w->mean_b));
  std::memcpy(p->log_std, w->log_std, sizeof(p->log_std));
  return GSM_OK;
}

// the head rows of the instance that serves a call
int n_actions(const gsm_policy_weights* w) { return w->n_actions; }
int n_actions(const gsm_policy_gauss_weights*) { return gsm::GD; }
int n_actions(const gsm_policy_eval_io* io) { return io->n_actions; }
int n_actions(const gsm_policy_gauss_eval_io*) { return gsm::GD; }

template <class IO> int check_rows(const IO* io, const char* who) {
  if (io->n_rows < 0 || io->max_nbrs < 1) return pfailf(GSM_ERR_INVALID_ARG, who, "bad n_rows / max_nbrs");
  if (io->n_rows > ((int64_t)1 << 31) * 128 - 128) return pfailf(GSM_ERR_INVALID_ARG, who, "n_rows too large");
  return GSM_OK;
}

// The checks the evaluate and backward entry points of both heads share; none touches the device.
template <class IO> int check_eval_io(const IO* io, const char* who) {
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
  return check_rows(io, who);
}
template <int KIND, class IO> gsm::EvalArgs<KIND> eval_args(const IO* io) {
  gsm::EvalArgs<KIND> a{};
  a.params = io->params; a.obs = io->obs; a.nbr_feat = io->nbr_feat; a.nbr_cnt = io->nbr_cnt;
  a.actions = io->actions; a.rows = io->rows;
  a.n_rows = io->n_rows; a.K = io->max_nbrs;
  return a;
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

template <int KIND, class W, class IO> int act_t(const W* w, const IO* io, int device, void* stream, const char* who) {
  typename gsm::Head<KIND>::Params p;
  if (const int st = pack(w, &p)) return st;
  if (!io || !io->obs || !io->nbr_feat || !io->nbr_cnt || !io->actions)
    return pfailf(GSM_ERR_INVALID_ARG, who, "obs, nbr_feat, nbr_cnt and actions are required");
  if (const int st = check_rows(io, who)) return st;
  gsm::ActorIO<KIND> k;
  k.obs = io->obs; k.nbr_feat = io->nbr_feat; k.nbr_cnt = io->nbr_cnt;
  k.actions = io->actions; k.logp = io->logp; k.values = io->values;
  if constexpr (KIND == gsm::HEAD_CAT) k.dist = io->logits; else k.dist = io->mean;
  k.n_rows = io->n_rows; k.row_offset = io->row_offset; k.seed = io->seed; k.step = io->step;
  k.K = io->max_nbrs; k.greedy = io->greedy;
  return on_device(device, who, [&] { return gsm::launch_actor<KIND>(p, k, n_actions(w), (cudaStream_t)stream); });
}

template <int KIND, class IO> int evaluate_t(const IO* io, int device, void* stream, const char* who) {
  if (const int st = check_eval_io(io, who)) return st;
  if (io->n_rows == 0) return GSM_OK;
  gsm::EvalArgs<KIND> a = eval_args<KIND>(io);
  a.logp = io->logp; a.entropy = io->entropy; a.values = io->values;
  return on_device(device, who, [&] { return gsm::launch_evaluate<KIND>(a, n_actions(io), (cudaStream_t)stream); });
}

// the *_workspace entry points; n_actions is checked for the categorical head only (the Gaussian passes GD)
template <int KIND, bool LOSS> int64_t workspace_t(int64_t n_rows, int n_actions, const char* who) {
  if (KIND == gsm::HEAD_CAT && n_actions != 5 && n_actions != 9)
    return pfailf(GSM_ERR_UNSUPPORTED, who, "n_actions must be 5 or 9");
  if (n_rows < 0) return pfailf(GSM_ERR_INVALID_ARG, who, "n_rows < 0");
  return gsm::for_na<KIND>(n_actions, [&](auto na) {   // per block: its partial gradient (then its statistics)
    constexpr int WS = gsm::PV<decltype(na)::value, KIND>::N + (LOSS ? gsm::PPO_WS_STATS : 0);
    return gsm::bwd_blocks(n_rows) * WS * (int64_t)sizeof(float);
  });
}

// gsm_policy_backward(_gauss) (LOSS_NONE: d_logp, d_entropy and d_values are the seeds),
// gsm_ppo_backward(_gauss) (LOSS_PPO: `loss` computes the seeds) and gsm_ppo_backward_normalized(_gauss)
// (LOSS_PPO_VNORM: on targets normalised with value_affine); ws_msg: the error for a short workspace
template <int KIND, int LOSS, class IO>
int backward_t(const IO* io, const gsm_ppo_loss_io* loss, const float* value_affine, const float* d_logp,
               const float* d_entropy, const float* d_values, float* grad, void* workspace, size_t workspace_bytes,
               int device, void* stream, const char* who, const char* ws_msg) {
  constexpr bool PPO = LOSS != gsm::LOSS_NONE;
  if (const int st = check_eval_io(io, who)) return st;
  if constexpr (PPO) { if (const int st = check_loss_io(loss, who)) return st; }
  if constexpr (LOSS == gsm::LOSS_PPO_VNORM) {
    if (!value_affine) return pfailf(GSM_ERR_INVALID_ARG, who, "value_affine is required");
  }
  if (!grad) return pfailf(GSM_ERR_INVALID_ARG, who, "grad is required");
  const int64_t need = workspace_t<KIND, PPO>(io->n_rows, n_actions(io), who);
  if (need > 0 && (!workspace || workspace_bytes < (size_t)need)) return pfailf(GSM_ERR_INVALID_ARG, who, ws_msg);
  if (io->n_rows == 0) return GSM_OK;
  gsm::BwdArgs<KIND, LOSS> a{};
  static_cast<gsm::EvalArgs<KIND>&>(a) = eval_args<KIND>(io);
  float* stats = nullptr;
  if constexpr (PPO) {
    a.old_logp = loss->old_logp; a.old_values = loss->old_values; a.returns = loss->returns; a.adv = loss->advantages;
    a.adv_moments = loss->adv_moments; a.lagrange = loss->lagrange;
    a.clip = loss->clip; a.value_clip = loss->value_clip;
    a.value_coef = loss->value_coef; a.entropy_coef = loss->entropy_coef;
    stats = loss->stats;
    if constexpr (LOSS == gsm::LOSS_PPO_VNORM) a.value_affine = value_affine;
  } else {
    a.d_logp = d_logp; a.d_entropy = d_entropy; a.d_values = d_values;
  }
  a.ws = (float*)workspace;
  return on_device(device, who, [&] {
    return gsm::for_na<KIND>(n_actions(io), [&](auto na) {
      return gsm::launch_backward<decltype(na)::value, KIND, LOSS>(a, grad, stats, (cudaStream_t)stream);
    });
  });
}

// gsm_gae (NORM = false) and gsm_gae_normalized (NORM: the values are denormalised with `affine`)
template <bool NORM>
int gae_t(const float* reward, const float* cost, const float* values, const uint8_t* done, int32_t n_steps,
          int64_t n_rows, int64_t slot_rows, float gamma, float lam, float* returns, float* advantages,
          const float* affine, int device, void* stream, const char* who) {
  if (!reward || !cost || !values || !done || !returns)
    return pfailf(GSM_ERR_INVALID_ARG, who, "reward, cost, values, done and returns are required");
  if constexpr (NORM) { if (!affine) return pfailf(GSM_ERR_INVALID_ARG, who, "value_affine is required"); }
  if (n_steps < 1 || n_rows < 0 || slot_rows < n_rows) return pfailf(GSM_ERR_INVALID_ARG, who, "bad sizes");
  if (const int ds = check_device(device, who)) return ds;
  if (n_rows == 0) return GSM_OK;
  DevGuard guard(device);
  if (!guard.ok) return pfailf(GSM_ERR_CUDA, who, "cudaSetDevice failed");
  gsm::GaeArgs<NORM> p{};
  static_cast<gsm::GaeParams&>(p) = {reward, cost, values, done, returns, advantages, n_rows, slot_rows, n_steps,
                                     gamma, lam};
  if constexpr (NORM) p.affine = affine;
  const int64_t threads = n_rows * GSM_POLICY_VALUE_HEADS;
  gsm::gae_kernel<NORM><<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return pfail(GSM_ERR_CUDA, cudaGetErrorString(e));
  return GSM_OK;
}
}  // namespace

extern "C" {

const char* gsm_policy_last_error(void) { return g_policy_err; }

int gsm_policy_act(const gsm_policy_weights* w, const gsm_policy_io* io, int device, void* stream) {
  return act_t<gsm::HEAD_CAT>(w, io, device, stream, "gsm_policy_act");
}

int gsm_policy_act_gauss(const gsm_policy_gauss_weights* w, const gsm_policy_gauss_io* io, int device,
                         void* stream) {
  return act_t<gsm::HEAD_GAUSS>(w, io, device, stream, "gsm_policy_act_gauss");
}

int gsm_policy_evaluate(const gsm_policy_eval_io* io, int device, void* stream) {
  return evaluate_t<gsm::HEAD_CAT>(io, device, stream, "gsm_policy_evaluate");
}

int gsm_policy_evaluate_gauss(const gsm_policy_gauss_eval_io* io, int device, void* stream) {
  return evaluate_t<gsm::HEAD_GAUSS>(io, device, stream, "gsm_policy_evaluate_gauss");
}

int64_t gsm_policy_backward_workspace(int64_t n_rows, int32_t n_actions) {
  return workspace_t<gsm::HEAD_CAT, false>(n_rows, n_actions, "gsm_policy_backward_workspace");
}

int64_t gsm_policy_backward_workspace_gauss(int64_t n_rows) {
  return workspace_t<gsm::HEAD_GAUSS, false>(n_rows, gsm::GD, "gsm_policy_backward_workspace_gauss");
}

int gsm_policy_backward(const gsm_policy_eval_io* io, const float* d_logp, const float* d_entropy,
                        const float* d_values, float* grad, void* workspace, size_t workspace_bytes,
                        int device, void* stream) {
  return backward_t<gsm::HEAD_CAT, gsm::LOSS_NONE>(io, nullptr, nullptr, d_logp, d_entropy, d_values, grad, workspace, workspace_bytes,
                                          device, stream, "gsm_policy_backward",
                                          "workspace smaller than gsm_policy_backward_workspace(n_rows, n_actions)");
}

int gsm_policy_backward_gauss(const gsm_policy_gauss_eval_io* io, const float* d_logp, const float* d_entropy,
                              const float* d_values, float* grad, void* workspace, size_t workspace_bytes,
                              int device, void* stream) {
  return backward_t<gsm::HEAD_GAUSS, gsm::LOSS_NONE>(io, nullptr, nullptr, d_logp, d_entropy, d_values, grad, workspace,
                                            workspace_bytes, device, stream, "gsm_policy_backward_gauss",
                                            "workspace smaller than gsm_policy_backward_workspace_gauss(n_rows)");
}

int64_t gsm_ppo_backward_workspace(int64_t n_rows, int32_t n_actions) {
  return workspace_t<gsm::HEAD_CAT, true>(n_rows, n_actions, "gsm_ppo_backward_workspace");
}

int64_t gsm_ppo_backward_workspace_gauss(int64_t n_rows) {
  return workspace_t<gsm::HEAD_GAUSS, true>(n_rows, gsm::GD, "gsm_ppo_backward_workspace_gauss");
}

int gsm_ppo_backward(const gsm_policy_eval_io* io, const gsm_ppo_loss_io* loss, float* grad, void* workspace,
                     size_t workspace_bytes, int device, void* stream) {
  return backward_t<gsm::HEAD_CAT, gsm::LOSS_PPO>(io, loss, nullptr, nullptr, nullptr, nullptr, grad, workspace, workspace_bytes, device,
                                         stream, "gsm_ppo_backward",
                                         "workspace smaller than the ppo backward workspace for n_rows");
}

int gsm_ppo_backward_gauss(const gsm_policy_gauss_eval_io* io, const gsm_ppo_loss_io* loss, float* grad,
                           void* workspace, size_t workspace_bytes, int device, void* stream) {
  return backward_t<gsm::HEAD_GAUSS, gsm::LOSS_PPO>(io, loss, nullptr, nullptr, nullptr, nullptr, grad, workspace, workspace_bytes,
                                           device, stream, "gsm_ppo_backward_gauss",
                                           "workspace smaller than the ppo backward workspace for n_rows");
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
  const gsm::AdamArgs a{params, grad, m, v, step, grad_norm, n, lr, beta1, beta2, eps, max_grad_norm};
  return on_device(device, who, [&] {
    gsm::adam_step_kernel<<<1, gsm::ADAM_THREADS, 0, (cudaStream_t)stream>>>(a);
    return (int)cudaGetLastError();
  });
}

int gsm_gae(const float* reward, const float* cost, const float* values, const uint8_t* done, int32_t n_steps,
            int64_t n_rows, int64_t slot_rows, float gamma, float lam, float* returns, float* advantages,
            int device, void* stream) {
  return gae_t<false>(reward, cost, values, done, n_steps, n_rows, slot_rows, gamma, lam, returns, advantages,
                      nullptr, device, stream, "gsm_gae");
}

int gsm_gae_normalized(const float* reward, const float* cost, const float* values, const uint8_t* done,
                       int32_t n_steps, int64_t n_rows, int64_t slot_rows, float gamma, float lam, float* returns,
                       float* advantages, const float* value_affine, int device, void* stream) {
  return gae_t<true>(reward, cost, values, done, n_steps, n_rows, slot_rows, gamma, lam, returns, advantages,
                     value_affine, device, stream, "gsm_gae_normalized");
}

int gsm_ppo_backward_normalized(const gsm_policy_eval_io* io, const gsm_ppo_loss_io* loss, const float* value_affine,
                                float* grad, void* workspace, size_t workspace_bytes, int device, void* stream) {
  return backward_t<gsm::HEAD_CAT, gsm::LOSS_PPO_VNORM>(io, loss, value_affine, nullptr, nullptr, nullptr, grad,
                                                        workspace, workspace_bytes, device, stream,
                                                        "gsm_ppo_backward_normalized",
                                                        "workspace smaller than the ppo backward workspace for n_rows");
}

int gsm_ppo_backward_normalized_gauss(const gsm_policy_gauss_eval_io* io, const gsm_ppo_loss_io* loss,
                                      const float* value_affine, float* grad, void* workspace,
                                      size_t workspace_bytes, int device, void* stream) {
  return backward_t<gsm::HEAD_GAUSS, gsm::LOSS_PPO_VNORM>(io, loss, value_affine, nullptr, nullptr, nullptr, grad,
                                                          workspace, workspace_bytes, device, stream,
                                                          "gsm_ppo_backward_normalized_gauss",
                                                          "workspace smaller than the ppo backward workspace for n_rows");
}

}  // extern "C"
