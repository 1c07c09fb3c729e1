// gsm_kernels.cuh — sm_100a kernels of the batched GS-MARL env hot path (SPEC.md).
//
// Stands in for MultiAgentGraphConstrainEnv.step/reset + World.step + the scenario
// callbacks (reference environment.py / core.py / scenarios/*.py,
// GSMARL.egg-info/SOURCES.txt:14,15,21-25 — withheld, see SPEC.md header).
//
// One fused kernel per env step: action force -> pairwise contact force -> damped Euler
// -> (polygon/line) in-warp linear assignment -> neighbour graph, obs, reward, cost, done.
// Two thread mappings, chosen on the host:
//   packed  (CTA_ENV=false): an env owns N*P consecutive lanes of ONE warp (P lanes per
//           agent), a warp carries 32/(N*P) envs, all exchange is warp-level
//           (shuffle / ballot / redux), no block barrier on the step path;
//   cta-env (CTA_ENV=true):  one env per CTA, groups of P lanes sweep the agents.
// Included by gsm_kernels_f32.cu (production) and gsm_kernels_f64.cu (verification,
// compiled with -fmad=false so every operation rounds once, like the oracle).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/gsmarl_b200.h"
#include "gsm_host.h"

namespace gsm {

constexpr int kThreads = 128;  // CTA size of the env kernel (4 warps)
__host__ __device__ constexpr unsigned low_mask(int n) { return n >= 32 ? 0xffffffffu : ((1u << (n & 31)) - 1u); }

template <typename T>
struct KParams {
  int64_t n_envs, env_offset;
  int N, L, E, K, W;
  int scenario, action_mode, n_actions, episode_length;
  int share_reward, cost_obstacles, own_goal_always;
  int envs_per_warp;  // packed mode
  T dt, one_minus_damp, cf, km, km_inv, Rs, w_dist, w_goal, goal_tol, poly_r;
  T discrete_u[GSM_MAX_DISCRETE][2];
  const T* size;           // [E]
  const uint8_t* eflag;    // [E] bit0 collide, bits1..2 type
  const T* mass;           // [N]
  const T* accel;          // [N]
  const T* max_speed;      // [N]
  const T* slot_table;     // [N][2] or null
  T* agent_state;          // [n_envs][N][4]
  T* lm_pos;               // [n_envs][L][2]
  int32_t* t;              // [n_envs]
  const uint8_t* mask;     // observe-after-reset: only envs with mask[i*stride] != 0
  int64_t mask_stride;
  // in-kernel auto-reset of fused rollouts (SPEC §8 draws, same counters as reset_kernel)
  int auto_reset;
  uint64_t seed;
  int32_t* episode;        // [n_envs]
  double ext[4];           // spawn half-extent per entity type
  const void* actions;
  T* obs; int32_t* nbr_idx; T* nbr_feat; int32_t* nbr_cnt; uint32_t* adj;
  T* reward; T* cost; uint8_t* done; int32_t* assign;
};

// ---- shared-memory carve-up (same arithmetic on host and device) ---------------------
struct SmemLayout {
  size_t off_size, off_agc, off_ag, off_lm, off_new, off_rew, off_slot, off_cmat, off_asg,
      off_stage, off_flag, stage_stride, stage_feat, total;
};
// epb: envs per CTA; groups: agent groups per CTA (kThreads / P); K: padded neighbour rows.
__host__ __device__ inline SmemLayout make_layout(int rb, int N, int L, int E, int K, int epb,
                                                  int groups, int lsa) {
  SmemLayout s;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += ((bytes + 15) / 16) * 16; return r; };
  s.off_size = take((size_t)E * rb);
  s.off_agc = take((size_t)N * 3 * rb);                  // mass, accel, max_speed
  s.off_ag = take((size_t)epb * N * 4 * rb);
  s.off_lm = take((size_t)epb * L * 2 * rb);
  s.off_new = take((size_t)epb * N * 4 * rb);
  s.off_rew = take((size_t)epb * N * rb);
  s.off_slot = take(lsa ? (size_t)epb * N * 2 * rb : 0);
  s.off_cmat = take(lsa ? (size_t)epb * N * N * rb : 0);
  s.off_asg = take((size_t)epb * N * 4);
  s.stage_feat = (((size_t)K * 4 + 15) / 16) * 16;       // idx rows first, then feat rows
  s.stage_stride = s.stage_feat + (((size_t)K * GSM_NBR_FEAT_DIM * rb + 15) / 16) * 16;
  s.off_stage = take((size_t)groups * s.stage_stride);
  s.off_flag = take((size_t)E);
  s.total = o;
  return s;
}

// ---- small device helpers ------------------------------------------------------------
__device__ __forceinline__ float r_sqrt(float x) { return sqrtf(x); }
__device__ __forceinline__ double r_sqrt(double x) { return sqrt(x); }
__device__ __forceinline__ float r_exp(float x) { return expf(x); }
__device__ __forceinline__ double r_exp(double x) { return exp(x); }
__device__ __forceinline__ float r_log1p(float x) { return log1pf(x); }
__device__ __forceinline__ double r_log1p(double x) { return log1p(x); }

// SPEC §3: numpy logaddexp(0, x).
template <typename T>
__device__ __forceinline__ T softplus(T x) {
  if (x > (T)0) return x + r_log1p(r_exp(-x));
  return r_log1p(r_exp(x));
}

__device__ __forceinline__ float shfl(unsigned m, float v, int src) { return __shfl_sync(m, v, src); }
__device__ __forceinline__ double shfl(unsigned m, double v, int src) { return __shfl_sync(m, v, src); }
__device__ __forceinline__ int shfl(unsigned m, int v, int src) { return __shfl_sync(m, v, src); }

// Minimum over the lanes of an arbitrary mask, via redux.sync on an order-preserving key.
__device__ __forceinline__ float mask_min(unsigned m, float v) {
  unsigned b = __float_as_uint(v);
  unsigned key = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  unsigned r = __reduce_min_sync(m, key);
  return __uint_as_float((r & 0x80000000u) ? (r & 0x7fffffffu) : ~r);
}
__device__ __forceinline__ double mask_min(unsigned m, double v) {
  unsigned long long b = (unsigned long long)__double_as_longlong(v);
  unsigned long long key = (b >> 63) ? ~b : (b | 0x8000000000000000ull);
  unsigned hi = (unsigned)(key >> 32), lo = (unsigned)key;
  unsigned mhi = __reduce_min_sync(m, hi);
  unsigned mlo = __reduce_min_sync(m, hi == mhi ? lo : 0xffffffffu);
  unsigned long long r = ((unsigned long long)mhi << 32) | mlo;
  r = (r >> 63) ? (r & 0x7fffffffffffffffull) : ~r;
  return __longlong_as_double((long long)r);
}

template <typename T> __device__ __forceinline__ T r_inf();
template <> __device__ __forceinline__ float r_inf<float>() { return __int_as_float(0x7f800000); }
template <> __device__ __forceinline__ double r_inf<double>() {
  return __longlong_as_double(0x7ff0000000000000ll);
}

// SPEC §8 draw of entity e of global env g in episode ep: the same integer stream and the same
// fp64 arithmetic as reset_kernel / the oracle, so an in-kernel reset is bit-identical.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t out[4]);
__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo);
__device__ __forceinline__ void spawn_draw_inline(uint64_t g, int ep, int e, uint64_t seed, double ext,
                                                  double& x, double& y) {
  uint32_t r[4];
  philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)ep, (uint32_t)e, (uint32_t)seed,
                (uint32_t)(seed >> 32), r);
  x = __dadd_rn(-ext, __dmul_rn(2.0 * ext, u53(r[0], r[1])));
  y = __dadd_rn(-ext, __dmul_rn(2.0 * ext, u53(r[2], r[3])));
}
// Cold path (once per episode end): kept out of line so that the 10 unrolled Philox rounds do
// not raise the register count of the step loops.
static __device__ __noinline__ void spawn_draw_f64(uint64_t g, int ep, int e, uint64_t seed, double ext,
                                            double* x, double* y) {
  spawn_draw_inline(g, ep, e, seed, ext, *x, *y);
}
template <typename T>
__device__ __forceinline__ void spawn_draw(uint64_t g, int ep, int e, uint64_t seed, double ext, T& x, T& y) {
  double dx, dy;
  spawn_draw_f64(g, ep, e, seed, ext, &dx, &dy);
  x = (T)dx; y = (T)dy;
}

// Production precision may drop contact terms that cannot change an fp32 result: for
// x = -(dist - dmin)/margin < -kFarCut the penetration is < margin * 2.1e-9 (SPEC §3 note).
template <typename T> struct Prec;
template <> struct Prec<float> { static constexpr bool kCut = true; };
template <> struct Prec<double> { static constexpr bool kCut = false; };
constexpr float kFarCut = 20.0f;

// Cooperative copy of `bytes` (multiple of 4) from shared to global by the P lanes of a
// group, with the widest vector both addresses allow.
template <int P>
__device__ __forceinline__ void group_copy(void* gdst, const void* ssrc, int bytes, int sub) {
  const uintptr_t ga = (uintptr_t)gdst;
  if (((ga | (uintptr_t)bytes) & 15) == 0) {
    for (int k = sub; k < (bytes >> 4); k += P) ((int4*)gdst)[k] = ((const int4*)ssrc)[k];
  } else if (((ga | (uintptr_t)bytes) & 7) == 0) {
    for (int k = sub; k < (bytes >> 3); k += P) ((int2*)gdst)[k] = ((const int2*)ssrc)[k];
  } else {
    for (int k = sub; k < (bytes >> 2); k += P) ((int*)gdst)[k] = ((const int*)ssrc)[k];
  }
}

// SPEC §5.  scipy rectangular_lsap (Crouse 2016) on an n x n matrix in shared memory,
// one lane per COLUMN (and per row): u/v/shortestPathCosts/path/row4col/col4row live in
// registers, the scan over `remaining` becomes one redux-min plus the tie rule (last
// unassigned minimum in `remaining` order, else first minimum), `remaining`'s
// swap-with-last removal is tracked as a per-lane position.  Lanes of `gm` with
// col >= n take part in the warp primitives only.  Returns col4row for row == col.
template <typename T>
__device__ int lsa_lanes(const T* __restrict__ C, int n, int col, unsigned gm, int base) {
  const T INF = r_inf<T>();
  T u_m = 0, v_m = 0;
  int col4row_m = -1, row4col_m = -1, path_m = -1;
  const bool is_col = col < n;
  for (int cur = 0; cur < n; cur++) {
    T minval = 0, spc = INF;
    int i = cur, nrem = n, sink = -1;
    int pos = n - 1 - col;
    bool inrem = is_col, sr_m = false, sc_m = false;
    for (int iter = 0; iter < n && sink == -1; iter++) {
      if (col == i) sr_m = true;
      const T u_i = shfl(gm, u_m, base + i);
      if (inrem) {
        const T r = minval + C[i * n + col] - u_i - v_m;
        if (r < spc) { path_m = i; spc = r; }
      }
      const T lowest = mask_min(gm, inrem ? spc : INF);
      if (lowest == INF) return -1;
      const bool cand = inrem && spc == lowest;
      const bool ucand = cand && row4col_m == -1;
      const unsigned bu = __ballot_sync(gm, ucand);
      int selpos;
      if (bu) selpos = __reduce_max_sync(gm, ucand ? pos : -1);
      else selpos = __reduce_min_sync(gm, cand ? pos : 0x3fffffff);
      const bool sel = inrem && pos == selpos;
      const int jl = __ffs(__ballot_sync(gm, sel)) - 1;
      minval = lowest;
      const int r4c = shfl(gm, row4col_m, jl);
      if (r4c == -1) sink = jl - base; else i = r4c;
      if (sel) { sc_m = true; inrem = false; }
      nrem--;
      if (inrem && pos == nrem) pos = selpos;
    }
    const T spc_row = shfl(gm, spc, base + (col4row_m >= 0 ? col4row_m : 0));
    if (is_col) {
      if (col == cur) u_m += minval;
      else if (sr_m) u_m += minval - spc_row;
    }
    if (sc_m) v_m -= minval - spc;
    if (sink < 0) return -1;                        // non-finite costs: give up, never hang
    int j = sink;
    for (int iter = 0; iter < n; iter++) {
      const int a = shfl(gm, path_m, base + j);
      if (col == j) row4col_m = a;
      const int tprev = shfl(gm, col4row_m, base + a);
      if (col == a) col4row_m = j;
      j = tprev;
      if (a == cur) break;
    }
  }
  return col4row_m;
}

// Segmented, lockstep form of lsa_lanes for several problems per warp.  Every lane of the
// warp calls it (full-mask primitives only).  A segment is a run of consecutive lanes
// starting at `base` that holds one problem; lane offset `off` < N of a segment is column
// `off`, row `off` AND slot `off` of scipy's `remaining` array (rem = column stored at that
// position), so the scan "last unassigned minimum in position order, else first minimum"
// is clz / ffs on two ballots.  Segments whose search has ended idle until the slowest one
// finishes (time = max, not sum, of the per-problem iteration counts).  All loops are bounded
// by N so that non-finite costs cannot hang the warp.  Returns col4row for row == off.
template <typename T, int N>
__device__ __forceinline__ int lsa_seg(const T* __restrict__ C, int off, int base, bool live) {
  constexpr unsigned FULL = 0xffffffffu;
  const T INF = r_inf<T>();
  const bool is_col = live && off < N;
  T u_m = 0, v_m = 0;
  int col4row_m = -1, row4col_m = -1, path_m = -1;
  for (int cur = 0; cur < N; cur++) {
    T minval = 0, spc = INF;
    int i = cur, nrem = N, sink = live ? -1 : 0;
    int rem = N - 1 - off;                          // remaining[] filled in reverse
    bool inrem = is_col, sr_m = false, sc_m = false;
    for (int iter = 0; iter < N && __any_sync(FULL, sink == -1); iter++) {
      const bool run = sink == -1;
      if (run && off == i) sr_m = true;
      const T u_i = shfl(FULL, u_m, base + i);
      if (run && inrem) {
        const T r = minval + C[i * N + off] - u_i - v_m;
        if (r < spc) { path_m = i; spc = r; }
      }
      const T mine = inrem ? spc : INF;
      T lowest = INF;
#pragma unroll
      for (int k = 0; k < N; k++) {
        const T o = shfl(FULL, mine, base + k);
        lowest = o < lowest ? o : lowest;
      }
      const int rc = off < N ? rem : 0;
      const T spc_of = shfl(FULL, spc, base + rc);
      const int r4c_of = shfl(FULL, row4col_m, base + rc);
      const bool cand = is_col && off < nrem && spc_of == lowest;
      const bool ucand = cand && r4c_of == -1;
      const unsigned bc = (__ballot_sync(FULL, cand) >> base) & low_mask(N);
      const unsigned bu = (__ballot_sync(FULL, ucand) >> base) & low_mask(N);
      const int it_sel = bu ? (31 - __clz(bu)) : (bc ? __ffs(bc) - 1 : 0);
      const int j = shfl(FULL, rem, base + it_sel);
      const int r4c_j = shfl(FULL, row4col_m, base + j);
      const int last = shfl(FULL, rem, base + nrem - 1);
      if (run) {
        minval = lowest;
        if (r4c_j == -1) sink = j; else i = r4c_j;
        if (off == j) { sc_m = true; inrem = false; }
        if (off == it_sel) rem = last;
        nrem--;
      }
    }
    const T spc_row = shfl(FULL, spc, base + (col4row_m >= 0 ? col4row_m : 0));
    if (is_col) {
      if (off == cur) u_m += minval;
      else if (sr_m) u_m += minval - spc_row;
    }
    if (sc_m) v_m -= minval - spc;
    int j = sink;
    bool going = live && sink >= 0;
    for (int iter = 0; iter < N && __any_sync(FULL, going); iter++) {
      const int a = shfl(FULL, path_m, base + j);
      const int tprev = shfl(FULL, col4row_m, base + a);
      if (going) {
        if (off == j) row4col_m = a;
        if (off == a) col4row_m = j;
        j = tprev;
        if (a == cur) going = false;
      }
    }
  }
  return col4row_m;
}

// ---- the fused env kernel ------------------------------------------------------------
// Lane roles: an agent is served by a group of P lanes; lane `sub` of the group handles the
// "other" entities o = sub, sub+P, ... (o indexes the E-1 entities != i), so for P >= E-1
// (navigation N=3: E-1 = 8 = P) every pair is one lane and the pair loops run once.
template <typename T, int P, bool CTA_ENV, bool PHYS>
__global__ void __launch_bounds__(kThreads) env_kernel(const __grid_constant__ KParams<T> p) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int N = p.N, L = p.L, E = p.E, K = p.K, W = p.W;
  const bool lsa = p.scenario != GSM_SCN_NAVIGATION;
  const int EPB = CTA_ENV ? 1 : p.envs_per_warp * (kThreads / 32);
  const SmemLayout lay = make_layout((int)sizeof(T), N, L, E, K, EPB, kThreads / P, lsa ? 1 : 0);
  T* s_size = (T*)(smem + lay.off_size);
  T* s_agc = (T*)(smem + lay.off_agc);
  T* s_ag = (T*)(smem + lay.off_ag);
  T* s_lm = (T*)(smem + lay.off_lm);
  T* s_new = (T*)(smem + lay.off_new);
  T* s_rew = (T*)(smem + lay.off_rew);
  T* s_slot = (T*)(smem + lay.off_slot);
  T* s_cmat = (T*)(smem + lay.off_cmat);
  int32_t* s_asg = (int32_t*)(smem + lay.off_asg);
  uint8_t* s_flag = smem + lay.off_flag;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int e = tid; e < E; e += kThreads) { s_size[e] = p.size[e]; s_flag[e] = p.eflag[e]; }
  for (int i = tid; i < N; i += kThreads) {
    s_agc[3 * i] = p.mass[i]; s_agc[3 * i + 1] = p.accel[i]; s_agc[3 * i + 2] = p.max_speed[i];
  }

  // ---- mapping -----------------------------------------------------------------------
  int env_l;          // env slot inside the CTA
  int64_t env;        // env index inside this handle
  bool active;        // this lane works on a real env
  int first_agent, agent_stride, sub, off;
  unsigned envmask, grpmask;
  int env_base_lane;
  if (CTA_ENV) {
    env_l = 0; env = blockIdx.x; active = true;
    first_agent = tid / P; agent_stride = kThreads / P; sub = tid % P; off = tid;
    envmask = 0xffffffffu; env_base_lane = 0;
    grpmask = low_mask(P) << ((lane - sub) & 31);
  } else {
    const int LPE = N * P, EPW = p.envs_per_warp;
    const int eiw = lane / LPE;
    off = lane - eiw * LPE;
    env_l = warp * EPW + eiw;
    env = (int64_t)blockIdx.x * EPB + env_l;
    active = eiw < EPW && env < p.n_envs;
    first_agent = off / P; agent_stride = N; sub = off % P;
    env_base_lane = eiw * LPE;
    envmask = low_mask(LPE) << (env_base_lane & 31);
    grpmask = low_mask(P) << ((lane - sub) & 31);
    if (!active) { first_agent = N; env_l = 0; }
  }
  if (p.mask != nullptr && active && p.mask[env * p.mask_stride] == 0) {
    // observe-after-reset on a subset: the whole env group (packed) / CTA (cta-env) drops out
    active = false; first_agent = N;
  }
  unsigned char* stage = smem + lay.off_stage + (size_t)(tid / P) * lay.stage_stride;
  int32_t* st_idx = (int32_t*)stage;
  T* st_feat = (T*)(stage + lay.stage_feat);

  // ---- stage state: coalesced, contiguous per warp (packed) / per CTA (cta-env) --------
  if (CTA_ENV) {
    const T* g_ag = p.agent_state + env * N * 4;
    const T* g_lm = p.lm_pos + env * L * 2;
    for (int k = tid; k < N * 4; k += kThreads) s_ag[k] = g_ag[k];
    for (int k = tid; k < L * 2; k += kThreads) s_lm[k] = g_lm[k];
  } else {
    const int EPW = p.envs_per_warp;
    const int64_t env0 = (int64_t)blockIdx.x * EPB + warp * EPW;
    int64_t nv = p.n_envs - env0;
    nv = nv < 0 ? 0 : (nv > EPW ? EPW : nv);
    const T* g_ag = p.agent_state + env0 * N * 4;
    const T* g_lm = p.lm_pos + env0 * L * 2;
    T* w_ag = s_ag + (size_t)warp * EPW * N * 4;
    T* w_lm = s_lm + (size_t)warp * EPW * L * 2;
    for (int k = lane; k < nv * N * 4; k += 32) w_ag[k] = g_ag[k];
    for (int k = lane; k < nv * L * 2; k += 32) w_lm[k] = g_lm[k];
  }
  __syncthreads();

  const T* e_ag = s_ag + (size_t)env_l * N * 4;
  const T* e_lm = s_lm + (size_t)env_l * L * 2;
  T* e_new = s_new + (size_t)env_l * N * 4;
  T* e_rew = s_rew + (size_t)env_l * N;
  int t_now = 0;
  if (active) t_now = p.t[env] + (PHYS ? 1 : 0);

  // ---- SPEC §2-4: force + integration ---------------------------------------------------
  if (PHYS) {
    for (int i = first_agent; i < N; i += agent_stride) {
      const T px = e_ag[4 * i], py = e_ag[4 * i + 1];
      T fx = 0, fy = 0;
      if (sub == 0) {
        T ux = 0, uy = 0;
        if (p.action_mode == GSM_ACT_DISCRETE) {
          const int a = ((const int32_t*)p.actions)[env * N + i];
          if (a >= 0 && a < p.n_actions) { ux = p.discrete_u[a][0]; uy = p.discrete_u[a][1]; }
        } else {
          const T* ap = (const T*)p.actions + (env * N + i) * 2;
          ux = ap[0]; uy = ap[1];
        }
        const T acc = s_agc[3 * i + 1];
        fx = acc * ux; fy = acc * uy;
      }
      if (s_flag[i] & 1) {
        const T si = s_size[i];
        for (int o = sub; o < E - 1; o += P) {
          const int j = o + (o >= i ? 1 : 0);
          if (!(s_flag[j] & 1)) continue;
          T qx, qy;
          if (j < N) { qx = e_ag[4 * j]; qy = e_ag[4 * j + 1]; }
          else { qx = e_lm[2 * (j - N)]; qy = e_lm[2 * (j - N) + 1]; }
          const T dx = px - qx, dy = py - qy;
          const T dist = r_sqrt(dx * dx + dy * dy);
          const T dmin = si + s_size[j];
          const T x = -(dist - dmin) / p.km;
          if (Prec<T>::kCut && x < (T)(-kFarCut)) continue;
          const T pen = softplus(x) * p.km;
          fx = fx + p.cf * dx / dist * pen;
          fy = fy + p.cf * dy / dist * pen;
        }
      }
      if (P > 1) {
#pragma unroll
        for (int m = P / 2; m >= 1; m >>= 1) {
          fx += __shfl_xor_sync(grpmask, fx, m);
          fy += __shfl_xor_sync(grpmask, fy, m);
        }
      }
      if (sub == 0) {
        T vx = e_ag[4 * i + 2] * p.one_minus_damp, vy = e_ag[4 * i + 3] * p.one_minus_damp;
        const T m = s_agc[3 * i];
        vx = vx + (fx / m) * p.dt;
        vy = vy + (fy / m) * p.dt;
        const T ms = s_agc[3 * i + 2];
        if (ms > (T)0) {
          const T sp = r_sqrt(vx * vx + vy * vy);
          if (sp > ms) { vx = vx / sp * ms; vy = vy / sp * ms; }
        }
        e_new[4 * i] = px + vx * p.dt; e_new[4 * i + 1] = py + vy * p.dt;
        e_new[4 * i + 2] = vx; e_new[4 * i + 3] = vy;
      }
    }
    if (CTA_ENV) __syncthreads(); else __syncwarp();
    // write the new state back, coalesced
    if (CTA_ENV) {
      T* g_ag = p.agent_state + env * N * 4;
      for (int k = tid; k < N * 4; k += kThreads) g_ag[k] = s_new[k];
      if (tid == 0) p.t[env] = t_now;
    } else {
      const int EPW = p.envs_per_warp;
      const int64_t env0 = (int64_t)blockIdx.x * EPB + warp * EPW;
      int64_t nv = p.n_envs - env0;
      nv = nv < 0 ? 0 : (nv > EPW ? EPW : nv);
      T* g_ag = p.agent_state + env0 * N * 4;
      const T* w_new = s_new + (size_t)warp * EPW * N * 4;
      for (int k = lane; k < nv * N * 4; k += 32) g_ag[k] = w_new[k];
      if (active && off == 0) p.t[env] = t_now;
    }
  }
  const T* cur = PHYS ? e_new : e_ag;

  // ---- SPEC §5: targets (assignment for polygon / line) --------------------------------
  if (lsa) {
    T* e_slot = s_slot + (size_t)env_l * N * 2;
    T* e_cm = s_cmat + (size_t)env_l * N * N;
    int32_t* e_asg = s_asg + (size_t)env_l * N;
    const bool solver = CTA_ENV ? (warp == 0) : active;
    const int col = CTA_ENV ? lane : off;
    const unsigned gm = CTA_ENV ? 0xffffffffu : envmask;
    if (solver) {
      if (col < N) {
        T sx, sy;
        if (p.scenario == GSM_SCN_POLYGON) {
          sx = e_lm[0] + p.poly_r * p.slot_table[2 * col];
          sy = e_lm[1] + p.poly_r * p.slot_table[2 * col + 1];
        } else {
          const T f = p.slot_table[2 * col];
          sx = e_lm[0] + f * (e_lm[2] - e_lm[0]);
          sy = e_lm[1] + f * (e_lm[3] - e_lm[1]);
        }
        e_slot[2 * col] = sx; e_slot[2 * col + 1] = sy;
        for (int i = 0; i < N; i++) {
          const T dx = sx - cur[4 * i], dy = sy - cur[4 * i + 1];
          e_cm[i * N + col] = r_sqrt(dx * dx + dy * dy);
        }
      }
      const int a = lsa_lanes<T>(e_cm, N, col, gm, env_base_lane);
      if (col < N) e_asg[col] = a;
    }
    if (CTA_ENV) __syncthreads(); else __syncwarp();
  }

  // ---- SPEC §6-7: graph, obs, reward, cost, done ---------------------------------------
  for (int i = first_agent; i < N; i += agent_stride) {
    const T px = cur[4 * i], py = cur[4 * i + 1], vx = cur[4 * i + 2], vy = cur[4 * i + 3];
    const int64_t row = env * N + i;
    const T si = s_size[i];
    int cnt = 0, ncol = 0;
    uint32_t word = 0;      // adjacency word under construction (lane sub == 0 keeps it)
    int wcur = 0;
    for (int o0 = 0; o0 < E - 1; o0 += P) {
      const int o = o0 + sub;
      const bool valid = o < E - 1;
      const int e = o + (o >= i ? 1 : 0);
      T dx = 0, dy = 0, dvx = 0, dvy = 0, dist = 0;
      bool nb = false, col = false;
      int fl = 0;
      if (valid) {
        T ex, ey, evx = 0, evy = 0;
        if (e < N) { ex = cur[4 * e]; ey = cur[4 * e + 1]; evx = cur[4 * e + 2]; evy = cur[4 * e + 3]; }
        else { ex = e_lm[2 * (e - N)]; ey = e_lm[2 * (e - N) + 1]; }
        dx = ex - px; dy = ey - py; dvx = evx - vx; dvy = evy - vy;
        dist = r_sqrt(dx * dx + dy * dy);
        fl = s_flag[e];
        nb = dist < p.Rs;
        if (p.own_goal_always && !lsa && e == N + i) nb = true;
        if (dist < si + s_size[e])
          col = (e < N) || (p.cost_obstacles && (fl >> 1) == GSM_ENT_OBSTACLE);
      }
      // neighbour compaction: ballot + popc prefix inside the group
      unsigned bits, cbits;
      if (P == 1) { bits = nb ? 1u : 0u; cbits = col ? 1u : 0u; }
      else {
        const int sh = (lane - sub) & 31;
        bits = (__ballot_sync(grpmask, nb) >> sh) & low_mask(P);
        cbits = (__ballot_sync(grpmask, col) >> sh) & low_mask(P);
      }
      const int pos = cnt + __popc(bits & low_mask(sub));
      if (nb && pos < K) {
        st_idx[pos] = e;
        T* f = st_feat + pos * GSM_NBR_FEAT_DIM;
        f[0] = dx; f[1] = dy; f[2] = dvx; f[3] = dvy; f[4] = dist; f[5] = (T)(fl >> 1);
      }
      cnt += __popc(bits);
      ncol += __popc(cbits);
      // adjacency words: a chunk's entity indices e_lo..e_hi are contiguous (self skipped),
      // ascending from chunk to chunk, and touch at most two 32-bit words.
      const int o_hi = (o0 + P - 1 < E - 2) ? o0 + P - 1 : E - 2;
      const int e_lo = o0 + (o0 >= i ? 1 : 0), e_hi = o_hi + (o_hi >= i ? 1 : 0);
      const int w_lo = e_lo >> 5, w_hi = e_hi >> 5;
      uint32_t c0 = (nb && (e >> 5) == w_lo) ? (1u << (e & 31)) : 0u;
      uint32_t c1 = (nb && (e >> 5) != w_lo) ? (1u << (e & 31)) : 0u;
      if (P > 1) { c0 = __reduce_or_sync(grpmask, c0); c1 = __reduce_or_sync(grpmask, c1); }
      if (w_lo != wcur) {
        if (sub == 0 && p.adj) p.adj[row * W + wcur] = word;
        word = 0; wcur = w_lo;
      }
      word |= c0;
      if (w_hi != w_lo) {
        if (sub == 0 && p.adj) p.adj[row * W + wcur] = word;
        word = c1; wcur = w_hi;
      }
    }
    if (sub == 0 && p.adj) {
      p.adj[row * W + wcur] = word;
      for (int w = wcur + 1; w < W; w++) p.adj[row * W + w] = 0u;
    }
    if (cnt > K) cnt = K;
    for (int k = cnt + sub; k < K; k += P) {
      st_idx[k] = -1;
      T* f = st_feat + k * GSM_NBR_FEAT_DIM;
#pragma unroll
      for (int q = 0; q < GSM_NBR_FEAT_DIM; q++) f[q] = 0;
    }
    if (P > 1) __syncwarp(grpmask);
    if (p.nbr_idx) group_copy<P>(p.nbr_idx + row * K, st_idx, K * 4, sub);
    if (p.nbr_feat)
      group_copy<P>(p.nbr_feat + row * K * GSM_NBR_FEAT_DIM, st_feat, K * GSM_NBR_FEAT_DIM * (int)sizeof(T), sub);
    if (P > 1) __syncwarp(grpmask);          // staging is reused by the group's next agent
    if (sub == 0) {
      T tx, ty;
      int asg = i;
      if (lsa) {
        asg = s_asg[(size_t)env_l * N + i];
        tx = s_slot[((size_t)env_l * N + asg) * 2]; ty = s_slot[((size_t)env_l * N + asg) * 2 + 1];
      } else {
        tx = e_lm[2 * i]; ty = e_lm[2 * i + 1];
      }
      if (p.nbr_cnt) p.nbr_cnt[row] = cnt;
      if (p.assign) p.assign[row] = asg;
      const T gx = tx - px, gy = ty - py;
      if (p.obs) {
        T* o = p.obs + row * GSM_OBS_DIM;
        o[0] = vx; o[1] = vy; o[2] = px; o[3] = py; o[4] = gx; o[5] = gy;
      }
      if (PHYS) {
        const T d = r_sqrt(gx * gx + gy * gy);
        const T r = ((T)0 - p.w_dist * d) + (d < p.goal_tol ? p.w_goal : (T)0);
        if (p.share_reward) e_rew[i] = r;
        else if (p.reward) p.reward[row] = r;
        if (p.cost) p.cost[row] = (T)ncol;
        if (p.done) p.done[row] = (uint8_t)(t_now >= p.episode_length);
      }
    }
  }
  if (PHYS && p.share_reward) {
    if (CTA_ENV) __syncthreads(); else __syncwarp();
    if (p.reward) {
      for (int i = first_agent; i < N; i += agent_stride) {
        if (sub != 0) continue;
        T s = e_rew[0];
        for (int k = 1; k < N; k++) s = s + e_rew[k];
        p.reward[env * N + i] = s / (T)N;
      }
    }
  }
}

// ---- SPEC §8: Philox4x32-10 reset, one thread per (env, entity) --------------------------
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
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
__device__ __forceinline__ double u53(uint32_t hi, uint32_t lo) {
  // (hi53 * 2^26 + lo) / 2^53: the division by a power of two is an exact multiply by 2^-53
  return __dmul_rn(__dadd_rn(__dmul_rn((double)(hi >> 5), 67108864.0), (double)(lo >> 6)),
                   1.0 / 9007199254740992.0);
}

struct ResetParams {
  int64_t n_envs, env_offset;
  int N, L;
  uint64_t seed;
  double ext[4];
  const uint8_t* eflag;
  const uint8_t* mask; int64_t mask_stride;
  void* agent_state; void* lm_pos; int32_t* t; int32_t* episode;
};

template <typename T>
__global__ void reset_kernel(const __grid_constant__ ResetParams p) {
  const int E = p.N + p.L;
  const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid >= p.n_envs * E) return;
  const int64_t env = gid / E;
  const int e = (int)(gid - env * E);
  if (p.mask && p.mask[env * p.mask_stride] == 0) return;
  const uint64_t g = (uint64_t)(p.env_offset + env);
  uint32_t r[4];
  philox4x32_10((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)p.episode[env], (uint32_t)e,
                (uint32_t)p.seed, (uint32_t)(p.seed >> 32), r);
  const double ext = p.ext[p.eflag[e] >> 1];
  // explicit _rn intrinsics: no FMA contraction, also in the fp32 translation unit
  const double x = __dadd_rn(-ext, __dmul_rn(2.0 * ext, u53(r[0], r[1])));
  const double y = __dadd_rn(-ext, __dmul_rn(2.0 * ext, u53(r[2], r[3])));
  if (e < p.N) {
    T* a = (T*)p.agent_state + (env * p.N + e) * 4;
    a[0] = (T)x; a[1] = (T)y; a[2] = 0; a[3] = 0;
  } else {
    T* l = (T*)p.lm_pos + (env * p.L + (e - p.N)) * 2;
    l[0] = (T)x; l[1] = (T)y;
  }
}

// Runs after reset_kernel (stream order): t = 0, episode += 1 for the reset envs.
template <typename T>
__global__ void reset_counters_kernel(int64_t n_envs, const uint8_t* mask, int64_t mask_stride,
                                      int32_t* t, int32_t* episode) {
  const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= n_envs) return;
  if (mask && mask[env * mask_stride] == 0) return;
  t[env] = 0;
  episode[env] += 1;
}

// ---- stand-alone batched LSA: one problem per G-lane group ---------------------------------
template <typename T>
__global__ void lsa_kernel(const T* __restrict__ cost, int32_t* __restrict__ col4row,
                           int64_t n_problems, int n, int G) {
  extern __shared__ __align__(16) unsigned char smem[];
  T* s_c = (T*)smem;
  const int tid = threadIdx.x, lane = tid & 31;
  const int per_cta = blockDim.x / G;
  const int pl = tid / G, col = tid % G;
  const int64_t prob = (int64_t)blockIdx.x * per_cta + pl;
  const int64_t p0 = (int64_t)blockIdx.x * per_cta;
  int64_t np = n_problems - p0;
  np = np > per_cta ? per_cta : np;
  for (int64_t k = tid; k < np * n * n; k += blockDim.x) s_c[k] = cost[p0 * n * n + k];
  __syncthreads();
  if (prob >= n_problems) return;
  const int base = lane - col;
  const unsigned gm = low_mask(G) << (base & 31);
  const int a = lsa_lanes<T>(s_c + (size_t)pl * n * n, n, col, gm, base);
  if (col < n) col4row[prob * n + col] = a;
}

}  // namespace gsm
