// gsm_kernels_wide.cuh — navigation kernel for small teams, "one lane per OTHER entity"
// (SPEC.md §2-8; reference environment.py / core.py / scenarios, SOURCES.txt:14,15,21-22 — withheld).
//
// env_steps_kernel (gsm_kernels_spec.cuh) gives an env N*P lanes: P lanes per agent, every lane
// owning one (agent, other) pair per chunk.  At navigation-3 (E = 9 entities, M = 8 others per
// agent) that is 12 lanes per env, 2 envs and 24 of 32 lanes per warp, and the per-warp overhead
// (cursors, action fetch, shuffles of the other agents' state, role stores) is paid per 2 envs.
// This kernel turns the layout by 90 degrees:
//   * an env owns GW = pow2(M) lanes; lane j is "other number j" of EVERY agent, the agents are the
//     (unrolled) chunks.  M = 8 fills a warp with 4 envs and all 32 lanes;
//   * the env's entities live in a shared-memory table (x, y, vx, vy): lane a < N OWNS agent a — it
//     alone integrates it (state in registers) and publishes it with one 16-byte store; a chunk reads
//     agent i and "its other" with two 16-byte loads.  No shuffle fetches a position, no select chain
//     picks one out of per-lane copies (the first version kept all agents in every lane: 75 of its
//     725 instructions per warp-step were that select chain);
//   * one ballot per agent covers its whole neighbourhood (all 4 envs at once), so the row of a
//     pair is known right after its own chunk — no second pass, no feature registers held;
//   * the contact force of step s+1 is a function of exactly the pair geometry the graph pass of
//     step s computes (same positions, same rounded distance: bit-identical in fp64 too), so the
//     separate force sweep disappears from the steady state: it runs on the first step of a launch
//     and after an in-kernel re-draw only;
//   * lane N-1+i holds agent i's own goal as its landmark, so its chunk-i geometry IS the goal
//     vector and the goal distance: reward and the goal half of obs cost no extra arithmetic;
//   * per-agent constants (size, mass, accel, max_speed, flags) and the staging layout travel in the
//     kernel parameter space; lane constants are chunk-independent (the launcher requires alike
//     agents) and pinned with a self-shuffle so that ptxas cannot rebuild them inside the step loop;
//   * every output of a warp-step is staged in shared memory and leaves as one bulk copy (nbr_feat)
//     plus coalesced 16-byte pieces (see WideSmem below).
// Arithmetic policy, output layout and auto-reset draws are env_steps_kernel's (fp32 softplus: SPEC §9
// deviation 6).  History and measurements: profiles/README.md, round 2.
#pragma once
#include "gsm_kernels_spec.cuh"
#include "gsm_bulk.cuh"

namespace gsm {

constexpr int kWideThreads = 128;
__host__ __device__ constexpr int wide_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }

template <typename T, int N, int E>
struct WideConsts {
  T size[E];
  T mass[N], mass_inv[N], accel[N], maxsp[N];
  int32_t eflag[E];
};

#ifndef GSM_WIDE_BLOCKS        // A/B: resident CTAs per SM the fp32 instance is compiled for
#define GSM_WIDE_BLOCKS 7
#endif
template <typename T> struct WideMinBlocks { static constexpr int value = sizeof(T) == 4 ? GSM_WIDE_BLOCKS : 1; };

// SPEC §3 softplus as ONE code path: max(x, 0) + log1p(exp(-|x|)).  Bit-identical to the two-branch
// form of gsm::softplus (x > 0: x + log1p(exp(-x)); else 0 + log1p(exp(x)) = log1p(exp(x)) exactly).
// fp64: libm exp / log1p, exactly the SPEC's operations.  fp32 (production; SPEC §9 deviation 6): the two
// SFU approximations, ex2.approx and lg2.approx on 1 + y — absolute error <= 2^-21 on softplus, i.e.
// <= contact_margin * 5e-7 on the penetration, far inside the 1e-4 bar (deviation 1 already drops 2.1e-9).
__device__ __forceinline__ float softplus1(float x) {
  float y, l;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(-fabsf(x) * 1.4426950408889634f));
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(1.0f + y));
  return fmaxf(x, 0.f) + 0.6931471805599453f * l;
}
__device__ __forceinline__ double softplus1(double x) { return fmax(x, 0.0) + r_log1p(r_exp(-fabs(x))); }

// Loop-invariant lane constants: ptxas prefers to REBUILD them inside the step loop (S2R, integer
// divisions, indexed constant loads: ~150 instructions per warp-step measured) over holding a register.
// A value that went through a shuffle cannot be rematerialised; it costs one SHFL per launch.
__device__ __forceinline__ int keep(int v) { return __shfl_sync(0xffffffffu, v, threadIdx.x & 31); }
__device__ __forceinline__ unsigned keep(unsigned v) { return __shfl_sync(0xffffffffu, v, threadIdx.x & 31); }
__device__ __forceinline__ float keep(float v) { return __shfl_sync(0xffffffffu, v, threadIdx.x & 31); }
__device__ __forceinline__ double keep(double v) { return __shfl_sync(0xffffffffu, v, threadIdx.x & 31); }

// Shared-memory access through 32-bit shared-space addresses held in (kept) registers: a generic pointer
// into the dynamic array makes ptxas rebuild the shared window base (S2UR + UMOV + ULEA) at every use.
__device__ __forceinline__ void sts(unsigned a, unsigned v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts(unsigned a, int v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts(unsigned a, float v) { asm volatile("st.shared.f32 [%0], %1;" :: "r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void sts(unsigned a, double v) { asm volatile("st.shared.f64 [%0], %1;" :: "r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ void sts2(unsigned a, float x, float y) { asm volatile("st.shared.v2.f32 [%0], {%1, %2};" :: "r"(a), "f"(x), "f"(y) : "memory"); }
__device__ __forceinline__ void sts2(unsigned a, double x, double y) { asm volatile("st.shared.v2.f64 [%0], {%1, %2};" :: "r"(a), "d"(x), "d"(y) : "memory"); }
__device__ __forceinline__ void sts4(unsigned a, float x, float y, float z, float w) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" :: "r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ void sts4(unsigned a, double x, double y, double z, double w) { sts2(a, x, y); sts2(a + 16, z, w); }
__device__ __forceinline__ void lds4(unsigned a, float& x, float& y, float& z, float& w) {
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x), "=f"(y), "=f"(z), "=f"(w) : "r"(a) : "memory");
}
__device__ __forceinline__ void lds4(unsigned a, double& x, double& y, double& z, double& w) {
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(x), "=d"(y) : "r"(a) : "memory");
  asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(z), "=d"(w) : "r"(a + 16) : "memory");
}
// Predicated stores (`@q st.shared`): a lane-dependent or pass-dependent store costs no branch region.
__device__ __forceinline__ void sts_if(bool on, unsigned a, unsigned v) {
  asm volatile("{ .reg .pred q; setp.ne.u32 q, %2, 0; @q st.shared.u32 [%0], %1; }" :: "r"(a), "r"(v), "r"((unsigned)on) : "memory");
}
__device__ __forceinline__ void sts2_if(bool on, unsigned a, float x, float y) {
  asm volatile("{ .reg .pred q; setp.ne.u32 q, %3, 0; @q st.shared.v2.f32 [%0], {%1, %2}; }" :: "r"(a), "f"(x), "f"(y), "r"((unsigned)on) : "memory");
}
__device__ __forceinline__ void sts2_if(bool on, unsigned a, double x, double y) {
  asm volatile("{ .reg .pred q; setp.ne.u32 q, %3, 0; @q st.shared.v2.f64 [%0], {%1, %2}; }" :: "r"(a), "d"(x), "d"(y), "r"((unsigned)on) : "memory");
}
// A select the compiler keeps as one SEL: a chain of ?: on a lane index otherwise becomes a jump table (BRX).
__device__ __forceinline__ unsigned selp(bool c, unsigned a, unsigned b) {
  unsigned r;
  asm("{ .reg .pred q; setp.ne.u32 q, %3, 0; selp.b32 %0, %1, %2, q; }" : "=r"(r) : "r"(a), "r"(b), "r"((unsigned)c));
  return r;
}
// Arith<T>::div computed on every lane, for a result that is then selected: the compiler keeps a volatile asm
// where it stands instead of sinking it into a branch region (fp32: the same div.approx.f32 that __fdividef
// emits, so the same bits).
__device__ __forceinline__ float div_eager(float a, float b) {
  float r; asm volatile("div.approx.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b)); return r;
}
__device__ __forceinline__ double div_eager(double a, double b) { return a / b; }
__device__ __forceinline__ float4 lds16(unsigned a) {
  float4 v; asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory"); return v;
}

template <typename T>
__device__ __forceinline__ T shfl_xor(T v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }

// Shared memory per warp:
//   * entity table [EPW envs][E] of (x, y, vx, vy): lane a < N owns agent a — it alone integrates it and
//     publishes it with one 16-byte store; every chunk reads agent i and "its other" with two 16-byte
//     loads.  No per-lane copies of all agents, no select chains, no position shuffles.
//   * two staging buffers [feat][idx][obs][cnt][adj][assign][reward][cost]: one warp-step's outputs are
//     eight contiguous, 16-byte aligned regions of the slot (env-major layout).  Rows are written with
//     STS; the feature block (77 % of the bytes) leaves as ONE bulk copy (cp.async.bulk.global.shared::cta,
//     UBLKCP) issued by one lane, the small blocks as coalesced 16-byte LDS + STG by a few lanes each.
//     The copies of step s drain while step s+1 is computed.
template <typename T> struct __align__(16) WideEnt { T x, y, vx, vy; };

struct WideSmem {              // byte offsets inside one staging buffer / one warp's block
  unsigned feat, idx, obs, cnt, adj, cost, rew, asg, buf;   // region offsets, buffer size
  unsigned ent, warp;                                         // entity table offset, bytes per warp
};
__host__ __device__ constexpr WideSmem wide_smem_layout(int rb, int N, int E, int K, int EPW) {
  WideSmem w{};
  unsigned o = 0;
  w.feat = o; o += (unsigned)(EPW * N * K * GSM_NBR_FEAT_DIM * rb);
  w.idx = o; o += ((unsigned)(EPW * N * K * 4) + 15u) & ~15u;    // N = 5 with odd K: pad, the vector stores below need 16
  w.obs = o; o += (unsigned)(EPW * N * GSM_OBS_DIM * rb);
  w.cnt = o; o += (unsigned)(EPW * N * 4);
  w.adj = o; o += (unsigned)(EPW * N * 4);
  w.cost = o; o += (unsigned)(EPW * N * rb);
  w.rew = o; o += (unsigned)(EPW * N * rb);
  w.asg = o; o += (unsigned)(EPW * N * 4);
  w.buf = (o + 15u) & ~15u;
  w.ent = 2 * w.buf;
  w.warp = w.ent + (unsigned)(EPW * E * 4 * rb);
  return w;
}
__host__ __device__ constexpr size_t wide_smem_bytes(int rb, int N, int E, int K, int EPW) {
  return (size_t)(kWideThreads / 32) * wide_smem_layout(rb, N, E, K, EPW).warp;
}

// MODE 0: step(s).  MODE 1: observe only (reset path, optional per-env mask).  MODE 2: steps with
// in-kernel auto-reset.  The launcher checks what the kernel assumes: every output pointer non-NULL;
// all agents share one size and one collide flag (the pair constants of a lane are then the same in
// every chunk); n_envs * N * K * 6 * sizeof(T) < 2^31 (32-bit offsets against 64-bit slot bases); in
// fp32 the five 4-byte-per-agent outputs share one slot stride.
// KT > 0: max_nbrs as a compile-time constant (every staging offset becomes an immediate); 0: p.K.
template <typename T, int N, int L, int MODE, int KT>
__global__ void __launch_bounds__(kWideThreads, WideMinBlocks<T>::value)
env_wide_kernel(const __grid_constant__ KParams<T> p, const int n_steps,
                const __grid_constant__ StepStrides ss,
                const __grid_constant__ WideConsts<T, N, N + L> wc,
                const __grid_constant__ WideSmem lay_rt) {
  constexpr int E = N + L, M = E - 1, GW = wide_pow2(M), EPW = 32 / GW;
  constexpr bool OBS = MODE == 1;
  constexpr bool BF = MODE == 2;                       // branch-free chunk body (see the chunk loop)
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int RB = (int)sizeof(T);
  constexpr int RS4 = EPW * N * 4, RST = EPW * N * RB;      // bytes of a per-agent 4-byte / real block of the warp
  // the per-agent scalar blocks of a warp-step leave in PS-byte pieces, one per lane (16 where the blocks allow, else 8)
  constexpr int PS = (RS4 % 16 == 0 && RST % 16 == 0) ? 16 : 8;
  constexpr int PC4 = RS4 / PS, PCT = RST / PS, NPIECE = 3 * PC4 + 2 * PCT;
  constexpr bool ROLE_OK = NPIECE <= 32;                   // else (N = 5 in fp64): the word-wise path
  static_assert(GW <= 32 && E <= 32, "an env must fit in one warp, adjacency in one word");
  static_assert(L >= N && 2 * N <= GW + 1 && N >= 3, "goal i is landmark i, held by lane N-1+i; lanes 0..2 stage scalars");
  static_assert(RS4 % 8 == 0 && RST % 8 == 0, "per-warp scalar blocks leave in 8- or 16-byte pieces");
  static_assert(EPW * N * M * 4 / 16 <= 64 && EPW * N * GSM_OBS_DIM * RB / 16 <= 64, "idx / obs blocks leave in <= 2 passes");
  typedef Arith<T> A;
  typedef WideEnt<T> Ent;
  typedef float4 V;                                        // a 16-byte piece
  extern __shared__ __align__(128) unsigned char wsm[];
  const int K = KT > 0 ? KT : p.K;
  const WideSmem lay = KT > 0 ? wide_smem_layout((int)sizeof(T), N, N + L, KT > 0 ? KT : 1, 32 / wide_pow2(N + L - 1)) : lay_rt;
  const int lane = keep((int)(threadIdx.x & 31)), warp = threadIdx.x >> 5;
  const int grp = lane / GW, j = lane % GW, shift = grp * GW;
  const int env_w0 = keep((int)(((int64_t)blockIdx.x * (kWideThreads / 32) + warp) * EPW));
  bool active = env_w0 + grp < p.n_envs;
  if (OBS && p.mask != nullptr && active) active = p.mask[(int64_t)(env_w0 + grp) * p.mask_stride] != 0;
  // idle groups read only env 0's actions (an input), start from a dummy state and never store (below)
  const int env = active ? env_w0 + grp : 0;
  const bool has = M == GW ? true : j < M;
  const bool own = j < N;                               // I own (integrate, publish) agent j
  const int ja = own ? j : 0;
  const unsigned act_bits = __ballot_sync(FULL, active);
  // staged bulk path: the warp's EPW envs all exist (and are unmasked) and every slot is 16-byte aligned
  const bool bulk = ROLE_OK && act_bits == FULL && ((EPW * N * K * 4) & 15) == 0 &&
      ((((uintptr_t)p.obs | (uintptr_t)p.nbr_idx | (uintptr_t)p.nbr_feat | (uintptr_t)p.nbr_cnt | (uintptr_t)p.adj |
         (uintptr_t)p.assign | (uintptr_t)p.reward | (uintptr_t)p.cost | (uintptr_t)ss.obs | (uintptr_t)ss.nbr_idx |
         (uintptr_t)ss.nbr_feat | (uintptr_t)ss.nbr_cnt | (uintptr_t)ss.adj | (uintptr_t)ss.assign |
         (uintptr_t)ss.reward | (uintptr_t)ss.cost) & 15) == 0);

  constexpr unsigned ES = (unsigned)sizeof(Ent);
  const unsigned sa_w = keep(smem_u32(wsm) + (unsigned)warp * lay.warp);                 // my warp's block (shared-space address)
  const unsigned sa_ent = keep(smem_u32(wsm) + (unsigned)warp * lay.warp + lay.ent + (unsigned)(grp * E) * ES);   // my env's entity table

  // ---- lane constants: my "other" is an agent in every chunk (j < N-1) or landmark j+1-N in every
  //      chunk, and the agents are alike, so its size / type / flags do not depend on the chunk ----------
  const int e_hi = has ? j + 1 : 0;                      // the other in chunks i <= j (i > j: e_hi - 1)
  const int fl_o = wc.eflag[e_hi];
  const T size_o = keep(wc.size[e_hi]), type_o = keep((T)(fl_o >> 1));
  // bit 0: contact pair, bit 1: counts as a collision, bits 8..: chunk in which my landmark is the agent's own goal (+1)
  const unsigned lfl = keep((unsigned)((has && (wc.eflag[0] & 1) && (fl_o & 1)) ? 1u : 0u) |
                            ((has && (e_hi < N || (p.cost_obstacles && (fl_o >> 1) == GSM_ENT_OBSTACLE))) ? 2u : 0u) |
                            (((has && p.own_goal_always && j >= N - 1 && j < 2 * N - 1) ? (unsigned)(j - (N - 1) + 1) : 0u) << 8));
  const bool cpair = lfl & 1u, colc = lfl & 2u;
  const int goal_i = (int)(lfl >> 8) - 1;

  // ---- state: my own agent in registers, everything in the entity table ---------------------------
  // An idle group starts with every entity at rest at the origin and t = 0.  Its values then evolve (t counts up,
  // coincident entities give NaN forces) but stay inside the group: `fin` and the episode-end minimum mask on
  // `active`, the force butterfly runs within the group, and every store is predicated on `active` / act_bits.
  T mx = 0, my = 0, mvx = 0, mvy = 0;
  if (active) {
    const T* a = p.agent_state + ((int64_t)env * N + ja) * 4;
    mx = a[0]; my = a[1]; mvx = a[2]; mvy = a[3];
  }
  if (own) sts4(sa_ent + (unsigned)j * ES, mx, my, mvx, mvy);
  if (has && j + 1 >= N) {                               // lane j also holds landmark j + 1 - N
    T lx = 0, ly = 0;
    if (active) { const T* l = p.lm_pos + ((int64_t)env * L + (j + 1 - N)) * 2; lx = l[0]; ly = l[1]; }
    sts4(sa_ent + (unsigned)(j + 1) * ES, lx, ly, (T)0, (T)0);
  }
  int t_now = active ? p.t[env] : 0;
  const bool auto_reset = MODE == 2 && p.auto_reset != 0;
  const T accel_m = keep(wc.accel[ja]), mass_m = keep(wc.mass[ja]), massinv_m = keep(wc.mass_inv[ja]), maxsp_m = keep(wc.maxsp[ja]);

  // ---- slot bases (warp-uniform), offsets of this warp / this lane ------------------------------------
  const unsigned char* b_act = (const unsigned char*)p.actions;
  unsigned char* b_obs = (unsigned char*)p.obs;
  unsigned char* b_idx = (unsigned char*)p.nbr_idx;
  unsigned char* b_feat = (unsigned char*)p.nbr_feat;
  unsigned char* b_done = (unsigned char*)p.done;
  const unsigned wrow0 = (unsigned)env_w0 * N;          // first agent row of the warp
  // the five per-agent scalar blocks leave as 16-byte pieces, staged contiguously in piece order
  // (cnt, adj, cost, reward, assign): lane q owns piece q
  unsigned char* c_role = nullptr;                       // my piece in global memory (advanced by its array's stride)
  int64_t role_stride = ss.nbr_cnt;                      // fp32: one stride for all five (launcher-checked)
  {
    const int q = lane;
    if (q < PC4) c_role = (unsigned char*)p.nbr_cnt + wrow0 * 4u + q * PS;
    else if (q < 2 * PC4) { c_role = (unsigned char*)p.adj + wrow0 * 4u + (q - PC4) * PS; if (RB != 4) role_stride = ss.adj; }
    else if (q < 2 * PC4 + PCT) { c_role = (unsigned char*)p.cost + wrow0 * (unsigned)RB + (q - 2 * PC4) * PS; if (RB != 4) role_stride = ss.cost; }
    else if (q < 2 * PC4 + 2 * PCT) { c_role = (unsigned char*)p.reward + wrow0 * (unsigned)RB + (q - 2 * PC4 - PCT) * PS; if (RB != 4) role_stride = ss.reward; }
    else if (q < NPIECE) { c_role = (unsigned char*)p.assign + wrow0 * 4u + (q - 2 * PC4 - 2 * PCT) * PS; if (RB != 4) role_stride = ss.assign; }
  }
  const bool role_on = lane < NPIECE && (!OBS || lane < 2 * PC4 || lane >= 2 * PC4 + 2 * PCT);
  // assign[i] = i never changes: both staging buffers get it once
  if (own) {
    sts(sa_w + lay.asg + (unsigned)(grp * N + j) * 4u, j);
    sts(sa_w + lay.buf + lay.asg + (unsigned)(grp * N + j) * 4u, j);
  }

  // action of my own agent, prefetched one step ahead
  const bool discrete = p.action_mode == GSM_ACT_DISCRETE;
  const unsigned act_off = keep(discrete ? ((unsigned)env * N + ja) * 4u : ((unsigned)env * N + ja) * 2u * (unsigned)RB);
  // 16-byte pieces of the idx / obs blocks: byte offsets of my piece in the slot and in the staging buffer
  const unsigned n_idx = (lay.obs - lay.idx) / 16, n_obs = (lay.cnt - lay.obs) / 16;
  const unsigned off_idx = keep(wrow0 * (unsigned)(K * 4) + (unsigned)lane * 16u), off_obs = keep(wrow0 * (unsigned)(GSM_OBS_DIM * RB) + (unsigned)lane * 16u);
  const unsigned off_done = keep((unsigned)env * N + (unsigned)ja);
  int act_next = 0;
  T actx_next = 0, acty_next = 0;
  if (!OBS) {
    if (discrete) act_next = *(const int32_t*)(b_act + act_off);
    else { actx_next = ((const T*)(b_act + act_off))[0]; acty_next = ((const T*)(b_act + act_off))[1]; }
  }
  __syncwarp();

  T fox = 0, foy = 0;                                    // contact force on my own agent for the NEXT integration
  // `pro` (warp-uniform): a prologue pass — geometry and contact forces of the CURRENT positions only,
  // no integration, no outputs, no step consumed.  The first pass of a launch and the pass after an
  // in-kernel re-draw are prologues; every other pass is one env step.  One copy of the code serves both.
  bool pro = !OBS;
  int step = 0;
  // staging buffer of the next output step: a loop-CARRIED address flipped by +-lay.buf (ptxas re-derives
  // `sa_w + offset` at every use when it can; it cannot re-derive a carried value)
  unsigned sb = sa_w;
  int sb_delta = (int)lay.buf;
  // lane-constant parts of my staging addresses (feature rows, idx rows, scalar role, obs rows of my env)
  const unsigned o_feat = keep((unsigned)(grp * N * K) * (unsigned)(GSM_NBR_FEAT_DIM * RB));
  const unsigned o_idx = keep(lay.idx + (unsigned)(grp * N * K) * 4u);
  const unsigned o_sc = keep(lay.cnt + (unsigned)(j < 3 ? j : 0) * (unsigned)RS4 + (unsigned)(grp * N) * 4u);
  const unsigned o_obs = keep(lay.obs + (unsigned)grp * (unsigned)(N * GSM_OBS_DIM * RB));
  // The hot loop runs up to step `stop` (warp-uniform): the launch's end or, with auto-reset, the first step
  // after which an env of the warp ends its episode (at least one step: an env that starts at or past its
  // episode's end is re-drawn after one).  It is counted once here and after every re-draw, so the loop has
  // no per-step vote.  Idle groups never end an episode.
  const auto segment_end = [&]() {
    int s = n_steps;
    if (MODE == 2 && auto_reset) {
      const int left = __reduce_min_sync(FULL, active ? p.episode_length - t_now : INT_MAX);
      s = step + max(1, min(left, n_steps - step));
    }
    return s;
  };
  int stop = segment_end();
  while (step < n_steps) {
   // hot loop: runs until `stop`
   for (;;) {
    if (!OBS && !pro) {
      // ---- SPEC §2 + §4 for my own agent (lanes j >= N integrate values that are never used or published) -
      T ux = actx_next, uy = acty_next;
      if (discrete) {
        const int a = act_next;
        ux = 0; uy = 0;
        if (a >= 0 && a < p.n_actions) { ux = p.discrete_u[a][0]; uy = p.discrete_u[a][1]; }
      }
      if (step + 1 < n_steps) b_act += ss.actions;      // the last step re-reads its own, valid, address
      if (discrete) act_next = *(const int32_t*)(b_act + act_off);
      else { actx_next = ((const T*)(b_act + act_off))[0]; acty_next = ((const T*)(b_act + act_off))[1]; }
      const T fx = accel_m * ux + fox, fy = accel_m * uy + foy;
      T nvx = mvx * p.one_minus_damp, nvy = mvy * p.one_minus_damp;
      nvx = nvx + A::div_const(fx, mass_m, massinv_m) * p.dt;
      nvy = nvy + A::div_const(fy, mass_m, massinv_m) * p.dt;
      if (maxsp_m > (T)0) {
        const T sp = A::sqrt(nvx * nvx + nvy * nvy);
        if (sp > maxsp_m) { nvx = A::div(nvx, sp) * maxsp_m; nvy = A::div(nvy, sp) * maxsp_m; }
      }
      mvx = nvx; mvy = nvy;
      mx = mx + nvx * p.dt; my = my + nvy * p.dt;
      t_now += 1;
      if (own) sts4(sa_ent + (unsigned)j * ES, mx, my, mvx, mvy);
      __syncwarp();
    }
    const bool st_on = !pro;                             // warp-uniform: this pass produces outputs
    const unsigned a_feat = sb + o_feat, a_idx = sb + o_idx, a_sc = sb + o_sc, sobs = sb + o_obs;
    // the bulk copy that read this buffer two steps ago must have finished reading it; the first
    // ballot below orders every lane's STS behind lane 0's wait
    if (st_on && bulk && lane == 0) bulk_wait_read<1>();

    // ---- SPEC §6-7: one chunk per agent; the pair's row is known after the chunk's own ballot -----
    T fcx[N], fcy[N];
    T gxs = 0, gys = 0, gd = 0;                          // lane N-1+i: goal vector / distance of agent i
    bool anyc = false;
#pragma unroll
    for (int i = 0; i < N; i++) {
      const int e = e_hi - (j < i ? 1 : 0);
      Ent si, so;
      lds4(sa_ent + (unsigned)i * ES, si.x, si.y, si.vx, si.vy);
      lds4(sa_ent + (unsigned)e * ES, so.x, so.y, so.vx, so.vy);
      const T dx = so.x - si.x, dy = so.y - si.y;
      const T dist = A::sqrt(dx * dx + dy * dy);
      const T dmin = wc.size[i] + size_o;
      const bool nb = (has && dist < p.Rs) || goal_i == i;
      const bool col = colc && dist < dmin;
      const unsigned bits = (__ballot_sync(FULL, nb) >> shift) & low_mask(GW);
      const unsigned cbits = (__ballot_sync(FULL, col) >> shift) & low_mask(GW);
      int cnt = __popc(bits);
      const int rank = __popc(bits & low_mask(j));
      const int pos = nb ? rank : cnt + (j - rank);
      // Two forms of the same stores and the same contact term, chosen per instance.  BF (auto-reset): every
      // lane writes its pair's row (values or zeros, by selects) and the scalars with predicated stores, and
      // computes the contact term and selects it — no branch regions.  Otherwise the branchy form: in the
      // plain / observe instances the branch-free one costs a register and a spill (<float,3,6,0,8>: 71 -> 72
      // registers, an 8 B stack) and runs 9 % slower as one launch (profiles/README.md, w7).
      if (BF) {
        // with K >= M every row lands inside the agent's K rows
        const bool row_on = st_on && has && (KT >= M || pos < K);
        sts_if(row_on, a_idx + (unsigned)pos * 4u + (unsigned)(i * K * 4), (unsigned)(nb ? e : -1));
        const unsigned f = a_feat + (unsigned)pos * (unsigned)(GSM_NBR_FEAT_DIM * RB) + (unsigned)(i * K * GSM_NBR_FEAT_DIM * RB);
        const T z = (T)0;
        sts2_if(row_on, f, nb ? dx : z, nb ? dy : z);
        sts2_if(row_on, f + 2 * RB, nb ? so.vx - si.vx : z, nb ? so.vy - si.vy : z);
        sts2_if(row_on, f + 4 * RB, nb ? dist : z, nb ? type_o : z);
      } else if (has && pos < K && st_on) {
        sts(a_idx + (unsigned)pos * 4u + (unsigned)(i * K * 4), nb ? e : -1);
        const unsigned f = a_feat + (unsigned)pos * (unsigned)(GSM_NBR_FEAT_DIM * RB) + (unsigned)(i * K * GSM_NBR_FEAT_DIM * RB);
        const T z = (T)0;
        if (nb) { sts2(f, dx, dy); sts2(f + 2 * RB, so.vx - si.vx, so.vy - si.vy); sts2(f + 4 * RB, dist, type_o); }
        else { sts2(f, z, z); sts2(f + 2 * RB, z, z); sts2(f + 4 * RB, z, z); }
      }
      if (cnt > K) cnt = K;
      // entity-indexed adjacency: open a zero bit at the agent's own index i
      const unsigned ebits = (bits & low_mask(i)) | ((bits & ~low_mask(i)) << 1);
      if (BF && RB == 4) {                                // lanes 0, 1, 2 stage cnt, adj, cost of agent i: three
        const unsigned v = selp(j == 0, (unsigned)cnt, selp(j == 1, ebits, __float_as_uint((float)__popc(cbits))));
        sts_if(st_on && j < 3, a_sc + (unsigned)(i * 4), v);   // equal 4-byte blocks, one store
      } else if (st_on && j < 3) {
        const unsigned ao = (unsigned)(grp * N + i);
        if (RB == 4) {
          const unsigned v = j == 0 ? (unsigned)cnt : (j == 1 ? ebits : __float_as_uint((float)__popc(cbits)));
          if (!OBS || j < 2) sts(a_sc + (unsigned)(i * 4), v);
        } else {
          if (j == 0) sts(sb + lay.cnt + ao * 4u, cnt);
          else if (j == 1) sts(sb + lay.adj + ao * 4u, ebits);
          else if (!OBS) sts(sb + lay.cost + ao * (unsigned)RB, (T)__popc(cbits));
        }
      }
      if (j == N - 1 + i) { gxs = dx; gys = dy; gd = dist; }   // my landmark is this agent's goal
      if (BF) {                                           // SPEC §3 for the next step, on the same geometry:
        // the force uses p_i - p_e = -d, exactly
        const T x = A::div_const(-(dist - dmin), p.km, p.km_inv);
        const bool term = cpair && !(Prec<T>::kCut && x < (T)(-kFarCut));
        const T pen = softplus1(x) * p.km;
        const T qx = div_eager(p.cf * (-dx), dist), qy = div_eager(p.cf * (-dy), dist);
        fcx[i] = term ? qx * pen : (T)0;
        fcy[i] = term ? qy * pen : (T)0;
        anyc = anyc || term;
      } else if (!OBS) {
        fcx[i] = 0; fcy[i] = 0;
        if (cpair) {
          const T x = A::div_const(-(dist - dmin), p.km, p.km_inv);
          if (!(Prec<T>::kCut && x < (T)(-kFarCut))) {
            const T pen = softplus1(x) * p.km;
            fcx[i] = A::div(p.cf * (-dx), dist) * pen;
            fcy[i] = A::div(p.cf * (-dy), dist) * pen;
            anyc = true;
          }
        }
      }
    }
    // Contact forces: butterfly all-reduce over the env's GW lanes (IEEE addition commutes: every lane of
    // the group ends with the same bits), each owner keeps its agent's sum.  All-zero partials sum to
    // exactly zero, so the butterfly is skipped when no lane of the warp has a term.
    if (!OBS && (pro || step + 1 < n_steps)) {
      fox = 0; foy = 0;
      if (__any_sync(FULL, anyc)) {
#pragma unroll
        for (int m = GW / 2; m >= 1; m >>= 1) {
#pragma unroll
          for (int i = 0; i < N; i++) { fcx[i] = fcx[i] + shfl_xor(fcx[i], m); fcy[i] = fcy[i] + shfl_xor(fcy[i], m); }
        }
#pragma unroll
        for (int i = 0; i < N; i++) if (ja == i) { fox = fcx[i]; foy = fcy[i]; }
      }
    }

    if (st_on) {
      // ---- per-agent outputs --------------------------------------------------------------------------
      if (own) { sts2(sobs + (unsigned)j * (GSM_OBS_DIM * RB), mvx, mvy); sts2(sobs + (unsigned)j * (GSM_OBS_DIM * RB) + 2 * RB, mx, my); }
      T rs = ((T)0 - p.w_dist * gd) + (gd < p.goal_tol ? p.w_goal : (T)0);
      if (p.share_reward && !OBS) {
        T s = shfl(FULL, rs, shift + N - 1);
#pragma unroll
        for (int k = 1; k < N; k++) s = s + shfl(FULL, rs, shift + N - 1 + k);
        rs = s / (T)N;
      }
      if (j >= N - 1 && j < 2 * N - 1) {
        const unsigned ao = (unsigned)(j - (N - 1));
        sts2(sobs + ao * (GSM_OBS_DIM * RB) + 4 * RB, gxs, gys);
        if (!OBS) sts(sb + lay.rew + ((unsigned)grp * N + ao) * (unsigned)RB, rs);
      }
      if (!OBS && own && active) b_done[off_done] = (uint8_t)(t_now >= p.episode_length);
      // ---- the staged blocks leave -----------------------------------------------------------------------
      if (bulk) {
        fence_async_smem();
        __syncwarp();
        if (lane == 0) {
          asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                       :: "l"(b_feat + wrow0 * (unsigned)(K * GSM_NBR_FEAT_DIM * RB)), "r"(sb), "r"(lay.idx) : "memory");
          bulk_commit();
        }
        V* const g_idx = (V*)(b_idx + off_idx);
        V* const g_obs = (V*)(b_obs + off_obs);
        const unsigned s_idx = sb + lay.idx + (unsigned)lane * 16u, s_obs = sb + lay.obs + (unsigned)lane * 16u;
        if (lane < n_idx) g_idx[0] = lds16(s_idx);
        if (lane + 32 < n_idx) g_idx[32] = lds16(s_idx + 512);
        if (lane < n_obs) g_obs[0] = lds16(s_obs);
        if (lane + 32 < n_obs) g_obs[32] = lds16(s_obs + 512);
        if (role_on) {
          if (PS == 16) *(V*)c_role = lds16(sb + lay.cnt + (unsigned)lane * 16u);
          else {
            float2 v8;
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v8.x), "=f"(v8.y) : "r"(sb + lay.cnt + (unsigned)lane * 8u) : "memory");
            *(float2*)c_role = v8;
          }
        }
      } else {
        // ragged / masked / unaligned warps: word-wise, per-env predicated
        __syncwarp();
        auto copy_words = [&](unsigned char* g, unsigned soff, unsigned bytes) {
          const unsigned wpe = bytes / (4 * EPW);         // words per env
          for (unsigned q = lane; q < bytes / 4; q += 32)
            if ((act_bits >> ((q / wpe) * GW)) & 1u) {
              unsigned v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(sb + soff + q * 4u) : "memory");
              ((uint32_t*)g)[q] = v;
            }
        };
        copy_words(b_feat + wrow0 * (unsigned)(K * GSM_NBR_FEAT_DIM * RB), lay.feat, lay.idx - lay.feat);
        copy_words(b_idx + wrow0 * (unsigned)(K * 4), lay.idx, (unsigned)(EPW * N * K * 4));
        copy_words(b_obs + wrow0 * (unsigned)(GSM_OBS_DIM * RB), lay.obs, lay.cnt - lay.obs);
        copy_words((unsigned char*)p.nbr_cnt + (int64_t)step * ss.nbr_cnt + wrow0 * 4u, lay.cnt, RS4);
        copy_words((unsigned char*)p.adj + (int64_t)step * ss.adj + wrow0 * 4u, lay.adj, RS4);
        copy_words((unsigned char*)p.assign + (int64_t)step * ss.assign + wrow0 * 4u, lay.asg, RS4);
        if (!OBS) {
          copy_words((unsigned char*)p.reward + (int64_t)step * ss.reward + wrow0 * (unsigned)RB, lay.rew, RST);
          copy_words((unsigned char*)p.cost + (int64_t)step * ss.cost + wrow0 * (unsigned)RB, lay.cost, RST);
        }
        __syncwarp();
      }
    }
    if (OBS) break;
    if (pro) { pro = false; continue; }                  // the prologue consumed no step
    b_obs += ss.obs; b_idx += ss.nbr_idx; b_feat += ss.nbr_feat; b_done += ss.done;
    c_role += role_stride;
    sb += sb_delta;
    sb_delta = -sb_delta;
    step++;
    if (step >= stop) break;
   }
   if (OBS) break;
   // ---- episode end inside a fused rollout: re-draw (the terminal outputs stay in their slot).  Cold:
   //      outside the hot loop, which it costs nothing ------------------------------------------------------
   if (MODE == 2 && auto_reset) {
     const bool fin = active && t_now >= p.episode_length;
     if (__any_sync(FULL, fin)) {
       __syncwarp();                                      // every lane has read the old table
       int ep = 0;
       if (fin) {
         // the episode counter and the landmarks are not held in registers across the hot loop: both are
         // read / written in global memory right here (once per episode).  Lane j draws entities j, j + GW,
         // ... (navigation-3: 9 entities on 8 lanes, two rounds), inline: no call, no stack frame
         const uint64_t genv = (uint64_t)(p.env_offset + env);
         ep = p.episode[env];
#pragma unroll 1
         for (int e = j; e < E; e += GW) {
           double dx, dy;
           spawn_draw_inline(genv, ep, e, p.seed, p.ext[wc.eflag[e] >> 1], dx, dy);
           const T x = (T)dx, y = (T)dy;
           sts4(sa_ent + (unsigned)e * ES, x, y, (T)0, (T)0);
           if (e < N) { mx = x; my = y; }                 // e = j: my own agent
           else { T* l = p.lm_pos + ((int64_t)env * L + (e - N)) * 2; l[0] = x; l[1] = y; }
         }
         mvx = 0; mvy = 0;
         t_now = 0;
       }
       __syncwarp();                                      // every lane of the env has read the old counter
       if (fin && j == 0) p.episode[env] = ep + 1;
       __syncwarp();
       pro = step < n_steps;                              // the new positions need their forces
       stop = segment_end();
     }
   }
  }
  if (bulk && lane == 0) bulk_wait_read<0>();            // shared memory must outlive the copy that reads it

  // ---- state back to HBM ------------------------------------------------------------------------------
  if (!OBS && active) {
    if (own) {
      T* a = p.agent_state + ((int64_t)env * N + j) * 4;
      st2<T>(a, mx, my); st2<T>(a + 2, mvx, mvy);
    }
    if (j == 0) p.t[env] = t_now;
  }
}

}  // namespace gsm
