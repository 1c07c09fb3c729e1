// gsm_api.cu — the C ABI of include/gsmarl_b200.h.
//
// Stands in for the vectorised-env boundary of the reference (env_wrappers.py /
// make_env.py / environment.py, GSMARL.egg-info/SOURCES.txt:11,12,15 — withheld).
// No torch types, no CPU fallback: every entry point either launches the sm_100a
// kernels of gsm_kernels.cuh or returns an error.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/gsmarl_b200.h"
#include "gsm_host.h"

namespace {

enum { IO_ACTIONS = 0, IO_OBS, IO_NBR_IDX, IO_NBR_FEAT, IO_NBR_CNT, IO_ADJ, IO_REWARD, IO_COST,
       IO_DONE, IO_ASSIGN, IO_COUNT };

thread_local std::string g_create_err;

void* io_get(const gsm_step_io& io, int k) {
  switch (k) {
    case IO_ACTIONS: return const_cast<void*>(io.actions);
    case IO_OBS: return io.obs;
    case IO_NBR_IDX: return io.nbr_idx;
    case IO_NBR_FEAT: return io.nbr_feat;
    case IO_NBR_CNT: return io.nbr_cnt;
    case IO_ADJ: return io.adj;
    case IO_REWARD: return io.reward;
    case IO_COST: return io.cost;
    case IO_DONE: return io.done;
    default: return io.assign;
  }
}
void io_set(gsm_step_io& io, int k, void* p) {
  switch (k) {
    case IO_ACTIONS: io.actions = p; break;
    case IO_OBS: io.obs = p; break;
    case IO_NBR_IDX: io.nbr_idx = (int32_t*)p; break;
    case IO_NBR_FEAT: io.nbr_feat = p; break;
    case IO_NBR_CNT: io.nbr_cnt = (int32_t*)p; break;
    case IO_ADJ: io.adj = (uint32_t*)p; break;
    case IO_REWARD: io.reward = p; break;
    case IO_COST: io.cost = p; break;
    case IO_DONE: io.done = (uint8_t*)p; break;
    default: io.assign = (int32_t*)p; break;
  }
}

}  // namespace

struct gsm_env {
  gsm::HostParams hp;
  gsm::LaunchPlan plan;
  int dtype, device, rb;
  gsm_io_sizes sz;
  size_t io_bytes[IO_COUNT];
  std::vector<void*> dev_allocs;
  cudaStream_t stream = nullptr;
  // host path: one device arena + one pinned arena, sub-buffers 256-B aligned
  unsigned char* d_arena = nullptr;
  unsigned char* h_arena = nullptr;
  size_t arena_off[IO_COUNT], arena_total = 0, arena_out_begin = 0;
  gsm_step_io d_io, h_io;
  uint8_t* d_mask = nullptr;
  // sparse export (arena host path): the pinned arena is MAPPED; a kernel writes the step's outputs into it
  // over PCIe and skips the padding rows of nbr_feat / nbr_idx (host rows >= cnt already hold 0 / -1)
  unsigned char* h_arena_dev = nullptr;   // device address of h_arena
  int32_t* d_prev_cnt = nullptr;          // [n_envs*N] neighbour rows the host copy currently holds per agent
  unsigned char* d_shadow = nullptr;      // device-side copy of what the host arena holds (same offsets): slowly
                                          // changing outputs leave as the 16-byte pieces that differ from it
  int host_sparse = 1;                    // GSM_HOST_DENSE=1 / gsm_set_host_outputs(..., sparse = 0): one dense D2H copy instead
  uint32_t host_out_mask = 0xffffffffu;   // bit k: output k (gsm_io index) is delivered to the host by the *_host calls
  int host_resync = 1;                    // next arena copy-out is dense and re-bases d_prev_cnt
  // rollout graph cache (one entry)
  cudaGraphExec_t graph_exec = nullptr;
  int graph_steps = 0;
  gsm_step_io graph_io;
  uint64_t graph_seed = 0;       // the captured reset_kernel launches carry the seed BY VALUE
  int graph_auto_reset = 0;
  int64_t launches = 0;
  uint64_t seed = 0;
  int auto_reset = 0;      // gsm_set_auto_reset: applies inside gsm_rollout only
  int64_t slot_envs = 0;   // gsm_set_slot_envs: envs per slot of the caller's [T][...] buffers (0: n_envs)
  std::string err;
};

namespace {

int fail(gsm_env* h, int status, const std::string& msg) {
  if (h) h->err = msg; else g_create_err = msg;
  return status;
}
int cuda_fail(gsm_env* h, int e, const char* what) {
  return fail(h, GSM_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString((cudaError_t)e));
}
#define GSM_CUDA(h, call)                                       \
  do {                                                          \
    cudaError_t e__ = (call);                                   \
    if (e__ != cudaSuccess) return cuda_fail(h, (int)e__, #call); \
  } while (0)

template <typename T>
int upload(gsm_env* h, const double* src, size_t n, void** out) {
  std::vector<T> tmp(n);
  for (size_t i = 0; i < n; i++) tmp[i] = (T)src[i];
  void* d = nullptr;
  GSM_CUDA(h, cudaMalloc(&d, n * sizeof(T) + 16));
  h->dev_allocs.push_back(d);
  GSM_CUDA(h, cudaMemcpy(d, tmp.data(), n * sizeof(T), cudaMemcpyHostToDevice));
  *out = d;
  return 0;
}
int upload_real(gsm_env* h, const double* src, size_t n, void** out) {
  return h->dtype == GSM_F32 ? upload<float>(h, src, n, out) : upload<double>(h, src, n, out);
}
int dev_alloc(gsm_env* h, size_t bytes, void** out) {
  void* d = nullptr;
  GSM_CUDA(h, cudaMalloc(&d, bytes + 16));
  GSM_CUDA(h, cudaMemset(d, 0, bytes + 16));
  h->dev_allocs.push_back(d);
  *out = d;
  return 0;
}

std::string validate(const gsm_config* c) {
  if (!c) return "cfg is NULL";
  if (c->struct_size != sizeof(gsm_config)) return "cfg.struct_size != sizeof(gsm_config)";
  if (c->abi_version != GSM_ABI_VERSION) return "cfg.abi_version mismatch";
  if (c->dtype != GSM_F32 && c->dtype != GSM_F64) return "cfg.dtype must be GSM_F32 or GSM_F64";
  if (c->scenario < GSM_SCN_NAVIGATION || c->scenario > GSM_SCN_LINE) return "unknown cfg.scenario";
  if (c->action_mode != GSM_ACT_DISCRETE && c->action_mode != GSM_ACT_CONTINUOUS) return "unknown cfg.action_mode";
  const int N = c->n_agents, L = c->n_landmarks, E = N + L;
  if (N < 1) return "n_agents must be >= 1";
  if (L < 0) return "n_landmarks must be >= 0";
  if (E > 1024) return "n_agents + n_landmarks must be <= 1024";
  if (c->max_nbrs < 1 || c->max_nbrs > (E > 1 ? E - 1 : 1)) return "max_nbrs must be in [1, N+L-1]";
  if (c->episode_length < 1) return "episode_length must be >= 1";
  if (!(c->dt > 0)) return "dt must be > 0";
  if (!(c->contact_margin > 0)) return "contact_margin must be > 0";
  if (!(c->damping >= 0 && c->damping <= 1)) return "damping must be in [0, 1]";
  if (!(c->sensing_radius >= 0)) return "sensing_radius must be >= 0";
  if (!std::isfinite(c->contact_force) || !std::isfinite(c->w_dist) || !std::isfinite(c->w_goal) ||
      !std::isfinite(c->goal_tol) || !std::isfinite(c->polygon_radius))
    return "non-finite scalar in cfg";
  if (!c->size || !c->collide || !c->type || !c->mass || !c->accel || !c->max_speed)
    return "size/collide/type/mass/accel/max_speed must not be NULL";
  if (c->action_mode == GSM_ACT_DISCRETE) {
    if (c->n_discrete_actions < 1 || c->n_discrete_actions > GSM_MAX_DISCRETE) return "n_discrete_actions out of range";
    if (!c->discrete_u) return "discrete_u must not be NULL";
  }
  for (int e = 0; e < E; e++) {
    if (c->type[e] < GSM_ENT_AGENT || c->type[e] > GSM_ENT_MARKER) return "entity type out of range";
    if ((e < N) != (c->type[e] == GSM_ENT_AGENT)) return "agents must be exactly the first n_agents entities";
    if (!(c->size[e] >= 0)) return "entity size must be >= 0";
  }
  for (int i = 0; i < N; i++)
    if (!(c->mass[i] > 0)) return "mass must be > 0";
  for (int k = 0; k < 4; k++)
    if (!(c->spawn_extent[k] >= 0)) return "spawn_extent must be >= 0";
  if (c->scenario == GSM_SCN_NAVIGATION) {
    if (L < N) return "navigation needs one goal per agent (n_landmarks >= n_agents)";
    for (int i = 0; i < N; i++)
      if (c->type[N + i] != GSM_ENT_GOAL) return "navigation: landmarks 0..N-1 must be goals";
  } else {
    if (N > GSM_MAX_LSA_N) return "polygon/line: n_agents must be <= GSM_MAX_LSA_N";
    if (!c->slot_table) return "polygon/line: slot_table must not be NULL";
    if (c->scenario == GSM_SCN_POLYGON && L != 1) return "polygon needs exactly 1 landmark";
    if (c->scenario == GSM_SCN_LINE && L != 2) return "line needs exactly 2 landmarks";
  }
  return "";
}

bool is_f32(const gsm_env* h) { return h->dtype == GSM_F32; }

int do_env(gsm_env* h, const gsm_step_io& io, int physics, const uint8_t* mask, int64_t stride,
           cudaStream_t st) {
  const int e = is_f32(h) ? gsm::launch_env_f32(h->hp, h->plan, io, physics, mask, stride, st)
                          : gsm::launch_env_f64(h->hp, h->plan, io, physics, mask, stride, st);
  if (e) return cuda_fail(h, e, "env kernel launch");
  h->launches += 1;
  return 0;
}

// Bytes between slot s and slot s+1 of rollout buffer k: the handle's own tensor size, or that of
// a wider [T][slot_envs][...] buffer this handle's envs are a contiguous slice of.
size_t slot_bytes(const gsm_env* h, int k) {
  if (h->slot_envs <= 0 || h->hp.n_envs <= 0) return h->io_bytes[k];
  return h->io_bytes[k] / (size_t)h->hp.n_envs * (size_t)h->slot_envs;
}

// One env step (physics + outputs): the size-specialised kernel when the handle has one.
int do_steps(gsm_env* h, const gsm_step_io& io, int n_steps, cudaStream_t st, int observe = 0,
             const uint8_t* mask = nullptr, int64_t mask_stride = 0) {
  for (int k = IO_OBS; k < IO_COUNT; k++)
    if (!io_get(io, k)) return -1000;   // the specialised kernel writes every output
  gsm::RolloutStrides rs;
  std::memset(&rs, 0, sizeof(rs));
  if (n_steps > 1) {
    rs.actions = (int64_t)slot_bytes(h, IO_ACTIONS); rs.obs = (int64_t)slot_bytes(h, IO_OBS);
    rs.nbr_idx = (int64_t)slot_bytes(h, IO_NBR_IDX); rs.nbr_feat = (int64_t)slot_bytes(h, IO_NBR_FEAT);
    rs.nbr_cnt = (int64_t)slot_bytes(h, IO_NBR_CNT); rs.adj = (int64_t)slot_bytes(h, IO_ADJ);
    rs.reward = (int64_t)slot_bytes(h, IO_REWARD); rs.cost = (int64_t)slot_bytes(h, IO_COST);
    rs.done = (int64_t)slot_bytes(h, IO_DONE); rs.assign = (int64_t)slot_bytes(h, IO_ASSIGN);
  }
  int e = -1;
  if (h->plan.team && !observe)
    e = is_f32(h) ? gsm::launch_team_f32(h->hp, io, n_steps, rs, st)
                  : gsm::launch_team_f64(h->hp, io, n_steps, rs, st);
  else if (h->plan.spec)
    e = is_f32(h) ? gsm::launch_spec_f32(h->hp, io, n_steps, rs, observe, mask, mask_stride, st)
                  : gsm::launch_spec_f64(h->hp, io, n_steps, rs, observe, mask, mask_stride, st);
  else if (h->plan.lane && !observe)
    e = is_f32(h) ? gsm::launch_lane_f32(h->hp, io, n_steps, rs, st)
                  : gsm::launch_lane_f64(h->hp, io, n_steps, rs, st);
  if (e > 0) return cuda_fail(h, e, "fused env kernel launch");
  if (e == 0) { h->launches += 1; return 0; }
  return -1000;      // no fused kernel for this handle / call
}

int do_step(gsm_env* h, const gsm_step_io& io, cudaStream_t st) {
  if (h->plan.spec || h->plan.lane) {
    const int r = do_steps(h, io, 1, st);
    if (r != -1000) return r;
  }
  return do_env(h, io, 1, nullptr, 0, st);
}

// Observation + graph of the current state (no physics), optionally for masked envs only.
int do_observe(gsm_env* h, const gsm_step_io& io, const uint8_t* mask, int64_t stride, cudaStream_t st) {
  if (h->plan.spec) {
    const int r = do_steps(h, io, 1, st, 1, mask, stride);
    if (r != -1000) return r;
  }
  return do_env(h, io, 0, mask, stride, st);
}

bool any_obs_output(const gsm_step_io& io) {
  return io.obs || io.nbr_idx || io.nbr_feat || io.nbr_cnt || io.adj || io.assign;
}

int ensure_host_path(gsm_env* h) {
  if (h->d_arena) return 0;
  size_t o = 0;
  for (int k = 0; k < IO_COUNT; k++) {
    h->arena_off[k] = o;
    o += ((h->io_bytes[k] + 255) / 256) * 256;
    if (k == IO_ACTIONS) h->arena_out_begin = o;
  }
  h->arena_total = o;
  GSM_CUDA(h, cudaMalloc((void**)&h->d_arena, o));
  GSM_CUDA(h, cudaMemset(h->d_arena, 0, o));
  GSM_CUDA(h, cudaHostAlloc((void**)&h->h_arena, o, cudaHostAllocMapped));
  std::memset(h->h_arena, 0, o);
  GSM_CUDA(h, cudaHostGetDevicePointer((void**)&h->h_arena_dev, h->h_arena, 0));
  GSM_CUDA(h, cudaMalloc((void**)&h->d_prev_cnt, (size_t)h->hp.n_envs * h->hp.N * 4 + 16));
  GSM_CUDA(h, cudaMemset(h->d_prev_cnt, 0, (size_t)h->hp.n_envs * h->hp.N * 4 + 16));
  GSM_CUDA(h, cudaMalloc((void**)&h->d_shadow, o));
  GSM_CUDA(h, cudaMemset(h->d_shadow, 0, o));
  if (const char* v = std::getenv("GSM_HOST_DENSE")) h->host_sparse = std::atoi(v) ? 0 : 1;
  h->host_resync = 1;
  GSM_CUDA(h, cudaMalloc((void**)&h->d_mask, (size_t)h->hp.n_envs * h->hp.N + 16));
  for (int k = 0; k < IO_COUNT; k++) {
    io_set(h->d_io, k, h->d_arena + h->arena_off[k]);
    io_set(h->h_io, k, h->h_arena + h->arena_off[k]);
  }
  return 0;
}

bool is_arena_io(const gsm_env* h, const gsm_step_io& io) {
  for (int k = 0; k < IO_COUNT; k++)
    if (io_get(io, k) != io_get(h->h_io, k)) return false;
  return true;
}

// ---- sparse export kernels (arena host path) ---------------------------------------------------------
// Of an agent's K neighbour rows only the first cnt are data: that block (cnt * row bytes, contiguous, at
// the start of the agent's K-row block) is written to the mapped host arena in 8-byte pieces together with the
// rows in [cnt, prev) — valid on the host from an earlier call, zeros now — and rows >= max(cnt, prev) already
// hold zeros there and are not touched.  A warp serves 4 agents per pass.
// Measured on B200 / PCIe gen5 (profiles/micro/mapped_d2h*.cu, 49152 agents x 8 rows x 24 B): dense DMA of
// nbr_feat 169 us; this kernel 116-121 us at 38-56 % valid rows (the link carries partial lines as small
// packets, so time follows the agent count more than the bytes); the same with 16-byte pieces 176 us (kept
// out); nbr_idx with 4-byte scattered writes cost +100 us per step, so it leaves dense with the small outputs.
struct RowsExport { const int32_t* cnt; int32_t* prev; const unsigned char* feat; unsigned char* h_feat; int64_t rows; int row_bytes, K; };
__device__ __forceinline__ void export_rows(const RowsExport& r, int block, int n_blocks) {
  const int32_t* __restrict__ cnt = r.cnt;
  int32_t* __restrict__ prev = r.prev;
  const unsigned char* __restrict__ feat = r.feat;
  unsigned char* __restrict__ h_feat = r.h_feat;
  const int64_t rows = r.rows;
  const int row_bytes = r.row_bytes, K = r.K;
  const int lane = threadIdx.x & 31;
  const int64_t w = ((int64_t)block * blockDim.x + threadIdx.x) >> 5, nw = ((int64_t)n_blocks * blockDim.x) >> 5;
  const int ab = K * row_bytes, ppa = ab / 8;                // bytes / 8-byte pieces per agent
  for (int64_t a0 = w * 4; a0 < rows; a0 += nw * 4) {
    for (int q = lane; q < 4 * ppa; q += 32) {
      const int64_t a = a0 + q / ppa;
      if (a >= rows) continue;
      const int o = (q % ppa) * 8;                            // byte offset inside the agent's block
      const size_t g = (size_t)a * ab + o;
      // one store path: rows in [cnt, prev) are copied too — the device tensor holds the zeros they must become
      // (measured 99 us against 115 us with a separate clearing branch, profiles/micro/mapped_d2h2.cu)
      const int c = cnt[a], pv = prev[a];
      if (o < (c > pv ? c : pv) * row_bytes) *(uint2*)(h_feat + g) = *(const uint2*)(feat + g);
    }
    __syncwarp();
    if (lane < 4 && a0 + lane < rows) prev[a0 + lane] = cnt[a0 + lane];
  }
}

// The other outputs leave in 16-byte pieces.  Slowly changing ones — nbr_idx (navigation-3: 18 % of the agents
// per step), nbr_cnt, adj, cost (mostly 0), done, assign — are compared with a device-side SHADOW of what the
// host already holds and only the pieces that differ are sent (profiles/micro/mapped_idx.cu: 20 % of the
// nbr_idx rows 16.7 us, the dense 1.57 MB block 35.8 us); obs and reward change everywhere and go out dense.
struct DenseCopies {
  const unsigned char* src[8]; unsigned char* dst[8]; unsigned char* shadow[8];   // shadow NULL: send every piece
  unsigned long long n16[8];
  int n;
};
__device__ __forceinline__ void export_dense(const DenseCopies& c, int block, int n_blocks) {
  for (int k = 0; k < c.n; k++) {
    const uint4* src = (const uint4*)c.src[k];
    uint4* dst = (uint4*)c.dst[k];
    uint4* sh = (uint4*)c.shadow[k];
    for (unsigned long long i = (unsigned long long)block * blockDim.x + threadIdx.x; i < c.n16[k];
         i += (unsigned long long)n_blocks * blockDim.x) {
      const uint4 v = src[i];
      if (sh) {
        const uint4 o = sh[i];
        if (v.x == o.x && v.y == o.y && v.z == o.z && v.w == o.w) continue;
        sh[i] = v;
      }
      dst[i] = v;
    }
  }
}

// ONE launch: blocks [0, rows_blocks) export the valid rows of nbr_feat, the others the 16-byte pieces
// (a second launch cost ~5 us on the critical path of a 200 us step).
__global__ void export_kernel(const __grid_constant__ RowsExport r, const __grid_constant__ DenseCopies c, const int rows_blocks) {
  if ((int)blockIdx.x < rows_blocks) export_rows(r, (int)blockIdx.x, rows_blocks);
  else export_dense(c, (int)blockIdx.x - rows_blocks, (int)gridDim.x - rows_blocks);
}

// D2H of the outputs of a host-path call.
int copy_out(gsm_env* h, const gsm_step_io& host_io, bool with_rcd) {
  if (is_arena_io(h, host_io)) {
    const auto wanted = [&](int k) {
      if (!(h->host_out_mask >> k & 1u)) return false;
      return with_rcd || !(k == IO_REWARD || k == IO_COST || k == IO_DONE);
    };
    const int64_t rows = h->hp.n_envs * h->hp.N;
    if (!h->host_sparse || h->host_resync) {
      // dense: every delivered output in full (one copy when nothing is masked out)
      if (h->host_out_mask == 0xffffffffu) {
        GSM_CUDA(h, cudaMemcpyAsync(h->h_arena + h->arena_out_begin, h->d_arena + h->arena_out_begin,
                                    h->arena_total - h->arena_out_begin, cudaMemcpyDeviceToHost, h->stream));
      } else {
        for (int k = IO_OBS; k < IO_COUNT; k++)
          if (h->host_out_mask >> k & 1u)
            GSM_CUDA(h, cudaMemcpyAsync(h->h_arena + h->arena_off[k], h->d_arena + h->arena_off[k], h->io_bytes[k],
                                        cudaMemcpyDeviceToHost, h->stream));
      }
      GSM_CUDA(h, cudaMemcpyAsync(h->d_prev_cnt, h->d_io.nbr_cnt, (size_t)rows * 4, cudaMemcpyDeviceToDevice, h->stream));
      GSM_CUDA(h, cudaMemcpyAsync(h->d_shadow + h->arena_out_begin, h->d_arena + h->arena_out_begin,
                                  h->arena_total - h->arena_out_begin, cudaMemcpyDeviceToDevice, h->stream));
      h->host_resync = 0;
    } else {
      DenseCopies dc;
      dc.n = 0;
      for (int k = IO_OBS; k < IO_COUNT; k++) {
        if (k == IO_NBR_FEAT || !wanted(k)) continue;
        dc.src[dc.n] = h->d_arena + h->arena_off[k];
        dc.dst[dc.n] = h->h_arena_dev + h->arena_off[k];
        dc.shadow[dc.n] = (k == IO_OBS || k == IO_REWARD) ? nullptr : h->d_shadow + h->arena_off[k];
        dc.n16[dc.n] = (h->io_bytes[k] + 15) / 16;            // sub-buffers are 256-byte aligned and padded
        dc.n++;
      }
      RowsExport re;
      re.cnt = h->d_io.nbr_cnt; re.prev = h->d_prev_cnt; re.feat = (const unsigned char*)h->d_io.nbr_feat;
      re.h_feat = h->h_arena_dev + h->arena_off[IO_NBR_FEAT]; re.rows = rows; re.row_bytes = GSM_NBR_FEAT_DIM * h->rb;
      re.K = h->hp.K;
      const int rows_blocks = wanted(IO_NBR_FEAT) ? 296 : 0, dense_blocks = dc.n ? 148 : 0;
      if (rows_blocks + dense_blocks) {
        export_kernel<<<rows_blocks + dense_blocks, 256, 0, h->stream>>>(re, dc, rows_blocks);
        GSM_CUDA(h, cudaGetLastError());
        h->launches += 1;
      }
    }
  } else {
    for (int k = IO_OBS; k < IO_COUNT; k++) {
      if (!with_rcd && (k == IO_REWARD || k == IO_COST || k == IO_DONE)) continue;
      void* dst = io_get(host_io, k);
      if (dst)
        GSM_CUDA(h, cudaMemcpyAsync(dst, io_get(h->d_io, k), h->io_bytes[k], cudaMemcpyDeviceToHost, h->stream));
    }
  }
  GSM_CUDA(h, cudaStreamSynchronize(h->stream));      // (polling cudaStreamQuery instead: no measurable gain)
  return 0;
}

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess; else prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

}  // namespace

extern "C" {

int gsm_abi_version(void) { return GSM_ABI_VERSION; }

const char* gsm_status_string(int status) {
  switch (status) {
    case GSM_OK: return "GSM_OK";
    case GSM_ERR_INVALID_ARG: return "GSM_ERR_INVALID_ARG";
    case GSM_ERR_CUDA: return "GSM_ERR_CUDA";
    case GSM_ERR_ABI: return "GSM_ERR_ABI";
    case GSM_ERR_UNSUPPORTED: return "GSM_ERR_UNSUPPORTED";
    case GSM_ERR_NO_DEVICE: return "GSM_ERR_NO_DEVICE";
    default: return "GSM_ERR_UNKNOWN";
  }
}

const char* gsm_last_error(const gsm_env* h) { return h ? h->err.c_str() : g_create_err.c_str(); }

int gsm_create(const gsm_config* cfg, int64_t n_envs, int64_t env_offset, int device, gsm_env** out) {
  if (!out) return fail(nullptr, GSM_ERR_INVALID_ARG, "out is NULL");
  *out = nullptr;
  if (cfg && (cfg->struct_size != sizeof(gsm_config) || cfg->abi_version != GSM_ABI_VERSION))
    return fail(nullptr, GSM_ERR_ABI, validate(cfg));
  const std::string v = validate(cfg);
  if (!v.empty()) return fail(nullptr, GSM_ERR_INVALID_ARG, v);
  if (n_envs < 1 || env_offset < 0) return fail(nullptr, GSM_ERR_INVALID_ARG, "n_envs must be >= 1, env_offset >= 0");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(nullptr, GSM_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  }
  if (device < 0 || device >= ndev) return fail(nullptr, GSM_ERR_INVALID_ARG, "device index out of range");
  DeviceGuard guard(device);
  gsm_env* h = new gsm_env();
  auto bail = [&](int st) { g_create_err = h->err; gsm_destroy(h); return st; };
  h->dtype = cfg->dtype; h->device = device; h->rb = cfg->dtype == GSM_F32 ? 4 : 8;
  const int N = cfg->n_agents, L = cfg->n_landmarks, E = N + L, K = cfg->max_nbrs;
  gsm::HostParams& hp = h->hp;
  std::memset(&hp, 0, sizeof(hp));
  hp.n_envs = n_envs; hp.env_offset = env_offset; hp.N = N; hp.L = L; hp.K = K;
  hp.scenario = cfg->scenario; hp.action_mode = cfg->action_mode;
  hp.n_actions = cfg->action_mode == GSM_ACT_DISCRETE ? cfg->n_discrete_actions : 0;
  hp.episode_length = cfg->episode_length; hp.share_reward = cfg->share_reward != 0;
  hp.cost_obstacles = cfg->cost_obstacles != 0; hp.own_goal_always = cfg->own_goal_always != 0;
  hp.dt = cfg->dt; hp.damping = cfg->damping; hp.cf = cfg->contact_force; hp.km = cfg->contact_margin;
  hp.Rs = cfg->sensing_radius; hp.w_dist = cfg->w_dist; hp.w_goal = cfg->w_goal;
  hp.goal_tol = cfg->goal_tol; hp.poly_r = cfg->polygon_radius;
  for (int a = 0; a < hp.n_actions; a++) {
    hp.discrete_u[a][0] = cfg->discrete_u[2 * a]; hp.discrete_u[a][1] = cfg->discrete_u[2 * a + 1];
  }
  for (int k = 0; k < 4; k++) hp.ext[k] = cfg->spawn_extent[k];

  const size_t rb = h->rb, ne = (size_t)n_envs;
  const int W = (E + 31) / 32;
  gsm_io_sizes& sz = h->sz;
  std::memset(&sz, 0, sizeof(sz));
  sz.actions = cfg->action_mode == GSM_ACT_DISCRETE ? ne * N * 4 : ne * N * 2 * rb;
  sz.obs = ne * N * GSM_OBS_DIM * rb; sz.nbr_idx = ne * N * K * 4;
  sz.nbr_feat = ne * N * K * GSM_NBR_FEAT_DIM * rb; sz.nbr_cnt = ne * N * 4; sz.adj = ne * N * W * 4;
  sz.reward = ne * N * rb; sz.cost = ne * N * rb; sz.done = ne * N; sz.assign = ne * N * 4;
  sz.agent_state = ne * N * 4 * rb; sz.landmark_pos = ne * L * 2 * rb; sz.step_count = ne * 4;
  sz.adj_words = W; sz.real_bytes = (int32_t)rb;
  const size_t iob[IO_COUNT] = {sz.actions, sz.obs, sz.nbr_idx, sz.nbr_feat, sz.nbr_cnt, sz.adj,
                                sz.reward, sz.cost, sz.done, sz.assign};
  std::memcpy(h->io_bytes, iob, sizeof(iob));

  int st;
  void* p = nullptr;
  if ((st = upload_real(h, cfg->size, E, &p))) return bail(st); hp.size = p;
  if ((st = upload_real(h, cfg->mass, N, &p))) return bail(st); hp.mass = p;
  if ((st = upload_real(h, cfg->accel, N, &p))) return bail(st); hp.accel = p;
  if ((st = upload_real(h, cfg->max_speed, N, &p))) return bail(st); hp.max_speed = p;
  if (cfg->scenario != GSM_SCN_NAVIGATION) {
    if ((st = upload_real(h, cfg->slot_table, (size_t)N * 2, &p))) return bail(st);
    hp.slot_table = p;
  }
  {
    std::vector<uint8_t> fl(E);
    for (int e = 0; e < E; e++) fl[e] = (uint8_t)((cfg->collide[e] ? 1 : 0) | (cfg->type[e] << 1));
    if ((st = dev_alloc(h, E, &p))) return bail(st);
    if (cudaMemcpy(p, fl.data(), E, cudaMemcpyHostToDevice) != cudaSuccess)
      return bail(fail(h, GSM_ERR_CUDA, "upload eflag"));
    hp.eflag = (const uint8_t*)p;
    hp.h_consts = (E <= gsm::kHostConstE && N <= gsm::kHostConstN) ? 1 : 0;
    if (hp.h_consts) {
      for (int e = 0; e < E; e++) { hp.h_size[e] = cfg->size[e]; hp.h_eflag[e] = fl[e]; }
      for (int i = 0; i < N; i++) { hp.h_mass[i] = cfg->mass[i]; hp.h_accel[i] = cfg->accel[i]; hp.h_maxsp[i] = cfg->max_speed[i]; }
    }
  }
  if ((st = dev_alloc(h, sz.agent_state, &p))) return bail(st); hp.agent_state = p;
  if ((st = dev_alloc(h, sz.landmark_pos ? sz.landmark_pos : 16, &p))) return bail(st); hp.lm_pos = p;
  if ((st = dev_alloc(h, sz.step_count, &p))) return bail(st); hp.t = (int32_t*)p;
  if ((st = dev_alloc(h, sz.step_count, &p))) return bail(st); hp.episode = (int32_t*)p;

  const int pe = is_f32(h) ? gsm::plan_f32(hp, &h->plan) : gsm::plan_f64(hp, &h->plan);
  if (pe) return bail(fail(h, GSM_ERR_UNSUPPORTED, "no launch plan for this configuration (shared memory / lane limits)"));
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess)
    return bail(fail(h, GSM_ERR_CUDA, "cudaStreamCreate"));
  std::memset(&h->d_io, 0, sizeof(h->d_io));
  std::memset(&h->h_io, 0, sizeof(h->h_io));
  std::memset(&h->graph_io, 0, sizeof(h->graph_io));
  *out = h;
  return GSM_OK;
}

int gsm_destroy(gsm_env* h) {
  if (!h) return GSM_OK;
  DeviceGuard guard(h->device);
  cudaDeviceSynchronize();
  if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
  for (void* p : h->dev_allocs) cudaFree(p);
  if (h->d_arena) cudaFree(h->d_arena);
  if (h->h_arena) cudaFreeHost(h->h_arena);
  if (h->d_prev_cnt) cudaFree(h->d_prev_cnt);
  if (h->d_shadow) cudaFree(h->d_shadow);
  if (h->d_mask) cudaFree(h->d_mask);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return GSM_OK;
}

int gsm_get_io_sizes(const gsm_env* h, gsm_io_sizes* out) {
  if (!h || !out) return GSM_ERR_INVALID_ARG;
  *out = h->sz;
  return GSM_OK;
}

int gsm_reset(gsm_env* h, uint64_t seed, const uint8_t* mask, int64_t mask_stride,
              const gsm_step_io* io, void* stream) {
  if (!h) return GSM_ERR_INVALID_ARG;
  if (mask && mask_stride < 1) return fail(h, GSM_ERR_INVALID_ARG, "mask_stride must be >= 1");
  DeviceGuard guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  h->seed = seed;
  const int e = is_f32(h) ? gsm::launch_reset_f32(h->hp, seed, mask, mask_stride, st)
                          : gsm::launch_reset_f64(h->hp, seed, mask, mask_stride, st);
  if (e) return cuda_fail(h, e, "reset kernel launch");
  h->launches += 2;
  if (io && any_obs_output(*io)) return do_observe(h, *io, mask, mask ? mask_stride : 0, st);
  return GSM_OK;
}

int gsm_step(gsm_env* h, const gsm_step_io* io, void* stream) {
  if (!h || !io) return GSM_ERR_INVALID_ARG;
  if (!io->actions) return fail(h, GSM_ERR_INVALID_ARG, "io.actions is NULL");
  DeviceGuard guard(h->device);
  return do_step(h, *io, (cudaStream_t)stream);
}

int gsm_observe(gsm_env* h, const gsm_step_io* io, void* stream) {
  if (!h || !io) return GSM_ERR_INVALID_ARG;
  DeviceGuard guard(h->device);
  return do_observe(h, *io, nullptr, 0, (cudaStream_t)stream);
}

int gsm_set_auto_reset(gsm_env* h, int enabled) {
  if (!h) return GSM_ERR_INVALID_ARG;
  if ((enabled != 0) != (h->auto_reset != 0) && h->graph_exec) {   // cached graph has the other behaviour
    cudaGraphExecDestroy(h->graph_exec);
    h->graph_exec = nullptr;
  }
  h->auto_reset = enabled != 0;
  return GSM_OK;
}

int gsm_set_slot_envs(gsm_env* h, int64_t slot_envs) {
  if (!h) return GSM_ERR_INVALID_ARG;
  if (slot_envs != 0 && slot_envs < h->hp.n_envs)
    return fail(h, GSM_ERR_INVALID_ARG, "slot_envs must be 0 or >= the handle's n_envs");
  if (slot_envs != h->slot_envs && h->graph_exec) {     // cached graph has the other strides
    cudaGraphExecDestroy(h->graph_exec);
    h->graph_exec = nullptr;
  }
  h->slot_envs = slot_envs;
  return GSM_OK;
}

int gsm_rollout(gsm_env* h, int32_t n_steps, const gsm_step_io* io, void* stream) {
  if (!h || !io || n_steps < 1) return GSM_ERR_INVALID_ARG;
  if (!io->actions) return fail(h, GSM_ERR_INVALID_ARG, "io.actions is NULL");
  DeviceGuard guard(h->device);
  // fused: all n_steps in one launch, state stays on chip; the specialised and the lane kernel
  // also re-draw finished envs in the kernel (auto-reset)
  if (h->plan.spec || h->plan.lane) {
    h->hp.auto_reset = h->auto_reset; h->hp.seed = h->seed;
    const int r = do_steps(h, *io, n_steps, (cudaStream_t)stream);
    h->hp.auto_reset = 0;
    if (r != -1000) return r;
  }
  if (h->auto_reset && !io->done) return fail(h, GSM_ERR_INVALID_ARG, "auto-reset rollout needs io.done");
  const bool hit = h->graph_exec && h->graph_steps == n_steps && h->graph_seed == h->seed &&
                   h->graph_auto_reset == h->auto_reset &&
                   std::memcmp(&h->graph_io, io, sizeof(gsm_step_io)) == 0;
  if (!hit) {
    if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; }
    const int64_t before = h->launches;
    GSM_CUDA(h, cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    int st = 0;
    for (int s = 0; s < n_steps && st == 0; s++) {
      gsm_step_io cur;
      for (int k = 0; k < IO_COUNT; k++) {
        unsigned char* b = (unsigned char*)io_get(*io, k);
        io_set(cur, k, b ? b + (size_t)s * slot_bytes(h, k) : nullptr);
      }
      st = do_step(h, cur, h->stream);
      if (st == 0 && h->auto_reset) {                  // masked re-draw of the envs that just finished
        const int e = is_f32(h) ? gsm::launch_reset_f32(h->hp, h->seed, cur.done, h->hp.N, h->stream)
                                : gsm::launch_reset_f64(h->hp, h->seed, cur.done, h->hp.N, h->stream);
        if (e) st = cuda_fail(h, e, "reset kernel launch");
      }
    }
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
    h->launches = before;
    if (st) { if (graph) cudaGraphDestroy(graph); return st; }
    if (ce != cudaSuccess) return cuda_fail(h, (int)ce, "cudaStreamEndCapture");
    ce = cudaGraphInstantiate(&h->graph_exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) return cuda_fail(h, (int)ce, "cudaGraphInstantiate");
    h->graph_steps = n_steps;
    h->graph_io = *io;
    h->graph_seed = h->seed;
    h->graph_auto_reset = h->auto_reset;
  }
  GSM_CUDA(h, cudaGraphLaunch(h->graph_exec, (cudaStream_t)stream));
  h->launches += (int64_t)n_steps * (h->auto_reset ? 3 : 1);
  return GSM_OK;
}

int gsm_set_state(gsm_env* h, const void* agent_state, const void* landmark_pos,
                  const int32_t* step_count, void* stream) {
  if (!h) return GSM_ERR_INVALID_ARG;
  DeviceGuard guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (agent_state) GSM_CUDA(h, cudaMemcpyAsync(h->hp.agent_state, agent_state, h->sz.agent_state, cudaMemcpyDefault, st));
  if (landmark_pos && h->sz.landmark_pos)
    GSM_CUDA(h, cudaMemcpyAsync(h->hp.lm_pos, landmark_pos, h->sz.landmark_pos, cudaMemcpyDefault, st));
  if (step_count) GSM_CUDA(h, cudaMemcpyAsync(h->hp.t, step_count, h->sz.step_count, cudaMemcpyDefault, st));
  return GSM_OK;
}

int gsm_get_state(gsm_env* h, void* agent_state, void* landmark_pos, int32_t* step_count, void* stream) {
  if (!h) return GSM_ERR_INVALID_ARG;
  DeviceGuard guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (agent_state) GSM_CUDA(h, cudaMemcpyAsync(agent_state, h->hp.agent_state, h->sz.agent_state, cudaMemcpyDefault, st));
  if (landmark_pos && h->sz.landmark_pos)
    GSM_CUDA(h, cudaMemcpyAsync(landmark_pos, h->hp.lm_pos, h->sz.landmark_pos, cudaMemcpyDefault, st));
  if (step_count) GSM_CUDA(h, cudaMemcpyAsync(step_count, h->hp.t, h->sz.step_count, cudaMemcpyDefault, st));
  return GSM_OK;
}

int gsm_set_episode(gsm_env* h, const int32_t* episode, void* stream) {
  if (!h) return GSM_ERR_INVALID_ARG;
  DeviceGuard guard(h->device);
  if (episode) GSM_CUDA(h, cudaMemcpyAsync(h->hp.episode, episode, h->sz.step_count, cudaMemcpyDefault, (cudaStream_t)stream));
  return GSM_OK;
}

int gsm_get_episode(gsm_env* h, int32_t* episode, void* stream) {
  if (!h) return GSM_ERR_INVALID_ARG;
  DeviceGuard guard(h->device);
  if (episode) GSM_CUDA(h, cudaMemcpyAsync(episode, h->hp.episode, h->sz.step_count, cudaMemcpyDefault, (cudaStream_t)stream));
  return GSM_OK;
}

int gsm_host_io(gsm_env* h, gsm_step_io* out) {
  if (!h || !out) return GSM_ERR_INVALID_ARG;
  DeviceGuard guard(h->device);
  const int st = ensure_host_path(h);
  if (st) return st;
  *out = h->h_io;
  return GSM_OK;
}

int gsm_set_host_outputs(gsm_env* h, uint32_t out_mask, int32_t sparse) {
  if (!h) return GSM_ERR_INVALID_ARG;
  out_mask |= 1u << IO_ACTIONS;
  out_mask |= ~((1u << IO_COUNT) - 1u);                      // unknown bits read as "on": 0xffffffff stays "everything"
  h->host_resync = 1;                                        // every call: also the way to recover an overwritten host arena
  h->host_out_mask = out_mask;
  h->host_sparse = sparse != 0;
  return GSM_OK;
}

int gsm_reset_host(gsm_env* h, uint64_t seed, const uint8_t* mask, int64_t mask_stride,
                   const gsm_step_io* io) {
  if (!h) return GSM_ERR_INVALID_ARG;
  DeviceGuard guard(h->device);
  int st = ensure_host_path(h);
  if (st) return st;
  const uint8_t* dmask = nullptr;
  if (mask && io && any_obs_output(*io) && !is_arena_io(h, *io))   // checked BEFORE anything is mutated: an error call has no side effect
    return fail(h, GSM_ERR_UNSUPPORTED, "masked gsm_reset_host needs the gsm_host_io buffers (partial rows are kept on the device copy)");
  if (mask) {
    if (mask_stride < 1 || mask_stride > h->hp.N) return fail(h, GSM_ERR_INVALID_ARG, "host mask_stride must be in [1, N]");
    GSM_CUDA(h, cudaMemcpyAsync(h->d_mask, mask, (size_t)(h->hp.n_envs - 1) * mask_stride + 1,
                                cudaMemcpyHostToDevice, h->stream));
    dmask = h->d_mask;
  }
  const bool want = io && any_obs_output(*io);
  st = gsm_reset(h, seed, dmask, mask_stride, want ? &h->d_io : nullptr, h->stream);
  if (st) return st;
  if (!want) { GSM_CUDA(h, cudaStreamSynchronize(h->stream)); return GSM_OK; }
  return copy_out(h, *io, false);
}

int gsm_step_host(gsm_env* h, const gsm_step_io* io) {
  if (!h || !io) return GSM_ERR_INVALID_ARG;
  if (!io->actions) return fail(h, GSM_ERR_INVALID_ARG, "io.actions is NULL");
  DeviceGuard guard(h->device);
  int st = ensure_host_path(h);
  if (st) return st;
  // (letting the step kernel read the actions from the mapped arena instead of this copy: no measurable gain)
  GSM_CUDA(h, cudaMemcpyAsync(const_cast<void*>(h->d_io.actions), io->actions, h->io_bytes[IO_ACTIONS],
                              cudaMemcpyHostToDevice, h->stream));
  st = do_step(h, h->d_io, h->stream);
  if (st) return st;
  return copy_out(h, *io, true);
}

int gsm_observe_host(gsm_env* h, const gsm_step_io* io) {
  if (!h || !io) return GSM_ERR_INVALID_ARG;
  DeviceGuard guard(h->device);
  int st = ensure_host_path(h);
  if (st) return st;
  st = do_observe(h, h->d_io, nullptr, 0, h->stream);
  if (st) return st;
  return copy_out(h, *io, false);
}

int gsm_set_state_host(gsm_env* h, const void* agent_state, const void* landmark_pos,
                       const int32_t* step_count) {
  if (!h) return GSM_ERR_INVALID_ARG;
  DeviceGuard guard(h->device);
  const int st = gsm_set_state(h, agent_state, landmark_pos, step_count, h->stream);
  if (st) return st;
  GSM_CUDA(h, cudaStreamSynchronize(h->stream));
  return GSM_OK;
}

int gsm_get_state_host(gsm_env* h, void* agent_state, void* landmark_pos, int32_t* step_count) {
  if (!h) return GSM_ERR_INVALID_ARG;
  DeviceGuard guard(h->device);
  const int st = gsm_get_state(h, agent_state, landmark_pos, step_count, h->stream);
  if (st) return st;
  GSM_CUDA(h, cudaStreamSynchronize(h->stream));
  return GSM_OK;
}

}  // extern "C"

namespace {
// The collect loop both heads share: step t's actor reads observation slot t and writes actions slot
// t (`act(t, obs, nbr_feat, nbr_cnt, actions)` enqueues it); gsm_step writes step outputs into slot t
// and observation outputs into slot t + 1; auto-reset re-draws finished envs into slot t + 1.
template <class Act>
int collect_loop(gsm_env* h, int32_t n_steps, const gsm_step_io* io, void* stream, Act&& act) {
  DeviceGuard guard(h->device);
  for (int t = 0; t < n_steps; t++) {
    gsm_step_io cur;     // step outputs: slot t; observation outputs: slot t + 1
    for (int k = 0; k < IO_COUNT; k++) {
      unsigned char* b = (unsigned char*)io_get(*io, k);
      const bool obs_like = k == IO_OBS || k == IO_NBR_IDX || k == IO_NBR_FEAT || k == IO_NBR_CNT ||
                            k == IO_ADJ || k == IO_ASSIGN;
      io_set(cur, k, b ? b + (size_t)(t + (obs_like ? 1 : 0)) * slot_bytes(h, k) : nullptr);
    }
    const float* obs = (const float*)((const unsigned char*)io->obs + (size_t)t * slot_bytes(h, IO_OBS));
    const float* feat = (const float*)((const unsigned char*)io->nbr_feat + (size_t)t * slot_bytes(h, IO_NBR_FEAT));
    const int32_t* cnt = (const int32_t*)((const unsigned char*)io->nbr_cnt + (size_t)t * slot_bytes(h, IO_NBR_CNT));
    int st = act(t, obs, feat, cnt, const_cast<void*>(cur.actions));
    if (st) return fail(h, st, gsm_policy_last_error());
    h->launches += 1;
    st = do_step(h, cur, (cudaStream_t)stream);
    if (st) return st;
    if (h->auto_reset) {   // the vec-env wrapper's reset-on-done: finished envs get their first observation in slot t+1
      st = gsm_reset(h, h->seed, cur.done, h->hp.N, &cur, stream);
      if (st) return st;
    }
  }
  return GSM_OK;
}

// The checks both collects share after the handle's kind; GSM_OK or the status to return.
int check_collect_io(gsm_env* h, const gsm_step_io* io, const char* who) {
  if (!io->actions || !io->obs || !io->nbr_feat || !io->nbr_cnt)
    return fail(h, GSM_ERR_INVALID_ARG, std::string(who) + " needs io.actions, io.obs, io.nbr_feat and io.nbr_cnt");
  if (h->auto_reset && !io->done) return fail(h, GSM_ERR_INVALID_ARG, "auto-reset collect needs io.done");
  return GSM_OK;
}
}  // namespace

extern "C" {

int gsm_collect(gsm_env* h, const gsm_policy_weights* w, int32_t n_steps, const gsm_step_io* io,
                float* logp, float* values, uint64_t seed, uint64_t first_step, int32_t greedy,
                void* stream) {
  if (!h || !io || !w || n_steps < 1) return GSM_ERR_INVALID_ARG;
  if (!is_f32(h) || h->hp.action_mode != GSM_ACT_DISCRETE)
    return fail(h, GSM_ERR_UNSUPPORTED, "gsm_collect needs a GSM_F32 handle with discrete actions");
  if (w->n_actions != h->hp.n_actions)
    return fail(h, GSM_ERR_INVALID_ARG, "gsm_collect: weights.n_actions != cfg.n_discrete_actions");
  if (const int st = check_collect_io(h, io, "gsm_collect")) return st;
  const int64_t rows = h->hp.n_envs * h->hp.N;
  const int64_t slot_rows = (h->slot_envs ? h->slot_envs : h->hp.n_envs) * h->hp.N;
  return collect_loop(h, n_steps, io, stream, [&](int t, const float* obs, const float* feat, const int32_t* cnt,
                                                  void* actions) {
    gsm_policy_io pio;
    pio.obs = obs; pio.nbr_feat = feat; pio.nbr_cnt = cnt;
    pio.actions = (int32_t*)actions;
    pio.logp = logp ? logp + (size_t)t * slot_rows : nullptr;
    pio.logits = nullptr;
    pio.values = values ? values + (size_t)t * slot_rows * GSM_POLICY_VALUE_HEADS : nullptr;
    pio.n_rows = rows;
    pio.row_offset = (uint64_t)h->hp.env_offset * (uint64_t)h->hp.N;
    pio.seed = seed; pio.step = first_step + (uint64_t)t;
    pio.max_nbrs = h->hp.K; pio.greedy = greedy;
    return gsm_policy_act(w, &pio, h->device, stream);
  });
}

int gsm_collect_gauss(gsm_env* h, const gsm_policy_gauss_weights* w, int32_t n_steps, const gsm_step_io* io,
                      float* logp, float* values, uint64_t seed, uint64_t first_step, int32_t greedy,
                      void* stream) {
  if (!h || !io || !w || n_steps < 1) return GSM_ERR_INVALID_ARG;
  if (!is_f32(h) || h->hp.action_mode != GSM_ACT_CONTINUOUS)
    return fail(h, GSM_ERR_UNSUPPORTED, "gsm_collect_gauss needs a GSM_F32 handle with continuous actions");
  if (const int st = check_collect_io(h, io, "gsm_collect_gauss")) return st;
  const int64_t rows = h->hp.n_envs * h->hp.N;
  const int64_t slot_rows = (h->slot_envs ? h->slot_envs : h->hp.n_envs) * h->hp.N;
  return collect_loop(h, n_steps, io, stream, [&](int t, const float* obs, const float* feat, const int32_t* cnt,
                                                  void* actions) {
    gsm_policy_gauss_io pio;
    pio.obs = obs; pio.nbr_feat = feat; pio.nbr_cnt = cnt;
    pio.actions = (float*)actions;
    pio.logp = logp ? logp + (size_t)t * slot_rows : nullptr;
    pio.mean = nullptr;
    pio.values = values ? values + (size_t)t * slot_rows * GSM_POLICY_VALUE_HEADS : nullptr;
    pio.n_rows = rows;
    pio.row_offset = (uint64_t)h->hp.env_offset * (uint64_t)h->hp.N;
    pio.seed = seed; pio.step = first_step + (uint64_t)t;
    pio.max_nbrs = h->hp.K; pio.greedy = greedy;
    return gsm_policy_act_gauss(w, &pio, h->device, stream);
  });
}

int64_t gsm_kernel_launches(const gsm_env* h) { return h ? h->launches : 0; }

int gsm_lsa(const void* cost, int32_t* col4row, int64_t n_problems, int32_t n, int32_t dtype,
            int device, void* stream) {
  if (!cost || !col4row || n_problems < 0 || n < 1 || n > GSM_MAX_LSA_N)
    return fail(nullptr, GSM_ERR_INVALID_ARG, "gsm_lsa: bad arguments");
  if (dtype != GSM_F32 && dtype != GSM_F64) return fail(nullptr, GSM_ERR_INVALID_ARG, "gsm_lsa: bad dtype");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(nullptr, GSM_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  }
  if (device < 0 || device >= ndev) return fail(nullptr, GSM_ERR_INVALID_ARG, "gsm_lsa: device index out of range");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(nullptr, GSM_ERR_CUDA, "gsm_lsa: cudaSetDevice failed");
  const int e = dtype == GSM_F32 ? gsm::launch_lsa_f32(cost, col4row, n_problems, n, (cudaStream_t)stream)
                                 : gsm::launch_lsa_f64(cost, col4row, n_problems, n, (cudaStream_t)stream);
  if (e) return cuda_fail(nullptr, e, "lsa kernel launch");
  return GSM_OK;
}

}  // extern "C"
