"""PPO-Lagrangian update on the device (SPEC.md §14): the loss fused into the learner backward, one Adam
step per minibatch and the cost multiplier.

The reference's learner (MACPO / MAPPO-Lagrangian, readme.md:37) is withheld, so this is a DECLARED
stand-in of the lineage's update: a clipped surrogate on the advantage A_reward - lambda A_cost (each head
normalised over the rollout), clipped value losses for both critics, an entropy bonus, gradient-norm
clipping and Adam; lambda follows the team episode cost against a limit.

    trainer = LagrangianPPO(actor, **presets.UNVERIFIED_PPO_LAG, seed=0)
    for it in range(n_iters):
        collect_fused(env, actor, buf, seed=it, first_step=it * T)
        buf["values"][-1] = actor.act(buf["obs"][-1], buf.graph(-1), want_values=True)[-1]
        buf.compute_returns(gamma, lam)
        totals = tracker.update(buf["reward"], buf["cost"], buf["done"])
        stats = trainer.update(buf)            # [ppo_epoch * num_mini_batch, 9] on the device, no host sync
        trainer.update_lagrange(totals)        # on the device
        actor.pack()                           # the collect kernels take the new weights

Per minibatch: `gsm_ppo_backward(_gauss)` (the §12 backward with the loss seeds computed in its phase A,
no separate forward) and `gsm_adam_step` (clip_grad_norm_ + Adam in one launch): three kernels.

With a value normaliser (SPEC.md §15, the lineage's `use_valuenorm`) the critics are trained on, and output,
normalised values:

    vnorm = ValueNorm(device, **presets.UNVERIFIED_VALUE_NORM)
    trainer = LagrangianPPO(actor, **presets.UNVERIFIED_PPO_LAG, value_norm=vnorm, seed=0)
    ...
        buf.compute_returns(gamma, lam, value_norm=vnorm)   # denormalises the collected values
        stats = trainer.update(buf)                         # one normaliser pass per epoch
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import abi
from .policy import GaussianGraphActor, GraphAttentionActor, _check, _eval_io

class ValueNorm:
    """The lineage's ValueNorm (utils/popart.py), one independent normaliser per critic head (SPEC.md §15).
    Owns `state` (fp64 [2, 3]: running mean, running mean of squares, debiasing term per head, from 0) and
    `affine` (fp32 [2, 2]: (mu_h, sigma_h) of the state), both on `device`.  Every hyper-parameter is a
    required keyword (`presets.UNVERIFIED_VALUE_NORM` holds the lineage's values)."""

    def __init__(self, device, *, beta, epsilon, var_floor):
        if not (0 <= beta < 1) or not (epsilon > 0 and var_floor > 0):
            raise ValueError("beta must lie in [0, 1), epsilon and var_floor must be > 0")
        self.beta, self.epsilon, self.var_floor = float(beta), float(epsilon), float(var_floor)
        dev = torch.device(device)
        if dev.type != "cuda":
            raise abi.GsmError("ValueNorm lives on a CUDA device: gs_marl_b200 has no CPU fallback")
        self.device = dev if dev.index is not None else torch.device("cuda", torch.cuda.current_device())
        self.state = torch.zeros(2, 3, dtype=torch.float64, device=self.device)
        # affine snapshots [n_mini_batch + 1, 2, 2] of the last update; `affine` is its last entry
        self._snaps = torch.tensor([[0.0, math.sqrt(self.var_floor)]] * 2, dtype=torch.float32,
                                   device=self.device)[None]
        self._ws = None

    @property
    def affine(self) -> torch.Tensor:
        """(mu_h, sigma_h) [2, 2] of the current state; a view that the next `update` rewrites."""
        return self._snaps[-1]

    def mean_std(self):
        """(mu [2], sigma [2]), fp32, per head (0: reward, 1: cost)."""
        return self.affine[:, 0], self.affine[:, 1]

    def normalize(self, x: torch.Tensor) -> torch.Tensor:
        """(x - mu_h) / sigma_h over x [..., 2], fp32: the rounding of the normalised backward's targets."""
        mu, sd = self.mean_std()
        return (x.float() - mu) / sd

    def denormalize(self, v: torch.Tensor) -> torch.Tensor:
        """fmaf(v, sigma_h, mu_h) over v [..., 2] (critic outputs to raw units): the rounding of
        gsm_gae_normalized.  The product is exact in fp64; the sum is rounded to odd there, which makes the
        final rounding to fp32 the single rounding of fmaf."""
        mu, sd = (t.double() for t in self.mean_std())
        p = v.double() * sd
        s = p + mu
        bp = s - mu
        err = (p - bp) + (mu - (s - bp))                      # s + err == p + mu exactly (TwoSum)
        even = (s.view(torch.int64) & 1) == 0
        toward = torch.where(err > 0, torch.full_like(s, math.inf), torch.full_like(s, -math.inf))
        return torch.where((err != 0) & even, torch.nextafter(s, toward), s).float()

    def update(self, returns: torch.Tensor, rows: torch.Tensor, num_mini_batch: int) -> torch.Tensor:
        """One epoch of updates: minibatch b = rows[b mb:(b + 1) mb], mb = len(rows) // num_mini_batch (the
        remainder is left out), in order.  Returns the affine snapshots [num_mini_batch, 2, 2], snapshot b
        taken after minibatch b's update; they stay valid until the next call.  Two launches, no host sync."""
        nmb = int(num_mini_batch)
        if returns.dtype != torch.float32 or returns.shape[-1] != 2 or not returns.is_contiguous():
            raise ValueError("returns must be a contiguous float32 [..., 2] tensor")
        if rows.dtype != torch.int64 or rows.dim() != 1 or not rows.is_contiguous():
            raise ValueError("rows must be a contiguous int64 vector")
        if returns.device != self.device or rows.device != self.device:
            raise ValueError(f"returns and rows must be on {self.device}")
        if nmb < 1 or rows.numel() < nmb:
            raise ValueError(f"{rows.numel()} rows cannot make {nmb} minibatches")
        mb = rows.numel() // nmb
        lib = abi.load_library()
        if self._snaps.shape[0] != nmb + 1:
            snaps = torch.empty(nmb + 1, 2, 2, dtype=torch.float32, device=self.device)
            snaps[-1] = self.affine
            self._snaps = snaps
        need = lib.gsm_value_norm_update_workspace(mb, nmb)
        if need < 0:
            raise ValueError(f"gsm_value_norm_update_workspace({mb}, {nmb}) = {need}")
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        io = abi.GsmValueNormIO()
        io.struct_size = C.sizeof(abi.GsmValueNormIO)
        io.state, io.affine = self.state.data_ptr(), self._snaps.data_ptr()
        io.returns, io.rows = returns.data_ptr(), rows.data_ptr()
        io.mb, io.n_mini_batch = mb, nmb
        io.beta, io.epsilon, io.var_floor = self.beta, self.epsilon, self.var_floor
        st = lib.gsm_value_norm_update(C.byref(io), self._ws.data_ptr(), self._ws.numel(), self.device.index or 0,
                                       C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
        if st != 0:
            raise abi.GsmError(f"gsm_value_norm_update: {lib.gsm_status_string(st).decode()}")
        return self._snaps[:nmb]

    def state_dict(self) -> dict:
        return {"state": self.state.clone(), "affine": self.affine.clone()}

    def load_state_dict(self, sd: dict):
        for k, shape, dt in (("state", (2, 3), torch.float64), ("affine", (2, 2), torch.float32)):
            if tuple(sd[k].shape) != shape or sd[k].dtype != dt:
                raise ValueError(f"value_norm {k}: {tuple(sd[k].shape)} {sd[k].dtype}, expected {shape} {dt}")
        self.state.copy_(sd["state"])
        self.affine.copy_(sd["affine"])


# the columns of `update`'s result: the GSM_PPO_STAT_FIELDS loss statistics, then the gradient norm
STAT_FIELDS = ("policy_loss", "value_loss_reward", "value_loss_cost", "entropy", "ratio", "clip_fraction",
               "approx_kl", "loss", "grad_norm")


class LagrangianPPO:
    """Owns the flat parameter vector (parameters_to_vector order), Adam's m, v and step, and lambda, all on
    the actor's device.  Every hyper-parameter is a required keyword (`presets.UNVERIFIED_PPO_LAG` holds
    lineage-typical values); the library has no defaults.

    value_norm: a `ValueNorm` (SPEC.md §15) or None.  With one, each epoch first updates it once per minibatch
    and each minibatch's value loss regresses the critics on normalize(R) under its snapshot; the buffer's
    returns must come from `compute_returns(..., value_norm=...)`.  The value-loss statistics are then in
    normalised units."""

    def __init__(self, actor, *, clip, value_clip, value_coef, entropy_coef, lr, betas, eps, max_grad_norm,
                 ppo_epoch, num_mini_batch, lagrangian_lr, cost_limit, lagrangian_init=0.0, seed, value_norm=None):
        if not isinstance(actor, (GraphAttentionActor, GaussianGraphActor)):
            raise TypeError("LagrangianPPO trains a GraphAttentionActor or a GaussianGraphActor")
        self._head = actor._desc
        self._act_dtype, self._act_tail = self._head.act_dtype, self._head.act_tail
        b1, b2 = (float(b) for b in betas)
        if not (clip > 0 and value_clip > 0):
            raise ValueError("clip and value_clip must be > 0")
        if not (value_coef >= 0 and entropy_coef >= 0):
            raise ValueError("value_coef and entropy_coef must be >= 0")
        if not (0 <= b1 < 1 and 0 <= b2 < 1) or not (lr >= 0 and eps >= 0 and max_grad_norm > 0):
            raise ValueError("betas must lie in [0, 1), lr and eps must be >= 0 and max_grad_norm > 0")
        if int(ppo_epoch) < 1 or int(num_mini_batch) < 1:
            raise ValueError("ppo_epoch and num_mini_batch must be >= 1")
        if not (lagrangian_lr >= 0 and lagrangian_init >= 0):
            raise ValueError("lagrangian_lr and lagrangian_init must be >= 0")
        self.actor = actor
        self.clip, self.value_clip = float(clip), float(value_clip)
        self.value_coef, self.entropy_coef = float(value_coef), float(entropy_coef)
        self.lr, self.betas, self.eps, self.max_grad_norm = float(lr), (b1, b2), float(eps), float(max_grad_norm)
        self.ppo_epoch, self.num_mini_batch = int(ppo_epoch), int(num_mini_batch)
        self.lagrangian_lr, self.cost_limit = float(lagrangian_lr), float(cost_limit)
        params = torch.nn.utils.parameters_to_vector(actor.parameters()).detach()
        if not params.is_cuda or params.dtype != torch.float32:
            raise abi.GsmError("the actor's parameters must be float32 CUDA tensors: gs_marl_b200 has no CPU fallback")
        self.device = params.device
        dev = self.device
        self.params = params.clone()
        self.grad = torch.zeros_like(self.params)
        self.m = torch.zeros_like(self.params)
        self.v = torch.zeros_like(self.params)
        self.step = torch.zeros(1, dtype=torch.int32, device=dev)
        self.lagrange = torch.full((1,), float(lagrangian_init), dtype=torch.float32, device=dev)
        self.adv_moments = torch.zeros(4, dtype=torch.float32, device=dev)
        self.generator = torch.Generator(device=dev)
        self.generator.manual_seed(int(seed))
        self._ws = None
        if value_norm is not None and (not isinstance(value_norm, ValueNorm) or value_norm.device != dev):
            raise ValueError(f"value_norm must be a ValueNorm on {dev}")
        self.value_norm = value_norm

    # ---- the pieces of one update -------------------------------------------------------------------
    def inputs(self, buf):
        """The buffer's tensors (a GraphRolloutBuffer or a dict with its keys) flattened to source rows
        [T * n_envs * N] (views, no copies)."""
        d = buf.data if hasattr(buf, "data") else buf
        if "returns" not in d or "advantages" not in d:
            raise ValueError("the buffer has no returns / advantages: call buf.compute_returns() before update")
        T = d["actions"].shape[0]
        obs, feat, cnt, act = d["obs"][:T], d["nbr_feat"][:T], d["nbr_cnt"][:T], d["actions"]
        if (obs.dtype != torch.float32 or feat.dtype != torch.float32 or cnt.dtype != torch.int32
                or act.dtype != self._act_dtype):
            raise TypeError("the learner kernels are fp32: obs / nbr_feat float32, nbr_cnt int32, actions "
                            + ("float32" if self._act_dtype == torch.float32 else "int32"))
        n = cnt.numel()
        x = dict(obs=obs.reshape(n, abi.GSM_OBS_DIM), feat=feat.reshape(n, feat.shape[-2], abi.GSM_NBR_FEAT_DIM),
                 cnt=cnt.reshape(n), act=act.reshape((n,) + self._act_tail), old_logp=d["logp"].reshape(n),
                 old_v=d["values"][:T].reshape(n, 2), ret=d["returns"].reshape(n, 2),
                 adv=d["advantages"].reshape(n, 2))
        for k, t in x.items():
            if t.device != self.device or not t.is_contiguous():
                raise ValueError(f"buffer tensor {k} must be contiguous on {self.device}")
        return x

    def set_advantage_moments(self, adv):
        """adv_moments = (mu_0, sigma_0, mu_1, sigma_1): fp64 mean and population std over every row, per head."""
        a = adv.reshape(-1, 2).double()
        mu = a.mean(0)
        sd = (a - mu).square().mean(0).sqrt()
        self.adv_moments.copy_(torch.stack([mu[0], sd[0], mu[1], sd[1]]).float())

    def backward(self, x, rows, stats, value_affine=None):
        """gsm_ppo_backward(_gauss) over the source rows `rows` (int64 [n], or None for all of x): self.grad =
        dL/dparams of the §14 loss at self.params, stats [8] = its statistics.  With value_affine (a device
        fp32 [2, 2] (mu_h, sigma_h)), gsm_ppo_backward_normalized(_gauss): the value targets are normalised
        with it (§15).  Two launches, no host sync."""
        lib = abi.load_library()
        dev = self.device
        n = rows.numel() if rows is not None else x["cnt"].numel()
        need = getattr(lib, self._head.ppo_workspace)(n, *self._head.ws_args)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(max(need, 1), dtype=torch.uint8, device=dev)
        io = _eval_io(self._head, self.params, x["obs"], x["feat"], x["cnt"], x["act"], rows)
        loss = abi.GsmPpoLossIO()
        loss.struct_size = C.sizeof(abi.GsmPpoLossIO)
        loss.old_logp, loss.old_values = x["old_logp"].data_ptr(), x["old_v"].data_ptr()
        loss.returns, loss.advantages = x["ret"].data_ptr(), x["adv"].data_ptr()
        loss.adv_moments, loss.lagrange, loss.stats = (self.adv_moments.data_ptr(), self.lagrange.data_ptr(),
                                                       stats.data_ptr())
        loss.clip, loss.value_clip = self.clip, self.value_clip
        loss.value_coef, loss.entropy_coef = self.value_coef, self.entropy_coef
        if value_affine is None:
            _check(lib, getattr(lib, self._head.ppo_backward)(C.byref(io), C.byref(loss), self.grad.data_ptr(),
                                                              self._ws.data_ptr(), self._ws.numel(), dev.index or 0,
                                                              self._stream()))
        else:
            _check(lib, getattr(lib, self._head.ppo_backward_normalized)(
                C.byref(io), C.byref(loss), value_affine.data_ptr(), self.grad.data_ptr(), self._ws.data_ptr(),
                self._ws.numel(), dev.index or 0, self._stream()))

    def adam_step(self, grad_norm):
        """gsm_adam_step on (self.params, self.grad, self.m, self.v, self.step); grad_norm: a device float [1]."""
        lib = abi.load_library()
        _check(lib, lib.gsm_adam_step(self.params.data_ptr(), self.grad.data_ptr(), self.m.data_ptr(),
                                      self.v.data_ptr(), self.step.data_ptr(), self.params.numel(), self.lr,
                                      self.betas[0], self.betas[1], self.eps, self.max_grad_norm,
                                      grad_norm.data_ptr(), self.device.index or 0, self._stream()))

    def minibatch_step(self, x, rows, stats, value_affine=None):
        """backward then adam_step; stats [9]: the loss statistics, then the gradient norm.  Three launches."""
        self.backward(x, rows, stats, value_affine)
        self.adam_step(stats[abi.GSM_PPO_STAT_FIELDS:])

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- the update ---------------------------------------------------------------------------------
    def update(self, buf) -> torch.Tensor:
        """ppo_epoch x num_mini_batch minibatch steps over the buffer filled by collect + compute_returns.
        Minibatches: a seeded device permutation of the T * n_envs * N rows per epoch, cut into
        num_mini_batch parts of rows // num_mini_batch (the remainder is left out, as in the lineage).  With a
        value normaliser, one `value_norm.update` over the epoch's permutation precedes its minibatches.
        Returns stats [ppo_epoch * num_mini_batch, 9] (STAT_FIELDS) on the device.  No host sync between the
        first and the last launch; call `actor.pack()` afterwards for the collect kernels."""
        x = self.inputs(buf)
        n = x["cnt"].numel()
        mb = n // self.num_mini_batch
        if mb < 1:
            raise ValueError(f"{n} rows cannot make {self.num_mini_batch} minibatches")
        dev = self.device
        with torch.cuda.device(dev), torch.no_grad():
            self.params.copy_(torch.nn.utils.parameters_to_vector(self.actor.parameters()))
            self.set_advantage_moments(x["adv"])
            out = torch.empty(self.ppo_epoch * self.num_mini_batch, len(STAT_FIELDS), dtype=torch.float32, device=dev)
            k = 0
            for _ in range(self.ppo_epoch):
                perm = torch.randperm(n, generator=self.generator, device=dev)
                if self.value_norm is None:
                    for b in range(self.num_mini_batch):
                        self.minibatch_step(x, perm[b * mb:(b + 1) * mb], out[k])
                        k += 1
                else:
                    snaps = self.value_norm.update(x["ret"], perm, self.num_mini_batch)
                    for b in range(self.num_mini_batch):
                        self.minibatch_step(x, perm[b * mb:(b + 1) * mb], out[k], snaps[b])
                        k += 1
            self.write_back()
        return out

    def write_back(self):
        """Copy the parameter vector into the actor's parameters (vector_to_parameters order, no aliasing)."""
        with torch.no_grad():
            o = 0
            for p in self.actor.parameters():
                p.copy_(self.params[o:o + p.numel()].view_as(p))
                o += p.numel()

    def update_lagrange(self, totals: torch.Tensor) -> torch.Tensor:
        """lambda <- max(0, lambda + lagrangian_lr (team cost mean - cost_limit)) in fp64, from an EpisodeTracker
        totals vector (one update's or a window's sum); unchanged when it holds no team episode.  On the device."""
        if totals.shape != (abi.GSM_EPISODE_STAT_FIELDS,) or totals.device != self.device:
            raise ValueError(f"totals must be the [{abi.GSM_EPISODE_STAT_FIELDS}] EpisodeTracker vector on {self.device}")
        t = totals.double()
        c = t[8]
        gap = t[11] / torch.where(c > 0, c, torch.ones_like(c)) - self.cost_limit
        new = (self.lagrange.double()[0] + self.lagrangian_lr * gap).clamp_min(0.0)
        self.lagrange.copy_(torch.where(c > 0, new, self.lagrange.double()[0]).float().reshape(1))
        return self.lagrange

    # ---- checkpoints ----------------------------------------------------------------------------------
    def state_dict(self) -> dict:
        sd = {"params": self.params.clone(), "m": self.m.clone(), "v": self.v.clone(), "step": self.step.clone(),
              "lagrange": self.lagrange.clone(), "adv_moments": self.adv_moments.clone(),
              "generator": self.generator.get_state()}
        if self.value_norm is not None:
            sd["value_norm"] = self.value_norm.state_dict()
        return sd

    def load_state_dict(self, sd: dict):
        if ("value_norm" in sd) != (self.value_norm is not None):
            raise ValueError("the checkpoint and this trainer disagree on having a value normaliser")
        for k in ("params", "m", "v", "step", "lagrange", "adv_moments"):
            dst = getattr(self, k)
            if tuple(sd[k].shape) != tuple(dst.shape) or sd[k].dtype != dst.dtype:
                raise ValueError(f"state {k}: {tuple(sd[k].shape)} {sd[k].dtype}, expected {tuple(dst.shape)} {dst.dtype}")
            dst.copy_(sd[k])
        if "generator" in sd:
            self.generator.set_state(sd["generator"])
        if self.value_norm is not None:
            self.value_norm.load_state_dict(sd["value_norm"])
        self.write_back()
