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
"""
from __future__ import annotations

import ctypes as C

import torch

from . import abi
from .policy import GaussianGraphActor, GraphAttentionActor, _check, _eval_io

# the columns of `update`'s result: the GSM_PPO_STAT_FIELDS loss statistics, then the gradient norm
STAT_FIELDS = ("policy_loss", "value_loss_reward", "value_loss_cost", "entropy", "ratio", "clip_fraction",
               "approx_kl", "loss", "grad_norm")


class LagrangianPPO:
    """Owns the flat parameter vector (parameters_to_vector order), Adam's m, v and step, and lambda, all on
    the actor's device.  Every hyper-parameter is a required keyword (`presets.UNVERIFIED_PPO_LAG` holds
    lineage-typical values); the library has no defaults."""

    def __init__(self, actor, *, clip, value_clip, value_coef, entropy_coef, lr, betas, eps, max_grad_norm,
                 ppo_epoch, num_mini_batch, lagrangian_lr, cost_limit, lagrangian_init=0.0, seed):
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

    def backward(self, x, rows, stats):
        """gsm_ppo_backward(_gauss) over the source rows `rows` (int64 [n], or None for all of x): self.grad =
        dL/dparams of the §14 loss at self.params, stats [8] = its statistics.  Two launches, no host sync."""
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
        _check(lib, getattr(lib, self._head.ppo_backward)(C.byref(io), C.byref(loss), self.grad.data_ptr(),
                                                          self._ws.data_ptr(), self._ws.numel(), dev.index or 0,
                                                          self._stream()))

    def adam_step(self, grad_norm):
        """gsm_adam_step on (self.params, self.grad, self.m, self.v, self.step); grad_norm: a device float [1]."""
        lib = abi.load_library()
        _check(lib, lib.gsm_adam_step(self.params.data_ptr(), self.grad.data_ptr(), self.m.data_ptr(),
                                      self.v.data_ptr(), self.step.data_ptr(), self.params.numel(), self.lr,
                                      self.betas[0], self.betas[1], self.eps, self.max_grad_norm,
                                      grad_norm.data_ptr(), self.device.index or 0, self._stream()))

    def minibatch_step(self, x, rows, stats):
        """backward then adam_step; stats [9]: the loss statistics, then the gradient norm.  Three launches."""
        self.backward(x, rows, stats)
        self.adam_step(stats[abi.GSM_PPO_STAT_FIELDS:])

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- the update ---------------------------------------------------------------------------------
    def update(self, buf) -> torch.Tensor:
        """ppo_epoch x num_mini_batch minibatch steps over the buffer filled by collect + compute_returns.
        Minibatches: a seeded device permutation of the T * n_envs * N rows per epoch, cut into
        num_mini_batch parts of rows // num_mini_batch (the remainder is left out, as in the lineage).
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
                for b in range(self.num_mini_batch):
                    self.minibatch_step(x, perm[b * mb:(b + 1) * mb], out[k])
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
        return {"params": self.params.clone(), "m": self.m.clone(), "v": self.v.clone(), "step": self.step.clone(),
                "lagrange": self.lagrange.clone(), "adv_moments": self.adv_moments.clone(),
                "generator": self.generator.get_state()}

    def load_state_dict(self, sd: dict):
        for k in ("params", "m", "v", "step", "lagrange", "adv_moments"):
            dst = getattr(self, k)
            if tuple(sd[k].shape) != tuple(dst.shape) or sd[k].dtype != dst.dtype:
                raise ValueError(f"state {k}: {tuple(sd[k].shape)} {sd[k].dtype}, expected {tuple(dst.shape)} {dst.dtype}")
            dst.copy_(sd[k])
        if "generator" in sd:
            self.generator.set_state(sd["generator"])
        self.write_back()
