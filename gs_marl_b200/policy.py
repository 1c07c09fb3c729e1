"""Graph-attention actor over the env's padded neighbour rows — SURVEY.md §8 row f3 (the GNN
encoder forward of gsmarl/algorithms over torch-geometric, requirements.txt:119; withheld).

The architecture is the DECLARED one of SPEC.md §10 (the reference's is unknown): parameters
shared by all agents,
    e = relu(W_e obs + b_e);  m_r = relu(W_n feat_r + b_n) for the nbr_cnt valid rows;
    a = softmax_r(w_a . m_r + b_a);  z = W_h [e ; sum_r a_r m_r] + b_h;
    action = argmax_k(z_k + Gumbel_k)   (Philox4x32-10; `greedy` -> argmax_k z_k).

`act` is ONE sm_100a kernel through the C ABI (`gsm_policy_act`): forward + sampling + log-prob,
only the valid neighbour rows are read.  There is no fallback: `act` raises without the library
or a device.  `evaluate_actions` is the learner pass (SPEC.md §12): log-prob of given actions,
entropy and both critics, differentiable through a forward kernel (`gsm_policy_evaluate`) and a
backward kernel (`gsm_policy_backward`).  `logits_autograd` is the same function in plain torch ops
(the reference formulation the kernels are tested against); it is not used by `act` or by
`collect_fused`.

`GaussianGraphActor` is the same embedding with a diagonal Gaussian head for continuous-action
worlds (SPEC.md §10b / §12b): mean = W_mu h + b_mu, a state-independent log_std, float actions
[..., 2] = mean + exp(log_std) eps (Box-Muller on the same Philox stream), with the same kernels'
`act`, `collect_fused` and `evaluate_actions` paths.  `dist_autograd` is its plain-torch reference.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import abi

H = abi.GSM_POLICY_HIDDEN


def _seeded_linear(g):
    """Linear(i, o) factory drawing U(-1/sqrt(i), 1/sqrt(i)) weights and biases from generator g."""
    def lin(o, i):
        l = torch.nn.Linear(i, o)
        with torch.no_grad():
            bound = 1.0 / np.sqrt(i)
            l.weight.copy_((torch.rand(o, i, generator=g) * 2 - 1) * bound)
            l.bias.copy_((torch.rand(o, generator=g) * 2 - 1) * bound)
        return l
    return lin


class _GraphEmbedding(torch.nn.Module):
    """What both actors share: the embedding h = [e; sum_r a_r m_r] in plain torch, the packing of its
    weights and the input checks of the kernel paths.  Subclasses register ego, nbr, att, their head
    and value, in that order (parameters_to_vector order is the learner's vector layout)."""

    def _put_embedding(self, w, put):
        put("ego_w", self.ego.weight); put("ego_b", self.ego.bias)
        put("nbr_w", self.nbr.weight); put("nbr_b", self.nbr.bias)
        put("att_w", self.att.weight.reshape(-1))
        w.att_b = float(self.att.bias.item())
        put("value_w", self.value.weight); put("value_b", self.value.bias)

    def packed(self):
        """The last `pack()` (call `pack()` again after an optimizer step)."""
        return self._packed if self._packed is not None else self.pack()

    def embed_autograd(self, obs, graph):
        feat, cnt = graph["nbr_feat"], graph["nbr_cnt"]
        K = feat.shape[-2]
        e = torch.relu(self.ego(obs))
        m = torch.relu(self.nbr(feat))
        valid = torch.arange(K, device=obs.device) < cnt[..., None]
        sc = self.att(m).squeeze(-1).masked_fill(~valid, float("-inf"))
        a = torch.softmax(sc, -1).nan_to_num(0.0)            # rows with cnt == 0: all -inf -> 0
        agg = (a[..., None] * m).sum(-2)
        return torch.cat([e, agg], -1)


def _pack_into(w, field, t, rows=None):
    a = np.ascontiguousarray(t.detach().to("cpu", torch.float32).numpy())
    dst = np.ctypeslib.as_array(getattr(w, field))
    if rows is None:
        dst[...] = a.reshape(dst.shape)
    else:
        dst[:rows] = a


def _check_act_inputs(obs, feat, cnt):
    """The input checks of `act`; returns the leading shape."""
    if not obs.is_cuda:
        raise abi.GsmError("CUDA tensors required: gs_marl_b200 has no CPU fallback")
    if obs.dtype != torch.float32 or feat.dtype != torch.float32 or cnt.dtype != torch.int32:
        raise TypeError("the actor kernel is fp32 (production mode): obs/nbr_feat float32, nbr_cnt int32")
    if not (obs.is_contiguous() and feat.is_contiguous() and cnt.is_contiguous()):
        raise ValueError("obs, nbr_feat and nbr_cnt must be contiguous")
    lead = tuple(cnt.shape)
    if obs.shape != lead + (abi.GSM_OBS_DIM,) or feat.shape[:-2] != lead or feat.shape[-1] != abi.GSM_NBR_FEAT_DIM:
        raise ValueError("obs / nbr_feat / nbr_cnt shapes disagree")
    return lead


def _check_eval_inputs(params, obs, feat, cnt, actions, rows, act_dtype, act_tail):
    """The input checks of `evaluate_actions` (actions: act_dtype, shape lead + act_tail); returns rows
    made contiguous."""
    if not (obs.is_cuda and feat.is_cuda and cnt.is_cuda and actions.is_cuda):
        raise abi.GsmError("CUDA tensors required: gs_marl_b200 has no CPU fallback")
    dev = obs.device
    if params.device != dev or any(t.device != dev for t in (feat, cnt, actions)):
        raise abi.GsmError(f"the actor's parameters and all inputs must be on {dev}")
    if (params.dtype != torch.float32 or obs.dtype != torch.float32 or feat.dtype != torch.float32
            or cnt.dtype != torch.int32 or actions.dtype != act_dtype):
        an = "float32" if act_dtype == torch.float32 else "int32"
        raise TypeError(f"the learner kernels are fp32: parameters/obs/nbr_feat float32, nbr_cnt int32, actions {an}")
    if not (obs.is_contiguous() and feat.is_contiguous() and cnt.is_contiguous() and actions.is_contiguous()):
        raise ValueError("obs, nbr_feat, nbr_cnt and actions must be contiguous")
    lead = tuple(cnt.shape)
    if (obs.shape != lead + (abi.GSM_OBS_DIM,) or feat.shape[:-2] != lead
            or feat.shape[-1] != abi.GSM_NBR_FEAT_DIM or tuple(actions.shape) != lead + act_tail):
        raise ValueError("obs / nbr_feat / nbr_cnt / actions shapes disagree")
    if rows is not None:
        if rows.dtype != torch.int64 or rows.dim() != 1 or rows.device != dev:
            raise ValueError(f"rows must be a 1-D int64 tensor on {dev}")
        rows = rows.contiguous()
        if rows.numel() and not torch.cuda.is_current_stream_capturing():
            lo, hi = torch.aminmax(rows)
            if int(lo) < 0 or int(hi) >= cnt.numel():
                raise IndexError(f"rows out of range [0, {cnt.numel()})")
    return rows


class GraphAttentionActor(_GraphEmbedding):
    action_mode = "discrete"

    def __init__(self, n_actions: int = 5, seed: int = 0):
        super().__init__()
        if n_actions not in (5, 9):
            raise ValueError("compiled actor instances exist for 5 and 9 actions")
        self.n_actions = n_actions
        lin = _seeded_linear(torch.Generator().manual_seed(seed))
        self.ego = lin(H, abi.GSM_OBS_DIM)
        self.nbr = lin(H, abi.GSM_NBR_FEAT_DIM)
        self.att = lin(1, H)
        self.head = lin(n_actions, 2 * H)
        self.value = lin(abi.GSM_POLICY_VALUE_HEADS, 2 * H)     # [0] reward critic, [1] cost critic
        self._packed = None

    # ---- weights -> the C struct (host memory; they ride in the kernel's parameter space) ----
    def pack(self) -> abi.GsmPolicyWeights:
        w = abi.GsmPolicyWeights()
        w.struct_size = C.sizeof(abi.GsmPolicyWeights)
        w.n_actions = self.n_actions
        put = lambda field, t, rows=None: _pack_into(w, field, t, rows)
        self._put_embedding(w, put)
        put("head_w", self.head.weight, self.n_actions); put("head_b", self.head.bias, self.n_actions)
        self._packed = w
        return w

    # ---- collect path: one kernel ------------------------------------------------------------
    @torch.no_grad()
    def act(self, obs, graph, seed: int = 0, step: int = 0, row_offset: int = 0, greedy: bool = False,
            want_logits: bool = False, want_values: bool = False, out=None):
        """obs [..., 6], graph['nbr_feat'] [..., K, 6], graph['nbr_cnt'] [...] (fp32 / int32 CUDA
        tensors, contiguous) -> actions int32 [...], logp fp32 [...], then logits [..., n_actions] if
        want_logits, then values [..., 2] (reward critic, cost critic) if want_values."""
        lib = abi.load_library()
        feat, cnt = graph["nbr_feat"], graph["nbr_cnt"]
        lead = _check_act_inputs(obs, feat, cnt)
        n_rows = cnt.numel()
        dev = obs.device
        if out is None:
            actions = torch.empty(lead, dtype=torch.int32, device=dev)
            logp = torch.empty(lead, dtype=torch.float32, device=dev)
        else:
            actions, logp = out
        logits = torch.empty(lead + (self.n_actions,), dtype=torch.float32, device=dev) if want_logits else None
        io = abi.GsmPolicyIO()
        io.obs, io.nbr_feat, io.nbr_cnt = obs.data_ptr(), feat.data_ptr(), cnt.data_ptr()
        io.actions, io.logp = actions.data_ptr(), logp.data_ptr()
        io.logits = logits.data_ptr() if want_logits else None
        values = (torch.empty(lead + (abi.GSM_POLICY_VALUE_HEADS,), dtype=torch.float32, device=dev)
                  if want_values else None)
        io.values = values.data_ptr() if want_values else None
        io.n_rows, io.row_offset, io.seed, io.step = n_rows, int(row_offset), int(seed), int(step)
        io.max_nbrs, io.greedy = int(feat.shape[-2]), int(bool(greedy))
        st = lib.gsm_policy_act(C.byref(self.packed()), C.byref(io), dev.index or 0,
                                C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        if st != 0:
            raise abi.GsmError(f"{lib.gsm_status_string(st).decode()}: {lib.gsm_policy_last_error().decode()}")
        return (actions, logp) + ((logits,) if want_logits else ()) + ((values,) if want_values else ())

    # ---- learner pass: two kernels, differentiable ----------------------------------------------
    def evaluate_actions(self, obs, graph, actions, rows=None):
        """log pi(actions), entropy and the two critics, differentiable w.r.t. the parameters.

        obs [..., 6], graph['nbr_feat'] [..., K, 6], graph['nbr_cnt'] [...] and actions [...]
        (fp32 / int32 contiguous CUDA tensors on the parameters' device) are the source rows.  rows:
        optional int64 1-D index into the flattened source rows (a shuffled minibatch read straight
        out of the rollout buffer, no gather of nbr_feat).  Returns logp [n], entropy [n] and values
        [n, 2] with n = the source shape, or [len(rows)].  logp and values are bit-identical to what
        `act` / `collect_fused` wrote for the same rows and actions.  The range check on `rows`
        synchronises and is skipped while a CUDA graph is being captured."""
        feat, cnt = graph["nbr_feat"], graph["nbr_cnt"]
        params = torch.nn.utils.parameters_to_vector(self.parameters())
        rows = _check_eval_inputs(params, obs, feat, cnt, actions, rows, torch.int32, ())
        return _EvaluateActions.apply(params, obs, feat, cnt, actions, rows, _CAT_LEARNER[self.n_actions])

    # ---- the same function in plain torch (reference formulation; not used by the kernels) ----
    def logits_autograd(self, obs, graph):
        return self.head(self.embed_autograd(obs, graph))

    def values_autograd(self, obs, graph):
        return self.value(self.embed_autograd(obs, graph))


class _LogStd(torch.nn.Module):
    """The Gaussian head's state-independent log standard deviation (the lineage's AddBias): a child
    module so that parameters_to_vector lists it between the head and the critics."""

    def __init__(self, dim: int):
        super().__init__()
        self.weight = torch.nn.Parameter(torch.zeros(dim))

    def forward(self):
        return self.weight


class GaussianGraphActor(_GraphEmbedding):
    """The graph-attention embedding with a diagonal Gaussian head for continuous-action worlds
    (SPEC.md §10b): ego, nbr, att, head = Linear(2H, 2) (the mean), log_std (initialised to 0), value.
    Actions are float32 [..., 2], not clipped or squashed."""
    action_mode = "continuous"

    def __init__(self, seed: int = 0):
        super().__init__()
        lin = _seeded_linear(torch.Generator().manual_seed(seed))
        self.ego = lin(H, abi.GSM_OBS_DIM)
        self.nbr = lin(H, abi.GSM_NBR_FEAT_DIM)
        self.att = lin(1, H)
        self.head = lin(abi.GSM_POLICY_GAUSS_DIM, 2 * H)
        self.log_std = _LogStd(abi.GSM_POLICY_GAUSS_DIM)
        self.value = lin(abi.GSM_POLICY_VALUE_HEADS, 2 * H)     # [0] reward critic, [1] cost critic
        self._packed = None

    def pack(self) -> abi.GsmPolicyGaussWeights:
        w = abi.GsmPolicyGaussWeights()
        w.struct_size = C.sizeof(abi.GsmPolicyGaussWeights)
        put = lambda field, t: _pack_into(w, field, t)
        self._put_embedding(w, put)
        put("mean_w", self.head.weight); put("mean_b", self.head.bias); put("log_std", self.log_std())
        self._packed = w
        return w

    @torch.no_grad()
    def act(self, obs, graph, seed: int = 0, step: int = 0, row_offset: int = 0, greedy: bool = False,
            want_mean: bool = False, want_values: bool = False, out=None):
        """obs [..., 6], graph['nbr_feat'] [..., K, 6], graph['nbr_cnt'] [...] (fp32 / int32 CUDA
        tensors, contiguous) -> actions float32 [..., 2], logp fp32 [...], then the mean [..., 2] if
        want_mean, then values [..., 2] (reward critic, cost critic) if want_values.  greedy: the mean."""
        lib = abi.load_library()
        feat, cnt = graph["nbr_feat"], graph["nbr_cnt"]
        lead = _check_act_inputs(obs, feat, cnt)
        dev = obs.device
        D = abi.GSM_POLICY_GAUSS_DIM
        if out is None:
            actions = torch.empty(lead + (D,), dtype=torch.float32, device=dev)
            logp = torch.empty(lead, dtype=torch.float32, device=dev)
        else:
            actions, logp = out
        mean = torch.empty(lead + (D,), dtype=torch.float32, device=dev) if want_mean else None
        values = (torch.empty(lead + (abi.GSM_POLICY_VALUE_HEADS,), dtype=torch.float32, device=dev)
                  if want_values else None)
        io = abi.GsmPolicyGaussIO()
        io.obs, io.nbr_feat, io.nbr_cnt = obs.data_ptr(), feat.data_ptr(), cnt.data_ptr()
        io.actions, io.logp, io.mean, io.values = actions.data_ptr(), logp.data_ptr(), _ptr(mean), _ptr(values)
        io.n_rows, io.row_offset, io.seed, io.step = cnt.numel(), int(row_offset), int(seed), int(step)
        io.max_nbrs, io.greedy = int(feat.shape[-2]), int(bool(greedy))
        _check(lib, lib.gsm_policy_act_gauss(C.byref(self.packed()), C.byref(io), dev.index or 0,
                                             C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        return (actions, logp) + ((mean,) if want_mean else ()) + ((values,) if want_values else ())

    def evaluate_actions(self, obs, graph, actions, rows=None):
        """log pi(actions), entropy and the two critics, differentiable w.r.t. the parameters, as
        `GraphAttentionActor.evaluate_actions` with float32 actions [..., 2]."""
        feat, cnt = graph["nbr_feat"], graph["nbr_cnt"]
        params = torch.nn.utils.parameters_to_vector(self.parameters())
        rows = _check_eval_inputs(params, obs, feat, cnt, actions, rows, torch.float32, (abi.GSM_POLICY_GAUSS_DIM,))
        return _EvaluateActions.apply(params, obs, feat, cnt, actions, rows, _GAUSS_LEARNER)

    # ---- the same function in plain torch (reference formulation; not used by the kernels) ----
    def dist_autograd(self, obs, graph):
        """torch.distributions.Normal(mean, exp(log_std)) per row and dimension."""
        mean = self.head(self.embed_autograd(obs, graph))
        return torch.distributions.Normal(mean, self.log_std().exp().expand_as(mean))

    def values_autograd(self, obs, graph):
        return self.value(self.embed_autograd(obs, graph))


class _Learner:
    """The learner entry points of one head: the eval-io struct and its head field, the C functions."""

    def __init__(self, io_cls, head_field, head_value, evaluate, backward, workspace):
        self.io_cls, self.head_field, self.head_value = io_cls, head_field, head_value
        self.evaluate, self.backward, self.workspace = evaluate, backward, workspace


_CAT_LEARNER = {a: _Learner(abi.GsmPolicyEvalIO, "n_actions", a, "gsm_policy_evaluate", "gsm_policy_backward",
                            lambda lib, n, a=a: lib.gsm_policy_backward_workspace(n, a)) for a in (5, 9)}
_GAUSS_LEARNER = _Learner(abi.GsmPolicyGaussEvalIO, "action_dim", abi.GSM_POLICY_GAUSS_DIM,
                          "gsm_policy_evaluate_gauss", "gsm_policy_backward_gauss",
                          lambda lib, n: lib.gsm_policy_backward_workspace_gauss(n))


def _eval_io(head, params, obs, feat, cnt, actions, rows):
    io = head.io_cls()
    io.struct_size = C.sizeof(head.io_cls)
    setattr(io, head.head_field, head.head_value)
    io.params, io.obs, io.nbr_feat = params.data_ptr(), obs.data_ptr(), feat.data_ptr()
    io.nbr_cnt, io.actions = cnt.data_ptr(), actions.data_ptr()
    io.rows = rows.data_ptr() if rows is not None else None
    io.n_rows = rows.numel() if rows is not None else cnt.numel()
    io.max_nbrs = int(feat.shape[-2])
    return io


def _ptr(t):
    return t.data_ptr() if t is not None else None


class _EvaluateActions(torch.autograd.Function):
    """forward: gsm_policy_evaluate(_gauss); backward: gsm_policy_backward(_gauss) (grad w.r.t. the
    parameter vector)."""

    @staticmethod
    def forward(ctx, params, obs, feat, cnt, actions, rows, head):
        lib = abi.load_library()
        params = params.contiguous()
        dev = obs.device
        shape = (rows.numel(),) if rows is not None else tuple(cnt.shape)
        logp = torch.empty(shape, dtype=torch.float32, device=dev)
        entropy = torch.empty(shape, dtype=torch.float32, device=dev)
        values = torch.empty(shape + (abi.GSM_POLICY_VALUE_HEADS,), dtype=torch.float32, device=dev)
        io = _eval_io(head, params, obs, feat, cnt, actions, rows)
        io.logp, io.entropy, io.values = logp.data_ptr(), entropy.data_ptr(), values.data_ptr()
        _check(lib, getattr(lib, head.evaluate)(C.byref(io), dev.index or 0,
                                                C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        ctx.save_for_backward(params, obs, feat, cnt, actions, rows)
        ctx.head = head
        ctx.set_materialize_grads(False)          # an unused output arrives as None -> NULL (zero)
        return logp, entropy, values

    @staticmethod
    def backward(ctx, d_logp, d_entropy, d_values):
        lib = abi.load_library()
        params, obs, feat, cnt, actions, rows = ctx.saved_tensors
        dev = obs.device
        io = _eval_io(ctx.head, params, obs, feat, cnt, actions, rows)
        if not io.n_rows:
            return torch.zeros_like(params), None, None, None, None, None, None
        grad = torch.empty_like(params)
        ws = torch.empty(ctx.head.workspace(lib, io.n_rows), dtype=torch.uint8, device=dev)
        d = [g.contiguous() if g is not None else None for g in (d_logp, d_entropy, d_values)]
        _check(lib, getattr(lib, ctx.head.backward)(C.byref(io), _ptr(d[0]), _ptr(d[1]), _ptr(d[2]), grad.data_ptr(),
                                            ws.data_ptr(), ws.numel(), dev.index or 0,
                                            C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        return grad, None, None, None, None, None, None


def _check(lib, st):
    if st != 0:
        raise abi.GsmError(f"{lib.gsm_status_string(st).decode()}: {lib.gsm_policy_last_error().decode()}")
