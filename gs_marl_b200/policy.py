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
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import abi

H = abi.GSM_POLICY_HIDDEN


class GraphAttentionActor(torch.nn.Module):
    def __init__(self, n_actions: int = 5, seed: int = 0):
        super().__init__()
        if n_actions not in (5, 9):
            raise ValueError("compiled actor instances exist for 5 and 9 actions")
        self.n_actions = n_actions
        g = torch.Generator().manual_seed(seed)

        def lin(o, i):
            l = torch.nn.Linear(i, o)
            with torch.no_grad():
                bound = 1.0 / np.sqrt(i)
                l.weight.copy_((torch.rand(o, i, generator=g) * 2 - 1) * bound)
                l.bias.copy_((torch.rand(o, generator=g) * 2 - 1) * bound)
            return l
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

        def put(field, t, rows=None):
            a = np.ascontiguousarray(t.detach().to("cpu", torch.float32).numpy())
            dst = np.ctypeslib.as_array(getattr(w, field))
            if rows is None:
                dst[...] = a.reshape(dst.shape)
            else:
                dst[:rows] = a
        put("ego_w", self.ego.weight); put("ego_b", self.ego.bias)
        put("nbr_w", self.nbr.weight); put("nbr_b", self.nbr.bias)
        put("att_w", self.att.weight.reshape(-1))
        w.att_b = float(self.att.bias.item())
        put("head_w", self.head.weight, self.n_actions); put("head_b", self.head.bias, self.n_actions)
        put("value_w", self.value.weight); put("value_b", self.value.bias)
        self._packed = w
        return w

    def packed(self) -> abi.GsmPolicyWeights:
        """The last `pack()` (call `pack()` again after an optimizer step)."""
        return self._packed if self._packed is not None else self.pack()

    # ---- collect path: one kernel ------------------------------------------------------------
    @torch.no_grad()
    def act(self, obs, graph, seed: int = 0, step: int = 0, row_offset: int = 0, greedy: bool = False,
            want_logits: bool = False, want_values: bool = False, out=None):
        """obs [..., 6], graph['nbr_feat'] [..., K, 6], graph['nbr_cnt'] [...] (fp32 / int32 CUDA
        tensors, contiguous) -> actions int32 [...], logp fp32 [...], then logits [..., n_actions] if
        want_logits, then values [..., 2] (reward critic, cost critic) if want_values."""
        lib = abi.load_library()
        feat, cnt = graph["nbr_feat"], graph["nbr_cnt"]
        if not obs.is_cuda:
            raise abi.GsmError("CUDA tensors required: gs_marl_b200 has no CPU fallback")
        if obs.dtype != torch.float32 or feat.dtype != torch.float32 or cnt.dtype != torch.int32:
            raise TypeError("the actor kernel is fp32 (production mode): obs/nbr_feat float32, nbr_cnt int32")
        if not (obs.is_contiguous() and feat.is_contiguous() and cnt.is_contiguous()):
            raise ValueError("obs, nbr_feat and nbr_cnt must be contiguous")
        lead = tuple(cnt.shape)
        n_rows = cnt.numel()
        if obs.shape != lead + (abi.GSM_OBS_DIM,) or feat.shape[:-2] != lead or feat.shape[-1] != abi.GSM_NBR_FEAT_DIM:
            raise ValueError("obs / nbr_feat / nbr_cnt shapes disagree")
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
        if not (obs.is_cuda and feat.is_cuda and cnt.is_cuda and actions.is_cuda):
            raise abi.GsmError("CUDA tensors required: gs_marl_b200 has no CPU fallback")
        dev = obs.device
        if params.device != dev or any(t.device != dev for t in (feat, cnt, actions)):
            raise abi.GsmError(f"the actor's parameters and all inputs must be on {dev}")
        if (params.dtype != torch.float32 or obs.dtype != torch.float32 or feat.dtype != torch.float32
                or cnt.dtype != torch.int32 or actions.dtype != torch.int32):
            raise TypeError("the learner kernels are fp32: parameters/obs/nbr_feat float32, nbr_cnt/actions int32")
        if not (obs.is_contiguous() and feat.is_contiguous() and cnt.is_contiguous() and actions.is_contiguous()):
            raise ValueError("obs, nbr_feat, nbr_cnt and actions must be contiguous")
        lead = tuple(cnt.shape)
        if (obs.shape != lead + (abi.GSM_OBS_DIM,) or feat.shape[:-2] != lead
                or feat.shape[-1] != abi.GSM_NBR_FEAT_DIM or tuple(actions.shape) != lead):
            raise ValueError("obs / nbr_feat / nbr_cnt / actions shapes disagree")
        if rows is not None:
            if rows.dtype != torch.int64 or rows.dim() != 1 or rows.device != dev:
                raise ValueError(f"rows must be a 1-D int64 tensor on {dev}")
            rows = rows.contiguous()
            if rows.numel() and not torch.cuda.is_current_stream_capturing():
                lo, hi = torch.aminmax(rows)
                if int(lo) < 0 or int(hi) >= cnt.numel():
                    raise IndexError(f"rows out of range [0, {cnt.numel()})")
        return _EvaluateActions.apply(params, obs, feat, cnt, actions, rows, self.n_actions)

    # ---- the same function in plain torch (reference formulation; not used by the kernels) ----
    def logits_autograd(self, obs, graph):
        return self.head(self.embed_autograd(obs, graph))

    def values_autograd(self, obs, graph):
        return self.value(self.embed_autograd(obs, graph))

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


def _eval_io(n_actions, params, obs, feat, cnt, actions, rows) -> abi.GsmPolicyEvalIO:
    io = abi.GsmPolicyEvalIO()
    io.struct_size, io.n_actions = C.sizeof(abi.GsmPolicyEvalIO), n_actions
    io.params, io.obs, io.nbr_feat = params.data_ptr(), obs.data_ptr(), feat.data_ptr()
    io.nbr_cnt, io.actions = cnt.data_ptr(), actions.data_ptr()
    io.rows = rows.data_ptr() if rows is not None else None
    io.n_rows = rows.numel() if rows is not None else cnt.numel()
    io.max_nbrs = int(feat.shape[-2])
    return io


def _ptr(t):
    return t.data_ptr() if t is not None else None


class _EvaluateActions(torch.autograd.Function):
    """forward: gsm_policy_evaluate; backward: gsm_policy_backward (grad w.r.t. the parameter vector)."""

    @staticmethod
    def forward(ctx, params, obs, feat, cnt, actions, rows, n_actions):
        lib = abi.load_library()
        params = params.contiguous()
        dev = obs.device
        shape = (rows.numel(),) if rows is not None else tuple(cnt.shape)
        logp = torch.empty(shape, dtype=torch.float32, device=dev)
        entropy = torch.empty(shape, dtype=torch.float32, device=dev)
        values = torch.empty(shape + (abi.GSM_POLICY_VALUE_HEADS,), dtype=torch.float32, device=dev)
        io = _eval_io(n_actions, params, obs, feat, cnt, actions, rows)
        io.logp, io.entropy, io.values = logp.data_ptr(), entropy.data_ptr(), values.data_ptr()
        _check(lib, lib.gsm_policy_evaluate(C.byref(io), dev.index or 0,
                                            C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        ctx.save_for_backward(params, obs, feat, cnt, actions, rows)
        ctx.n_actions = n_actions
        ctx.set_materialize_grads(False)          # an unused output arrives as None -> NULL (zero)
        return logp, entropy, values

    @staticmethod
    def backward(ctx, d_logp, d_entropy, d_values):
        lib = abi.load_library()
        params, obs, feat, cnt, actions, rows = ctx.saved_tensors
        dev = obs.device
        io = _eval_io(ctx.n_actions, params, obs, feat, cnt, actions, rows)
        if not io.n_rows:
            return torch.zeros_like(params), None, None, None, None, None, None
        grad = torch.empty_like(params)
        ws = torch.empty(lib.gsm_policy_backward_workspace(io.n_rows, ctx.n_actions), dtype=torch.uint8, device=dev)
        d = [g.contiguous() if g is not None else None for g in (d_logp, d_entropy, d_values)]
        _check(lib, lib.gsm_policy_backward(C.byref(io), _ptr(d[0]), _ptr(d[1]), _ptr(d[2]), grad.data_ptr(),
                                            ws.data_ptr(), ws.numel(), dev.index or 0,
                                            C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        return grad, None, None, None, None, None, None


def _check(lib, st):
    if st != 0:
        raise abi.GsmError(f"{lib.gsm_status_string(st).decode()}: {lib.gsm_policy_last_error().decode()}")
