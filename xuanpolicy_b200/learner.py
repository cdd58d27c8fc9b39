"""PPOCLIP_Learner drop-in (and the A2C / PG / PPO-KL / PPG learners that share its machinery).

Mirrors PPOCLIP_Learner (xuance/torch/learners/policy_gradient/ppoclip_learner.py:4-65) and its base Learner
(xuance/torch/learners/learner.py:10-52): same constructor, `update(obs_batch, act_batch, ret_batch, value_batch,
adv_batch, old_logp) -> info`, `save_model`, `load_model`, `iterations`.

`update` (compat — what an unmodified PPOCLIP_Agent calls): forwards the policy's torch modules, runs the loss
forward + backward w.r.t. the network outputs in one hand-written kernel (csrc/ppo_loss.cu), back-propagates through
the torch MLP and uses the caller's torch optimizer / scheduler exactly like the reference.
`update_from_buffer` / `stage_*` (native — what our vectorised agent calls): minibatch gather fused with the first MLP
layer, the hidden layers on the tcgen05 dense kernels with the loss in their epilogue (csrc/dense_tc.cu), hand-written
dgrad / wgrad into one flat gradient buffer, clip + Adam + LinearLR on the device (csrc/optim.cu); env-sharded, the
gradient exchange is a kernel over NVLink peer memory fused with the norm pass (csrc/peer_comm.cu; NCCL all-reduce as
the fallback).  No host synchronisation: the info scalars stay on the device until `info()` is asked for them.
"""
import os

import numpy as np
import torch

from . import ops
from . import dist as xdist
from .fused_mlp import FusedActorCritic
from .policies import old_dist_params


def _dist_params(a_dist):
    """('categorical', logits) or ('gaussian', mu, std) from a reference-shaped distribution wrapper
    (xuance/torch/utils/distributions.py:39-101: CategoricalDistribution.get_param / DiagGaussianDistribution.get_param)."""
    p = a_dist.get_param()
    if isinstance(p, (tuple, list)):
        return "gaussian", p[0], p[1]
    return "categorical", p, None


class FlatAdamState:
    """Flat fp32 views of the policy's parameters / gradients + Adam moments for csrc/optim.cu.

    Parameters are re-pointed at slices of one buffer (values preserved), `.grad` at slices of another, so
    torch autograd accumulates straight into the flat gradient and one NCCL all-reduce covers every tensor.
    Hyper-parameters are read from the torch optimizer / LinearLR scheduler the caller built
    (xuance/torch/runners/runner_drl.py:71-73)."""

    def __init__(self, policy, optimizer, scheduler):
        params = [p for p in policy.parameters() if p.requires_grad]
        dev = params[0].device
        pad4 = lambda k: (k + 3) // 4 * 4          # every tensor starts 16-byte aligned (float4 epilogue kernels)
        n = sum(pad4(p.numel()) for p in params)
        self.n = n
        self.n_params = sum(p.numel() for p in params)
        self.flat_param = torch.zeros(n, dtype=torch.float32, device=dev)
        self.flat_grad = torch.zeros(n, dtype=torch.float32, device=dev)
        self.grad_sum = None                        # peer mode: the cross-rank sum lands here (local memory)
        off = 0
        for p in params:
            k = p.numel()
            self.flat_param[off:off + k].copy_(p.data.reshape(-1))
            p.data = self.flat_param[off:off + k].view_as(p.data)
            p.grad = self.flat_grad[off:off + k].view_as(p.data)
            off += pad4(k)
        self.params = params
        self.grad_views = [p.grad for p in params]
        group = optimizer.param_groups[0]
        if group.get("weight_decay", 0) != 0 or group.get("amsgrad", False) or group.get("maximize", False):
            raise NotImplementedError("fused Adam supports plain Adam (no weight decay / amsgrad / maximize)")
        self.lr0 = float(group.get("initial_lr", group["lr"]))
        self.beta1, self.beta2 = (float(b) for b in group["betas"])
        self.eps = float(group["eps"])
        self.end_factor, self.total_iters = 1.0, 0
        if scheduler is not None:
            if not isinstance(scheduler, torch.optim.lr_scheduler.LinearLR) or scheduler.start_factor != 1.0:
                raise NotImplementedError("fused Adam supports LinearLR(start_factor=1.0) as built by the reference runner")
            self.end_factor, self.total_iters = float(scheduler.end_factor), int(scheduler.total_iters)
        self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
        self.step = torch.zeros(1, dtype=torch.int64, device=dev)
        self.workspace = torch.zeros(8 + 1024, dtype=torch.float64, device=dev)
        self.lr = torch.full((1,), self.lr0, dtype=torch.float32, device=dev)
        self.gnorm = torch.zeros(1, dtype=torch.float32, device=dev)

    def backward_into(self, outputs, grad_outputs):
        """d(loss)/d(params) straight into the flat gradient: `torch.autograd.grad` (fresh gradient tensors, no
        per-parameter accumulate kernels) followed by one multi-tensor copy.  Parameters that are not reached from
        `outputs` (e.g. logstd, whose gradient the loss kernel produces directly) get zero."""
        grads = torch.autograd.grad(outputs, self.params, grad_outputs, allow_unused=True)
        dst = [v for v, g in zip(self.grad_views, grads) if g is not None]
        src = [g for g in grads if g is not None]
        torch._foreach_copy_(dst, src)
        for v, g in zip(self.grad_views, grads):
            if g is None:
                v.zero_()

    def can_split(self, fused):
        """True if `adam` can rewrite `fused`'s operand copies in the same launch (its weights live in the flat buffer)."""
        return fused is not None and fused.la1.weight.data_ptr() >= self.flat_param.data_ptr()

    def adam(self, grad, fused=None, grad_scale=1.0, split=True):
        """Second pass of the step (scalars already in `workspace`).  With the tensor-core MLP active (`fused`) and `split`
        the same launch rewrites the tf32 hi/lo operand copies of the two hidden-layer weights (`fused.splits_fresh`
        tells the next forward that no separate split launch is needed); otherwise the copies are marked stale."""
        if split and self.can_split(fused):
            ops.adam_apply_split(self.flat_param, grad, self.exp_avg, self.exp_avg_sq, self.beta1, self.beta2, self.eps,
                                 grad_scale, self.workspace, fused.la1.weight.data, fused.wa_hi, fused.wa_lo,
                                 fused.lc1.weight.data, fused.wc_hi, fused.wc_lo, fused.wt_hi, fused.wt_lo)
            fused.splits_fresh = True
        else:
            ops.adam_apply(self.flat_param, grad, self.exp_avg, self.exp_avg_sq, self.beta1, self.beta2, self.eps,
                           grad_scale, self.workspace)
            if fused is not None:
                fused.splits_fresh = False

    def apply_peer(self, peer, max_norm, grad_scale=1.0, fused=None, split=True):
        """Env-sharded step: ONE kernel pushes this rank's gradient to every peer over NVLink, sums the W gradients in rank
        order and takes the norm of the sum (csrc/peer_comm.cu); the Adam kernel then consumes the sum."""
        if self.grad_sum is None:
            self.grad_sum = torch.zeros_like(self.flat_param)
        ops.peer_allreduce_grad_norm(peer, self.flat_grad, self.grad_sum, peer.tickets, self.step, self.lr0, self.end_factor,
                                     self.total_iters, self.beta1, self.beta2, self.eps, max_norm, grad_scale,
                                     self.workspace, lr_out=self.lr, gnorm_out=self.gnorm)
        self.adam(self.grad_sum, fused, grad_scale, split)

    def apply(self, max_norm, grad_scale=1.0):
        ops.clip_adam_step(self.flat_param, self.flat_grad, self.exp_avg, self.exp_avg_sq, self.step, self.lr0,
                           self.end_factor, self.total_iters, self.beta1, self.beta2, self.eps, max_norm, grad_scale,
                           self.workspace, lr_out=self.lr, gnorm_out=self.gnorm)


class PPOCLIP_Learner:
    def __init__(self, policy, optimizer, scheduler=None, device=None, model_dir="./", vf_coef=0.25, ent_coef=0.005,
                 clip_range=0.25, clip_grad_norm=0.25, use_grad_clip=True, value_clip=None):
        self.policy, self.optimizer, self.scheduler = policy, optimizer, scheduler
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("xuanpolicy_b200.PPOCLIP_Learner runs on a CUDA device only (no CPU fallback)")
        self.model_dir = model_dir
        self.iterations = 0
        self.vf_coef, self.ent_coef, self.clip_range = vf_coef, ent_coef, clip_range
        self.clip_grad_norm, self.use_grad_clip = clip_grad_norm, use_grad_clip
        self.value_clip = float(value_clip) if value_clip else 0.0   # opt-in; the reference has none (SURVEY App. F.1)
        self._scalars = torch.zeros(8, dtype=torch.float64, device=self.device)
        self._flat = None
        self._fused = None          # FusedActorCritic: the MLP on the tcgen05 dense kernels (native path, large batches)
        self.use_fused_mlp = os.environ.get("XB_FUSED_MLP", "1") != "0"
        self._mb = {}
        self.world_size, self.process_group = 1, None
        self._peer = None           # dist.PeerComm when env-sharded over NVLink peer memory
        self._dls64 = None          # fp64 log-std gradient written by the fused loss epilogue

    # ---------------------------------------------------------------------------------------------- checkpoints
    def save_model(self, model_path):
        torch.save(self.policy.state_dict(), model_path)

    def load_model(self, path, seed=1):
        for f in os.listdir(path):
            if "seed_%s" % seed in f:
                path = os.path.join(path, f)
                break
        names = sorted(n for n in os.listdir(path) if n != "obs_rms.npy")
        state = torch.load(os.path.join(path, names[-1]), map_location=self.device)
        self.policy.load_state_dict(state)
        if self._fused is not None:
            self._fused.splits_fresh = False      # the tf32 operand copies no longer match the weights
        return path

    # ---------------------------------------------------------------------------------------------- training state
    def state_tensors(self):
        """The learner's share of the agent's training state (PPOCLIP_Agent._state_tensors): the fused Adam's flat
        parameters, moments, step and learning rate, and the log scalars of the last update.  A learner whose torch
        optimiser steps (no flat state) holds its parameters in the policy: those are listed instead."""
        fl = self._flat
        named = {"learner.scalars": self._scalars}
        if fl is not None:
            named.update({"learner.flat_param": fl.flat_param, "learner.exp_avg": fl.exp_avg,
                          "learner.exp_avg_sq": fl.exp_avg_sq, "learner.step": fl.step, "learner.lr": fl.lr})
        else:
            named.update(("policy." + k, v) for k, v in self.policy.state_dict().items())
        return named

    def host_state(self):
        """Host-side training state: the update counter, and the torch optimiser's and scheduler's state where the torch
        optimiser is the one that steps."""
        st = {"iterations": self.iterations}
        if self._flat is None:
            st["optimizer"] = self.optimizer.state_dict()
            if self.scheduler is not None:
                st["scheduler"] = self.scheduler.state_dict()
        return st

    def load_host_state(self, st):
        self.iterations = st["iterations"]
        if "optimizer" in st:
            self.optimizer.load_state_dict(st["optimizer"])
        if "scheduler" in st:
            self.scheduler.load_state_dict(st["scheduler"])

    # ---------------------------------------------------------------------------------------------- loss kernel
    def _loss_backward(self, a_dist, v_pred, act, ret, adv, old_logp, val_old, inv_batch, idx=None, T=0, N=0,
                       adv_stats=None, adv_count=0, packed=None, flat=None, fused=None):
        """Fused loss fwd+bwd on the network outputs, then the MLP backward: torch autograd (into `.grad`, or — with
        `flat` — straight into the flat gradient buffer) or, with `fused`, the hand-written dgrad/wgrad kernels."""
        base = torch.autograd.backward if flat is None else flat.backward_into

        def backward(outs, grads):      # (an actor-only policy's stand-in value output is not part of the graph)
            live = [(o, g) for o, g in zip(outs, grads) if o.requires_grad]
            base([o for o, _ in live], [g for _, g in live])
        if fused is not None:      # (categorical: the loss kernel's two logit gradients are a softmax pair)
            backward = lambda outs, grads: fused.backward(grads[0], grads[1], softmax_pair=True)
        kind, p0, p1 = _dist_params(a_dist)
        v = v_pred.detach().contiguous()
        dv = torch.empty_like(v)
        common = dict(clip_range=self.clip_range, vf_coef=self.vf_coef, ent_coef=self.ent_coef, inv_batch=inv_batch,
                      idx=idx, T=T, N=N, val_old=val_old if self.value_clip > 0 else None, adv_stats=adv_stats,
                      adv_count=adv_count, value_clip=self.value_clip, packed=packed)
        if kind == "categorical":
            logits = p0.detach().contiguous()
            dlogits = torch.empty_like(logits)
            ops.ppo_loss_categorical(logits, v, act, ret, adv, old_logp, dlogits, dv, self._scalars, **common)
            backward([p0, v_pred], [dlogits, dv])
        else:
            mu = p0.detach().contiguous()
            std = p1
            param = getattr(getattr(self.policy, "actor", None), "logstd", None)   # gaussian.py:25
            direct = param is not None and param.requires_grad and param.numel() == mu.shape[1]
            logstd = param.detach() if direct else std.detach().log().contiguous()
            dmu = torch.empty_like(mu)
            dls = torch.empty(mu.shape[1], dtype=torch.float64, device=mu.device)
            ops.ppo_loss_gaussian(mu, logstd, v, act, ret, adv, old_logp, dmu, dls, dv, self._scalars, **common)
            if direct and fused is not None and flat is not None:   # fp64 -> fp32 log-std gradient inside the tail launch
                fused.backward(dmu, dv, dls, flat.grad_views[[id(q) for q in flat.params].index(id(param))])
            elif direct:           # the kernel's dL/dlogstd goes straight into the parameter's gradient
                backward([p0, v_pred], [dmu, dv])
                if flat is not None:
                    flat.grad_views[[id(q) for q in flat.params].index(id(param))].copy_(dls)
                elif param.grad is None:
                    param.grad = dls.to(param.dtype)
                else:
                    param.grad.add_(dls.to(param.dtype))
            elif std.requires_grad:  # d/dstd = d/dlogstd / std ; autograd carries it back to the logstd parameter
                backward([p0, v_pred, std], [dmu, dv, (dls / std.detach().double()).to(std.dtype)])
            else:
                backward([p0, v_pred], [dmu, dv])

    # ---------------------------------------------------------------------------------------------- compat update
    def update(self, obs_batch, act_batch, ret_batch, value_batch, adv_batch, old_logp):
        self.iterations += 1
        dev = self.device

        def dv_(x):
            return torch.as_tensor(x, device=dev).to(torch.float32).contiguous()

        with torch.cuda.device(dev):
            act, ret, val, adv = dv_(act_batch), dv_(ret_batch), dv_(value_batch), dv_(adv_batch)
            olp = dv_(old_logp) if old_logp is not None else None
            obs = torch.as_tensor(obs_batch, device=dev)
            B = ret.shape[0]
            out = self.policy(obs)
            a_dist = out[1]
            # actor-only policies (PG) have no critic: a zero value head that receives (and ignores) a zero gradient
            v_pred = out[2] if len(out) > 2 else torch.zeros(B, device=dev, requires_grad=True)
            self.optimizer.zero_grad()
            self._loss_backward(a_dist, v_pred, act.reshape(B, -1) if act.dim() > 1 else act, ret, adv, olp, val, 1.0 / B)
            if self.use_grad_clip:
                torch.nn.utils.clip_grad_norm_(self.policy.parameters(), self.clip_grad_norm)
            self.optimizer.step()
            if self.scheduler is not None:
                self.scheduler.step()
            lr = self.optimizer.state_dict()["param_groups"][0]["lr"]
            s = self._scalars.cpu().numpy() / B
        return {"actor-loss": float(-s[0]), "critic-loss": float(s[1]), "entropy": float(s[2]), "learning_rate": lr,
                "predict_value": float(s[3]), "clip_ratio": torch.tensor(s[4], dtype=torch.float32)}

    # ---------------------------------------------------------------------------------------------- native update
    def enable_fused_optimizer(self, process_group=None):
        """Switch to the flat-buffer fused clip+Adam+LinearLR step (native path).  The torch optimizer handed to
        the constructor is only read for its hyper-parameters from here on."""
        if process_group is not None or (torch.distributed.is_available() and torch.distributed.is_initialized()):
            self.process_group = process_group
            self.world_size = torch.distributed.get_world_size(process_group)
        if self._flat is None:
            self._flat = FlatAdamState(self.policy, self.optimizer, self.scheduler)
            if self.world_size > 1 and os.environ.get("XB_PEER_COMM", "1") != "0":
                self._open_peer_comm(self._flat.n)
            if self.use_fused_mlp and FusedActorCritic.plan(self.policy) is not None:
                self._fused = FusedActorCritic(self.policy)
        return self._flat

    def _open_peer_comm(self, n):
        """This rank's NVLink-visible comm block (dist.PeerComm).  Falls back to the NCCL all-reduce path (with a
        warning) when CUDA IPC is unavailable."""
        from .dist import PeerComm
        try:
            self._peer = PeerComm(n, self.device, self.process_group)
        except Exception as e:            # pragma: no cover - depends on the container's IPC permissions
            import warnings
            warnings.warn("peer-memory exchange unavailable (%s); using NCCL all-reduces" % (e,))
            self._peer = None

    def _minibatch_buffers(self, B, obs_dim):
        key = (B, obs_dim)
        if key not in self._mb:
            self._mb[key] = dict(obs=torch.empty((B, obs_dim), dtype=torch.float32, device=self.device),
                                 scal=torch.empty((B, 4), dtype=torch.float32, device=self.device),
                                 stats=torch.zeros(2, dtype=torch.float64, device=self.device))
        return self._mb[key]

    def stage_gather(self, memory, idx, compute_stats=True):
        """Stage 1 of a native update: gather the MLP input rows and (unless the caller already has the global ones)
        the minibatch advantage statistics."""
        mb = self._minibatch_buffers(idx.numel(), memory.obs_dim)
        want = memory.use_advnorm and compute_stats
        fused = self._fused if (self._fused is not None and idx.numel() >= FusedActorCritic.MIN_ROWS) else None
        mb["trunk_done"] = False
        # the first MLP layer: by the gather launch (xb_gather_trunk_fwd) or its own launch; XB_TRUNK_IN_FWD=1 generates it inside
        # the hidden-layer launch instead (xb_mlp_fwd_from_obs_train, bit-identical) — measured SLOWER at 65 536 x 128 (45 us
        # against 16.4 + 31.8 - 11.3 for gather+trunk, forward, plain gather: the operand warps become the forward's bottleneck)
        mb["trunk_in_fwd"] = fused is not None and fused.fwd_from_obs_ok() and os.environ.get("XB_TRUNK_IN_FWD", "0") == "1"
        if (fused is not None and memory.packed and self.value_clip <= 0 and fused.obs_dim <= 4 and not mb["trunk_in_fwd"]
                and os.environ.get("XB_GATHER_TRUNK", "1") != "0"):
            # gather + the MLP's first layer in one launch: the gathered rows feed the layer from registers
            b = fused._buffers(idx.numel())
            ops.gather_trunk_fwd(idx, memory.n_size, memory.n_envs, memory._rec, memory.obs_dim, fused.l0.weight.data,
                                 fused.l0.bias.data, fused.slope, mb["obs"], mb["scal"], b["h1"],
                                 stats=mb["stats"] if want else None, h1_signs=b.get("h1s"))
            mb["trunk_done"] = True
        elif memory.packed and self.value_clip <= 0:   # one 32-byte record per sample: obs + {act, old_logp, adv, ret}
            ops.gather_records(idx, memory.n_size, memory.n_envs, memory._rec, memory.obs_dim, mb["obs"], mb["scal"],
                               stats=mb["stats"] if want else None)
        else:
            ops.gather_obs(idx, memory.n_size, memory.n_envs, memory._obs, memory.obs_dim, mb["obs"],
                           b_adv=memory._adv if want else None, stats=mb["stats"] if want else None)
        return mb

    def stage_forward_backward(self, memory, idx, mb, stats=None):
        """Stage 2: torch MLP forward, fused gather+loss+backward kernel, torch MLP backward into the flat gradient.
        `stats` (fp64 [2], optional): the GLOBAL-minibatch (sum adv, sum adv^2) when the caller exchanged them itself."""
        B = idx.numel()
        fused = self._fused if (self._fused is not None and B >= FusedActorCritic.MIN_ROWS) else None
        if self._fused is not None:
            # single rank: the tail launch of the fused backward also takes the gradient norm (stage_optimizer then only
            # applies Adam); env-sharded, the norm belongs to the cross-rank sum and is taken by the peer kernel instead
            single = self.world_size == 1 and os.environ.get("XB_TAIL_NORM", "1") != "0"
            self._fused.norm_sink = (self._flat, self.clip_grad_norm if self.use_grad_clip else 0.0) if (fused is not None and single) else None
            self._fused.norm_done = False
        stats = (stats if stats is not None else mb["stats"]) if memory.use_advnorm else None
        if fused is not None and self._fused_loss_ok(memory, fused):
            # the loss forward + backward ride in the epilogue of the hidden-layer launch (csrc/dense_tc.cu FusedLoss)
            logstd = fused.policy.actor.logstd.detach() if fused.gaussian else None
            if fused.gaussian and self._dls64 is None:
                self._dls64 = torch.zeros(1, dtype=torch.float64, device=self.device)
            loss = dict(scal=mb["scal"], adv_stats=stats, adv_count=B * self.world_size, clip_range=self.clip_range,
                        vf_coef=self.vf_coef, ent_coef=self.ent_coef, inv_batch=1.0 / (B * self.world_size), logstd=logstd,
                        scalars=self._scalars, dlogstd=self._dls64 if fused.gaussian else None)
            # (rank-1 head gradients: the backward reads the hidden activations only through their sign words — not stored)
            fused.forward(mb["obs"], refresh=not fused.splits_fresh, trunk_done=mb.get("trunk_done", False), loss=loss,
                          keep_y=not fused.can_skip_y(softmax_pair=not fused.gaussian),
                          trunk_in_kernel=mb.get("trunk_in_fwd", False))
            b = fused._last[1]
            if fused.gaussian:
                flat = self._flat
                dls32 = flat.grad_views[[id(q) for q in flat.params].index(id(fused.policy.actor.logstd))]
                fused.backward(b["dact"], b["dv"], self._dls64, dls32)
            else:
                fused.backward(b["dact"], b["dv"], softmax_pair=True)
            return
        if fused is not None:                        # tcgen05 dense kernels; weights re-split after every Adam step
            act_out, v_pred = fused.forward(mb["obs"], refresh=not fused.splits_fresh, trunk_done=mb.get("trunk_done", False),
                                            trunk_in_kernel=mb.get("trunk_in_fwd", False))
            a_dist = fused.dist_params(act_out)
        else:
            out = self.policy(mb["obs"])
            a_dist = out[1]
            v_pred = out[2] if len(out) > 2 else torch.zeros(B, dtype=torch.float32, device=self.device)   # actor-only (PG)
        if memory.packed and self.value_clip <= 0:   # scalars already gathered, compact and coalesced
            self._loss_backward(a_dist, v_pred, None, None, None, None, None, 1.0 / (B * self.world_size),
                                adv_stats=stats, adv_count=B * self.world_size, packed=mb["scal"], flat=self._flat,
                                fused=fused)
        else:                                        # gather fused into the loss kernel
            self._loss_backward(a_dist, v_pred, memory._act, memory._ret, memory._adv, memory._logp, memory._val,
                                1.0 / (B * self.world_size), idx=idx, T=memory.n_size, N=memory.n_envs,
                                adv_stats=stats, adv_count=B * self.world_size, flat=self._flat, fused=fused)

    def _fused_loss_ok(self, memory, fused):
        """The loss can ride in the forward kernel's epilogue when the minibatch scalars are the packed float4 rows, there is
        no value clipping, and the actor head is Gaussian with one action dim and a directly-held log-std, or 2 logits."""
        if os.environ.get("XB_FUSED_LOSS", "1") == "0" or not (memory.packed and self.value_clip <= 0 and self._flat is not None):
            return False
        if fused.gaussian:
            p = getattr(fused.policy.actor, "logstd", None)
            return fused.A == 1 and p is not None and p.requires_grad and p.numel() == 1
        return fused.A == 2

    def stage_optimizer(self):
        """Stage 3: global-norm clip + Adam + LinearLR on the flat buffers (one fused device step).  Env-sharded over peer
        memory, the gradient exchange happens INSIDE this stage (fused with the norm pass)."""
        max_norm = self.clip_grad_norm if self.use_grad_clip else 0.0
        fused, split = self._fused, os.environ.get("XB_ADAM_SPLIT", "1") != "0"
        if self._peer is not None:
            self._flat.apply_peer(self._peer, max_norm, 1.0, fused, split)
        elif fused is not None and fused.norm_done:     # norm + step scalars came out of the backward tail launch
            self._flat.adam(self._flat.flat_grad, fused, 1.0, split)
            fused.norm_done = False
        else:
            self._flat.apply(max_norm, 1.0)
            if self._fused is not None:
                self._fused.splits_fresh = False

    def adam_resplits(self):
        """True if every `stage_optimizer` of the current configuration rewrites the fused MLP's tf32 operand copies
        (adam_apply_split): the peer-memory path and the single-rank tail-norm path, with XB_ADAM_SPLIT on.  False for
        the NCCL fallback / XB_TAIL_NORM=0 (clip_adam_step) and XB_ADAM_SPLIT=0 — there the first minibatch of every
        epoch must re-split (agent._epoch_start)."""
        if self._fused is None or self._flat is None or os.environ.get("XB_ADAM_SPLIT", "1") == "0":
            return False
        if not self._flat.can_split(self._fused):
            return False
        if self._peer is not None:
            return True
        return self.world_size == 1 and os.environ.get("XB_TAIL_NORM", "1") != "0" and self._fused_tail_norm_possible()

    def _fused_tail_norm_possible(self):
        f = self._fused
        return f is not None and not f.fold3 and (not f.gaussian or (getattr(f.policy.actor, "logstd", None) is not None
                                                     and f.policy.actor.logstd.numel() == 1))

    def update_from_buffer(self, memory, idx):
        """One PPO-Clip SGD step on the minibatch `idx` (CUDA int64 flat indices) of a native buffer.
        Env-sharded data parallel: the two collectives are the (sum, sumsq) of advantages and the flat gradient."""
        self.iterations += 1
        if self._flat is None:
            self.enable_fused_optimizer()
        mb = self.stage_gather(memory, idx)
        if self.world_size > 1 and memory.use_advnorm:
            xdist.allreduce_adv_stats(mb["stats"], self.process_group)
        self.stage_forward_backward(memory, idx, mb)
        if self.world_size > 1 and self._peer is None:
            xdist.allreduce_flat_grad(self._flat.flat_grad, self.process_group)
        self.stage_optimizer()

    def info(self, batch_size):
        """Host copy of the last update's log scalars (one sync; the native loop calls it once per rollout)."""
        s = self._scalars.cpu().numpy() / batch_size
        lr = float(self._flat.lr.item()) if self._flat is not None else self.optimizer.param_groups[0]["lr"]
        if self._flat is not None and self._flat.total_iters > 0:   # the reference reports the lr AFTER scheduler.step()
            it = min(int(self._flat.step.item()), self._flat.total_iters)
            lr = self._flat.lr0 * (1.0 + (self._flat.end_factor - 1.0) * it / self._flat.total_iters)
        return {"actor-loss": float(-s[0]), "critic-loss": float(s[1]), "entropy": float(s[2]), "learning_rate": lr,
                "predict_value": float(s[3]), "clip_ratio": torch.tensor(s[4], dtype=torch.float32)}


class A2C_Learner(PPOCLIP_Learner):
    """A2C_Learner drop-in (xuance/torch/learners/policy_gradient/a2c_learner.py:4-50): same constructor and
    `update(obs_batch, act_batch, ret_batch, adv_batch)`.  Same fused loss kernel with the A2C surrogate
    (`clip_range <= 0`: a_loss = -(adv * log_prob).mean()); the reference always clips the gradient norm (:36)."""

    def __init__(self, policy, optimizer, scheduler=None, device=None, model_dir="./", vf_coef=0.25, ent_coef=0.005,
                 clip_grad=None):
        super().__init__(policy, optimizer, scheduler, device, model_dir, vf_coef=vf_coef, ent_coef=ent_coef,
                         clip_range=0.0, clip_grad_norm=clip_grad, use_grad_clip=clip_grad is not None)
        self.clip_grad = clip_grad

    def update(self, obs_batch, act_batch, ret_batch, adv_batch):
        info = super().update(obs_batch, act_batch, ret_batch, ret_batch, adv_batch, None)
        info.pop("clip_ratio")
        return info


class PG_Learner(PPOCLIP_Learner):
    """PG_Learner drop-in (xuance/torch/learners/policy_gradient/pg_learner.py:4-45): actor-only policy
    (`policy(obs) -> (outputs, dist)`), a_loss = -(returns * log_prob).mean(), no value term."""

    def __init__(self, policy, optimizer, scheduler=None, device=None, model_dir="./", ent_coef=0.005, clip_grad=None):
        super().__init__(policy, optimizer, scheduler, device, model_dir, vf_coef=0.0, ent_coef=ent_coef, clip_range=0.0,
                         clip_grad_norm=clip_grad, use_grad_clip=clip_grad is not None)
        self.clip_grad = clip_grad

    def update(self, obs_batch, act_batch, ret_batch):
        info = super().update(obs_batch, act_batch, ret_batch, ret_batch, ret_batch, None)
        return {k: info[k] for k in ("actor-loss", "entropy", "learning_rate")}


# ---------------------------------------------------------------------------------------------------- PPO-KL / PPG
class _DistLossLearner(PPOCLIP_Learner):
    """Shared machinery of the learners whose loss needs the old action distribution (csrc/dist_loss.cu)."""

    def _dist_loss_backward(self, a_dist, v_pred, aux_v, act, ret, adv, old_dists, *, clip_range, surr_coef, kl_coef,
                            vf_coef, ent_coef, aux_coef=0.0, kl_coef_dev=None):
        """Runs the fused loss kernel on the network outputs and back-propagates through the torch MLP.  Only the
        outputs that carry a non-zero coefficient are back-propagated, so untouched sub-networks keep `grad = None`
        and the torch optimizer skips them exactly like the reference's `loss.backward()` does."""
        dev = self.device
        kind, p0, p1 = _dist_params(a_dist)
        okind, o0, o1 = old_dist_params(old_dists, dev)
        if okind != kind:
            raise TypeError("KL divergence needs two distributions of the same type")   # distributions.py:64-65
        B = ret.shape[0]
        v = v_pred.detach().contiguous()
        dv = torch.empty_like(v)
        aux = aux_v.detach().contiguous() if aux_v is not None else None
        daux = torch.empty_like(aux) if (aux is not None and aux_coef != 0.0) else None
        kw = dict(clip_range=clip_range, surr_coef=surr_coef, kl_coef=kl_coef, vf_coef=vf_coef, ent_coef=ent_coef,
                  inv_batch=1.0 / B, kl_coef_dev=kl_coef_dev, aux_v=aux, aux_coef=aux_coef, daux=daux)
        actor_live = surr_coef != 0.0 or kl_coef != 0.0 or ent_coef != 0.0
        outs, grads = [], []
        if vf_coef != 0.0:
            outs.append(v_pred)
            grads.append(dv)
        if daux is not None:
            outs.append(aux_v)
            grads.append(daux)
        if kind == "categorical":
            logits = p0.detach().contiguous()
            dlogits = torch.empty_like(logits)
            ops.dist_loss_categorical(logits, o0.reshape(B, -1), v, act.reshape(B), ret, adv, dlogits, dv, self._scalars, **kw)
            if actor_live:
                outs.append(p0)
                grads.append(dlogits)
            torch.autograd.backward(outs, grads)
            return B
        mu = p0.detach().contiguous()
        A = mu.shape[1]
        std = p1
        param = getattr(getattr(self.policy, "actor", None), "logstd", None)   # gaussian.py:25
        direct = param is not None and param.requires_grad and param.numel() == A
        logstd = param.detach() if direct else std.detach().log().contiguous()
        dmu = torch.empty_like(mu)
        dls = torch.empty(A, dtype=torch.float64, device=dev)
        old_std = o1.reshape(B, A) if o1.numel() == B * A else o1.reshape(A)
        ops.dist_loss_gaussian(mu, logstd, o0.reshape(B, A), old_std, v, act.reshape(B, A), ret, adv, dmu, dls, dv,
                               self._scalars, **kw)
        if actor_live:
            outs.append(p0)
            grads.append(dmu)
            if not direct and std.requires_grad:
                outs.append(std)
                grads.append((dls / std.detach().double()).to(std.dtype))
        torch.autograd.backward(outs, grads)
        if actor_live and direct:
            g = dls.to(param.dtype)
            param.grad = g if param.grad is None else param.grad.add_(g)
        return B * A

    def _prep(self, *arrays):
        return [torch.as_tensor(x, device=self.device).to(torch.float32).contiguous() for x in arrays]

    def _step(self, scheduler=True):
        self.optimizer.step()
        if scheduler and self.scheduler is not None:
            self.scheduler.step()
        return self.optimizer.state_dict()["param_groups"][0]["lr"]


class PPOKL_Learner(_DistLossLearner):
    """PPOKL_Learner drop-in (xuance/torch/learners/policy_gradient/ppokl_learner.py:5-61): same constructor and
    `update(obs_batch, act_batch, ret_batch, adv_batch, old_dists)`.  Loss + backward w.r.t. the network outputs
    in one kernel; the adaptive KL coefficient (:39-43) lives on the device (`kl_coef` reads it back).  No gradient
    clipping, like the reference."""

    def __init__(self, policy, optimizer, scheduler=None, device=None, model_dir="./", vf_coef=0.25, ent_coef=0.005,
                 target_kl=0.25):
        super().__init__(policy, optimizer, scheduler, device, model_dir, vf_coef=vf_coef, ent_coef=ent_coef,
                         clip_range=0.0, clip_grad_norm=None, use_grad_clip=False)
        self.target_kl = target_kl
        self._kl_coef_dev = torch.ones(1, dtype=torch.float32, device=self.device)

    def state_tensors(self):
        return dict(super().state_tensors(), **{"learner.kl_coef": self._kl_coef_dev})

    @property
    def kl_coef(self):
        return float(self._kl_coef_dev.item())

    @kl_coef.setter
    def kl_coef(self, value):
        self._kl_coef_dev.fill_(float(value))

    def update(self, obs_batch, act_batch, ret_batch, adv_batch, old_dists):
        self.iterations += 1
        with torch.cuda.device(self.device):
            act, ret, adv = self._prep(act_batch, ret_batch, adv_batch)
            B = ret.shape[0]
            _, a_dist, v_pred = self.policy(torch.as_tensor(obs_batch, device=self.device))
            kl_used = self._kl_coef_dev.clone()
            self.optimizer.zero_grad()
            kl_count = self._dist_loss_backward(a_dist, v_pred, None, act, ret, adv, old_dists, clip_range=0.0,
                                                surr_coef=1.0, kl_coef=1.0, vf_coef=self.vf_coef, ent_coef=self.ent_coef,
                                                kl_coef_dev=self._kl_coef_dev)
            ops.kl_coef_adapt(self._scalars, self._kl_coef_dev, self.target_kl, kl_count)   # takes effect next update
            lr = self._step()
            s = self._scalars.cpu().numpy()
            kl = float(s[5]) / kl_count
            a_loss = -float(s[0]) / B + float(kl_used.item()) * kl
        return {"actor-loss": a_loss, "critic-loss": float(s[1]) / B, "entropy": float(s[2]) / B, "learning_rate": lr,
                "kl": kl, "predict_value": float(s[3]) / B}


class PPG_Learner(_DistLossLearner):
    """PPG_Learner drop-in (xuance/torch/learners/policy_gradient/ppg_learner.py:5-91): same constructor and the
    three phase updates `update_policy / update_critic / update_auxiliary(obs, act, ret, adv, old_dists)` over a
    policy returning `(outputs, a_dist, v, aux_v)`.  Each phase is one launch of the generic kernel of
    csrc/dist_loss.cu with that phase's coefficients.

    `process_group` (or `enable_sharding`): env-sharded data parallelism over W ranks, each updating on its equal share of the
    minibatch.  Rank 0's parameters are broadcast once; after every phase's backward the gradients the phase reached are
    averaged over the ranks (xb_peer_allreduce_mean over NVLink peer memory; an NCCL all-reduce when XB_PEER_COMM=0 or CUDA IPC
    is unavailable), so the caller's torch optimiser takes the same step on every rank.  Parameters the phase did not reach
    keep `grad = None` and the optimiser skips them, as it does for the reference's `loss.backward()`."""

    def __init__(self, policy, optimizer, scheduler=None, device=None, model_dir="./", ent_coef=0.005, clip_range=0.25,
                 kl_beta=1.0, process_group=None):
        super().__init__(policy, optimizer, scheduler, device, model_dir, vf_coef=0.0, ent_coef=ent_coef,
                         clip_range=clip_range, clip_grad_norm=None, use_grad_clip=False)
        self.kl_beta = kl_beta
        self.policy_iterations = 0
        self.value_iterations = 0
        self.read_back = True       # False: the phase update returns {} without reading the log scalars back (no sync)
        self._shard = None          # (params, flat gradient in, flat mean out, their per-parameter views) when env-sharded
        if process_group is not None:
            self.enable_sharding(process_group)

    def host_state(self):
        return dict(super().host_state(), policy_iterations=self.policy_iterations, value_iterations=self.value_iterations)

    def load_host_state(self, st):
        super().load_host_state(st)
        self.policy_iterations, self.value_iterations = st["policy_iterations"], st["value_iterations"]

    def enable_sharding(self, process_group=None):
        """Switch to env-sharded updates when `process_group` (default: the initialised default group) has W > 1 ranks."""
        d = torch.distributed
        if self._shard is not None or (process_group is None and not (d.is_available() and d.is_initialized())):
            return
        world = d.get_world_size(process_group)
        if world == 1:
            return
        self.process_group, self.world_size = process_group, world
        params = [p for p in self.policy.parameters() if p.requires_grad]
        for p in params:                    # replicated policy: every rank starts from rank 0's parameters
            xdist.broadcast_parameters(p.data, 0, process_group)
        pad4 = lambda k: (k + 3) // 4 * 4   # the peer kernels move float4s
        offs = np.cumsum([0] + [pad4(p.numel()) for p in params])
        g_in = torch.zeros(int(offs[-1]), dtype=torch.float32, device=self.device)
        g_out = torch.zeros_like(g_in)
        view = lambda buf: [buf[o:o + p.numel()].view_as(p) for o, p in zip(offs, params)]
        self._shard = (params, g_in, g_out, view(g_in), view(g_out))
        if os.environ.get("XB_PEER_COMM", "1") != "0":
            self._open_peer_comm(g_in.numel())

    def _average_grads(self):
        """The gradients this phase reached -> one flat buffer -> mean over the ranks -> back into `.grad`."""
        params, g_in, g_out, v_in, v_out = self._shard
        live = [k for k, p in enumerate(params) if p.grad is not None]
        torch._foreach_copy_([v_in[k] for k in live], [params[k].grad for k in live])
        if self._peer is not None:
            ops.peer_allreduce_mean(self._peer, g_in, g_out)
        else:
            xdist.allreduce_flat_grad(g_in, self.process_group)
            torch.mul(g_in, 1.0 / self.world_size, out=g_out)
        torch._foreach_copy_([params[k].grad for k in live], [v_out[k] for k in live])

    def _backward_step(self, *args, scheduler=True, **kw):
        """_dist_loss_backward, the cross-rank gradient mean when env-sharded, then the optimiser (and scheduler) step."""
        count = self._dist_loss_backward(*args, **kw)
        if self._shard is not None:
            self._average_grads()
        return count, self._step(scheduler)

    def _forward(self, obs_batch):
        return self.policy(torch.as_tensor(obs_batch, device=self.device))

    def update_policy(self, obs_batch, act_batch, ret_batch, adv_batch, old_dists):
        with torch.cuda.device(self.device):
            act, ret, adv = self._prep(act_batch, ret_batch, adv_batch)
            B = ret.shape[0]
            _, a_dist, v, _ = self._forward(obs_batch)
            self.optimizer.zero_grad()
            _, lr = self._backward_step(a_dist, v, None, act, ret, adv, old_dists, clip_range=self.clip_range, surr_coef=1.0,
                                        kl_coef=0.0, vf_coef=0.0, ent_coef=self.ent_coef)
            self.policy_iterations += 1
            if not self.read_back:
                return {}
            s = self._scalars.cpu().numpy() / B
        return {"actor-loss": float(-s[0]), "entropy": float(s[2]), "learning_rate": lr,
                "clip_ratio": torch.tensor(s[4], dtype=torch.float32)}

    def update_critic(self, obs_batch, act_batch, ret_batch, adv_batch, old_dists):
        with torch.cuda.device(self.device):
            act, ret, adv = self._prep(act_batch, ret_batch, adv_batch)
            B = ret.shape[0]
            _, a_dist, v, _ = self._forward(obs_batch)
            self.optimizer.zero_grad()
            self._backward_step(a_dist, v, None, act, ret, adv, old_dists, clip_range=0.0, surr_coef=0.0, kl_coef=0.0,
                                vf_coef=1.0, ent_coef=0.0, scheduler=False)     # the reference steps no scheduler here (:63)
            self.value_iterations += 1
            if not self.read_back:
                return {}
            s = self._scalars.cpu().numpy() / B
        return {"critic-loss": float(s[1])}

    def update_auxiliary(self, obs_batch, act_batch, ret_batch, adv_batch, old_dists):
        with torch.cuda.device(self.device):
            act, ret, adv = self._prep(act_batch, ret_batch, adv_batch)
            B = ret.shape[0]
            _, a_dist, v, aux_v = self._forward(obs_batch)
            self.optimizer.zero_grad()
            kl_count, _ = self._backward_step(a_dist, v, aux_v, act, ret, adv, old_dists, clip_range=0.0, surr_coef=0.0,
                                              kl_coef=self.kl_beta, vf_coef=1.0, ent_coef=0.0, aux_coef=1.0,
                                              scheduler=False)                            # (:84)
            if not self.read_back:
                return {}
            s = self._scalars.cpu().numpy()
        return {"kl-loss": float(s[6]) / B + self.kl_beta * float(s[5]) / kl_count + float(s[1]) / B}

    def update(self):
        pass
