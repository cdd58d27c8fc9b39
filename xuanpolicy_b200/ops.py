"""Torch-tensor front-end of the C ABI: derives raw device pointers + the current CUDA stream and calls
libxb200.  No arithmetic happens here and nothing falls back to torch ops: a CPU tensor is an error.

Every function only enqueues work on `torch.cuda.current_stream()` (graph-capturable).
"""
import torch

from . import _lib

ENV_KINDS = {"CartPole-v1": 0, "CartPole-v0": 0, "Pendulum-v1": 1, "gym:MountainCar-v0": 2, "Acrobot-v1": 3, "MountainCar-v0": 4,
             "gym:MountainCarContinuous-v0": 5, "MountainCarContinuous-v0": 6}
# env kinds with a Box action: float32 actions [N] in and out of the env kernels; every other kind takes int64 actions
CONTINUOUS_KINDS = frozenset({1, 5, 6})
GAE_VARIANTS = {"auto": 0, "ldg": 1, "tma": 2}


def _p(t, dtype=None):
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.XB200Error("xb200 kernels take CUDA tensors (got a %s tensor); there is no CPU path" % t.device)
    if not t.is_contiguous():
        raise _lib.XB200Error("xb200 kernels take contiguous tensors")
    if dtype is not None and t.dtype != dtype:
        raise _lib.XB200Error("expected dtype %s, got %s" % (dtype, t.dtype))
    return t.data_ptr()


def continuous_kind(kind):
    """True for the env kinds whose action is one float32 per env (include/xb200.h XB_ENV_*)."""
    return kind in CONTINUOUS_KINDS


def _stream():
    return torch.cuda.current_stream().cuda_stream


F32, F64, I64, I32, U8 = torch.float32, torch.float64, torch.int64, torch.int32, torch.uint8


def _act_dtype(kind):
    return F32 if continuous_kind(kind) else I64


def env_reset(kind, state, rng, elapsed, ep_score, obs, n_draws):
    N = elapsed.numel()
    _lib.call("xb_env_reset", kind, _p(state, F64), _p(rng, I64), _p(elapsed, I32), _p(ep_score, F64), _p(obs, F32),
              n_draws, N, _stream())


def env_step(kind, state, rng, elapsed, ep_score, actions, obs, next_obs, rew, term, trunc, reset_obs, ep_step_out,
             ep_score_out, max_steps, ep_stats=None):
    N = elapsed.numel()
    _lib.call("xb_env_step", kind, _p(state, F64), _p(rng, I64), _p(elapsed, I32), _p(ep_score, F64),
              _p(actions, _act_dtype(kind)), _p(obs, F32), _p(next_obs, F32), _p(rew, F32), _p(term, U8),
              _p(trunc, U8), _p(reset_obs, F32), _p(ep_step_out, I32), _p(ep_score_out, F64), _p(ep_stats, F64), max_steps,
              N, _stream())


def rollout_step(kind, act_param, logstd, val, seed, counter, offset, state, rng, elapsed, ep_score, obs, next_obs, rew,
                 term, trunc, reset_obs, ep_step_out, ep_score_out, ep_stats, max_steps, x_in, act_out, logp_out, obs_row,
                 act_row, rew_row, val_row, term_row, trunc_row, logp_row, rew_std=None, rew_clip=0.0, boot_src=None,
                 boot_row=None, trig_cache=None, stats=None, dist_row=None):
    """sample + env step + store of one vector step in one launch (see xb_rollout_step in include/xb200.h).
    `stats` (dict, optional): running statistics carried by the launch — obs_in / obs_out (normaliser states), obs_dim,
    obs_clip, ret_state, returns, gamma, mask_terminal, partials, ticket; `rew_std` is then also rewritten for the next step.
    `dist_row` (optional, f32 [N, W]): receives the parameters of the distribution each action was drawn from."""
    N = elapsed.numel()
    st = stats or {}
    _lib.call("xb_rollout_step", kind, _p(act_param, F32), _p(logstd, F32), _p(val, F32), int(seed), _p(counter, I64),
              int(offset), _p(state, F64), _p(rng, I64), _p(elapsed, I32), _p(ep_score, F64), _p(obs, F32),
              _p(next_obs, F32), _p(rew, F32), _p(term, U8), _p(trunc, U8), _p(reset_obs, F32), _p(ep_step_out, I32),
              _p(ep_score_out, F64), _p(ep_stats, F64), max_steps, _p(x_in, F32), _p(act_out, _act_dtype(kind)),
              _p(logp_out, F32), _p(obs_row, F32), _p(act_row, F32), _p(rew_row, F32), _p(val_row, F32),
              _p(term_row, F32), _p(trunc_row, U8), _p(logp_row, F32), _p(rew_std, F32), float(rew_clip), _p(boot_src, F32),
              _p(boot_row, F32), _p(trig_cache, F64), _p(st.get("obs_in"), F64), _p(st.get("obs_out"), F64),
              int(st.get("obs_dim", 0)), float(st.get("obs_clip", 0.0)), _p(st.get("ret_state"), F64),
              _p(rew_std if st.get("returns") is not None else None, F32), _p(st.get("returns"), F64),
              float(st.get("gamma", 0.0)), int(bool(st.get("mask_terminal", True))), _p(st.get("partials"), F64),
              _p(st.get("ticket"), I32), _p(st.get("sums_out"), F64), _p(dist_row, F32), N, _stream())


def eval_step(kind, act_param, logstd, key, step, state, rng, elapsed, ep_score, next_obs, trig_cache, max_steps, scores, count,
              test_episode, partials, workspace, obs_state=None, obs_state_cand=None, obs_dim=0, act_tape=None, local_count=None,
              score_step=None, record=None):
    """Sample + env step + episode queue + observation statistics of one evaluation step in one launch (xb_eval_step).
    local_count / score_step / record: the env-sharded form (this rank's queue, step tags and step record)."""
    N = elapsed.numel()
    if score_step is not None and score_step.numel() < scores.numel():
        raise _lib.XB200Error("score_step needs one entry per queue slot (%d < %d)" % (score_step.numel(), scores.numel()))
    _lib.call("xb_eval_step", kind, _p(act_param, F32), _p(logstd, F32), _p(key, I64), _p(step, I64), _p(state, F64),
              _p(rng, I64), _p(elapsed, I32), _p(ep_score, F64), _p(next_obs, F32), _p(trig_cache, F64), max_steps,
              _p(act_tape, _act_dtype(kind)), act_tape.shape[0] if act_tape is not None else 0, _p(scores, F64),
              _p(count, I64), _p(test_episode, I64), scores.numel(), _p(obs_state, F64), _p(obs_state_cand, F64), int(obs_dim),
              _p(partials, F64), _p(workspace, I64), _p(local_count, I64), _p(score_step, I32), _p(record, F64), N, _stream())


def sincos_f64(x):
    s, c = torch.empty_like(x), torch.empty_like(x)
    _lib.call("xb_sincos_f64", _p(x, F64), _p(s, F64), _p(c, F64), x.numel(), _stream())
    return s, c


def store(obs, act, rew, val, term, trunc, logp, obs_row, act_row, rew_row, val_row, term_row, trunc_row, logp_row,
          rew_std=None, rew_clip=0.0):
    N = rew.numel()
    is_i64 = act.dtype == I64
    act_dim = 1 if is_i64 else act.numel() // N
    _lib.call("xb_store", _p(obs, F32), _p(act), int(is_i64), act_dim, _p(rew, F32), _p(val, F32), _p(term, U8),
              _p(trunc, U8), _p(logp, F32), _p(obs_row, F32), _p(act_row, F32), _p(rew_row, F32), _p(val_row, F32),
              _p(term_row, F32), _p(trunc_row, U8), _p(logp_row, F32), _p(rew_std, F32), float(rew_clip),
              obs.shape[-1] // 4, N, _stream())


def gae(rew, val, term, boot_last, adv, ret, gamma, lam, trunc=None, boot=None, stats=None, use_gae=True, variant="auto"):
    T, N = rew.shape
    _lib.call("xb_gae", _p(rew, F32), _p(val, F32), _p(term, F32), _p(trunc, U8), _p(boot, F32), _p(boot_last, F32),
              _p(adv, F32), _p(ret, F32), _p(stats, F64), T, N, float(gamma), float(lam), int(bool(use_gae)),
              GAE_VARIANTS[variant], _stream())


def gather_obs(idx, T, N, b_obs, obs_dim, obs_out, b_adv=None, stats=None):
    _lib.call("xb_gather_obs", _p(idx, I64), idx.numel(), T, N, _p(b_obs, F32), obs_dim, _p(b_adv, F32),
              _p(obs_out, F32), _p(stats, F64), _stream())


def gather_batch(idx, T, N, b_obs, obs_dim, b_act, act_dim, b_ret, b_val, b_adv, b_logp, obs_out, act_out, ret_out,
                 val_out, adv_out, logp_out, stats=None):
    _lib.call("xb_gather_batch", _p(idx, I64), idx.numel(), T, N, _p(b_obs, F32), obs_dim, _p(b_act, F32), act_dim,
              _p(b_ret, F32), _p(b_val, F32), _p(b_adv, F32), _p(b_logp, F32), _p(obs_out, F32), _p(act_out, F32),
              _p(ret_out, F32), _p(val_out, F32), _p(adv_out, F32), _p(logp_out, F32), _p(stats, F64), _stream())


def gather_rows(idx, T, N, src, out):
    """out[i, :] = src[step, env, :] for the reference's flat index k -> (env = k // T, step = k % T): any per-transition
    [T, N, W] array through the generic row slot of xb_gather_batch."""
    W = src.shape[2]
    _lib.call("xb_gather_batch", _p(idx, I64), idx.numel(), T, N, None, 1, _p(src, F32), W, None, None, None, None, None,
              _p(out, F32), None, None, None, None, None, _stream())


def normalize_adv(adv, stats, count):
    _lib.call("xb_normalize_adv", _p(adv, F32), _p(stats, F64), count, adv.numel(), _stream())


def _scalars(packed, act, ret, adv, old_logp):
    """Raw pointers + stride of the per-sample scalars: separate arrays (stride 1) or a packed [B, 4] float4 tensor
    {act, old_logp, adv, ret} as produced by gather_records (stride 4)."""
    if packed is None:
        return _p(act, F32), _p(ret, F32), _p(adv, F32), _p(old_logp, F32), 1
    base = _p(packed, F32)
    return base, base + 12, base + 8, base + 4, 4


def ppo_loss_categorical(logits, v_pred, act, ret, adv, old_logp, dlogits, dv, scalars, clip_range, vf_coef, ent_coef,
                         inv_batch, idx=None, T=0, N=0, val_old=None, adv_stats=None, adv_count=0, value_clip=0.0,
                         packed=None):
    B, A = logits.shape
    pa, pr, pv, pl, stride = _scalars(packed, act, ret, adv, old_logp)
    _lib.call("xb_ppo_loss_categorical", _p(idx, I64), B, T, N, _p(logits, F32), A, _p(v_pred, F32), pa, pr, pv, pl,
              _p(val_old, F32), _p(adv_stats, F64), adv_count, float(clip_range), float(vf_coef), float(ent_coef),
              float(value_clip), float(inv_batch), stride, _p(dlogits, F32), _p(dv, F32), _p(scalars, F64), _stream())


def ppo_loss_gaussian(mu, logstd, v_pred, act, ret, adv, old_logp, dmu, dlogstd_acc, dv, scalars, clip_range, vf_coef,
                      ent_coef, inv_batch, idx=None, T=0, N=0, val_old=None, adv_stats=None, adv_count=0, value_clip=0.0,
                      packed=None):
    B, A = mu.shape
    pa, pr, pv, pl, stride = _scalars(packed, act, ret, adv, old_logp)
    _lib.call("xb_ppo_loss_gaussian", _p(idx, I64), B, T, N, _p(mu, F32), _p(logstd, F32), A, _p(v_pred, F32), pa, pr, pv,
              pl, _p(val_old, F32), _p(adv_stats, F64), adv_count, float(clip_range), float(vf_coef), float(ent_coef),
              float(value_clip), float(inv_batch), stride, _p(dmu, F32), _p(dlogstd_acc, F64), _p(dv, F32),
              _p(scalars, F64), _stream())


def dist_loss_categorical(logits, old_logits, v_pred, act, ret, adv, dlogits, dv, scalars, clip_range, surr_coef, kl_coef,
                          vf_coef, ent_coef, inv_batch, kl_coef_dev=None, aux_v=None, aux_coef=0.0, daux=None):
    """PPO-KL / PPG losses on Categorical outputs with the old logits (see xb_dist_loss_categorical)."""
    B, A = logits.shape
    _lib.call("xb_dist_loss_categorical", B, _p(logits, F32), _p(old_logits, F32), A, _p(v_pred, F32), _p(aux_v, F32),
              _p(act, F32), _p(ret, F32), _p(adv, F32), float(clip_range), float(surr_coef), float(kl_coef),
              _p(kl_coef_dev, F32), float(vf_coef), float(ent_coef), float(aux_coef), float(inv_batch), _p(dlogits, F32),
              _p(dv, F32), _p(daux, F32), _p(scalars, F64), _stream())


def dist_loss_gaussian(mu, logstd, old_mu, old_std, v_pred, act, ret, adv, dmu, dlogstd_acc, dv, scalars, clip_range,
                       surr_coef, kl_coef, vf_coef, ent_coef, inv_batch, kl_coef_dev=None, aux_v=None, aux_coef=0.0,
                       daux=None):
    """PPO-KL / PPG losses on diagonal-Gaussian outputs; old_std is [B, A] or one shared row [A]."""
    B, A = mu.shape
    _lib.call("xb_dist_loss_gaussian", B, _p(mu, F32), _p(logstd, F32), _p(old_mu, F32), _p(old_std, F32),
              1 if old_std.dim() == 2 else 0, A, _p(v_pred, F32), _p(aux_v, F32), _p(act, F32), _p(ret, F32), _p(adv, F32),
              float(clip_range), float(surr_coef), float(kl_coef), _p(kl_coef_dev, F32), float(vf_coef), float(ent_coef),
              float(aux_coef), float(inv_batch), _p(dmu, F32), _p(dlogstd_acc, F64), _p(dv, F32), _p(daux, F32),
              _p(scalars, F64), _stream())


def kl_coef_adapt(scalars, kl_coef_dev, target_kl, count):
    _lib.call("xb_kl_coef_adapt", _p(scalars, F64), _p(kl_coef_dev, F32), float(target_kl), int(count), _stream())


def ppokl_loss_packed(idx, T, N, scal, old_dist, act_out, logstd, v_pred, adv_stats, adv_count, vf_coef, ent_coef, inv_batch,
                      kl_coef, kl_used, target_kl, adapt, kl_count, dact, dv, dlogstd, scalars, kl_sum_out=None):
    """PPO-KL loss forward + backward on packed minibatch rows with the adaptive coefficient (xb_ppokl_loss_packed).
    `old_dist`: the rollout's [T, N, 2] pairs; adapt=False leaves the coefficient to xb_ppokl_kl_adapt."""
    gaussian = logstd is not None
    _lib.call("xb_ppokl_loss_packed", _p(idx, I64), idx.numel(), int(T), int(N), _p(scal, F32), _p(old_dist, F32),
              _p(act_out, F32), _p(logstd, F32), int(gaussian), _p(v_pred, F32), _p(adv_stats, F64), int(adv_count),
              float(vf_coef), float(ent_coef), float(inv_batch), _p(kl_coef, F32), _p(kl_used, F32), float(target_kl),
              int(bool(adapt)), int(kl_count), _p(kl_sum_out, F64), _p(dact, F32), _p(dv, F32), _p(dlogstd, F64), _p(scalars, F64), _stream())


def ppokl_kl_adapt(kl_sum, kl_coef, kl_used, target_kl, count):
    _lib.call("xb_ppokl_kl_adapt", _p(kl_sum, F64), _p(kl_coef, F32), _p(kl_used, F32), float(target_kl), int(count),
              _stream())


def pack_records(b_obs, b_act, b_logp, b_adv, b_ret, rec):
    _lib.call("xb_pack_records", _p(b_obs, F32), _p(b_act, F32), _p(b_logp, F32), _p(b_adv, F32), _p(b_ret, F32),
              _p(rec, F32), b_adv.numel(), _stream())


def gather_records(idx, T, N, rec, obs_dim, obs_out, scal_out, stats=None):
    _lib.call("xb_gather_records", _p(idx, I64), idx.numel(), T, N, _p(rec, F32), obs_dim, _p(obs_out, F32),
              _p(scal_out, F32), _p(stats, F64), _stream())


def gather_trunk_fwd(idx, T, N, rec, obs_dim, w0, b0, slope, obs_out, scal_out, h1, stats=None, h1_signs=None):
    """gather_records + the MLP's first layer in one launch (xb_gather_trunk_fwd).  h1_signs: int32 [B, H / 32] sign words."""
    _lib.call("xb_gather_trunk_fwd", _p(idx, I64), idx.numel(), T, N, _p(rec, F32), obs_dim, _p(w0, F32), _p(b0, F32),
              float(slope), w0.shape[0], _p(obs_out, F32), _p(scal_out, F32), _p(stats, F64), _p(h1, F32), _p(h1_signs, I32),
              _stream())


def sample_categorical(logits, seed, counter, offset, act_out, logp_out):
    N, A = logits.shape
    _lib.call("xb_sample_categorical", _p(logits, F32), A, seed, _p(counter, I64), offset, _p(act_out, I64),
              _p(logp_out, F32), N, _stream())


def sample_gaussian(mu, logstd, seed, counter, offset, act_out, logp_out):
    N, A = mu.shape
    _lib.call("xb_sample_gaussian", _p(mu, F32), _p(logstd, F32), A, seed, _p(counter, I64), offset, _p(act_out, F32),
              _p(logp_out, F32), N, _stream())


def random_permutation(out, seed, counter=None, offset=0):
    """out[i] = P(i): a keyed pseudo-random permutation of 0..n-1 written in one launch (xb_random_permutation)."""
    _lib.call("xb_random_permutation", _p(out, I64), out.numel(), int(seed), _p(counter, I64), int(offset), _stream())


def counter_add(counter, inc=1):
    _lib.call("xb_counter_add", _p(counter, I64), inc, _stream())


def clip_adam_step(param, grad, exp_avg, exp_avg_sq, step_dev, lr0, lr_end_factor, lr_total_iters, beta1, beta2, eps,
                   max_norm, grad_scale, workspace, lr_out=None, gnorm_out=None):
    _lib.call("xb_clip_adam_step", _p(param, F32), _p(grad, F32), _p(exp_avg, F32), _p(exp_avg_sq, F32), param.numel(),
              _p(step_dev, I64), float(lr0), float(lr_end_factor), int(lr_total_iters), float(beta1), float(beta2),
              float(eps), float(max_norm), float(grad_scale), _p(workspace, F64), _p(lr_out, F32), _p(gnorm_out, F32),
              _stream())


def peer_allreduce_grad_norm(peer, grad_in, grad_out, tickets, step_dev, lr0, lr_end_factor, lr_total_iters, beta1, beta2, eps,
                             max_norm, grad_scale, workspace, lr_out=None, gnorm_out=None):
    """Cross-GPU gradient sum over peer memory fused with the gradient-norm pass (xb_peer_allreduce_grad_norm)."""
    _lib.call("xb_peer_allreduce_grad_norm", peer.bases, peer.rank, peer.world, peer.n, _p(grad_in, F32), _p(grad_out, F32),
              _p(tickets, I32),
              _p(step_dev, I64), float(lr0), float(lr_end_factor), int(lr_total_iters), float(beta1), float(beta2),
              float(eps), float(max_norm), float(grad_scale), _p(workspace, F64), _p(lr_out, F32), _p(gnorm_out, F32),
              _stream())


def adam_apply(param, grad, exp_avg, exp_avg_sq, beta1, beta2, eps, grad_scale, workspace):
    _lib.call("xb_adam_apply", _p(param, F32), _p(grad, F32), _p(exp_avg, F32), _p(exp_avg_sq, F32), param.numel(),
              float(beta1), float(beta2), float(eps), float(grad_scale), _p(workspace, F64), _stream())


def adam_apply_split(param, grad, exp_avg, exp_avg_sq, beta1, beta2, eps, grad_scale, workspace, w0, hi0, lo0, w1, hi1, lo1,
                     thi, tlo):
    """Adam step + the tf32 operand split of the hidden-layer weights w0 / w1 (views INTO `param`) in one launch."""
    N, K = w0.shape
    off = lambda w: (w.data_ptr() - param.data_ptr()) // 4
    _lib.call("xb_adam_apply_split", _p(param, F32), _p(grad, F32), _p(exp_avg, F32), _p(exp_avg_sq, F32), param.numel(),
              float(beta1), float(beta2), float(eps), float(grad_scale), _p(workspace, F64), off(w0), _p(hi0, F32),
              _p(lo0, F32), off(w1), _p(hi1, F32), _p(lo1, F32), N, K, _p(thi, F32), _p(tlo, F32), _stream())


def peer_allreduce_mean(peer, grad_in, grad_out):
    """grad_out = the mean over ranks of every rank's grad_in (fp32 [peer.n]), summed in rank order over peer memory and
    bit-identical on every rank (xb_peer_allreduce_mean)."""
    _lib.call("xb_peer_allreduce_mean", peer.bases, peer.rank, peer.world, peer.n, _p(grad_in, F32), _p(grad_out, F32),
              _p(peer.tickets, I32), _stream())


def peer_allreduce_f64(peer, n, out, offset=0):
    """out[:n] = sum over ranks of doubles [offset, offset + n) of each rank's comm-block statistics."""
    _lib.call("xb_peer_allreduce_f64", peer.bases, peer.rank, peer.world, int(offset), int(n), _p(out, F64),
              _p(peer.tickets, I32), _stream())


def peer_allreduce_merge(peer, src, n, out, inbox_offset, obs_in=None, obs_out=None, obs_dim=0, ret_state=None, rew_std=None):
    """One-barrier push exchange of `src[:n]` (out[:n] = totals over ranks) + the normaliser merge (xb_peer_allreduce_merge)."""
    _lib.call("xb_peer_allreduce_merge", peer.bases, peer.rank, peer.world, _p(src, F64), int(n), int(inbox_offset), _p(out, F64),
              _p(peer.tickets, I32), _p(obs_in, F64), _p(obs_out, F64), int(obs_dim), _p(ret_state, F64), _p(rew_std, F32), _stream())


def peer_eval_merge(peer, record, totals, count, test_episode, inbox_offset, obs_state=None, obs_state_cand=None, obs_dim=0):
    """The exchange that completes one env-sharded evaluation step: the ranks' records (fp64 [2D + 4]) summed in rank order into
    `totals`, the global episode count advanced, the observation statistics merged while the loop goes on (xb_peer_eval_merge)."""
    if totals.numel() < record.numel():
        raise _lib.XB200Error("totals needs %d doubles" % record.numel())
    _lib.call("xb_peer_eval_merge", peer.bases, peer.rank, peer.world, _p(record, F64), record.numel(), int(inbox_offset),
              _p(totals, F64), _p(count, I64), _p(test_episode, I64), _p(obs_state, F64), _p(obs_state_cand, F64), int(obs_dim),
              _p(peer.tickets, I32), _stream())


def adv_stats_minibatches(idx, n_minibatches, B, T, N, adv, stride, stats):
    _lib.call("xb_adv_stats_minibatches", _p(idx, I64), int(n_minibatches), int(B), int(T), int(N), _p(adv, F32), int(stride),
              _p(stats, F64), _stream())


def act_bias_bwd(dy, y, slope, dz, dbias, workspace):
    B, H = dy.shape
    _lib.call("xb_act_bias_bwd", _p(dy, F32), _p(y, F32), float(slope), _p(dz, F32), _p(dbias, F32), _p(workspace, F32),
              B, H, _stream())


def moments4(x, sums, workspace):
    """sums[:2D + 1] = column sums, column sums of squares and the row count of x [N, D], D = 4 or 8."""
    _lib.call("xb_moments4", _p(x, F32), x.shape[1], _p(sums, F64), _p(workspace, F64), x.shape[0], _stream())


def rms_normalize(x, dim, sums, state_in, state_out, clip, out, n_merged_rows):
    _lib.call("xb_rms_normalize", _p(x, F32), dim, _p(sums, F64), _p(state_in, F64), _p(state_out, F64), float(clip),
              _p(out, F32), x.shape[0], int(n_merged_rows), _stream())


def rms_apply(x, dim, state_new, state_old, n_new_rows, clip, out):
    _lib.call("xb_rms_apply", _p(x, F32), x.shape[1], int(dim), _p(state_new, F64), _p(state_old, F64), int(n_new_rows),
              float(clip), _p(out, F32), x.shape[0], _stream())


def rms_update_rows(x, dim, state_in, state_out, partials, ticket):
    _lib.call("xb_rms_update_rows", _p(x, F32), x.shape[1], int(dim), x.shape[0], _p(state_in, F64), _p(state_out, F64),
              _p(partials, F64), _p(ticket, I32), _stream())


def rms_merge_sums(sums, obs_in, obs_out, dim, ret_state, rew_std):
    """Merges one step's cross-rank totals sums [2D + 4] (D = 4 or 8 floats per observation row) into the normalisers."""
    _lib.call("xb_rms_merge_sums", _p(sums, F64), sums.numel(), _p(obs_in, F64), _p(obs_out, F64), int(dim), _p(ret_state, F64),
              _p(rew_std, F32), _stream())


def returns_track(returns, rew, term, trunc, gamma, sums, workspace, mask_terminal=True):
    _lib.call("xb_returns_track", _p(returns, F64), _p(rew, F32), _p(term, U8), _p(trunc, U8), float(gamma),
              1 if mask_terminal else 0, _p(sums, F64), _p(workspace, F64), returns.numel(), _stream())


def rms_merge_scalar(sums, state, rew_std):
    _lib.call("xb_rms_merge_scalar", _p(sums, F64), _p(state, F64), _p(rew_std, F32), _stream())


def bias_act_fwd(y, bias, slope):
    B, H = y.shape
    _lib.call("xb_bias_act_fwd", _p(y, F32), _p(bias, F32), float(slope), B, H, _stream())


def head_fwd(h, weight, bias, out):
    B, H = h.shape
    _lib.call("xb_head_fwd", _p(h, F32), _p(weight, F32), _p(bias, F32), _p(out, F32), B, H, weight.shape[0], _stream())


def head_bwd_act(dout, y, weight2, slope, dz, db1, dw2, db2, workspace):
    B, H = y.shape
    _lib.call("xb_head_bwd_act", _p(dout, F32), _p(y, F32), _p(weight2, F32), float(slope), _p(dz, F32), _p(db1, F32),
              _p(dw2, F32), _p(db2, F32), _p(workspace, F32), B, H, weight2.shape[0], _stream())


# ------------------------------------------------------------------------------------------------ tcgen05 dense layers
def _rows_ld(x):
    """(data pointer, row pitch in floats) of a 2-D fp32 tensor whose rows are contiguous (e.g. a column slice)."""
    if not x.is_cuda or x.dtype != F32 or x.dim() != 2 or x.stride(1) != 1:
        raise _lib.XB200Error("expected a CUDA fp32 matrix with contiguous rows")
    return x.data_ptr(), x.stride(0)


def dense_split_weights(W, hi, lo, thi=None, tlo=None, toff=0):
    N, K = W.shape
    _lib.call("xb_dense_split_weights", _p(W, F32), N, K, _p(hi, F32), _p(lo, F32), _p(thi, F32), _p(tlo, F32),
              thi.shape[1] if thi is not None else 0, toff, _stream())


def dense_split_weights2(w0, hi0, lo0, w1, hi1, lo1, thi, tlo):
    N, K = w0.shape
    _lib.call("xb_dense_split_weights2", _p(w0, F32), _p(hi0, F32), _p(lo0, F32), _p(w1, F32), _p(hi1, F32), _p(lo1, F32),
              N, K, _p(thi, F32), _p(tlo, F32), _stream())


def dense_fwd(x, w_hi, w_lo, bias, slope, y, head_w=None, head_b=None, head_out=None, b_resident=True):
    M, K = x.shape
    N = w_hi.shape[0]
    _lib.call("xb_dense_fwd", _p(x, F32), M, K, _p(w_hi, F32), _p(w_lo, F32), N, _p(bias, F32), float(slope), _p(y, F32),
              _p(head_w, F32), _p(head_b, F32), head_w.shape[0] if head_w is not None else 0, _p(head_out, F32),
              1 if b_resident else 0, _stream())


def dense_fwd2(x, slope, layer0, layer1, b_resident=True, prep=None, sign_out=None):
    """layerK = (w_hi, w_lo, bias, y, head_w, head_b, head_out): two layers on the same input in one launch.
    prep = (W0, W1, thi, tlo): also write the mask-form dgrad weight operand (see xb_dense_fwd2 in include/xb200.h).
    sign_out: int32 [M, 2 * N / 32] activation sign words for dense_dgrad(signs=...)."""
    pw0, pw1, pthi, ptlo = prep if prep is not None else (None, None, None, None)
    M, K = x.shape
    N = layer0[0].shape[0]
    args = []
    for w_hi, w_lo, bias, y, head_w, head_b, head_out in (layer0, layer1):
        args += [_p(w_hi, F32), _p(w_lo, F32), _p(bias, F32), _p(y, F32), _p(head_w, F32), _p(head_b, F32),
                 head_w.shape[0] if head_w is not None else 0, _p(head_out, F32)]
    _lib.call("xb_dense_fwd2", _p(x, F32), M, K, N, float(slope), *args, 1 if b_resident else 0, _p(pw0, F32), _p(pw1, F32),
              _p(pthi, F32), _p(ptlo, F32), _p(sign_out, I32), _stream())


def dense_fwd2_loss(x, slope, layer0, layer1, scal, adv_stats, adv_count, clip_range, vf_coef, ent_coef, inv_batch, logstd,
                    dact, dv, partials, ticket, scalars, dlogstd, b_resident=True, prep=None, sign_out=None):
    """dense_fwd2 with the PPO loss forward + backward fused into its epilogue (xb_dense_fwd2_loss)."""
    pw0, pw1, pthi, ptlo = prep if prep is not None else (None, None, None, None)
    M, K = x.shape
    N = layer0[0].shape[0]
    args = []
    for w_hi, w_lo, bias, y, head_w, head_b, head_out in (layer0, layer1):
        args += [_p(w_hi, F32), _p(w_lo, F32), _p(bias, F32), _p(y, F32), _p(head_w, F32), _p(head_b, F32),
                 head_w.shape[0], _p(head_out, F32)]
    _lib.call("xb_dense_fwd2_loss", _p(x, F32), M, K, N, float(slope), *args, 1 if b_resident else 0, _p(scal, F32),
              _p(adv_stats, F64), int(adv_count), float(clip_range), float(vf_coef), float(ent_coef), float(inv_batch),
              _p(logstd, F32), _p(dact, F32), _p(dv, F32), _p(partials, F64), _p(ticket, I32), _p(scalars, F64),
              _p(dlogstd, F64), _p(pw0, F32), _p(pw1, F32), _p(pthi, F32), _p(ptlo, F32), _p(sign_out, I32), _stream())


def mlp_fwd_from_obs(obs, w0, b0, slope, layer0, layer1, norm=None, weights_stable=False):
    """Whole actor-critic forward in one launch; layerK = (w_hi, w_lo, bias, y or None, head_w, head_b, head_out).
    norm = (state_new, state_old, n_new_rows, clip): `obs` is raw and is normalised in front of the trunk layer.
    weights_stable: the launch right before this one on the stream writes no weight array (XB_FWD_WEIGHTS_STABLE)."""
    nn, no, nr, nc = norm if norm is not None else (None, None, 0, 0.0)
    ptr, ld = _rows_ld(obs)
    args = []
    for w_hi, w_lo, bias, y, head_w, head_b, head_out in (layer0, layer1):
        args += [_p(w_hi, F32), _p(w_lo, F32), _p(bias, F32), _p(y, F32), _p(head_w, F32), _p(head_b, F32),
                 head_w.shape[0], _p(head_out, F32)]
    _lib.call("xb_mlp_fwd_from_obs", ptr, ld, obs.shape[1], _p(w0, F32), _p(b0, F32), obs.shape[0], w0.shape[0],
              float(slope), *args, _p(nn, F64), _p(no, F64), int(nr), float(nc), 1 if weights_stable else 0, _stream())


def mlp_fwd_from_obs_train(obs, w0, b0, slope, layer0, layer1, h1_out, loss=None, prep=None, sign_out=None):
    """Training forward with the trunk layer generated in the kernel (xb_mlp_fwd_from_obs_train): layerK as in dense_fwd2,
    h1_out receives the trunk activations; loss = (scal, adv_stats, adv_count, clip_range, vf_coef, ent_coef, inv_batch, logstd,
    dact, dv, partials, ticket, scalars, dlogstd) fuses the PPO loss into the epilogue."""
    pw0, pw1, pthi, ptlo = prep if prep is not None else (None, None, None, None)
    ptr, ld = _rows_ld(obs)
    args = []
    for w_hi, w_lo, bias, y, head_w, head_b, head_out in (layer0, layer1):
        args += [_p(w_hi, F32), _p(w_lo, F32), _p(bias, F32), _p(y, F32), _p(head_w, F32), _p(head_b, F32),
                 head_w.shape[0], _p(head_out, F32)]
    if loss is None:
        largs = [None, None, 0, 0.0, 0.0, 0.0, 0.0, None, None, None, None, None, None, None]
    else:
        scal, adv_stats, adv_count, clip_range, vf_coef, ent_coef, inv_batch, logstd, dact, dv, partials, ticket, scalars, dls = loss
        largs = [_p(scal, F32), _p(adv_stats, F64), int(adv_count), float(clip_range), float(vf_coef), float(ent_coef),
                 float(inv_batch), _p(logstd, F32), _p(dact, F32), _p(dv, F32), _p(partials, F64), _p(ticket, I32),
                 _p(scalars, F64), _p(dls, F64)]
    _lib.call("xb_mlp_fwd_from_obs_train", ptr, ld, obs.shape[1], _p(w0, F32), _p(b0, F32), obs.shape[0], w0.shape[0],
              float(slope), *args, _p(h1_out, F32), *largs, _p(pw0, F32), _p(pw1, F32), _p(pthi, F32), _p(ptlo, F32),
              _p(sign_out, I32), _stream())


def dense_dgrad(y0, dout0, w2_0, y1, dout1, w2_1, wt_hi, wt_lo, h1, slope, dz1, wt_form=0, signs=None, h1_signs=None):
    """signs: int32 [M, (K0 + K1) / 32] sign words of [y0 | y1] (dense_fwd2's sign_out); the kernel then does not read y0 / y1."""
    M, K0 = y0.shape
    _lib.call("xb_dense_dgrad", _p(y0, F32), _p(dout0, F32), _p(w2_0, F32), w2_0.shape[0], K0, _p(y1, F32),
              _p(dout1, F32), _p(w2_1, F32), w2_1.shape[0] if w2_1 is not None else 0,
              y1.shape[1] if y1 is not None else 0, M, _p(wt_hi, F32), _p(wt_lo, F32), wt_hi.shape[0], _p(h1, F32),
              float(slope), _p(dz1, F32), int(wt_form), _p(signs, I32), _p(h1_signs, I32), _stream())


def dense_wgrad_workspace(h_in, device):
    n = _lib.load().xb_dense_wgrad_workspace_floats(int(h_in))
    return torch.empty(n, dtype=F32, device=device)


def dense_wgrad(y0, dout0, w2_0, y1, dout1, w2_1, x, slope, workspace, dW0, db0, dw2_0, db2_0, dW1=None, db1=None,
                dw2_1=None, db2_1=None):
    B, H_out = y0.shape
    _lib.call("xb_dense_wgrad", _p(y0, F32), _p(dout0, F32), _p(w2_0, F32), w2_0.shape[0], _p(y1, F32), _p(dout1, F32),
              _p(w2_1, F32), w2_1.shape[0] if w2_1 is not None else 0, _p(x, F32), B, H_out, x.shape[1], float(slope),
              _p(workspace, F32), _p(dW0, F32), _p(db0, F32), _p(dw2_0, F32), _p(db2_0, F32), _p(dW1, F32), _p(db1, F32),
              _p(dw2_1, F32), _p(db2_1, F32), _stream())


# ------------------------------------------------------------------------------------------------ trunk layer (SIMT)
def mlp_trunk_fwd(obs, w0, b0, slope, h1, h1_signs=None):
    ptr, ld = _rows_ld(obs)
    _lib.call("xb_mlp_trunk_fwd", ptr, ld, obs.shape[1], _p(w0, F32), _p(b0, F32), float(slope), _p(h1, F32),
              obs.shape[0], w0.shape[0], _p(h1_signs, I32), _stream())


def mlp_trunk_wgrad_workspace(obs_dim, h, device):
    return torch.empty(_lib.load().xb_mlp_trunk_wgrad_workspace_floats(int(obs_dim), int(h)), dtype=F32, device=device)


def mlp_trunk_wgrad(dz1, obs, workspace, dw0, db0):
    ptr, ld = _rows_ld(obs)
    _lib.call("xb_mlp_trunk_wgrad", _p(dz1, F32), ptr, ld, obs.shape[1], _p(workspace, F32), _p(dw0, F32), _p(db0, F32),
              obs.shape[0], dz1.shape[1], _stream())


def dense_wgrad_bin(signs, dout0, nh0, dout1, nh1, x, h_out, workspace):
    """Binary-form weight-gradient partials (xb_dense_wgrad_bin): rank-1 head gradients, activation sign words instead of Y."""
    B, h_in = x.shape
    _lib.call("xb_dense_wgrad_bin", _p(signs, I32), signs.shape[1], _p(dout0, F32), nh0, _p(dout1, F32), nh1, _p(x, F32), B,
              h_out, h_in, _p(workspace, F32), _stream())


def mlp_backward_tail(wgrad_ws, h_out, h_in, nh0, nh1, grads0, grads1, trunk_ws, obs_dim, dwt, dbt, dls64=None, dls32=None,
                      norm=None, bin_form=None):
    """grads0/grads1 = (dW, db, dw2, db2) of the actor / critic; finishes xb_dense_wgrad + xb_mlp_trunk_wgrad partials.
    norm = (workspace, step_dev, lr0, lr_end_factor, lr_total_iters, beta1, beta2, max_norm, grad_scale, lr_out, gnorm_out):
    also take the global gradient norm and derive the clipped-Adam scalars in the same launch.
    bin_form = (W0, b0, w2_0, W1, b1, w2_1, slope): the partials come from dense_wgrad_bin (xb_mlp_backward_tail_bin)."""
    parts = _lib.load().xb_mlp_trunk_wgrad_parts()
    args = [_p(wgrad_ws, F32), h_out, h_in, 2 if grads1 is not None else 1, nh0, nh1,
            *[_p(g, F32) for g in grads0], *([_p(g, F32) for g in grads1] if grads1 is not None else [None] * 4),
            _p(trunk_ws, F32), parts, obs_dim, _p(dwt, F32), _p(dbt, F32), _p(dls64, F64), _p(dls32, F32),
            dls64.numel() if dls64 is not None else 0]
    if bin_form is not None:
        ws, step_dev, lr0, end_factor, total_iters, beta1, beta2, max_norm, grad_scale, lr_out, gnorm_out = \
            norm if norm is not None else (None, None, 0.0, 1.0, 1, 0.9, 0.999, 0.0, 1.0, None, None)
        W0, b0, w2_0, W1, b1, w2_1, slope = bin_form
        _lib.call("xb_mlp_backward_tail_bin", *args, _p(ws, F64), _p(step_dev, I64), float(lr0), float(end_factor),
                  int(total_iters), float(beta1), float(beta2), float(max_norm), float(grad_scale), _p(lr_out, F32),
                  _p(gnorm_out, F32), _p(W0, F32), _p(b0, F32), _p(w2_0, F32), _p(W1, F32), _p(b1, F32), _p(w2_1, F32),
                  float(slope), _stream())
    elif norm is None:
        _lib.call("xb_mlp_backward_tail", *args, _stream())
    else:
        ws, step_dev, lr0, end_factor, total_iters, beta1, beta2, max_norm, grad_scale, lr_out, gnorm_out = norm
        _lib.call("xb_mlp_backward_tail_norm", *args, _p(ws, F64), _p(step_dev, I64), float(lr0), float(end_factor),
                  int(total_iters), float(beta1), float(beta2), float(max_norm), float(grad_scale), _p(lr_out, F32),
                  _p(gnorm_out, F32), _stream())


def head3_fold(w3, b3, w2, b2):
    _lib.call("xb_head3_fold", _p(w3, F32), _p(b3, F32), _p(w2, F32), _p(b2, F32), w3.shape[1], _stream())


def head3_unfold_grads(gw3, gb3):
    _lib.call("xb_head3_unfold_grads", _p(gw3, F32), _p(gb3, F32), gw3.shape[1], _stream())
