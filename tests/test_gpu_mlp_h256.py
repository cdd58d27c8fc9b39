"""The tensor-core MLP at hidden width 256 (the network of the largest benchmark configuration) against fp64 references.

At H = 256 the update runs code that H = 128 never reaches: 16 sign words per row, the SS-form dgrad at K = 512, the
binary-form weight gradient with two operand-warp groups and two output halves per source (csrc/dense_tc.cu
dense_wgrad_bin_kernel<256>), the `bw[1]` branch and the 256-column G rows of wgrad_reduce_kernel, and adam_apply_split
with a 512-wide transposed operand.  Every reference here is plain torch in float64 on the same parameters; the LeakyReLU
pattern comes from the kernel's saved activations or sign words, so that units with |z| < 1e-6 cannot flip between fp32
and fp64.  Bars: tests/test_gpu_dense.py's MAX_BAR / RMS_BAR for single operations, north_star's 1e-4 for whole-network
param.grad and loss scalars."""
import math

import pytest
import torch

from tests.helpers import MAX_BAR, RMS_BAR
from tests.helpers import rel_err as _rel
from tests.helpers import rel_rms_err as _rel_rms

pytestmark = pytest.mark.gpu

SLOPE = 0.01
GRAD_BAR = 1e-4


def _spaces(env_id):
    import xuanpolicy_b200 as xb
    from xuanpolicy_b200 import spaces
    if env_id == "Box2":                      # a 2-D Gaussian action: general-form dgrad, three-MMA wgrad with nh0 = 2
        return spaces.Box(-1.0, 1.0, (3,)), spaces.Box(-2.0, 2.0, (2,))
    return xb.make_spaces(env_id)


def _fused(env_id, H, seed):
    """A policy of width H whose .grad are views of a flat buffer (as the learner holds them), and its fused MLP."""
    from xuanpolicy_b200.fused_mlp import FusedActorCritic
    from xuanpolicy_b200.learner import FlatAdamState
    from xuanpolicy_b200.policies import make_policy
    obs_space, act_space = _spaces(env_id)
    policy = make_policy(obs_space, act_space, hidden=(H,), device="cuda", seed=seed)
    with torch.no_grad():                     # biases are zero-initialised by the reference; make them count
        for p in policy.parameters():
            if p.dim() == 1:
                p.add_(0.1 * torch.randn_like(p))
    FlatAdamState(policy, torch.optim.Adam(policy.parameters(), 1e-3), None)
    assert FusedActorCritic.plan(policy) is not None
    fused = FusedActorCritic(policy)
    assert fused.H == H
    return policy, fused


def _obs(fused, B, gen):
    return torch.randn(B, 8, device="cuda", generator=gen)[:, :fused.obs_dim]     # rows with a pitch, as the buffer holds them


def _sign_bits(signs, H):
    """[B, 2H] bool from the forward's sign words: bit l of word s * H/32 + c is feature 32 c + l of source s."""
    w = signs.long() & 0xFFFFFFFF
    bits = (w[:, :, None] >> torch.arange(32, device=w.device)) & 1
    return bits.bool().reshape(signs.shape[0], 32 * signs.shape[1])


def _check_sign_words(b, H):
    B = b["h1"].shape[0]
    assert b["signs"].shape == (B, 2 * H // 32)
    bits = _sign_bits(b["signs"], H)
    assert torch.equal(bits[:, :H], b["ya"] > 0) and torch.equal(bits[:, H:], b["yc"] > 0)


def _ref_forward(P, obs, buf, head, slope=SLOPE):
    """fp64 actor / critic outputs of the reference's module graph, with the kernel's activation pattern."""
    lk = lambda z, y: z * torch.where(y > 0, 1.0, slope).double()
    h1 = lk(obs.double() @ P["representation.model.0.weight"].t() + P["representation.model.0.bias"], buf["h1"])
    ya = lk(h1 @ P[head + ".0.weight"].t() + P[head + ".0.bias"], buf["ya"])
    yc = lk(h1 @ P["critic.model.0.weight"].t() + P["critic.model.0.bias"], buf["yc"])
    return ya @ P[head + ".2.weight"].t() + P[head + ".2.bias"], (yc @ P["critic.model.2.weight"].t() + P["critic.model.2.bias"])[:, 0]


# ------------------------------------------------------------------------------------------------ 1. sign words
@pytest.mark.parametrize("env_id,B", [("Pendulum-v1", 65536), ("CartPole-v1", 4096 + 33), ("Acrobot-v1", 2048 + 77)])
def test_sign_words_at_h256_match_the_activations(env_id, B):
    """16 words per row; every row, the last partial 128-row tile's included, is written (the buffer starts all ones)."""
    policy, fused = _fused(env_id, 256, seed=5)
    assert fused.sign_bits
    obs = _obs(fused, B, torch.Generator(device="cuda").manual_seed(B))
    b = fused._buffers(B)
    b["signs"].fill_(-1)
    b["ya"].fill_(float("nan"))
    b["yc"].fill_(float("nan"))
    fused.forward(obs)
    torch.cuda.synchronize()
    assert torch.isfinite(b["ya"]).all() and torch.isfinite(b["yc"]).all()
    _check_sign_words(b, 256)
    print("%s B=%d: %d rows in the last tile, %.3f of the activations > 0"
          % (env_id, B, B % 128 or 128, float((b["ya"] > 0).double().mean())))


# ------------------------------------------------------------------------------------------------ 2. binary-form wgrad
_FWD = {}


def _forward_for_wgrad(H, B):
    """A Pendulum policy of width H and one forward at B rows (h1, ya, yc, sign words), shared by the binary-form cases."""
    if (H, B) not in _FWD:
        policy, fused = _fused("Pendulum-v1", H, seed=11)
        fused.forward(_obs(fused, B, torch.Generator(device="cuda").manual_seed(B + H)))
        _FWD[(H, B)] = (fused, fused._buf[B])
    return _FWD[(H, B)]


_BIN_CASES = [(256, B, n_src, nh0) for B in (65536, 8192 + 33, 1000, 100) for n_src in (1, 2) for nh0 in (1, 2)]


@pytest.mark.parametrize("H,B,n_src,nh0", _BIN_CASES + [(128, 1000, 2, 1), (128, 1000, 1, 2)])
def test_binary_form_wgrad_matches_fp64_autograd(H, B, n_src, nh0):
    """xb_dense_wgrad_bin + xb_mlp_backward_tail_bin on the sign words of a real forward and rank-1 head gradients (nh0 = 2:
    a softmax pair, second column = -first) against fp64 autograd of y = leaky(h1 W^T + b), out = y w2^T + b2.
    B = 1000 and 100 leave CTAs without a k-block (148 CTAs over 2 or 4 jobs of 32-row blocks): their partials must be
    zeros, so the workspace starts as NaN.

    The rms bar is 2 x RMS_BAR, as for the three-MMA wgrad in tests/test_gpu_dense.py.  Each CTA sums its share of the batch
    in the tensor core's fp32 accumulator, which truncates; at H = 256 with two sources the 148 CTAs split over 4 jobs, so
    each one sums ~1 770 rows of a 65 536-row batch (twice the chain of H = 128).  Measured on a B200 (1000 W) at B = 65 536,
    two sources: dW max 4.7e-5, rms 6.6e-6 (cuBLAS fp32 on the same data: max 1.2e-5); at B <= 8 225 every rms <= 1.4e-6."""
    from xuanpolicy_b200 import ops
    fused, b = _forward_for_wgrad(H, B)
    gen = torch.Generator(device="cuda").manual_seed(1000 * B + 10 * n_src + nh0)
    r = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    bits = _sign_bits(b["signs"], H)
    e0 = r(B, 1) / B
    srcs = [dict(lin=fused.la1, bits=bits[:, :H], dout=e0 if nh0 == 1 else torch.cat([e0, -e0], 1).contiguous(),
                 w2=(r(nh0, H) / H ** 0.5).contiguous(), b2=r(nh0))]
    if n_src == 2:
        srcs.append(dict(lin=fused.lc1, bits=bits[:, H:], dout=r(B, 1) / B, w2=fused.lc2.weight.data, b2=fused.lc2.bias.data))
    ws = ops.dense_wgrad_workspace(H, "cuda").fill_(float("nan"))
    nan = lambda *s: torch.full(s, float("nan"), device="cuda")
    outs = [[nan(H, H), nan(H), nan(s["w2"].shape[0], H), nan(s["w2"].shape[0])] for s in srcs]
    s0, s1 = srcs[0], srcs[1] if n_src == 2 else None
    ops.dense_wgrad_bin(b["signs"], s0["dout"], nh0, s1["dout"] if s1 else None, 1, b["h1"], H, ws)
    bin_form = (s0["lin"].weight.data, s0["lin"].bias.data, s0["w2"], s1["lin"].weight.data if s1 else None,
                s1["lin"].bias.data if s1 else None, s1["w2"] if s1 else None, SLOPE)
    ops.mlp_backward_tail(ws, H, H, nh0, 1, outs[0], outs[1] if s1 else None, None, fused.obs_dim, None, None, bin_form=bin_form)
    torch.cuda.synchronize()
    errs = []
    for s, o in zip(srcs, outs):
        W = s["lin"].weight.detach().double().requires_grad_(True)
        bb = s["lin"].bias.detach().double().requires_grad_(True)
        w2 = s["w2"].double().requires_grad_(True)
        b2 = s["b2"].double().requires_grad_(True)
        z = b["h1"].double() @ W.t() + bb
        out = (z * torch.where(s["bits"], 1.0, SLOPE).double()) @ w2.t() + b2
        ref = torch.autograd.grad(out, [W, bb, w2, b2], s["dout"].double())
        # cuBLAS fp32 on the same data, for scale
        dz32 = (s["dout"] @ s["w2"]) * torch.where(s["bits"], 1.0, SLOPE)
        cublas = _rel(dz32.t() @ b["h1"], ref[0])
        for name, got, want in zip(("dW", "db", "dw2", "db2"), o, ref):
            assert torch.isfinite(got).all(), name
            errs.append((name, _rel(got, want), _rel_rms(got, want)))
        if s["w2"].shape[0] == 2:             # the softmax pair's second head row is the negative of the first, exactly
            assert torch.equal(o[2][1], -o[2][0]) and torch.equal(o[3][1], -o[3][0])
        print("H=%d B=%d source %d/%d nh=%d: %s  (cuBLAS fp32 dW: max %.2e)" % (H, B, len(errs) // 4, n_src, s["w2"].shape[0], "  ".join(
            "%s %.2e/%.2e" % e for e in errs[-4:]), cublas))
    for name, emax, erms in errs:
        assert emax < MAX_BAR and erms < 2 * RMS_BAR, (name, emax, erms)


# ------------------------------------------------------------------------------------------------ 3. dgrad
@pytest.mark.parametrize("env_id,M", [(e, M) for e in ("Pendulum-v1", "CartPole-v1") for M in (65536, 4096 + 3, 2048 + 77)])
def test_dgrad_at_h256_matches_fp64(env_id, M):
    """dZ1 of the SS-form dgrad (K = 2H = 512; H = 256 reads ya / yc, not sign words): the mask form (w2-scaled weight
    operand, one head or a softmax pair) and the general form (dz generated element by element; for nh0 = 2 also with two
    independent logit gradients) against fp64, pattern from the saved activations.  Measured on a B200 (1000 W): max <= 3.0e-5,
    rms 4.2e-6 (cuBLAS fp32 on the same data: max 6.3e-6, rms 3.1e-7) — each output sums K = 2H = 512 products in the tensor
    core's truncating fp32 accumulator, twice the chain of H = 128."""
    policy, fused = _fused(env_id, 256, seed=7)
    gen = torch.Generator(device="cuda").manual_seed(M)
    fused.forward(_obs(fused, M, gen))
    assert fused._mask_ready and not fused.sign_dgrad
    b = fused._last[1]
    A = fused.A
    d0 = torch.randn(M, 1, device="cuda", generator=gen) / M
    pair = d0 if A == 1 else torch.cat([d0, -d0], 1).contiguous()
    dv2 = torch.randn(M, 1, device="cuda", generator=gen) / M
    cases = [("mask", pair, True), ("general", pair, False)]
    if A == 2:
        cases.append(("general, free pair", torch.randn(M, 2, device="cuda", generator=gen) / M, False))
    w = lambda m: m.weight.detach().double()
    mk = lambda y: torch.where(y > 0, 1.0, SLOPE).double()
    errs = []
    for name, dact, mask in cases:
        fused._mask_ready = mask
        b["dz1"] = torch.full((M, 256), float("nan"), device="cuda")
        fused.stage_dgrad(b, dact, dv2, softmax_pair=mask)
        torch.cuda.synchronize()
        ref = ((dact.double() @ w(fused.la2)) * mk(b["ya"]) @ w(fused.la1)
               + (dv2.double() @ w(fused.lc2)) * mk(b["yc"]) @ w(fused.lc1)) * mk(b["h1"])
        f = lambda m: m.weight.detach()
        m32 = lambda y: torch.where(y > 0, 1.0, SLOPE)
        cublas = (((dact @ f(fused.la2)) * m32(b["ya"])) @ f(fused.la1) + ((dv2 @ f(fused.lc2)) * m32(b["yc"])) @ f(fused.lc1)) * m32(b["h1"])
        assert torch.isfinite(b["dz1"]).all(), name
        errs.append((name, _rel(b["dz1"], ref), _rel_rms(b["dz1"], ref), _rel(cublas, ref), _rel_rms(cublas, ref)))
        print("%s M=%d %-18s max %.2e rms %.2e  (cuBLAS fp32: max %.2e rms %.2e)" % ((env_id, M) + errs[-1]))
    for name, emax, erms, _, _ in errs:
        assert emax < MAX_BAR and erms < RMS_BAR, (name, emax, erms)


# ------------------------------------------------------------------------------------------------ 4. whole backward
@pytest.mark.parametrize("env_id,B", [("CartPole-v1", 4096 + 33), ("CartPole-v1", 65536), ("Acrobot-v1", 8192 + 5),
                                      ("MountainCar-v0", 4096 + 33), ("Box2", 4096 + 77), ("Box2", 65536),
                                      ("Pendulum-v1", 65536), ("Pendulum-v1", 4096 + 33)])
def test_fused_backward_at_h256_matches_fp64_autograd(env_id, B):
    """FusedActorCritic.forward -> backward at H = 256 for every head the plan accepts: a softmax pair (CartPole, binary wgrad,
    mask dgrad), the folded Discrete(3) head (Acrobot, MountainCar: 6 and 8 observation floats in the trunk weight gradient),
    a 2-D Gaussian (general dgrad, three-MMA wgrad with nh0 = 2) and the 1-D Gaussian.  Every param.grad within 1e-4;
    measured on a B200 (1000 W), worst 8.3e-5 (critic hidden weight, 2-D Gaussian at B = 65 536: a sum over the batch of
    random value gradients that cancels)."""
    policy, fused = _fused(env_id, 256, seed=3)
    gen = torch.Generator(device="cuda").manual_seed(B)
    obs = _obs(fused, B, gen)
    act_out, v = fused.forward(obs)
    buf = fused._buf[B]
    names = [n for n, _ in policy.named_parameters()]
    P = {n: q.detach().double().requires_grad_(True) for n, q in policy.named_parameters()}
    ref_act, ref_v = _ref_forward(P, obs, buf, "actor.mu" if fused.gaussian else "actor.model", fused.slope)
    A = ref_act.shape[1]
    if fused.fold3:                           # the kernels report folded logits (third one 0): same softmax
        assert _rel(torch.log_softmax(act_out.double(), 1), torch.log_softmax(ref_act, 1)) < GRAD_BAR
    else:
        assert _rel(act_out, ref_act) < GRAD_BAR
    assert _rel(v, ref_v) < GRAD_BAR
    if fused.gaussian:
        dact, pair = torch.randn(B, A, device="cuda", generator=gen) / B, False
    elif A == 2:
        d0 = torch.randn(B, 1, device="cuda", generator=gen) / B
        dact, pair = torch.cat([d0, -d0], 1).contiguous(), True
    else:                                     # a softmax-loss gradient: rows sum to zero
        d = torch.randn(B, A, device="cuda", generator=gen) / B
        dact, pair = (d - d.mean(1, keepdim=True)).contiguous(), True
    dv = torch.randn(B, device="cuda", generator=gen) / B
    grads = torch.autograd.grad([ref_act, ref_v], [P[n] for n in names], [dact.double(), dv.double()], allow_unused=True)
    mine = dict(policy.named_parameters())
    for n, gref in zip(names, grads):
        if gref is not None:                  # (logstd: its gradient comes from the loss kernel, not from the MLP)
            mine[n].grad.fill_(float("nan"))
    fused.backward(dact, dv, softmax_pair=pair)
    torch.cuda.synchronize()
    assert fused._bin_now == (env_id in ("CartPole-v1", "Pendulum-v1"))
    errs = {n: _rel(mine[n].grad, gref) for n, gref in zip(names, grads) if gref is not None}
    print("%s B=%d: %s" % (env_id, B, "  ".join("%s %.1e" % (n.replace(".weight", ".w").replace(".bias", ".b"), e)
                                                 for n, e in errs.items())))
    for n, e in errs.items():
        assert e < GRAD_BAR, (n, e)


# ------------------------------------------------------------------------------------------------ 5. one learner update
def _ref_loss(P, obs, buf, scal, gauss, hp):
    """fp64 restatement of PPOCLIP_Learner.update's loss (clipped surrogate, value loss, entropy) and its log scalars."""
    act_out, v = _ref_forward(P, obs, buf, "actor.mu" if gauss else "actor.model")
    a, old_logp, adv, ret = scal.double().unbind(1)
    if gauss:
        logstd = P["actor.logstd"][0]
        logp = -(a - act_out[:, 0]) ** 2 / (2 * torch.exp(2 * logstd)) - logstd - 0.5 * math.log(2 * math.pi)
        ent = (0.5 + 0.5 * math.log(2 * math.pi) + logstd).expand_as(logp)
    else:
        lp = torch.log_softmax(act_out, 1)
        logp = lp.gather(1, a.long()[:, None])[:, 0]
        ent = -(lp.exp() * lp).sum(1)
    c = hp["clip_range"]
    ratio = torch.exp(logp - old_logp)
    a_loss = -torch.minimum(ratio.clamp(1 - c, 1 + c) * adv, ratio * adv).mean()
    c_loss = ((v - ret) ** 2).mean()
    e_loss = ent.mean()
    info = {"actor-loss": a_loss, "critic-loss": c_loss, "entropy": e_loss, "predict_value": v.mean(),
            "clip_ratio": ((ratio < 1 - c) | (ratio > 1 + c)).double().mean()}
    return a_loss - hp["ent_coef"] * e_loss + hp["vf_coef"] * c_loss, {k: float(x) for k, x in info.items()}


def _ref_adam_step(P, grads, m, v, t, lr, max_norm, beta1=0.9, beta2=0.999, eps=1e-5):
    """clip_grad_norm_ (when max_norm > 0) + torch.optim.Adam's step, in fp64."""
    if max_norm > 0:
        total = torch.sqrt(sum((g ** 2).sum() for g in grads.values()))
        coef = min(1.0, float(max_norm / (total + 1e-6)))
        grads = {n: g * coef for n, g in grads.items()}
    out = {}
    for n, g in grads.items():
        m[n] = beta1 * m[n] + (1 - beta1) * g
        v[n] = beta2 * v[n] + (1 - beta2) * g * g
        denom = (v[n].sqrt() / math.sqrt(1 - beta2 ** t)) + eps
        out[n] = P[n] - lr / (1 - beta1 ** t) * m[n] / denom
    return out


@pytest.mark.parametrize("clip", [False, True])
@pytest.mark.parametrize("env_id,B", [("Pendulum-v1", 65536), ("CartPole-v1", 16384 + 33)])
def test_learner_update_at_h256_matches_fp64_reference_update(env_id, B, clip):
    """Two native updates through PPOCLIP_Learner with the fused optimiser, on the path of the fused-loss golden test: loss in
    the forward epilogue (xb_dense_fwd2_loss at N = 256), gradient norm + Adam scalars in the backward tail launch,
    stage_optimizer -> adam_apply_split (N = K = 256, transposed operand 512 wide).  The reference is an fp64 restatement of
    PPOCLIP_Learner.update: loss, clip_grad_norm_ (max_norm = half the first gradient's norm, so the clip acts), Adam
    (eps = 1e-5) and LinearLR.  Checked: info scalars and every param.grad (1e-4), parameters after each step (1e-5), and
    the operand copies the Adam launch wrote, which the second update consumes, bit-equal to a fresh split.

    Each reference step starts from the parameters the native step before it produced (the Adam moments stay the
    reference's): the critic weight gradient is a sum over the batch that cancels (ret - v is zero-mean here), so the
    ~1e-6 fp32 difference of the parameters after step 1 alone moves it by ~1.5e-4 of its scale at B = 16 417."""
    import xuanpolicy_b200 as xb
    from xuanpolicy_b200 import ops
    from xuanpolicy_b200.policies import make_policy
    hp = dict(vf_coef=0.25, ent_coef=0.01, clip_range=0.2)
    lr0, total_iters = 4e-4, 1000
    obs_space, act_space = xb.make_spaces(env_id)
    gauss = env_id == "Pendulum-v1"
    pol = make_policy(obs_space, act_space, hidden=(256,), device="cuda", seed=13)
    gen = torch.Generator(device="cuda").manual_seed(B)
    with torch.no_grad():                     # off the symmetric init (logits, log-std), biases non-zero
        for p in pol.parameters():
            p.add_(0.05 * torch.randn(p.shape, device="cuda", generator=gen))
        obs = torch.randn(B, obs_space.shape[0], device="cuda", generator=gen)
        _, dist, v0 = pol(obs)
        if gauss:
            mu, std = dist.get_param()
            act = mu + std * torch.randn(mu.shape, device="cuda", generator=gen)
            logp0 = dist.log_prob(act)
            act = act[:, 0]
        else:
            act = torch.multinomial(torch.softmax(dist.get_param(), 1), 1, generator=gen)[:, 0].float()
            logp0 = dist.log_prob(act)
        old_logp = logp0 + 0.1 * torch.randn(B, device="cuda", generator=gen)
        adv = torch.randn(B, device="cuda", generator=gen)
        ret = v0 + torch.randn(B, device="cuda", generator=gen)
    scal = torch.stack([act, old_logp, adv, ret], 1).contiguous()           # the packed minibatch rows
    opt = torch.optim.Adam(pol.parameters(), lr0, eps=1e-5)
    sched = torch.optim.lr_scheduler.LinearLR(opt, start_factor=1.0, end_factor=0.0, total_iters=total_iters)
    learner = xb.PPOCLIP_Learner(pol, opt, sched, "cuda", "/tmp", use_grad_clip=clip, **hp)
    flat = learner.enable_fused_optimizer()
    fused = learner._fused
    assert fused is not None and fused.H == 256
    names = [n for n, _ in pol.named_parameters()]
    mine = dict(pol.named_parameters())
    m = {n: torch.zeros_like(q, dtype=torch.float64) for n, q in mine.items()}
    v = {n: torch.zeros_like(q, dtype=torch.float64) for n, q in mine.items()}
    dls64 = torch.zeros(1, dtype=torch.float64, device="cuda") if gauss else None
    loss = dict(scal=scal, adv_stats=None, adv_count=B, inv_batch=1.0 / B, logstd=pol.actor.logstd.detach() if gauss else None,
                scalars=learner._scalars, dlogstd=dls64, **hp)
    max_norm = None
    for t in (1, 2):
        assert fused.splits_fresh == (t == 2)     # the second forward runs on the copies the Adam launch wrote
        fused.forward(obs, refresh=not fused.splits_fresh, loss=loss)
        b = fused._last[1]
        torch.cuda.synchronize()
        _check_sign_words(b, 256)
        P = {n: q.detach().double() for n, q in mine.items()}
        Pg = {n: x.clone().requires_grad_(True) for n, x in P.items()}
        ref_loss, ref_info = _ref_loss(Pg, obs, b, scal, gauss, hp)
        ref_grads = dict(zip(names, torch.autograd.grad(ref_loss, [Pg[n] for n in names])))
        if max_norm is None:
            max_norm = 0.5 * float(torch.sqrt(sum((g ** 2).sum() for g in ref_grads.values()))) if clip else 0.0
            learner.clip_grad_norm = max_norm
        fused.norm_sink = (flat, max_norm)
        if gauss:
            dls32 = flat.grad_views[[id(q) for q in flat.params].index(id(pol.actor.logstd))]
            fused.backward(b["dact"], b["dv"], dls64, dls32)
        else:
            fused.backward(b["dact"], b["dv"], softmax_pair=True)
        assert fused.norm_done
        torch.cuda.synchronize()
        gerr = {n: _rel(mine[n].grad, ref_grads[n]) for n in names}
        learner.stage_optimizer()
        assert fused.splits_fresh
        info = learner.info(B)
        ierr = {k: abs(float(info[k]) - r) / max(1.0, abs(r)) for k, r in ref_info.items()}
        lr = lr0 * (1.0 - (t - 1) / total_iters)
        P = _ref_adam_step(P, ref_grads, m, v, t, lr, max_norm)
        perr = {n: _rel(mine[n].detach(), P[n]) for n in names}
        steps = {n: float((mine[n].detach().double() - P[n]).abs().max()) / lr for n in names}
        print("%s B=%d clip=%s step %d: grad %.2e (%s)  info %.2e (%s)  param %.2e (%s, %.2e lr)"
              % (env_id, B, clip, t, max(gerr.values()), max(gerr, key=gerr.get), max(ierr.values()), max(ierr, key=ierr.get),
                 max(perr.values()), max(perr, key=perr.get), max(steps.values())))
        for n, e in gerr.items():
            assert e < GRAD_BAR, (t, n, e)
        for k, e in ierr.items():
            assert e < GRAD_BAR, (t, k, e)
        for n, e in perr.items():
            assert e < 1e-5, (t, n, e)
        # the hi / lo operand copies the Adam launch wrote are those a fresh split of the updated weights gives
        fresh = [torch.empty_like(x) for x in (fused.wa_hi, fused.wa_lo, fused.wc_hi, fused.wc_lo, fused.wt_hi, fused.wt_lo)]
        ops.dense_split_weights2(fused.la1.weight.data, fresh[0], fresh[1], fused.lc1.weight.data, fresh[2], fresh[3],
                                 fresh[4], fresh[5])
        for x, y in zip((fused.wa_hi, fused.wa_lo, fused.wc_hi, fused.wc_lo, fused.wt_hi, fused.wt_lo), fresh):
            assert torch.equal(x, y)


# ------------------------------------------------------------------------------------------------ 6. end to end
@pytest.mark.parametrize("env_id", ["CartPole-v1", "Acrobot-v1"])
def test_native_agent_at_h256_uses_the_tensor_core_mlp(env_id):
    """The device-resident PPO loop with a width-256 network on the discrete envs (yaml defaults: obs / reward normalisation
    on), tensor-core MLP for the rollout forward and the updates, against the same loop with the torch MLP (XB_FUSED_MLP=0):
    same trajectories (discrete actions), parameters within fp32 tolerance after two rollouts and eight updates."""
    import os
    from xuanpolicy_b200.configs import build_ppo
    out = []
    for fused in ("1", "0"):
        os.environ["XB_FUSED_MLP"] = fused
        try:
            agent = build_ppo(env_id, parallels=1024, n_steps=8, n_epoch=2, n_minibatch=2, shuffle="device", seed=6,
                              use_obsnorm=True, use_rewnorm=True, representation_hidden_size=[256],
                              actor_hidden_size=[256], critic_hidden_size=[256])
        finally:
            os.environ.pop("XB_FUSED_MLP", None)
        f = agent.learner._fused
        assert (f is not None) == (fused == "1") and agent._fused_step and agent._fused_norm
        if f is not None:
            assert f.H == 256 and f.fold3 == (env_id == "Acrobot-v1") and agent.batch_size >= f.MIN_ROWS
        agent.train(8)
        info = agent.train(8)
        out.append((agent.memory._act.clone(), agent.memory._obs.clone(), agent.learner._flat.flat_param.clone(), info))
    assert torch.equal(out[0][0], out[1][0])                                   # same actions -> same trajectory
    assert torch.allclose(out[0][1], out[1][1], atol=1e-5, rtol=1e-5)
    print("%s: max parameter difference %.2e" % (env_id, float((out[0][2] - out[1][2]).abs().max())))
    assert torch.allclose(out[0][2], out[1][2], atol=2e-5, rtol=2e-4), (out[0][2] - out[1][2]).abs().max()
    assert abs(out[0][3]["critic-loss"] - out[1][3]["critic-loss"]) <= 1e-4 * max(1.0, abs(out[1][3]["critic-loss"]))
