"""tcgen05 3xTF32 dense kernels (csrc/dense_tc.cu) against fp64 torch references of the same layers.

The layers are those of the reference's actor-critic MLP (xuance/torch/representations/mlp.py:40-51,
policies/gaussian.py:17-24,41-48): Linear + LeakyReLU(0.01) blocks followed by a narrow head.  Bars: forward
activations and head outputs <= 2e-6 of the output scale (fp32-level, far inside the 1e-4 loss/gradient tolerance);
plain TF32 would sit at ~1e-3.
"""
import pytest
import torch

# (bars: see tests/helpers.py)
from tests.helpers import MAX_BAR, RMS_BAR
from tests.helpers import rel_err as _rel
from tests.helpers import rel_rms_err as _rel_rms

pytestmark = pytest.mark.gpu

SLOPE = 0.01


def _split(W, transposed_into=None, toff=0):
    from xuanpolicy_b200 import ops
    hi, lo = torch.empty_like(W), torch.empty_like(W)
    if transposed_into is None:
        ops.dense_split_weights(W, hi, lo)
    else:
        ops.dense_split_weights(W, hi, lo, transposed_into[0], transposed_into[1], toff)
    return hi, lo


@pytest.mark.parametrize("M,K,N,n_head,resident", [
    (65536, 128, 128, 1, True), (65536, 128, 128, 2, False), (8192, 128, 128, 0, True), (333, 128, 128, 1, True),
    (128 * 149 + 7, 64, 64, 2, True), (4096, 256, 256, 1, False), (65536, 256, 256, 2, False), (1000, 64, 128, 1, True),
])
def test_dense_fwd_matches_fp64(M, K, N, n_head, resident):
    from xuanpolicy_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M + K + N)
    x = torch.randn(M, K, device="cuda", generator=g)
    W = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    b = torch.randn(N, device="cuda", generator=g) * 0.1
    hw = torch.randn(max(n_head, 1), N, device="cuda", generator=g) / N ** 0.5
    hb = torch.randn(max(n_head, 1), device="cuda", generator=g)
    hi, lo = _split(W)
    assert torch.equal(hi + lo, W)
    y = torch.full((M, N), float("nan"), device="cuda")
    ho = torch.full((M, max(n_head, 1)), float("nan"), device="cuda")
    if n_head:
        ops.dense_fwd(x, hi, lo, b, SLOPE, y, hw[:n_head].contiguous(), hb[:n_head].contiguous(), ho, b_resident=resident)
    else:
        ops.dense_fwd(x, hi, lo, b, SLOPE, y, b_resident=resident)
    torch.cuda.synchronize()
    ref = torch.nn.functional.leaky_relu(x.double() @ W.double().t() + b.double(), SLOPE)
    assert torch.isfinite(y).all()
    cublas = torch.nn.functional.leaky_relu(x @ W.t() + b, SLOPE)
    print("fwd M=%d K=%d N=%d: max %.2e rms %.2e  (cuBLAS fp32: max %.2e rms %.2e)"
          % (M, K, N, _rel(y, ref), _rel_rms(y, ref), _rel(cublas, ref), _rel_rms(cublas, ref)))
    assert _rel(y, ref) < MAX_BAR and _rel_rms(y, ref) < RMS_BAR
    if n_head:
        href = ref @ hw[:n_head].double().t() + hb[:n_head].double()
        assert _rel(ho[:, :n_head], href) < MAX_BAR


@pytest.mark.parametrize("M,H,nh0,nh1", [(65536, 128, 1, 1), (4099, 128, 2, 1), (2048, 64, 2, 1), (8192, 256, 1, 1),
                                         (4096, 128, 1, 0)])
def test_dense_dgrad_matches_fp64_autograd(M, H, nh0, nh1):
    """dZ1 = d(loss)/d(pre-activation of the trunk layer) given dL/d(head outputs) of the actor and critic branches."""
    from xuanpolicy_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M + H)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    z1 = r(M, H)
    h1 = torch.nn.functional.leaky_relu(z1, SLOPE)
    Wa, Wc = r(H, H) / H ** 0.5, r(H, H) / H ** 0.5
    wa2, wc2 = r(nh0, H) / H ** 0.5, r(max(nh1, 1), H) / H ** 0.5
    douta, doutc = r(M, nh0), r(M, max(nh1, 1))
    # fp64 autograd reference
    z1d = z1.double().requires_grad_(True)
    h1d = torch.nn.functional.leaky_relu(z1d, SLOPE)
    ya = torch.nn.functional.leaky_relu(h1d @ Wa.double().t(), SLOPE)
    yc = torch.nn.functional.leaky_relu(h1d @ Wc.double().t(), SLOPE)
    outs, gouts = [ya @ wa2.double().t()], [douta.double()]
    if nh1:
        outs.append(yc @ wc2.double().t())
        gouts.append(doutc.double())
    ref, = torch.autograd.grad(outs, z1d, gouts)
    # kernel inputs: the saved fp32 activations
    ya32, yc32 = ya.detach().float().contiguous(), yc.detach().float().contiguous()
    K = H * (2 if nh1 else 1)
    thi, tlo = torch.zeros(H, K, device="cuda"), torch.zeros(H, K, device="cuda")
    _split(Wa, (thi, tlo), 0)
    if nh1:
        _split(Wc, (thi, tlo), H)
    dz1 = torch.full((M, H), float("nan"), device="cuda")
    if nh1:
        ops.dense_dgrad(ya32, douta, wa2, yc32, doutc, wc2, thi, tlo, h1, SLOPE, dz1)
    else:
        ops.dense_dgrad(ya32, douta, wa2, None, None, None, thi, tlo, h1, SLOPE, dz1)
    torch.cuda.synchronize()
    assert torch.isfinite(dz1).all()
    # entries whose fp32 activation sign differs from the fp64 graph's (|y| ~ 1e-8) are excluded by construction: same y
    print("dgrad M=%d H=%d: max %.2e rms %.2e" % (M, H, _rel(dz1, ref), _rel_rms(dz1, ref)))
    assert _rel(dz1, ref) < MAX_BAR and _rel_rms(dz1, ref) < RMS_BAR


@pytest.mark.parametrize("B,H,nh0,nh1", [(65536, 128, 1, 1), (4099, 128, 2, 1), (8192, 256, 1, 1), (4096, 128, 1, 0),
                                         (100, 128, 1, 1), (8192 + 33, 256, 2, 1)])
def test_dense_wgrad_matches_fp64_autograd(B, H, nh0, nh1):
    """dW, db of the actor / critic hidden layers and dw2, db2 of their heads, from the saved activations."""
    from xuanpolicy_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(B + H + 1)
    r = lambda *s: torch.randn(*s, device="cuda", generator=g)
    h1 = torch.nn.functional.leaky_relu(r(B, H), SLOPE)
    srcs = []
    for nh in (nh0, nh1):
        if nh == 0:
            srcs.append(None)
            continue
        W = (r(H, H) / H ** 0.5).double().requires_grad_(True)
        b = (r(H) * 0.1).double().requires_grad_(True)
        w2 = (r(nh, H) / H ** 0.5).double().requires_grad_(True)
        b2 = r(nh).double().requires_grad_(True)
        dout = r(B, nh)
        y = torch.nn.functional.leaky_relu(h1.double() @ W.t() + b, SLOPE)
        out = y @ w2.t() + b2
        grads = torch.autograd.grad(out, [W, b, w2, b2], dout.double())
        srcs.append(dict(y=y.detach().float().contiguous(), dout=dout, w2=w2.detach().float().contiguous(), ref=grads))
    ws = ops.dense_wgrad_workspace(H, "cuda")
    outs = []
    for s_ in srcs:
        if s_ is None:
            outs.append([None] * 4)
        else:
            nh = s_["w2"].shape[0]
            outs.append([torch.full((H, H), float("nan"), device="cuda"), torch.full((H,), float("nan"), device="cuda"),
                         torch.full((nh, H), float("nan"), device="cuda"), torch.full((nh,), float("nan"), device="cuda")])
    a, c = srcs
    ops.dense_wgrad(a["y"], a["dout"], a["w2"], c["y"] if c else None, c["dout"] if c else None, c["w2"] if c else None,
                    h1, SLOPE, ws, *outs[0], *outs[1])
    torch.cuda.synchronize()
    for s_, o in zip(srcs, outs):
        if s_ is None:
            continue
        for name, got, ref in zip(("dW", "db", "dw2", "db2"), o, s_["ref"]):
            assert torch.isfinite(got).all(), name
            print("wgrad B=%d H=%d %s: max %.2e rms %.2e" % (B, H, name, _rel(got, ref), _rel_rms(got, ref)))
            assert _rel(got, ref) < MAX_BAR and _rel_rms(got, ref) < 2 * RMS_BAR, name
