"""Shared helpers for the parity tests (test infrastructure)."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    d = {k: z[k] for k in z.files}
    if "meta" in d:
        d["meta"] = json.loads(str(d["meta"]))
    return d


def replay_buffer_protocol(buf, g):
    """Drives a DummyOnPolicyBuffer-shaped object with the agent's store/finish_path protocol
    (ppoclip_agent.py:68-100) using the golden's recorded rollout."""
    T, N = g["rew"].shape
    for t in range(T):
        buf.store(g["obs"][t], g["act"][t], g["rew"][t], g["val"][t], g["term"][t], {"old_logp": g["logp"][t]})
        if buf.full:
            for i in range(N):
                buf.finish_path(0.0 if g["term"][t, i] else g["boot"][t, i], i)
            break
        for i in range(N):
            if g["term"][t, i] or g["trunc"][t, i]:
                buf.finish_path(0.0 if g["term"][t, i] else g["boot"][t, i], i)


def gae_close(a, b, rtol=1e-5):
    """|a-b| <= rtol*max(|b|, rms(b)) (advantages cross zero; SURVEY.md §8(c))."""
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    scale = np.maximum(np.abs(b), np.sqrt(np.mean(b * b)))
    return bool(np.all(np.abs(a - b) <= rtol * scale)), float(np.max(np.abs(a - b) / scale))


def rel_err(a, ref):
    """max_i |a_i - ref_i| / max(|ref_i|, rms(ref)) of two torch tensors — the metric the GAE parity test uses (values
    cross zero)."""
    ref = ref.double()
    rms = ref.pow(2).mean().sqrt().clamp_min(1e-30)
    return float(((a.double() - ref).abs() / rms.maximum(ref.abs())).max())


def rel_rms_err(a, ref):
    """rms(a - ref) / rms(ref) of two torch tensors."""
    ref = ref.double()
    return float((a.double() - ref).pow(2).mean().sqrt() / ref.pow(2).mean().sqrt().clamp_min(1e-30))


# Bars of the tensor-core dense kernels against fp64 (rel_err, rel_rms_err).  The tensor core accumulates in fp32 with
# truncation, so the worst element of ~10^7 sits near 1e-5 of the output scale (cuBLAS fp32 SIMT: ~1e-6; single-pass
# TF32: ~1e-3); the rms error is ~1e-6.  Both are far inside north_star's 1e-4 loss/gradient tolerance.
MAX_BAR, RMS_BAR = 5e-5, 5e-6


def rel_close(a, b, rtol):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    denom = max(float(np.sqrt(np.mean(b * b))), 1e-30)
    err = float(np.max(np.abs(a - b)) / denom)
    return err <= rtol, err
