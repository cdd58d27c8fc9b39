"""bench.roofline_of: the `roofline` object of the JSON line names the roof that bounds the dominant kernel (CPU only)."""
import pytest

import bench

# The kernel fractions below were taken against this TF32 ceiling (1/2 x the measured bf16 burst of a B200, DESIGN.md);
# pinned so the test does not depend on which peaks file, if any, the machine running it has.
TF32_PEAK = 832.0


@pytest.fixture(autouse=True)
def _pinned_tf32_peak(monkeypatch):
    monkeypatch.setattr(bench, "measured_tf32_peak", lambda: TF32_PEAK)


def _kd(**kw):
    base = {"ms": 0.0347, "achieved_gbs": 2008.6, "frac": 0.307, "bytes_per_launch": 69730304, "launches_per_step": 64}
    base.update(kw)
    return base


def test_tensor_bound_kernel_reports_the_tensor_roof_and_keeps_the_hbm_numbers():
    kd = _kd(gemm_tflops=123.7, tf32_passes=3, tensor_pipe_tflops_tf32=371.2, tensor_frac_of_tf32_peak=0.446)
    r = bench.roofline_of("dense_dgrad_tc", kd, 6534.5, "measured (MEASURED_PEAKS.json)", 38046719)
    assert r["kernel"] == "dense_dgrad_tc" and r["bound"] == "tensor" and r["unit"] == "TFLOP/s"
    assert r["achieved"] == 371.2 and abs(r["frac"] - 0.446) < 1e-12 and r["traffic"] == 38046719
    assert abs(r["achieved"] / r["peak"] - r["frac"]) < 0.01          # frac = achieved / peak (rounded inputs)
    assert r["hbm"]["unit"] == "GB/s" and r["hbm"]["frac"] == 0.307 and r["hbm"]["peak"] == 6534.5


def test_hbm_bound_kernel_reports_the_hbm_roof():
    kd = _kd(achieved_gbs=5922.3, frac=0.906)
    r = bench.roofline_of("gae_tma", kd, 6534.5, "measured (MEASURED_PEAKS.json)", None)
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and r["achieved"] == 5922.3 and r["peak"] == 6534.5 and r["frac"] == 0.906
    assert r["traffic"] is None and r["tensor"] == {}
