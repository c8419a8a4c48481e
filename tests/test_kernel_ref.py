"""CPU checks of tests/kernel_ref.py (the rounding-faithful reference of the tensor-core path) and of its per-element checker."""
import numpy as np
import pytest

import kernel_ref as kr
from conftest import GOLDEN_FA, GOLDEN_PILEUP, golden_case
from oracle import clair3_oracle as orc
from test_gpu_layer_parity import BOUNDS


def _relerr(a, b):          # the aggregate check the GPU tests used for taps before the per-element harness
    return float(np.linalg.norm(a.astype(np.float64) - b) / (np.linalg.norm(b) + 1e-30))


def _forward(meta, sd, x, exact):
    ref = kr.KernelRef(sd, exact=exact)
    return ref.pileup(x) if meta["kind"] == "pileup" else ref.fa(x)


@pytest.mark.parametrize("name", GOLDEN_PILEUP + GOLDEN_FA)
def test_exact_reference_is_the_oracle(name):
    z, meta, sd, x = golden_case(name)
    taps = {}
    fwd = orc.pileup_forward if meta["kind"] == "pileup" else orc.fa_forward
    y = fwd(sd, x, meta["add_indel_length"], taps=taps)
    got = _forward(meta, sd, x, exact=True)
    assert np.abs(got["y"] - y).max() < 1e-12
    for k, v in got.items():
        if k == "y":
            continue
        want = taps[k] - sd["L4.bias"] if k == "l4_pre" else taps[k]       # the stage excludes the L4 bias, like the tap
        assert np.abs(v - want).max() < 1e-12, k


@pytest.mark.parametrize("name", GOLDEN_PILEUP + GOLDEN_FA)
def test_rounded_reference_meets_the_stated_tolerance(name):
    """fp16 rounding at the kernels' storage points stays within the fp16 tensor-core path's stated tolerance of the fp32
    reference: max |dp| <= 2e-2, mean |dp| <= 2e-3, arg-max agreement >= 99 % per head."""
    z, meta, sd, x = golden_case(name)
    y = _forward(meta, sd, x, exact=False)["y"]
    d = np.abs(y - z["y"])
    assert d.max() <= 2e-2 and d.mean() <= 2e-3, (d.max(), d.mean())
    for lo, hi in [(0, 21), (21, 24), (24, 57), (57, 90)]:
        if hi <= y.shape[1]:
            assert (y[:, lo:hi].argmax(1) == z["y"][:, lo:hi].argmax(1)).mean() >= 0.99


# ------------------------------------------------------------------------------------------------ checker sensitivity
def _flags(stage, got, ref, bound_key, axes, mean_axis=None, mean_key=None):
    try:
        kr.check_stage(stage, got, ref, BOUNDS[bound_key], axes, mean_axis, BOUNDS[mean_key] if mean_key else None)
    except AssertionError as e:
        return str(e)
    return None


def test_checker_flags_small_injected_faults():
    z, meta, sd, x = golden_case("p24")
    ref = kr.KernelRef(sd)
    t = ref.pileup(x)
    lstm_axes = ("site", "step", "unit")
    assert _flags("lstm2", t["lstm2"], t["lstm2"], "lstm2_f16x2", lstm_axes, 1, "lstm2_mean") is None

    # one LSTM2 element off by 0.05
    g = t["lstm2"].copy()
    g[1, 17, 200] += 0.05
    msg = _flags("lstm2", g, t["lstm2"], "lstm2_f16x2", lstm_axes, 1, "lstm2_mean")
    assert msg is not None and "site 1, step 17, unit 200" in msg, msg
    assert _relerr(g[:2], z["tap_lstm2"]) < 2e-2          # ... which the old aggregate check accepts

    # one hidden unit off by 0.02 at every step (a wrong bias in one unit)
    g = t["lstm2"].copy()
    g[0, :, 37] += 0.02
    msg = _flags("lstm2", g, t["lstm2"], "lstm2_f16x2", lstm_axes, 1, "lstm2_mean")
    assert msg is not None and "site 0" in msg and "unit 37" in msg, msg
    assert _relerr(g[:2], z["tap_lstm2"]) < 2e-2

    # one 64-wide k-chunk missing from one L4 output
    h = t["lstm2"].reshape(len(x), -1)
    w4 = ref.weight16(sd["L4.weight"])
    site, out = 5, 17
    parts = [h[site, k:k + 64] @ w4[out, k:k + 64] for k in range(0, h.shape[1], 64)]
    k = int(np.argmax(np.abs(parts)))
    g = t["l4_pre"].copy()
    g[site, out] -= parts[k]
    msg = _flags("l4_pre", g, t["l4_pre"], "l4_pre", ("site", "unit"))
    assert msg is not None and "site 5, unit 17" in msg, msg

    # two sites swapped (a site-to-lane mapping error)
    g = t["lstm1"].copy()
    g[[3, 4]] = g[[4, 3]]
    assert _flags("lstm1", g, t["lstm1"], "lstm1", lstm_axes, 1, "lstm1_mean") is not None

    # one conv pixel taken from its neighbour (a border / pixel mapping error)
    z, meta, sd, x = golden_case("f8")
    c1 = kr.KernelRef(sd).conv1(x[:2]).transpose(0, 2, 3, 1)       # NHWC, as the taps
    g = c1.copy()
    g[1, 10, 5] = g[1, 10, 6]
    msg = _flags("conv1", g, c1, "conv", ("site", "row", "col", "channel"))
    assert msg is not None and "site 1, row 10, col 5" in msg, msg


def test_checker_reports_nan():
    a = np.zeros((2, 3))
    b = a.copy()
    b[1, 2] = np.nan
    with pytest.raises(AssertionError, match="site 1, unit 2"):
        kr.check_stage("s", b, a, 1.0, ("site", "unit"))


# ------------------------------------------------------------------------------------------------ LSTM1's hi/lo input split
def test_hi_lo_split_is_exact_up_to_67552():
    """hi = satfinite_f16(x) stops at 65 504, lo = satfinite_f16(x - hi) is exact while x - hi <= 2 048."""
    x = np.arange(0, 131009, dtype=np.int64)
    for sign in (1, -1):
        hi, lo = kr.split_counts(sign * x)
        exact = hi + lo == sign * x
        assert exact[:67553].all()
        assert not exact[67553]
        assert int((~exact).sum()) == 58337
        assert np.abs(hi + lo - sign * x).max() == 16
