"""Stage-isolated, per-element parity of the tensor-core kernels against the rounding-faithful reference (tests/kernel_ref.py).

Every stage is fed the GPU's own tap of the previous stage.  Taps hold the exact fp16 (or fp32) values the next kernel reads,
so an error found in a stage was made by that stage's kernel.  Taps cover the first chunk of a call only, so every tapped call
here stays within one chunk (1024 pileup sites, 256 full-alignment sites).

Bounds are absolute, per element; each sits next to the maximum measured on a B200 by this file (the full per-stage
statistics of that run are committed as profiles/r3_layer_parity.json).  A run writes its own statistics to
layer_parity.json in the directory named by the environment variable C3B_LAYER_PARITY_DIR, when it is set.
"""
import json
import os

import numpy as np
import pytest
import torch

import kernel_ref as kr

pytestmark = pytest.mark.gpu

REPORT = {}

# Per-element bounds.  Each is set from the maximum measured on a B200 (1000 W power limit) by the first run of this file,
# 2026-10-17, and sits within 4x of it; the a-priori estimate comes first.
BOUNDS = {
    # LSTM layers: fp32 accumulation order (~1e-6 on the pre-activations) plus MUFU tanh.approx (|rel| <= 2^-10.7 on the
    # fp32 path, fp16 packed pre-activations and activations on the f16x2 path), fed back through 33 steps; h is stored fp16, so
    # one fp16 ulp of |h| <= 1 (2^-11) flips wherever the two sides straddle a rounding boundary.  Estimate: a few 1e-3.
    # "_f16x2": the packed fp16 gate activations (the CTA-pair kernels, and lstm_tc.cu with option lstm_mufu16 = 1)
    "lstm1": 1.5e-3,       # measured 4.9e-4 = one fp16 ulp in [0.5, 1) (lstm_tc.cu, fp32 MUFU: the default)
    "lstm1_f16x2": 1e-2,   # measured 3.42e-3 (lstm1_impl = 1, and lstm_mufu16 = 1)
    "lstm2": 1.5e-3,       # measured 4.9e-4 (lstm2_impl = 0, fp32 MUFU)
    "lstm2_f16x2": 6e-3,   # measured 1.95e-3 (lstm2_impl = 1, the default; counts up to 67 552), 1.71e-3 otherwise
    # the same errors averaged over the 33 steps of one (site, unit): rounding noise shrinks, a systematic offset stays
    "lstm1_mean": 4e-3,    # measured 1.25e-3 (lstm1_impl=1)
    "lstm2_mean": 2.5e-3,  # measured 7.2e-4 (lstm1_impl=1)
    # L4 without bias on identical fp16 operands: only fp32 accumulation order over K = 10 560 (pileup) / 3 584 (FA) terms,
    # ~sqrt(K) * 2^-24 * |partial sums| ~ 1e-6 to 1e-5.
    "l4_pre": 1e-4,        # measured 3.9e-5 (pileup, counts up to 67 552)
    # tail from the GPU's L4 accumulator: __expf SELU, fp16 a4 / a5 operands that may round the other way (one fp16 ulp of an
    # activation moves a logit by ~|w| * 2^-11), fp32 softmax.  Estimate ~1e-4 to 1e-3 on probabilities.
    "y": 4e-3,             # measured 1.17e-3 (full alignment, C8, depth 89, 256 sites)
    # convs: fp32 accumulation order, then fp16 output rounding: one ulp of the largest map value (2^-7 in [8, 16)).
    "conv": 2e-2,          # measured 7.8e-3 = one fp16 ulp in [8, 16)
    # residual blocks: two convs with the fp16 mid map in between; a mid value that rounds the other way moves the output by
    # ~|w| * ulp, so one or two output ulps.
    "res_block": 5e-2,     # measured 1.56e-2 = one fp16 ulp in [16, 32)
    # fp32 debug path against plain fp64 (exact reference): fp32 rounding only, ~1e-6 relative.
    "fp32_lstm": 3e-6,     # measured 7.8e-7
    "fp32_conv": 8e-5,     # measured 2.4e-5 (res_block3, values up to ~100)
    "fp32_l4_pre": 4e-5,   # measured 1.2e-5
    "fp32_y": 6e-6,        # measured 1.7e-6
}


def _record(key, st):
    REPORT[key] = st
    out = os.environ.get("C3B_LAYER_PARITY_DIR")
    if out:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "layer_parity.json"), "w") as f:
            json.dump(REPORT, f, indent=1, sort_keys=True)
    print("LAYER", key, json.dumps(st))


def _check(variant, stage, got, ref, bound_key, axes, mean_axis=None, mean_key=None):
    # stats are recorded before the assertion so a failing run still reports every stage it reached
    st = kr.stage_stats(got, ref)
    if mean_axis is not None:
        st["max_mean"] = float(np.abs((np.asarray(got, np.float64) - ref).mean(axis=mean_axis)).max())
    _record("%s/%s" % (variant, stage), st)
    kr.check_stage("%s/%s" % (variant, stage), got, ref, BOUNDS[bound_key], axes, mean_axis,
                   BOUNDS[mean_key] if mean_key else None)


def _model(kind, sd, channels, add_indel, **opts):
    from clair3_b200.model import Clair3_F, Clair3_P
    cls = Clair3_P if kind == "pileup" else Clair3_F
    m = cls(add_indel_length=add_indel, predict=True, input_channels=channels)
    m.set_option("taps", 1)
    for k, v in opts.items():
        m.set_option(k, v)
    m.to(torch.device("cuda"))
    m.eval()
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    return m


def _run(m, x, host):
    return (m(torch.from_numpy(x)) if host else m(torch.from_numpy(x).cuda())).cpu().numpy()


# ---------------------------------------------------------------------------------------------------------------- pileup
def _pileup_stages(variant, ref, m, x, y, fp32=False, opts={}):
    n = len(x)
    mufu16 = opts.get("lstm_mufu16", 0)
    k1 = "lstm1_f16x2" if opts.get("lstm1_impl", 0) == 1 or mufu16 else "lstm1"
    k2 = "lstm2_f16x2" if opts.get("lstm2_impl", 1) == 1 or mufu16 else "lstm2"
    g1 = m.tap("lstm1").reshape(n, 33, 256)
    g2 = m.tap("lstm2").reshape(n, 33, 320)
    z4 = m.tap("l4_pre").reshape(n, -1)
    p = "fp32_" if fp32 else ""
    _check(variant, "lstm1", g1, ref.lstm1(x), "fp32_lstm" if fp32 else k1, ("site", "step", "unit"),
           None if fp32 else 1, None if fp32 else "lstm1_mean")
    _check(variant, "lstm2", g2, ref.lstm2(g1), "fp32_lstm" if fp32 else k2, ("site", "step", "unit"),
           None if fp32 else 1, None if fp32 else "lstm2_mean")
    _check(variant, "l4_pre", z4, ref.l4_pre(g2), p + "l4_pre", ("site", "unit"))
    _check(variant, "y", y, ref.y(z4), p + "y", ("site", "output"))


PILEUP_VARIANTS = {
    "default": {},
    "host": {},                                              # host buffers: the latency variants (LSTM1 tile 16 at these sizes)
    "tile16_wg1": dict(lstm_tile=16, lstm_wg=1),
    "tile16_wg2": dict(lstm_tile=16, lstm_wg=2),
    "tile32_wg1": dict(lstm_tile=32, lstm_wg=1),
    "tile32_wg2": dict(lstm_tile=32, lstm_wg=2),
    "mufu16": dict(lstm_mufu16=1),                            # packed tanh.approx.f16x2 (the default is the fp32 MUFU path)
    "lstm1_pair": dict(lstm1_impl=1),
    "lstm2_rows_tile16": dict(lstm2_impl=0, lstm_tile=16),
    "lstm2_rows_tile32": dict(lstm2_impl=0, lstm_tile=32),
}


@pytest.mark.parametrize("out_dim", [24, 90])
@pytest.mark.parametrize("variant", list(PILEUP_VARIANTS))
def test_pileup_stages_per_element(variant, out_dim):
    """Sizes 1024, 300, 129 and 1: the odd 128-site tile counts put the CTA pair's peer on padding."""
    from clair3_b200 import synth
    add_indel = out_dim == 90
    sd = synth.pileup_state_dict(add_indel, seed=131)
    x = synth.pileup_inputs(1024, seed=131)
    m = _model("pileup", sd, 18, add_indel, **PILEUP_VARIANTS[variant])
    ref = kr.KernelRef(sd)
    for n in (1024, 300, 129, 1):
        y = _run(m, x[:n], variant == "host")
        _pileup_stages("pileup_%s_out%d_n%d" % (variant, out_dim, n), ref, m, x[:n], y, opts=PILEUP_VARIANTS[variant])


def test_pileup_deep_counts_meet_the_lstm1_bound():
    """Counts up to 67 552, the largest the hi/lo split of LSTM1's input columns carries exactly (hi saturates at 65 504,
    lo is exact up to 2 048)."""
    from clair3_b200 import synth
    sd = synth.pileup_state_dict(False, seed=133)
    x = synth.pileup_inputs(512, seed=133).astype(np.int64) * 600
    x[1::2] //= 600                                          # every other site keeps its normal depth
    x = np.clip(x, -67552, 67552)
    x[0, 0, :6] = [67552, -67552, 65504, 65505, 66000, 67551]
    assert np.abs(x).max() == 67552
    x = x.astype(np.int32)
    m = _model("pileup", sd, 18, False)
    y = _run(m, x, False)
    with np.errstate(over="ignore"):                        # exp overflow in the reference's saturated sigmoids
        _pileup_stages("pileup_deep_67552", kr.KernelRef(sd), m, x, y)


def test_pileup_fp32_path_against_fp64():
    from clair3_b200 import synth
    sd = synth.pileup_state_dict(True, seed=135)
    x = synth.pileup_inputs(256, seed=135)
    m = _model("pileup", sd, 18, True, precision=1)
    y = _run(m, x, False)
    _pileup_stages("pileup_fp32_n256", kr.KernelRef(sd, exact=True), m, x, y, fp32=True)


# ---------------------------------------------------------------------------------------------------------------- full alignment
def _fa_stages(variant, ref, m, x, y, fp32=False):
    n, depth = x.shape[0], x.shape[1]
    hh, ww = [depth], [33]
    for _ in range(3):
        hh.append((hh[-1] - 1) // 2 + 1)
        ww.append((ww[-1] - 1) // 2 + 1)
    chans = [64, 128, 256]
    axes = ("site", "row", "col", "channel")
    conv_key, res_key = ("fp32_conv", "fp32_conv") if fp32 else ("conv", "res_block")

    def tap(name, level):
        return m.tap(name).reshape(n, hh[level + 1], ww[level + 1], chans[level]).transpose(0, 3, 1, 2)   # NHWC -> NCHW

    def nhwc(a):
        return a.transpose(0, 2, 3, 1)

    prev = None
    for level, (stem, block) in enumerate((("conv1", "res_block1"), ("conv3", "res_block2"), ("conv5", "res_block3"))):
        g_stem, g_block = tap(stem, level), tap(block, level)
        want = ref.conv1(x) if level == 0 else ref.stem(prev, level)
        _check(variant, stem, nhwc(g_stem), nhwc(want), conv_key, axes)
        _check(variant, block, nhwc(g_block), nhwc(ref.res_block(g_stem, level)), res_key, axes)
        prev = g_block
    sp = m.tap("spp").reshape(n, -1)
    want_sp = ref.spp(prev)
    _record("%s/spp" % variant, kr.stage_stats(sp, want_sp))
    if fp32:
        kr.check_stage("%s/spp" % variant, sp, want_sp, BOUNDS["fp32_conv"], ("site", "feature"))
    else:
        # a max over identical fp16 values: bitwise equal
        assert np.array_equal(sp, want_sp.astype(np.float32)), "%s/spp: %d features differ" % (variant, int((sp != want_sp).sum()))
    z4 = m.tap("l4_pre").reshape(n, -1)
    p = "fp32_" if fp32 else ""
    _check(variant, "l4_pre", z4, ref.l4_pre(sp), p + "l4_pre", ("site", "unit"))
    _check(variant, "y", y, ref.y(z4), p + "y", ("site", "output"))


FA_CASES = {"c8_d89_n256": (8, 89, 256), "c9_d89_n129": (9, 89, 129), "c8_d55_n44": (8, 55, 44), "c8_d89_n1": (8, 89, 1)}


@pytest.mark.parametrize("case", list(FA_CASES))
@pytest.mark.parametrize("pconv_impl", [0, 1])
def test_full_alignment_stages_per_element(pconv_impl, case):
    from clair3_b200 import synth
    channels, depth, n = FA_CASES[case]
    sd = synth.fa_state_dict(True, channels=channels, seed=141)
    x = synth.fa_inputs(n, depth=depth, channels=channels, seed=141)
    m = _model("fa", sd, channels, True, pconv_impl=pconv_impl)
    y = _run(m, x, False)
    _fa_stages("fa_pconv%d_%s" % (pconv_impl, case), kr.KernelRef(sd), m, x, y)


def test_full_alignment_fp32_path_against_fp64():
    from clair3_b200 import synth
    sd = synth.fa_state_dict(True, channels=8, seed=143)
    x = synth.fa_inputs(64, depth=89, channels=8, seed=143)
    m = _model("fa", sd, 8, True, precision=1)
    y = _run(m, x, False)
    _fa_stages("fa_fp32_n64", kr.KernelRef(sd, exact=True), m, x, y, fp32=True)


# ---------------------------------------------------------------------------------------------------------------- invariance
@pytest.mark.parametrize("kind", ["pileup", "fa"])
def test_taps_and_repeats_do_not_change_the_answer(kind):
    """Turning taps on only adds stores; a repeated call recomputes the same values: both bitwise."""
    from clair3_b200 import synth
    if kind == "pileup":
        sd, x, ch = synth.pileup_state_dict(False, seed=151), synth.pileup_inputs(700, seed=151), 18
    else:
        sd, x, ch = synth.fa_state_dict(True, channels=8, seed=152), synth.fa_inputs(200, depth=89, channels=8, seed=152), 8
    m_on = _model(kind, sd, ch, kind == "fa")
    m_off = _model(kind, sd, ch, kind == "fa", taps=0)
    y_on, y_off = _run(m_on, x, False), _run(m_off, x, False)
    assert np.array_equal(y_on, y_off)
    names = ("lstm1", "lstm2", "l4_pre") if kind == "pileup" else ("conv1", "res_block1", "conv3", "res_block2", "conv5",
                                                                    "res_block3", "spp", "l4_pre")
    taps = {k: m_on.tap(k) for k in names}
    for _ in range(3):
        assert np.array_equal(_run(m_on, x, False), y_on)
        for k in names:
            assert np.array_equal(m_on.tap(k), taps[k]), k
