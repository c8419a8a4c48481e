"""GPU parity tests (run on the B200 box: ``pytest -m gpu``).  Everything goes through the C-ABI
(``libclair3b200.so`` via cffi); the checker is the oracle / the golden vectors minted from the reference.

Tolerances (stated, SURVEY.md §8c):
  * fp32 debug kernels vs the fp32 reference:   max |dp| <= 1e-4 on probabilities, taps rel-L2 <= 1e-4
  * fp16-operand tensor-core kernels vs the fp32 reference: max |dp| <= 2e-2, mean |dp| <= 2e-3, taps rel-L2 <= 2e-2,
    >= 99% arg-max agreement per head.
"""
import numpy as np
import pytest
import torch

from conftest import GOLDEN_FA, GOLDEN_PILEUP, golden_case

pytestmark = pytest.mark.gpu

FP32, TC = 1, 0
HEAD_SLICES = [(0, 21), (21, 24), (24, 57), (57, 90)]


def _relerr(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / (np.linalg.norm(b) + 1e-30))


def _model(meta, sd, precision, **opts):
    from clair3_b200.model import Clair3_F, Clair3_P
    cls = Clair3_P if meta["kind"] == "pileup" else Clair3_F
    ch = 18 if meta["kind"] == "pileup" else meta["channels"]
    m = cls(add_indel_length=meta["add_indel_length"], predict=True, input_channels=ch)
    m.set_option("precision", precision)
    m.set_option("taps", 1)
    for k, v in opts.items():
        m.set_option(k, v)
    m.to(torch.device("cuda"))
    m.eval()
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    return m


def _check_probs(y, ref, max_tol, mean_tol, argmax_frac):
    assert y.shape == ref.shape
    assert np.isfinite(y).all()
    d = np.abs(y - ref)
    assert d.max() <= max_tol, "max |dp| %.3e" % d.max()
    assert d.mean() <= mean_tol, "mean |dp| %.3e" % d.mean()
    for lo, hi in HEAD_SLICES:
        if hi <= y.shape[1]:
            assert np.allclose(y[:, lo:hi].sum(1), 1.0, atol=1e-4)
            agree = (y[:, lo:hi].argmax(1) == ref[:, lo:hi].argmax(1)).mean()
            assert agree >= argmax_frac, "argmax agreement %.3f" % agree


@pytest.mark.parametrize("name", GOLDEN_PILEUP + GOLDEN_FA)
def test_fp32_kernels_match_reference(name):
    z, meta, sd, x = golden_case(name)
    m = _model(meta, sd, FP32)
    y = m(torch.from_numpy(x).cuda()).cpu().numpy()
    _check_probs(y, z["y"], 1e-4, 1e-5, 1.0)
    for tap in ("lstm1", "lstm2", "spp", "l4_pre"):
        if "tap_" + tap in z.files:
            got = m.tap(tap).reshape(x.shape[0], -1)
            want = z["tap_" + tap]
            if tap == "l4_pre":       # library tap excludes the L4 bias
                got = got + sd["L4.bias"][None, :]
            n = want.shape[0]
            assert _relerr(got[:n].reshape(want.shape), want) < 1e-4, tap


@pytest.mark.parametrize("name", GOLDEN_PILEUP + GOLDEN_FA)
def test_tensor_core_kernels_match_reference(name):
    z, meta, sd, x = golden_case(name)
    m = _model(meta, sd, TC)
    y = m(torch.from_numpy(x).cuda()).cpu().numpy()
    for tap in ("lstm1", "lstm2", "spp", "l4_pre"):
        if "tap_" + tap in z.files:
            got = m.tap(tap).reshape(x.shape[0], -1)
            want = z["tap_" + tap]
            if tap == "l4_pre":
                got = got + sd["L4.bias"][None, :]
            n = want.shape[0]
            assert _relerr(got[:n].reshape(want.shape), want) < 2e-2, tap
    _check_probs(y, z["y"], 2e-2, 2e-3, 0.99)


def test_tensor_core_conv_taps_match_reference():
    z, meta, sd, x = golden_case("f8")
    m = _model(meta, sd, TC)
    m(torch.from_numpy(x).cuda())
    for tap in ("conv1", "res_block1", "conv3", "res_block2", "conv5", "res_block3"):
        want = z["tap_" + tap]                         # [1,C,H,W]
        got = m.tap(tap).reshape(x.shape[0], want.shape[2], want.shape[3], want.shape[1])[:1].transpose(0, 3, 1, 2)
        assert _relerr(got, want) < 2e-2, tap


def test_ragged_empty_and_host_buffers():
    z, meta, sd, x = golden_case("p24")
    m = _model(meta, sd, TC)
    full = m(torch.from_numpy(x).cuda()).cpu().numpy()
    # host in / host out (the _torch_predict shape: numpy in, numpy out)
    taps = {k: m.tap(k) for k in ("lstm1", "lstm2", "l4_pre")}
    y_host = m(torch.from_numpy(x))
    assert y_host.device.type == "cpu"
    # host buffers select the latency variants (LSTM1 tile width, projection grid): bit-identical by construction
    assert np.array_equal(y_host.numpy(), full)
    for k, v in taps.items():
        assert np.array_equal(m.tap(k), v), k
    # ragged batches: any B >= 1, every site independent of its batch neighbours
    for b in (1, 7, 33):
        yb = m(torch.from_numpy(x[:b]).cuda()).cpu().numpy()
        assert np.array_equal(yb, full[:b])
    assert m(torch.from_numpy(x[:0]).cuda()).shape == (0, 24)
    # chunked internal passes give the same answer
    m.set_option("chunk_sites", 16)
    assert np.array_equal(m(torch.from_numpy(x).cuda()).cpu().numpy(), full)


def test_lstm_tiles_agree():
    z, meta, sd, x = golden_case("p24")
    outs = []
    for tile in (16, 32, 64):
        m = _model(meta, sd, TC, lstm_tile=tile)
        outs.append(m(torch.from_numpy(x).cuda()).cpu().numpy())
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])


@pytest.mark.parametrize("tile", [16, 32, 64])
def test_lstm_warpgroup_layouts_agree(tile):
    """One or two epilogue warpgroups per LSTM sub-tile (option lstm_wg) run the same per-cell arithmetic: identical output."""
    z, meta, sd, x = golden_case("p90")
    outs = []
    for wg in (1, 2):
        m = _model(meta, sd, TC, lstm_tile=tile, lstm_wg=wg)
        outs.append(m(torch.from_numpy(x).cuda()).cpu().numpy())
    assert np.array_equal(outs[0], outs[1])
    _check_probs(outs[1], z["y"], 2e-2, 2e-3, 0.99)


def test_fp32_mufu_variant_matches_reference():
    """The packed tanh.approx.f16x2 gate path (default) and the fp32 tanh.approx path both meet the stated tolerance."""
    z, meta, sd, x = golden_case("p24")
    for flag in (0, 1):
        m = _model(meta, sd, TC, lstm_mufu16=flag)
        y = m(torch.from_numpy(x).cuda()).cpu().numpy()
        _check_probs(y, z["y"], 2e-2, 2e-3, 0.99)


def test_forward_async_pinned_host_pipeline():
    z, meta, sd, x = golden_case("p24")
    m = _model(meta, sd, TC)
    ref = m(torch.from_numpy(x).cuda()).cpu().numpy()
    xs = [torch.from_numpy(x).pin_memory() for _ in range(3)]
    ys = [torch.empty((x.shape[0], 24), dtype=torch.float32).pin_memory() for _ in range(3)]
    streams = [torch.cuda.Stream() for _ in range(3)]
    for i in range(6):
        with torch.cuda.stream(streams[i % 3]):
            m.forward_async(xs[i % 3], ys[i % 3])
    torch.cuda.synchronize()
    for y in ys:
        assert np.array_equal(y.numpy(), ref)


@pytest.mark.parametrize("tile", [16, 64])
def test_concurrent_streams_are_consistent(tile):
    """Forwards of one model in flight on 8 CUDA streams (each with its own workspace) must equal the single-stream
    result.  Regression test for a race found this way: an epilogue thread copied h_t chunks written by other threads
    before they had been written (timing-dependent, only visible under memory contention)."""
    from clair3_b200 import synth
    sd = synth.pileup_state_dict(False, seed=0)
    meta = dict(kind="pileup", add_indel_length=False)
    m = _model(meta, sd, TC, lstm_tile=tile)
    xd = [torch.from_numpy(synth.pileup_inputs(1024, seed=100 + i)).cuda() for i in range(8)]
    ref = [m(x).cpu().numpy() for x in xd]
    streams = [torch.cuda.Stream() for _ in range(8)]
    for rep in range(4):
        outs = [None] * 8
        for i in range(8):
            with torch.cuda.stream(streams[i]):
                outs[i] = m(xd[i])
        torch.cuda.synchronize()
        for i in range(8):
            assert np.array_equal(outs[i].cpu().numpy(), ref[i])


def test_input_dtypes_agree():
    z, meta, sd, x = golden_case("p24_int8")
    m = _model(meta, sd, TC)
    names = ("lstm1", "lstm2", "l4_pre")
    outs, taps = [], []
    for dt in (np.int8, np.int32, np.float32):
        outs.append(m(torch.from_numpy(x.astype(dt)).cuda()).cpu().numpy())
        taps.append({k: m.tap(k) for k in names})
    # every dtype converts to the same fp32 count before the hi/lo split: identical operands, identical answer
    for i in (1, 2):
        assert np.array_equal(outs[0], outs[i])
        for k in names:
            assert np.array_equal(taps[0][k], taps[i][k]), k


def test_strict_state_dict_errors():
    from clair3_b200._ffi import C3BError
    z, meta, sd, x = golden_case("p24")
    bad = dict(sd)
    bad.pop("L4.bias")
    with pytest.raises(C3BError, match="Missing key"):
        _model(meta, bad, TC)
    bad = dict(sd)
    bad["nonsense.weight"] = np.zeros(3, dtype=np.float32)
    with pytest.raises(C3BError, match="Unexpected key"):
        _model(meta, bad, TC)
    bad = dict(sd)
    bad["L4.weight"] = np.zeros((128, 10), dtype=np.float32)
    with pytest.raises(C3BError, match="size mismatch"):
        _model(meta, bad, TC)


def test_large_batch_properties():
    """BASELINE.json full sizes through size-independent properties: rows are probability vectors, every site is
    independent of its batch neighbours (permutation equivariance), and the fp32 and fp16 tensor-core paths agree."""
    from clair3_b200 import synth
    sd = synth.pileup_state_dict(False, seed=11)
    x = synth.pileup_inputs(1024, seed=11)
    meta = dict(kind="pileup", add_indel_length=False)
    m = _model(meta, sd, TC)
    y = m(torch.from_numpy(x).cuda()).cpu().numpy()
    assert np.isfinite(y).all() and np.allclose(y[:, :21].sum(1), 1, atol=1e-4) and np.allclose(y[:, 21:].sum(1), 1, atol=1e-4)
    perm = np.random.default_rng(0).permutation(1024)
    yp = m(torch.from_numpy(x[perm]).cuda()).cpu().numpy()
    assert np.array_equal(yp, y[perm])
    m32 = _model(meta, sd, FP32)
    y32 = m32(torch.from_numpy(x[:256]).cuda()).cpu().numpy()
    assert np.abs(y[:256] - y32).max() < 2e-2

    sdf = synth.fa_state_dict(True, channels=8, seed=12)
    xf = synth.fa_inputs(256, depth=89, channels=8, seed=12)
    metaf = dict(kind="fa", add_indel_length=True, channels=8)
    mf = _model(metaf, sdf, TC)
    yf = mf(torch.from_numpy(xf).cuda()).cpu().numpy()
    assert np.isfinite(yf).all()
    for lo, hi in HEAD_SLICES:
        assert np.allclose(yf[:, lo:hi].sum(1), 1, atol=1e-4)
    permf = np.random.default_rng(1).permutation(256)
    ypf = mf(torch.from_numpy(xf[permf]).cuda()).cpu().numpy()
    assert np.array_equal(ypf, yf[permf])
    # all-zero rows beyond read depth (calloc'ed tensors): an all-zero site must still give finite probabilities
    z0 = mf(torch.zeros((4, 89, 33, 8), dtype=torch.int8).cuda()).cpu().numpy()
    assert np.isfinite(z0).all()
