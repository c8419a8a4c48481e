"""Test helper: a rounding-faithful restatement of the fp16 tensor-core forward pass, stage by stage, for per-element parity
checks of the kernels (tests/test_gpu_layer_parity.py).  Never imported by the package.

Built from oracle/clair3_oracle.py's primitives (sigmoid, selu, softmax, im2col, pyramid pooling).  It computes in float64
but rounds to fp16 exactly where the CUDA path stores fp16; what is left between it and a kernel is fp32 accumulation order
and the MUFU ``tanh.approx`` of the LSTM epilogues.  ``exact=True`` turns every rounding off: the stages then restate the
oracle itself (to fp64 reassociation).

Rounding points, weight side (``finalize_impl`` in clair3_b200/csrc/c3b_api.cu):
  * LSTM1: W_ih, W_hh and the fp32 sum b_ih + b_hh (the constant-1 input column), each times the gate scale (0.5 for the
    pre-halved sigmoid rows i, f, o; 1 for g), cast to fp16 (c3b_api.cu:413-421, pair image :438-446);
  * LSTM2: W_hh * gate scale to fp16 (:464-468, pair image :509-512); the projection's W_ih * gate scale to fp16
    (:474-478, :495-497), its bias (b_ih + b_hh) * gate scale stays fp32 (:465, :493);
  * convs: BatchNorm folded in fp32 (eps 1e-3), conv1's 1/100 folded into the fp32 weight, then fp16; bias fp32 (:524-550);
  * tail: L4 / L5 / Y weights fp16, biases fp32 (:354-370).
Rounding points, activation side:
  * LSTM1 input counts: hi = satfinite_f16(x), lo = satfinite_f16(x - hi) (lstm_tc.cu:481-483), exact for |x| <= 67 552;
  * h1 / h2 at every step (lstm_tc.cu:401 and :418, lstm2x_tc.cu:327: the next step's operand and the stored tap);
  * LSTM2 pre-gates pg = fp16(W_ih h1 + b) (proj_tc.cu:162-165, :173-174);
  * every feature map: bias (+ residual) + ReLU then fp16 (pconv_tc.cu:116-123, pconv2_tc.cu:119-131), including the
    residual block's mid map; the input int8 counts are exact in fp16 (fa_tc.cu:39,44);
  * SPP: max over fp16 values, stored fp16 (fa_tc.cu:66) - no rounding;
  * tail: SELU(L4 + b4) and SELU(L5 + b5) as fp16 operands (tail_tc.cu:192, :211); Y + by -> SELU -> softmax in fp32.
"""
import numpy as np

from oracle import clair3_oracle as orc

F16_MAX = 65504.0
HEADS = [("L5_1", "Y_gt21_logits"), ("L5_2", "Y_genotype_logits"),
         ("L5_3", "Y_indel_length_logits_1"), ("L5_4", "Y_indel_length_logits_2")]
CONVS = [("conv1.conv", "conv1.bn", 2), ("res_block1.0.conv1", "res_block1.0.bn1", 1), ("res_block1.0.conv2", "res_block1.0.bn2", 1),
         ("conv3.conv", "conv3.bn", 2), ("res_block2.0.conv1", "res_block2.0.bn1", 1), ("res_block2.0.conv2", "res_block2.0.bn2", 1),
         ("conv5.conv", "conv5.bn", 2), ("res_block3.0.conv1", "res_block3.0.bn1", 1), ("res_block3.0.conv2", "res_block3.0.bn2", 1)]


def f16(a):
    """Round to fp16 (round-to-nearest-even, saturating at +-65504 like cvt.rn.satfinite) and return float64."""
    a = np.asarray(a, dtype=np.float64)
    return np.clip(a, -F16_MAX, F16_MAX).astype(np.float16).astype(np.float64)


def split_counts(x):
    """The LSTM1 ingest's hi/lo split of raw counts (lstm_tc.cu:474-484): the count goes to fp32, hi = satfinite_f16(x),
    lo = satfinite_f16(x - hi) computed in fp32.  Returns (hi, lo) as float64; hi + lo == x exactly for |x| <= 67 552."""
    xf = np.asarray(x).astype(np.float32)
    hi = np.clip(xf, -F16_MAX, F16_MAX).astype(np.float16)
    lo = np.clip(xf - hi.astype(np.float32), -F16_MAX, F16_MAX).astype(np.float16)
    return hi.astype(np.float64), lo.astype(np.float64)


def _gate_scale(h):
    """Per gate row: 0.5 for the pre-halved sigmoid gates (i, f, o), 1 for g."""
    gs = np.full(4 * h, 0.5, dtype=np.float32)
    gs[2 * h:3 * h] = 1.0
    return gs


class KernelRef:
    """Weights prepared once per state_dict, the way c3b_finalize packs them; one method per stage."""

    def __init__(self, sd, exact=False):
        self.exact = exact
        self.sd = sd
        self.out_dim = 90 if "L5_3.weight" in sd else 24
        self.nheads = 4 if self.out_dim == 90 else 2
        self._w = {}

    # -- rounding primitives (no-ops when exact)
    def act16(self, a):
        return np.asarray(a, np.float64) if self.exact else f16(a)

    def weight16(self, w32, scale=None):
        """fp32 host value (times an fp32 scale) -> fp16 operand, returned in the unscaled domain as float64."""
        w32 = np.asarray(w32, np.float32)
        if scale is None:
            return np.asarray(w32, np.float64) if self.exact else f16(w32)
        if self.exact:
            return np.asarray(w32, np.float64)
        return f16(w32 * scale) / scale.astype(np.float64)     # the scale is a power of two: dividing back is exact

    # -- pileup
    def _lstm_w(self, layer, d):
        key = ("lstm", layer, d)
        if key not in self._w:
            sfx = "_l0_reverse" if d else "_l0"
            sd = self.sd
            wih = np.asarray(sd[f"{layer}.weight_ih{sfx}"], np.float32)
            whh = np.asarray(sd[f"{layer}.weight_hh{sfx}"], np.float32)
            dt = np.float64 if self.exact else np.float32             # the host sums the two biases in fp32
            bias = np.asarray(sd[f"{layer}.bias_ih{sfx}"], dt) + np.asarray(sd[f"{layer}.bias_hh{sfx}"], dt)
            gs = _gate_scale(whh.shape[1])
            if layer == "LSTM1" and not self.exact:
                b = self.weight16(bias, gs)                  # the bias is a weight column of the gate GEMM
            else:
                b = np.asarray(bias, np.float64)             # the projection's bias stays fp32 (fp32 * 0.5 is exact)
            self._w[key] = (self.weight16(wih, gs[:, None]), self.weight16(whh, gs[:, None]), b)
        return self._w[key]

    def _recurrence(self, xw, whh, reverse):
        """xw: [B,T,4H] input part of the pre-activations; h (fp16 operand) and c (fp32 register) recurrence."""
        B, T, G = xw.shape
        H = G // 4
        h = np.zeros((B, H))
        c = np.zeros((B, H))
        out = np.zeros((B, T, H))
        for t in (range(T - 1, -1, -1) if reverse else range(T)):
            g = xw[:, t] + h @ whh.T
            i = orc.sigmoid(g[:, :H])
            f = orc.sigmoid(g[:, H:2 * H])
            gg = np.tanh(g[:, 2 * H:3 * H])
            o = orc.sigmoid(g[:, 3 * H:])
            c = f * c + i * gg
            h = self.act16(o * np.tanh(c))
            out[:, t] = h
        return out

    def lstm1(self, x):
        """x: [B,33,C] raw counts -> h1 [B,33,256]."""
        if self.exact:
            xin = np.asarray(x).astype(np.float64)
        else:
            hi, lo = split_counts(x)
            xin = None
        outs = []
        for d in (0, 1):
            wih, whh, b = self._lstm_w("LSTM1", d)
            xw = (xin @ wih.T if xin is not None else hi @ wih.T + lo @ wih.T) + b
            outs.append(self._recurrence(xw, whh, d == 1))
        return np.concatenate(outs, axis=-1)

    def lstm2(self, h1):
        """h1: [B,33,256] (fp16 values) -> h2 [B,33,320]."""
        outs = []
        for d in (0, 1):
            wih, whh, b = self._lstm_w("LSTM2", d)
            gs = _gate_scale(whh.shape[1]).astype(np.float64)
            pg = self.act16((np.asarray(h1, np.float64) @ wih.T + b) * gs) / gs      # stored pre-halved, as fp16
            outs.append(self._recurrence(pg, whh, d == 1))
        return np.concatenate(outs, axis=-1)

    # -- shared tail
    def l4_pre(self, feats):
        """feats: [B,K] (flattened LSTM2 output or SPP features) -> L4 accumulator without bias [B,d4]."""
        if "L4" not in self._w:
            self._w["L4"] = self.weight16(self.sd["L4.weight"])
        return np.asarray(feats, np.float64).reshape(len(feats), -1) @ self._w["L4"].T

    def y(self, z4):
        """L4 accumulator without bias -> probabilities [B, 24|90]."""
        sd = self.sd
        a4 = self.act16(orc.selu(np.asarray(z4, np.float64) + np.asarray(sd["L4.bias"], np.float64)))
        outs = []
        for l5, yk in HEADS[:self.nheads]:
            a5 = self.act16(orc.selu(a4 @ self.weight16(sd[f"{l5}.weight"]).T + np.asarray(sd[f"{l5}.bias"], np.float64)))
            z = orc.selu(a5 @ self.weight16(sd[f"{yk}.weight"]).T + np.asarray(sd[f"{yk}.bias"], np.float64))
            outs.append(orc.softmax(z))
        return np.concatenate(outs, axis=1)

    def pileup(self, x):
        """Whole pileup pass; returns the stage outputs keyed like the library's taps, plus "y"."""
        t = {"lstm1": self.lstm1(x)}
        t["lstm2"] = self.lstm2(t["lstm1"])
        t["l4_pre"] = self.l4_pre(t["lstm2"])
        t["y"] = self.y(t["l4_pre"])
        return t

    # -- full alignment (maps NCHW, as the oracle)
    def _conv_w(self, i):
        if ("conv", i) not in self._w:
            conv, bn, stride = CONVS[i]
            sd = self.sd
            w, cb = np.asarray(sd[conv + ".weight"], np.float32), np.asarray(sd[conv + ".bias"], np.float32)
            g, be = np.asarray(sd[bn + ".weight"], np.float32), np.asarray(sd[bn + ".bias"], np.float32)
            mu, var = np.asarray(sd[bn + ".running_mean"], np.float32), np.asarray(sd[bn + ".running_var"], np.float32)
            if self.exact:
                s = np.asarray(g, np.float64) / np.sqrt(np.asarray(var, np.float64) + orc.BN_EPS)
                wf = w.astype(np.float64) * s[:, None, None, None] / (orc.NORMALIZE_NUM if i == 0 else 1.0)
                bf = (cb.astype(np.float64) - mu) * s + be
            else:
                s = g / np.sqrt(var + np.float32(orc.BN_EPS))                      # fp32, as the host folding
                bf = ((cb - mu) * s + be).astype(np.float64)
                wf = w * s[:, None, None, None]
                if i == 0:
                    wf = wf * np.float32(1.0 / orc.NORMALIZE_NUM)
                wf = f16(wf)
            self._w[("conv", i)] = (wf.reshape(wf.shape[0], -1), bf, stride)
        return self._w[("conv", i)]

    def conv(self, x, i, residual=None, chunk=32):
        """Conv i of CONVS on an NCHW map: fp32 accumulate, + bias (+ residual), ReLU, fp16 store."""
        w, b, stride = self._conv_w(i)
        x = np.asarray(x, np.float64)
        outs = []
        for s0 in range(0, len(x), chunk):
            cols, ho, wo = orc._im2col3x3(x[s0:s0 + chunk], stride)
            y = (cols @ w.T + b).transpose(0, 3, 1, 2)
            if residual is not None:
                y = y + residual[s0:s0 + chunk]
            outs.append(self.act16(np.maximum(y, 0)))
        return np.concatenate(outs)

    def conv1(self, x):
        """x: [B,depth,33,C] int8 NHWC -> conv1 map [B,64,h,w] (1/100 folded into the weights)."""
        return self.conv(np.asarray(x).astype(np.float64).transpose(0, 3, 1, 2), 0)

    def res_block(self, x, level):
        mid = self.conv(x, 3 * level + 1)
        return self.conv(mid, 3 * level + 2, residual=np.asarray(x, np.float64))

    def stem(self, x, level):
        return self.conv(x, 3 * level)

    def spp(self, x):
        return orc.pyramid_pool(np.asarray(x, np.float64))

    def fa(self, x):
        """Whole full-alignment pass; returns the stage outputs keyed like the library's taps (maps NCHW), plus "y"."""
        t = {"conv1": self.conv1(x)}
        t["res_block1"] = self.res_block(t["conv1"], 0)
        t["conv3"] = self.stem(t["res_block1"], 1)
        t["res_block2"] = self.res_block(t["conv3"], 1)
        t["conv5"] = self.stem(t["res_block2"], 2)
        t["res_block3"] = self.res_block(t["conv5"], 2)
        t["spp"] = self.spp(t["res_block3"])
        t["l4_pre"] = self.l4_pre(t["spp"])
        t["y"] = self.y(t["l4_pre"])
        return t


# ---------------------------------------------------------------------------------------------------- per-element checker
def stage_stats(got, ref):
    d = np.abs(np.asarray(got, np.float64) - np.asarray(ref, np.float64)).ravel()
    return {"n": int(d.size), "max": float(d.max()) if d.size else 0.0,
            "p99_99": float(np.quantile(d, 0.9999)) if d.size else 0.0,
            "rms": float(np.sqrt(np.mean(d * d))) if d.size else 0.0}


def check_stage(stage, got, ref, bound, axes, mean_axis=None, mean_bound=None):
    """Per-element comparison of one stage.  ``axes`` names the dimensions (e.g. ("site", "step", "unit")).  Fails with the
    worst element (its index by name and both values) when |got - ref| > bound anywhere.  With ``mean_axis`` the signed error
    averaged along that axis must also stay within ``mean_bound``: rounding errors average out, a systematic offset (a wrong
    bias, a shifted unit) does not.  Returns the stage's error statistics."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    assert got.shape == ref.shape, (stage, got.shape, ref.shape)
    assert len(axes) == got.ndim, (stage, axes, got.shape)
    st = stage_stats(got, ref)
    err = got - ref
    bad = ~(np.abs(err) <= bound)                      # NaN counts as bad
    if bad.any():
        idx = np.unravel_index(int(np.argmax(np.where(np.isnan(err), np.inf, np.abs(err)))), err.shape)
        where = ", ".join("%s %d" % (a, i) for a, i in zip(axes, idx))
        raise AssertionError("%s: %d element(s) beyond %.3g; worst at %s: got %.7g, ref %.7g (|d| = %.3g); max %.3g, p99.99 %.3g, "
                             "rms %.3g" % (stage, int(bad.sum()), bound, where, got[idx], ref[idx], abs(err[idx]), st["max"],
                                          st["p99_99"], st["rms"]))
    if mean_axis is not None:
        m = np.abs(err.mean(axis=mean_axis))
        st["max_mean"] = float(m.max())
        if not (m <= mean_bound).all():
            idx = np.unravel_index(int(np.argmax(m)), m.shape)
            rest = [a for k, a in enumerate(axes) if k != mean_axis]
            where = ", ".join("%s %d" % (a, i) for a, i in zip(rest, idx))
            raise AssertionError("%s: error averaged over %s is %.3g at %s (bound %.3g): a systematic offset"
                                 % (stage, axes[mean_axis], m[idx], where, mean_bound))
    return st
