"""CPU: oracle/ref_port.py — the reference's Quantizer and layer classes restated on the oracle, which
the parity and fuzz tests compare with where oracle/_ref/ is not staged — driven through its
classes against the vectors the live reference produced (tests/golden/make_golden.py).  Same bars
as tests/test_oracle_golden.py: outputs and input gradients bit-exact, parameter gradients within
1e-6 relative."""
import math
import types

import pytest
import torch

from oracle import ref_port
from tests import helpers as H

ref = ref_port.load()


class _RecordedNoise:
    """torch.randint_like -> the reference's recorded {0,1} draw for a tensor of that shape (the
    reference draws its noise in backward, gdnsq.py:54)."""

    def __init__(self, *bits):
        self.by_shape = {tuple(b.shape): b for b in bits if b is not None}

    def __enter__(self):
        self._orig = torch.randint_like
        torch.randint_like = lambda t, high, **kw: self.by_shape[tuple(t.shape)].to(t.dtype).clone()
        return self

    def __exit__(self, *a):
        torch.randint_like = self._orig


def _close(a, b, what):
    H.assert_close_rel(a, b, 1e-6, what, abs_floor=1e-7)


@pytest.mark.parametrize("name", H.golden_names("act_"))
def test_noisy_act_golden(name):
    c = H.load_golden(name)
    act = ref.NoisyAct(signed=c["signed"])
    with torch.no_grad():
        act.log_act_s.fill_(float(c["log_act_s"])); act.log_act_q.fill_(float(c["log_act_q"]))
        act.act_b.fill_(float(c["act_b"]))
    act.train()
    x = c["x"].clone().requires_grad_(True)
    with _RecordedNoise(c["noise_bits"]):
        y = act(x)
        y.backward(c["go"])
    H.assert_bit_exact(y, c["y"], "y")
    H.assert_bit_exact(x.grad, c["gx"], "gx")
    _close(act.log_act_s.grad, c["g_log_act_s"], "g_log_act_s")
    _close(act.log_act_q.grad, c["g_log_act_q"], "g_log_act_q")
    if c["signed"]:
        _close(act.act_b.grad, c["g_act_b"], "g_act_b")
    act.eval()
    with torch.no_grad():
        H.assert_bit_exact(act(c["x"]), c["y"], "y eval")
    H.assert_bit_exact(act.bw, c["bw"], "bw")


@pytest.mark.parametrize("name", H.golden_names("w_"))
def test_noisy_conv2d_weight_golden(name):
    c = H.load_golden(name)
    o, i, kh, kw = c["weight"].shape
    conv = ref.NoisyConv2d(i, o, (kh, kw), bias=True, quant_bias="bq" in c,
                           qscheme=ref.QScheme.PER_CHANNEL if c["per_channel"] else ref.QScheme.PER_TENSOR,
                           qnmethod=ref.QNMethod[c["method"]])
    with torch.no_grad():
        conv.weight.copy_(c["weight"]); conv.bias.copy_(c["bias"]); conv.log_wght_s.copy_(c["log_wght_s"])
    conv.train()
    with _RecordedNoise(c.get("noise_bits"), c.get("noise_bits_bias")):
        wq, bq = conv.quantized_weight()
        loss = (wq * c["go"]).sum()
        if "bq" in c:
            loss = loss + (bq * c["go_bias"]).sum()
        loss.backward()
    H.assert_bit_exact(wq, c["wq"], "wq")
    _close(conv.weight.grad, c["g_weight"], "g_weight")
    _close(conv.log_wght_s.grad, c["g_log_wght_s"], "g_log_wght_s")
    if "bq" in c:
        H.assert_bit_exact(bq, c["bq"], "bq")
        _close(conv.bias.grad, c["g_bias"], "g_bias")


def test_noisy_linear_golden():
    c = H.load_golden("lin_pt_lsq")
    lin = ref.NoisyLinear(c["weight"].shape[1], c["weight"].shape[0], bias=True,
                          qscheme=ref.QScheme.PER_TENSOR, qnmethod=ref.QNMethod.LSQ)
    with torch.no_grad():
        lin.weight.copy_(c["weight"]); lin.bias.copy_(c["bias"]); lin.log_wght_s.copy_(c["log_wght_s"])
    lin.train()
    x = c["x"].clone().requires_grad_(True)
    y = lin(x)
    y.backward(c["go"])
    H.assert_bit_exact(y, c["y"], "y")
    H.assert_bit_exact(x.grad, c["gx"], "gx")
    _close(lin.weight.grad, c["g_weight"], "g_weight")
    _close(lin.bias.grad, c["g_bias"], "g_bias")
    _close(lin.log_wght_s.grad, c["g_log_wght_s"], "g_log_wght_s")


def test_quantizer_codes_golden():
    c = H.load_golden("quantizer_codes_lsq")
    x, scale, zp = (c[k].clone().requires_grad_(True) for k in ("x", "scale", "zp"))
    Q = ref.Quantizer(types.SimpleNamespace(training=True), scale, zp, -math.inf, math.inf,
                      qnmethod=ref.QNMethod.LSQ)
    codes = Q.quantize(x)
    codes.backward(c["gcodes"])
    H.assert_bit_exact(codes, c["codes"], "codes")
    H.assert_bit_exact(x.grad, c["gx"], "gx")
    _close(scale.grad, c["g_scale"], "g_scale")
    _close(zp.grad, c["g_zp"], "g_zp")
