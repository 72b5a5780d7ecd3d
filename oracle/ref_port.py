"""The reference's quantizer API restated on ``oracle/fq_oracle.py``.  TEST INFRASTRUCTURE ONLY.

``ref_loader.load_ops()`` imports the unmodified reference from ``oracle/_ref/``, which is not part
of this repository.  Where it is not staged, the parity and fuzz tests compare with this module
instead: the same names (``Quantizer``, ``QNMethod``, ``QScheme``, ``gdnsq.QNSTE / QNLSQ / QNAEWGS``,
``NoisyAct``, ``NoisyConv2d``, ``NoisyLinear``), constructors, parameters and initial values, and
the arithmetic of ``fq_oracle`` — the reference's ATen ops in the reference's order, pinned
against the reference's own outputs by ``tests/golden/*.npz`` (``tests/test_oracle_golden.py``).
Like the reference, the noise of the GDNSQ estimators is drawn in backward through
``torch.randint_like``, so the tests' noise patches apply unchanged.
"""
from __future__ import annotations

import types
from enum import Enum

import torch
from torch import inf, nn
import torch.nn.functional as F

from . import fq_oracle as O

QNMethod = Enum("QNMethod", {"STE": 0, "EWGS": 1, "AEWGS": 2, "LSQ": 3})     # gdnsq_utils.py:9-13
QScheme = Enum("QScheme", {"PER_TENSOR": 0, "PER_CHANNEL": 1})               # aux/types.py


class _QN:
    """QNoise.apply(v, s) (gdnsq.py:11-147): round(v) - v with the estimator's backward."""
    method = O.STE

    @classmethod
    def apply(cls, value, scale):
        return O._RoundNoise.apply(value, scale, cls.method, None)


gdnsq = types.SimpleNamespace(
    QNSTE=type("QNSTE", (_QN,), {"method": O.STE}),
    QNLSQ=type("QNLSQ", (_QN,), {"method": O.LSQ}),
    QNAEWGS=type("QNAEWGS", (_QN,), {"method": O.AEWGS}),
    reduce_to_shape=O.reduce_to_shape)


class Quantizer:
    """gdnsq.py:159-229."""

    def __init__(self, module, scale, zero_point, min_val, max_val, rnoise_ratio=-1.0,
                 qnmethod=QNMethod.STE):
        self.module, self.scale, self.zero_point = module, scale, zero_point
        self.min_val, self.max_val, self.qnmethod = min_val, max_val, qnmethod
        self.positive_scale = torch.all(torch.as_tensor(scale) > 0).item()

    def quantize(self, value):
        if not self.positive_scale:
            return torch.clamp(value, min=self.min_val, max=self.max_val) - self.zero_point
        codes = O.quantize(value, self.scale, self.zero_point, self.min_val, self.max_val, self.qnmethod)
        if not self.module.training:
            O.check_codes(codes, self.scale, self.zero_point, self.min_val, self.max_val)
        return codes

    def dequantize(self, codes):
        if not self.positive_scale:
            return codes + self.zero_point
        return O.dequantize(codes, self.scale, self.zero_point)


class NoisyAct(nn.Module):
    """layers/gdnsq_act.py:9-55."""

    def __init__(self, init_s=-10, init_q=10, signed=True, noise_ratio=1, disable=False,
                 qnmethod=QNMethod.STE):
        super().__init__()
        self.disable, self.signed, self.qnmethod = disable, signed, qnmethod
        zero_point = 0.0 if not signed else -torch.exp2(torch.tensor(init_q - 1).float())
        self.log_act_q = nn.Parameter(torch.tensor([init_q]).float(), requires_grad=True)
        self.act_b = nn.Parameter(torch.tensor([zero_point]).float(), requires_grad=bool(signed))
        self.log_act_s = nn.Parameter(torch.tensor([init_s]).float(), requires_grad=True)
        self.bw = torch.tensor(0.0)

    def forward(self, x):
        if self.disable:
            return x
        s = torch.exp2(self.log_act_s)
        q = torch.exp2(self.log_act_q)
        Q = Quantizer(self, s, self.act_b, self.act_b, self.act_b + q - s, qnmethod=self.qnmethod)
        codes = Q.quantize(x)
        if not self.training:
            self.bw = O.act_bit_width(codes)
        return Q.dequantize(codes)


def _log_s_param(qscheme, rows, log_s_init):
    if qscheme == QScheme.PER_CHANNEL:
        return nn.Parameter(torch.empty((rows, 1, 1, 1)).fill_(log_s_init), requires_grad=True)
    return nn.Parameter(torch.Tensor([log_s_init]), requires_grad=True)


class NoisyConv2d(nn.Conv2d):
    """layers/gdnsq_conv2d.py:13-98: the bias quantizer reuses the weight's scale and row minimum."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1, groups=1,
                 bias=True, padding_mode="zeros", device=None, dtype=None, qscheme=QScheme.PER_TENSOR,
                 log_s_init=-12, rand_noise=False, quant_bias=False, qnmethod=QNMethod.AEWGS):
        super().__init__(in_channels, out_channels, kernel_size, stride, padding, dilation, groups,
                         bias, padding_mode, device, dtype)
        self.qscheme, self.quant_bias, self.qnmethod = qscheme, quant_bias, qnmethod
        self.log_wght_s = _log_s_param(qscheme, out_channels, log_s_init)
        if qscheme == QScheme.PER_CHANNEL:
            self.log_b_s = nn.Parameter(torch.empty(1).fill_(log_s_init), requires_grad=True)
        self._noise_ratio = nn.Parameter(torch.Tensor([1]), requires_grad=False)

    def quantized_weight(self):
        """(weight_q, bias_q) the convolution sees."""
        s = torch.exp2(self.log_wght_s)
        if self.qscheme == QScheme.PER_CHANNEL:
            zp = self.weight.amin((1, 2, 3), keepdim=True)
        else:
            zp = self.weight.amin()
        Q = Quantizer(self, s, zp, -inf, inf, qnmethod=self.qnmethod)
        weight = Q.dequantize(Q.quantize(self.weight))
        bias = self.bias
        if self.quant_bias:
            Qb = Quantizer(self, s.ravel(), zp.ravel(), -inf, inf, qnmethod=self.qnmethod)
            bias = Qb.dequantize(Qb.quantize(self.bias))
        return weight, bias

    def forward(self, input):
        return self._conv_forward(input, *self.quantized_weight())


class NoisyLinear(nn.Linear):
    """layers/gdnsq_linear.py:13-76 (per-channel takes amin((1, 2, 3)) of the 2-D weight and fails,
    as in the reference)."""

    def __init__(self, in_features, out_features, bias=True, device=None, dtype=None,
                 qscheme=QScheme.PER_TENSOR, log_s_init=-12, rand_noise=False, qnmethod=QNMethod.STE):
        super().__init__(in_features, out_features, bias, device, dtype)
        self.qscheme, self.qnmethod = qscheme, qnmethod
        self.log_wght_s = _log_s_param(qscheme, out_features, log_s_init)
        self._noise_ratio = nn.Parameter(torch.Tensor([1]), requires_grad=False)

    def forward(self, input):
        s = torch.exp2(self.log_wght_s)
        if self.qscheme == QScheme.PER_CHANNEL:
            zp = self.weight.amin((1, 2, 3), keepdim=True)
        else:
            zp = self.weight.amin()
        Q = Quantizer(self, s, zp, -inf, inf, qnmethod=self.qnmethod)
        return F.linear(input, Q.dequantize(Q.quantize(self.weight)), self.bias)


def load():
    """The namespace ``ref_loader.load_ops()`` returns, on the oracle."""
    return types.SimpleNamespace(gdnsq=gdnsq, QNMethod=QNMethod, QScheme=QScheme, Quantizer=Quantizer,
                                 NoisyAct=NoisyAct, NoisyConv2d=NoisyConv2d, NoisyLinear=NoisyLinear,
                                 root=None, level="port")
