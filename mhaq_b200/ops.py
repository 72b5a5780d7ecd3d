"""Autograd-level entry points of the B200 fake-quant path.

``fake_quant`` is the fused replacement for the reference's
``Q.dequantize(Q.quantize(x))`` (src/quantization/gdnsq/gdnsq.py:189-229);
``quantize_codes`` is ``Q.quantize(x)`` alone.  Both run ONE sm_100a kernel in
forward and ONE in backward (plus a tiny finalize), through the C ABI in
``include/mhaq_fq.h``.  CUDA tensors only; there is no CPU path.
"""
from __future__ import annotations

import ctypes
import math
import dataclasses
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import torch
import torch.distributed as dist

from . import _lib
from ._lib import lib, check

_check_rc = check   # for functions whose `check` argument shadows it

METHOD_IDS = {"STE": 0, "EWGS": 1, "AEWGS": 2, "LSQ": 3}


def _method_id(method) -> int:
    """Accepts the reference's QNMethod enum (gdnsq_utils.py:9-13), its name or its value."""
    if isinstance(method, int):
        mid = method
    elif isinstance(method, str):
        mid = METHOD_IDS[method]
    else:  # Enum
        mid = int(method.value)
    if mid not in (0, 1, 2, 3):
        raise AttributeError(f"Unknown method {method}!")
    return mid


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream() -> int:
    # raw cudaStream_t of torch's current stream; ~50x cheaper than torch.cuda.current_stream()
    # (which builds a Stream object) — this is called for every kernel launch
    return torch._C._cuda_getCurrentRawStream(torch.cuda.current_device())


def _require_cuda(x: torch.Tensor) -> None:
    if not x.is_cuda:
        raise RuntimeError(
            "mhaq_b200 fake-quant kernels are CUDA (sm_100a) only; got a "
            f"{x.device.type} tensor. There is no CPU fallback."
        )
    if x.dtype != torch.float32:
        raise RuntimeError(f"mhaq_b200 fake-quant is fp32 only, got {x.dtype}")


def _is_dense(x: torch.Tensor, axis: Optional[int]) -> bool:
    """True if the kernels can walk x's storage directly as [n_rows][n_inner]: row-major, or
    channels_last (NHWC / NDHWC strides) when the parameters are per-tensor (any dense
    permutation is one flat row) or per dim-0 channel (each dim-0 slice is still one dense
    block of numel/shape[0] elements).  cuDNN's fast convolution kernels want channels_last
    activations; taking them as they are avoids a layout copy either side of every quantizer."""
    if x.is_contiguous():
        return True
    if axis not in (None, 0):
        return False
    if x.dim() == 4:
        return x.is_contiguous(memory_format=torch.channels_last)
    if x.dim() == 5:
        return x.is_contiguous(memory_format=torch.channels_last_3d)
    return False


def _dense(x: torch.Tensor, axis: Optional[int]) -> torch.Tensor:
    return x if _is_dense(x, axis) else x.contiguous()


def _rows2d(t: torch.Tensor) -> torch.Tensor:
    """[rows = shape[0], inner] view of a tensor that is dense per dim-0 slice, in storage order."""
    rows = t.shape[0]
    if t.is_contiguous():
        return t.view(rows, -1)
    inner = t.numel() // rows
    return t.as_strided((rows, inner), (inner, 1))


def _unrows(t2d: torch.Tensor, like: torch.Tensor) -> torch.Tensor:
    """Inverse of _rows2d: a [rows, inner] storage-order result seen with `like`'s shape/strides."""
    if like.is_contiguous():
        return t2d.view_as(like)
    return t2d.as_strided(like.shape, like.stride())


def _like_layout(t: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """`t` (same shape as x) in x's memory layout, copying only if the strides differ."""
    if t.stride() == x.stride():
        return t
    return torch.empty_like(x).copy_(t)


class Geometry:
    """[n_rows][n_inner] view of a tensor and the channel layout of its parameters."""

    __slots__ = ("n_rows", "n_inner", "n_ch", "axis")

    def __init__(self, n_rows: int, n_inner: int, n_ch: int, axis: Optional[int]):
        self.n_rows, self.n_inner, self.n_ch, self.axis = n_rows, n_inner, n_ch, axis

    def param_shape(self, x_shape: Sequence[int]) -> Tuple[int, ...]:
        if self.axis is None:
            return (1,)
        return tuple(x_shape[d] if d == self.axis else 1 for d in range(len(x_shape)))


def infer_geometry(x: torch.Tensor, params: Sequence[Optional[torch.Tensor]]) -> Geometry:
    """Find the (single) channel axis the parameters broadcast along.

    Per-tensor: every parameter has one element.  Per-channel: a parameter of
    shape like (O,1,1,1) against x (O,I,kh,kw) — channel axis 0 — or (O,)
    against a bias (O,).  (gdnsq_conv2d.py:53-56, 80-88.)
    """
    axis = None
    for p in params:
        if p is None or p.numel() == 1:
            continue
        shape = list(p.shape)
        # right-align like broadcasting
        shape = [1] * (x.dim() - len(shape)) + shape
        if len(shape) != x.dim():
            raise RuntimeError(f"parameter shape {tuple(p.shape)} does not broadcast to {tuple(x.shape)}")
        nz = [d for d, s in enumerate(shape) if s != 1]
        if len(nz) != 1 or shape[nz[0]] != x.shape[nz[0]]:
            raise RuntimeError(
                f"parameter shape {tuple(p.shape)}: only one broadcast (channel) axis is supported"
            )
        if axis is not None and axis != nz[0]:
            raise RuntimeError("parameters disagree on the channel axis")
        axis = nz[0]
    n = x.numel()
    if axis is None:
        return Geometry(1, n, 1, None)
    n_ch = x.shape[axis]
    n_inner = 1
    for d in range(axis + 1, x.dim()):
        n_inner *= x.shape[d]
    n_rows = n // n_inner if n_inner else 0
    return Geometry(n_rows, n_inner, n_ch, axis)


def _prep_param(p, x: torch.Tensor, name: str):
    """-> (flat fp32 contiguous CUDA tensor or None, stride 0/1)."""
    if p is None:
        return None, 0
    if not torch.is_tensor(p):
        v = float(p)
        if name == "lo" and v == -math.inf:
            return None, 0
        if name == "hi" and v == math.inf:
            return None, 0
        p = torch.full((1,), v, dtype=torch.float32, device=x.device)
    if p.device != x.device:
        p = p.to(x.device)
    if p.dtype != torch.float32:
        p = p.float()
    if not p.is_contiguous():
        p = p.contiguous()
    # only the data pointer and the element count are used: no detach / reshape views needed
    return p, (0 if p.numel() == 1 else 1)


_ws_bytes_cache = {}


def _ws_bytes(geo: Geometry) -> int:
    key = (geo.n_rows, geo.n_inner)
    v = _ws_bytes_cache.get(key)
    if v is None:
        if len(_ws_bytes_cache) > 4096:
            _ws_bytes_cache.clear()
        v = _ws_bytes_cache[key] = int(lib.mhaq_fq_workspace_bytes(geo.n_rows, geo.n_inner))
    return v


def _workspace(x: torch.Tensor, geo: Geometry) -> torch.Tensor:
    """A fresh scratch buffer (callers that keep several in flight, CUDA-graph capture)."""
    return torch.empty(_ws_bytes(geo) // 8, dtype=torch.float64, device=x.device)


# Per-(device, stream[, graph capture]) scratch of the backward pass.  Calls ordered on one stream may share
# the record workspace (kernel k+1 writes it after finalize k has read it) and the ticket
# counters (zero on entry, restored to zero by the kernel: include/mhaq_fq.h), so the eager
# training path allocates nothing per call.  Bounded: the least recently used stream's entry is
# dropped beyond _ARENA_MAX streams.
_ARENA_MAX = 16
_ticket_need_cache = {}
_arenas = {}


class _Arena:
    __slots__ = ("ws", "tickets")

    def __init__(self):
        self.ws = None
        self.tickets = None


def _arena(x: torch.Tensor) -> _Arena:
    raw = torch._C._cuda_getCurrentRawStream(x.device.index)
    # A capture gets an arena of its own (key: the capture id): the graph may be replayed on any
    # stream later, concurrently with eager launches on the stream it was captured from, so its
    # ticket buffer must not be the stream's.  (Its zero-fill is captured once per graph; the
    # memory comes from the graph's private pool and stays reserved for the graph's lifetime.)
    cap = int(lib.mhaq_fq_stream_capture_id(raw)) if torch.cuda.is_current_stream_capturing() else 0
    key = (x.device.index, raw, cap)
    a = _arenas.get(key)
    if a is None:
        if len(_arenas) >= _ARENA_MAX:
            _arenas.pop(next(iter(_arenas)))
        a = _arenas[key] = _Arena()
    elif len(_arenas) > 1:
        _arenas[key] = _arenas.pop(key)          # most recently used last
    return a


def _tickets(x: torch.Tensor, geo: Geometry, a: Optional[_Arena] = None) -> torch.Tensor:
    # per-channel tickets + the flat backward's record region (include/mhaq_fq.h)
    n_ch = geo.n_ch if geo.n_ch > 0 else 1
    need = _ticket_need_cache.get(n_ch)
    if need is None:
        if len(_ticket_need_cache) > 4096:
            _ticket_need_cache.clear()
        need = _ticket_need_cache[n_ch] = int(lib.mhaq_fq_ticket_count(geo.n_rows, geo.n_inner, n_ch))
    if a is None:
        a = _arena(x)
    buf = a.tickets
    if buf is None or buf.numel() < need:
        n = max(32768, 1 << (int(need) - 1).bit_length())
        buf = a.tickets = torch.zeros(n, dtype=torch.int32, device=x.device)
    return buf


def _shared_workspace(x: torch.Tensor, geo: Geometry, a: Optional[_Arena] = None) -> torch.Tensor:
    """The stream's reusable record workspace (a CUDA-graph capture has an arena of its own, so a
    captured call never aliases scratch that eager calls keep using)."""
    need = _ws_bytes(geo) // 8
    if a is None:
        a = _arena(x)
    buf = a.ws
    if buf is None or buf.numel() < need:
        n = max(1 << 15, 1 << (int(need) - 1).bit_length())
        buf = a.ws = torch.empty(n, dtype=torch.float64, device=x.device)
    return buf


def _next_philox(device: torch.device) -> Tuple[int, int]:
    """Draw a fresh (seed, offset) pair from torch's CUDA generator of `device`."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    gen = torch.cuda.default_generators[idx]
    seed = gen.initial_seed()
    off = gen.get_offset()
    gen.set_offset(off + 4)
    return seed & 0xFFFFFFFFFFFFFFFF, off // 4


# Optional device-resident Philox state (uint64[2] = seed, step): makes the
# backward CUDA-graph capturable because nothing host-side changes per step.
_philox_dev = {}


_philox_call = {}


def set_device_philox_state(state: Optional[torch.Tensor]) -> None:
    """state: int64 CUDA tensor [2] = (seed, stream base) read by the kernels at run time.
    With a device-resident state nothing host-side changes from step to step, so a training
    step can be captured in a CUDA graph: advance ``state[1]`` on the device once per step
    (by at least the number of quantizer backward calls in a step) and call
    ``reset_philox_call_counter()`` at the start of every step so each backward call gets
    the same per-call stream index in every (captured or eager) step."""
    if state is None:
        _philox_dev.clear()
        _philox_call.clear()
        return
    assert state.is_cuda and state.dtype == torch.int64 and state.numel() == 2
    _philox_dev[state.device.index] = state
    _philox_call[state.device.index] = 0


def reset_philox_call_counter() -> None:
    for k in _philox_call:
        _philox_call[k] = 0


PARAMS_LINEAR, PARAMS_ACT_LOG, PARAMS_WEIGHT_LOG, PARAMS_UNIT = 0, 1, 2, 3


class _Launch:
    """Flattened, validated launch description shared by forward and backward."""

    mode = PARAMS_LINEAR
    stats_over_all = False

    def __init__(self, x, scale, zp, lo, hi):
        _require_cuda(x)
        self.geo = infer_geometry(x, [p for p in (scale, zp, lo, hi) if torch.is_tensor(p)])
        self.scale, self.ss = _prep_param(scale, x, "scale")
        self.zp, self.zs = _prep_param(zp, x, "zp")
        self.lo, self.ls = _prep_param(lo, x, "lo")
        self.hi, self.hs = _prep_param(hi, x, "hi")
        if self.scale is None or self.zp is None:
            raise RuntimeError("scale and zero_point are required")
        # Reference quirk: QNAEWGS averages its statistics over the dims where the scale has
        # size 1 (reduce_to_shape, gdnsq.py:150-152).  A per-channel scale WITHOUT singleton
        # dims — the quantized bias: value (O,), scale (O,) (gdnsq_conv2d.py:86-94) — gives an
        # empty dim tuple, and torch.mean(dim=()) reduces over everything: the statistics are
        # then per TENSOR although scale / zero point stay per channel.
        self.stats_over_all = (torch.is_tensor(scale) and scale.dim() > 0 and scale.numel() > 1
                               and all(n != 1 for n in scale.shape))

    @classmethod
    def act_log(cls, x, log_act_s, log_act_q, act_b):
        """MHAQ_FQ_PARAMS_ACT_LOG: the kernels read the three NoisyAct parameters directly."""
        _require_cuda(x)
        L = cls.__new__(cls)
        L.mode = PARAMS_ACT_LOG
        L.geo = Geometry(1, x.numel(), 1, None)
        L.scale, L.ss = _prep_param(log_act_s, x, "scale")
        L.zp, L.zs = _prep_param(act_b, x, "zp")
        L.lo, L.ls = _prep_param(log_act_q, x, "lo_param")
        L.hi, L.hs = None, 0
        if not (L.scale.numel() == L.zp.numel() == L.lo.numel() == 1):
            raise RuntimeError("NoisyAct parameters must have one element each")
        return L

    @classmethod
    def weight_log(cls, w, log_wght_s, zp_rows):
        """MHAQ_FQ_PARAMS_WEIGHT_LOG: per-channel (dim 0) log-scale, zero point per row."""
        _require_cuda(w)
        L = cls.__new__(cls)
        L.mode = PARAMS_WEIGHT_LOG
        rows = w.shape[0]
        L.geo = Geometry(rows, w.numel() // rows if rows else 0, rows, 0)
        L.scale, L.ss = _prep_param(log_wght_s, w, "scale")
        L.zp, L.zs = _prep_param(zp_rows, w, "zp")
        L.lo = L.hi = None
        L.ls = L.hs = 0
        if L.scale.numel() != rows or L.zp.numel() != rows:
            raise RuntimeError("per-channel weight parameters must have one entry per row of dim 0")
        return L

    @classmethod
    def unit(cls, v, scale):
        """MHAQ_FQ_PARAMS_UNIT: `v` is already scaled (the two-step `v + QN*.apply(v, s)` form);
        `scale` only fixes the channel layout of the estimator's scale gradient."""
        _require_cuda(v)
        L = cls.__new__(cls)
        L.mode = PARAMS_UNIT
        L.geo = infer_geometry(v, [scale])
        L.scale, L.ss = _prep_param(scale, v, "scale")
        L.zp, L.zs = L.scale, L.ss
        L.lo = L.hi = None
        L.ls = L.hs = 0
        L.stats_over_all = (scale.dim() > 0 and scale.numel() > 1 and all(n != 1 for n in scale.shape))
        return L

    def params(self):
        return (_ptr(self.scale), _ptr(self.zp), _ptr(self.lo), _ptr(self.hi),
                self.ss, self.zs, self.ls, self.hs, self.mode)


def _forward_impl(x, L: _Launch, want_y: bool, want_codes: bool, want_minmax: bool):
    geo = L.geo
    y = torch.empty_like(x) if want_y else None
    codes = torch.empty_like(x) if want_codes else None
    mm = None
    ws = None
    if x.numel() > 0:
        if want_minmax:
            ws = _workspace(x, geo)
        check(lib.mhaq_fq_fwd_f32(_ptr(x), _ptr(y), _ptr(codes), *L.params(),
                                  geo.n_rows, geo.n_inner, geo.n_ch, _ptr(ws), _stream()),
              "mhaq_fq_fwd_f32")
        if want_minmax:
            mm = torch.empty(5, dtype=torch.float32, device=x.device)
            check(lib.mhaq_fq_minmax_finalize(_ptr(ws), geo.n_rows, geo.n_inner, _ptr(mm), _stream()),
                  "mhaq_fq_minmax_finalize")
    return y, codes, mm


def launches_per_fwd_bwd(x, scale, zp, lo, hi, method) -> int:
    """How many kernels of this library one fake_quant forward + backward launches for these
    operands: forward, backward, finalize (+ the AEWGS statistics kernel and its finalize)."""
    mid = _method_id(method)
    geo = infer_geometry(x, [p for p in (scale, zp, lo, hi) if torch.is_tensor(p)])
    single = lib.mhaq_fq_bwd_single_launch(geo.n_rows, geo.n_inner, geo.n_ch, mid, 0)
    return (2 if single else 3) + (2 if mid == METHOD_IDS["AEWGS"] else 0)


def _reduce_to_param(g: torch.Tensor, param, geo: Geometry, x_shape):
    """[n_ch] channel gradients -> gradient shaped like `param` (sum_to_size)."""
    if not torch.is_tensor(param):
        return None
    if param.numel() == 1 and g.numel() > 1:
        g = g.sum()
    return g.reshape(param.shape).to(param.dtype)


def aewgs_stats(go, x, L: _Launch, code_grad: bool) -> torch.Tensor:
    """Packed per-channel means [3*n_ch] = (num, e2, me), all-reduced once (AVG) under DDP.

    Reference: three reductions + three all_reduce calls (gdnsq.py:118-129)."""
    geo = L.geo
    ws = _workspace(x, geo)
    stats = torch.empty(3 * geo.n_ch, dtype=torch.float32, device=x.device)
    check(lib.mhaq_fq_aewgs_stats_f32(_ptr(go), _ptr(x), *L.params(), geo.n_rows, geo.n_inner,
                                      geo.n_ch, int(code_grad), _ptr(ws), _stream()),
          "mhaq_fq_aewgs_stats_f32")
    check(lib.mhaq_fq_aewgs_stats_finalize_f32(_ptr(ws), geo.n_rows, geo.n_inner, geo.n_ch,
                                               _ptr(stats), _stream()),
          "mhaq_fq_aewgs_stats_finalize_f32")
    if L.stats_over_all and geo.n_ch > 1:
        # channels hold equally many elements, so the mean over everything is the mean of the
        # channel means; every channel then uses the same (num, e2, me)
        stats = stats.view(3, geo.n_ch).mean(dim=1, keepdim=True).expand(3, geo.n_ch).reshape(-1).contiguous()
    return allreduce_packed_stats(stats)


def allreduce_packed_stats(stats: torch.Tensor) -> torch.Tensor:
    """The one exchange step on the path: AVG all-reduce of the packed [3*n_ch] AEWGS
    statistics (num | e2 | me) — one collective where the reference issues three
    (gdnsq.py:126-129).  No-op outside a process group."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.AVG)
    return stats


def _noise_source(x, method: int, noise, philox):
    """-> (explicit noise tensor in x's layout or None, seed, offset, device Philox state or None)
    for one backward call: an explicit tensor (parity runs), a given (seed, offset), the
    device-resident state (CUDA graphs) or a fresh draw from torch's CUDA generator."""
    seed = offset = 0
    pdev = None
    if noise is not None:
        if noise.shape != x.shape or noise.dtype != torch.float32 or not noise.is_cuda:
            raise RuntimeError("explicit noise must be an fp32 CUDA tensor shaped like the input")
        noise = _like_layout(noise, x)
    elif method != METHOD_IDS["LSQ"]:
        if philox is not None:
            seed, offset = philox
        else:
            pd = _philox_dev.get(x.device.index)
            if pd is not None:
                pdev = pd            # kernel: seed = pd[0], offset = pd[1] + this call's index
                offset = _philox_call[x.device.index]
                _philox_call[x.device.index] = offset + 1
            else:
                seed, offset = _next_philox(x.device)
    return noise, seed, offset, pdev


def _backward_impl(go, x, L: _Launch, method: int, code_grad: bool, noise, need_gx: bool,
                   philox=None, acc=None):
    geo = L.geo
    go = _like_layout(go, x)
    gx = torch.empty_like(x) if need_gx else None
    n_ch = geo.n_ch
    if x.numel() == 0:
        return gx, torch.zeros(4, n_ch, dtype=torch.float32, device=x.device)
    out = torch.empty(4, n_ch, dtype=torch.float32, device=x.device)   # fully written by the kernel
    if method == METHOD_IDS["AEWGS"] and geo.axis is None and x.dim() >= 2 and L.scale.dim() == 1:
        if L.mode not in (PARAMS_LINEAR, PARAMS_UNIT):
            # (the log-domain modes return log-domain gradients of ONE channel; the dim-0 quirk
            # needs per-position channels — the layers route AEWGS through the linear operands)
            raise NotImplementedError("per-tensor AEWGS needs the linear parameter mode")
        return _backward_aewgs_dim0(go, x, L, code_grad, noise, need_gx, philox)
    stats = aewgs_stats(go, x, L, code_grad) if method == METHOD_IDS["AEWGS"] else None
    arena = _arena(x)
    ws = _shared_workspace(x, geo, arena)
    noise, seed, offset, pdev = _noise_source(x, method, noise, philox)
    tk = _tickets(x, geo, arena)
    # one C call: backward + deterministic reduction (ONE kernel for per-tensor STE / LSQ,
    # otherwise the streaming backward followed by the finalize kernel)
    if acc is None:
        check(lib.mhaq_fq_bwd_fused_f32(_ptr(go), _ptr(x), _ptr(gx), *L.params(),
                                        geo.n_rows, geo.n_inner, geo.n_ch, method, int(code_grad),
                                        _ptr(noise), seed, offset, _ptr(pdev), _ptr(stats), _ptr(ws), _ptr(tk),
                                        _ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]), _stream()),
              "mhaq_fq_bwd_fused_f32")
    else:
        # acc = gradients the same four parameters receive along other paths of the graph
        # (quantization/gdnsq/_funnel.py): added in the kernel, no accumulation launch
        check(lib.mhaq_fq_bwd_fused_acc_f32(_ptr(go), _ptr(x), _ptr(gx), *L.params(),
                                            geo.n_rows, geo.n_inner, geo.n_ch, method, int(code_grad),
                                            _ptr(noise), seed, offset, _ptr(pdev), _ptr(stats), _ptr(ws), _ptr(tk),
                                            _ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]),
                                            _ptr(acc[0]), _ptr(acc[1]), _ptr(acc[2]), _ptr(acc[3]), _stream()),
              "mhaq_fq_bwd_fused_acc_f32")
    return gx, out


def _backward_aewgs_dim0(go, x, L: _Launch, code_grad, noise, need_gx, philox):
    """Per-tensor AEWGS, reference quirk 9: with a scale of shape (1,) `reduce_to_shape`
    (gdnsq.py:150-152) averages over dim 0 ONLY, i.e. the statistics (hence delta) are per
    inner position, shared across dim 0.  Run the per-channel kernels on the transposed view
    [P = numel/shape[0]][O = shape[0]] with channel = inner position and broadcast scalar
    parameters, then transpose the input gradient back.  (Small weight tensors in practice.)"""
    O_, P_ = x.shape[0], x.numel() // x.shape[0]
    xt = x.reshape(O_, P_).t().contiguous()
    got = go.reshape(O_, P_).t().contiguous()
    nt = None if noise is None else noise.reshape(O_, P_).t().contiguous()
    Lt = _Launch.__new__(_Launch)
    Lt.mode = L.mode
    Lt.geo = Geometry(P_, O_, P_, 0)
    Lt.scale, Lt.ss, Lt.zp, Lt.zs = L.scale, 0, L.zp, 0
    Lt.lo, Lt.ls, Lt.hi, Lt.hs = L.lo, 0, L.hi, 0
    for p in (L.scale, L.zp, L.lo, L.hi):
        if p is not None and p.numel() != 1:
            raise NotImplementedError("per-tensor AEWGS expects scalar parameters")
    gxt, out = _backward_impl(got, xt, Lt, METHOD_IDS["AEWGS"], code_grad, nt, need_gx, philox)
    gx = None if gxt is None else gxt.t().reshape(x.shape).contiguous()
    return gx, out.sum(dim=1, keepdim=True)


class _FakeQuantFn(torch.autograd.Function):
    """y = dequantize(quantize(x)); saves only x and the O(channels) parameters."""

    @staticmethod
    def forward(ctx, x, scale, zp, lo, hi, method, noise, philox, code_only):
        L = _Launch(x, scale, zp, lo, hi)
        # (per-tensor AEWGS re-views the tensor along dim 0, reference quirk 9: row-major only)
        x = x.contiguous() if method == METHOD_IDS["AEWGS"] and L.geo.axis is None else _dense(x, L.geo.axis)
        y, codes, _ = _forward_impl(x, L, want_y=not code_only, want_codes=code_only,
                                    want_minmax=False)
        prm = (scale, zp, lo, hi)
        ctx.save_for_backward(x, *(p for p in prm if torch.is_tensor(p)))
        ctx.is_t = tuple(torch.is_tensor(p) for p in prm)
        # the flattened parameter views of L alias the saved tensors' storage: reuse the launch
        # description in backward instead of re-deriving it (host overhead matters for the
        # small tensors of CIFAR-sized models)
        ctx.L = L
        ctx.method, ctx.noise, ctx.philox, ctx.code_only = method, noise, philox, code_only
        return codes if code_only else y

    @staticmethod
    def backward(ctx, go):
        saved = ctx.saved_tensors          # also performs autograd's in-place-modification check
        x = saved[0]
        L = ctx.L
        need = ctx.needs_input_grad
        gx, out = _backward_impl(go, x, L, ctx.method, ctx.code_only, ctx.noise, need[0], ctx.philox)
        geo = L.geo
        grads = [gx if need[0] else None]
        k = 1
        for i, is_t in enumerate(ctx.is_t):
            if is_t:
                p = saved[k]
                k += 1
                grads.append(_reduce_to_param(out[i], p, geo, x.shape) if need[1 + i] else None)
            else:
                grads.append(None)
        return (*grads, None, None, None, None)


def fake_quant(x, scale, zero_point, min_val=None, max_val=None, method="STE", noise=None,
               philox=None):
    """Fused fake-quantization with the reference's gradients.

    Forward (bit-exact to gdnsq.py:197-208, 229):
        y = rint((clamp(x, min_val, max_val) - zero_point) / scale) * scale + zero_point
    Backward: gradients for x, scale, zero_point, min_val, max_val exactly as
    autograd derives them for the reference graph with estimator ``method``
    (QNSTE / QNEWGS / QNAEWGS / QNLSQ).  ``noise``: explicit {-0.5,+0.5} tensor
    standing in for ``randint_like(v,2)-0.5`` (parity runs); default draws it
    in-kernel from Philox keyed by torch's CUDA generator.
    """
    return _FakeQuantFn.apply(x, scale, zero_point, min_val, max_val, _method_id(method), noise,
                              philox, False)


def quantize_codes(x, scale, zero_point, min_val=None, max_val=None, method="STE", noise=None,
                   philox=None):
    """``Quantizer.quantize`` alone: integer-valued fp32 codes, differentiable."""
    return _FakeQuantFn.apply(x, scale, zero_point, min_val, max_val, _method_id(method), noise,
                              philox, True)


def quantize_eval(x, scale, zero_point, min_val=None, max_val=None, want_y=True, want_codes=False):
    """No-grad forward that also returns (min code, max code, #non-finite codes) as a
    3-element CUDA tensor — the eval-mode extras of gdnsq.py:211-217 / gdnsq_act.py:51-54
    in the same pass."""
    x = x.detach()
    L = _Launch(x, scale, zero_point, min_val, max_val)
    return _forward_impl(_dense(x, L.geo.axis), L, want_y, want_codes, True)


class _RoundingNoiseFn(torch.autograd.Function):
    """The reference's QNoise family (gdnsq.py:11-147) as a stand-alone op: forward
    ``round(v) - v`` on an already-scaled value, backward the estimator's (grad_v, grad_scale)."""

    @staticmethod
    def forward(ctx, v, scale, method, noise, philox):
        L = _Launch.unit(v, scale)
        v = v.contiguous() if method == METHOD_IDS["AEWGS"] and L.geo.axis is None else _dense(v, L.geo.axis)
        _, codes, _ = _forward_impl(v, L, want_y=False, want_codes=True, want_minmax=False)
        ctx.save_for_backward(v, scale)
        ctx.L, ctx.method, ctx.noise, ctx.philox = L, method, noise, philox
        return codes.sub_(v) if codes is not None else torch.empty_like(v)

    @staticmethod
    def backward(ctx, go):
        v, scale = ctx.saved_tensors
        need = ctx.needs_input_grad
        # codes = v + noise: the backward kernel, fed d/d codes = go, returns d codes/dv * go;
        # the identity branch (the `v +` of gdnsq.py:208) is not part of this op
        gx, out = _backward_impl(go, v, ctx.L, ctx.method, True, ctx.noise, need[0], ctx.philox)
        gv = None
        if need[0]:
            gv = gx.sub_(_like_layout(go, v))
        gs = _reduce_to_param(out[0], scale, ctx.L.geo, v.shape) if need[1] else None
        return gv, gs, None, None, None


def rounding_noise(v, scale, method="STE", noise=None, philox=None):
    """``QN<method>.apply(v, scale)`` of the reference: ``round(v) - v`` with the estimator's
    gradients (gdnsq.py:35-57 STE, 63-84 LSQ, 90-107 EWGS, 113-147 AEWGS)."""
    _require_cuda(v)
    if not torch.is_tensor(scale):
        scale = torch.full((1,), float(scale), dtype=torch.float32, device=v.device)
    return _RoundingNoiseFn.apply(v, scale, _method_id(method), noise, philox)


def philox_noise(shape_like: torch.Tensor, scale_like=None, seed: int = 0, offset: int = 0):
    """Materialise the kernels' noise stream r in {-0.5,+0.5} for `shape_like` (tests)."""
    _require_cuda(shape_like)
    geo = infer_geometry(shape_like, [scale_like] if torch.is_tensor(scale_like) else [])
    r = torch.empty_like(shape_like, memory_format=torch.contiguous_format)
    if r.numel():
        check(lib.mhaq_fq_noise_f32(_ptr(r), geo.n_rows, geo.n_inner, seed, offset, None, _stream()),
              "mhaq_fq_noise_f32")
    return r


def row_stats(x2d: torch.Tensor):
    """(row_min, row_max, n_at_min, n_at_max) of a [rows, inner] view in one pass."""
    _require_cuda(x2d)
    x2d = x2d.contiguous()
    rows, inner = x2d.shape
    o = torch.empty(4, rows, dtype=torch.float32, device=x2d.device)
    check(lib.mhaq_fq_rowstat_f32(_ptr(x2d), rows, inner, _ptr(o[0]), _ptr(o[1]), _ptr(o[2]),
                                  _ptr(o[3]), _stream()), "mhaq_fq_rowstat_f32")
    return o[0], o[1], o[2], o[3]


def row_stats_backward(gx, x2d, row_min=None, n_at_min=None, g_min=None, row_max=None,
                       n_at_max=None, g_max=None):
    """gx + amin/amax backward in one pass: adds g_min[row]/n_at_min[row] to every element equal
    to the row minimum (torch's even split among ties) and likewise for the maximum."""
    _require_cuda(x2d)
    x2d = x2d.contiguous()
    rows, inner = x2d.shape
    out = torch.empty_like(x2d)
    c = lambda t: None if t is None else t.contiguous()
    gx, row_min, n_at_min, g_min, row_max, n_at_max, g_max = map(
        c, (gx, row_min, n_at_min, g_min, row_max, n_at_max, g_max))
    check(lib.mhaq_fq_rowstat_bwd_f32(_ptr(gx), _ptr(x2d), rows, inner, _ptr(row_min), _ptr(n_at_min),
                                      _ptr(g_min), _ptr(row_max), _ptr(n_at_max), _ptr(g_max),
                                      _ptr(out), _stream()), "mhaq_fq_rowstat_bwd_f32")
    return out


class _WeightFakeQuantFn(torch.autograd.Function):
    """Per-channel weight quantizer with the zero point fused in:
        zp = row minimum of the weight (gdnsq_conv2d.py:80-81), wq = fake_quant(w, s, zp)
    Outputs (wq, row_min, row_max): the row range is what ModelHelper.get_model_values
    (model_helper.py:24-25) needs, so the weight is reduced ONCE per step instead of three
    times, and the three amin/amax backward passes (even split among ties) collapse into one
    scatter fused with the input gradient."""

    @staticmethod
    def forward(ctx, w, scale, method, noise, philox):
        ctx.set_materialize_grads(False)
        w = _dense(w, 0)
        rows = w.shape[0]
        mn, mx, cmn, cmx = row_stats(_rows2d(w))
        pshape = (rows,) + (1,) * (w.dim() - 1)
        L = _Launch(w, scale, mn.view(pshape), None, None)
        wq, _, _ = _forward_impl(w, L, True, False, False)
        ctx.save_for_backward(w, scale, mn, mx, cmn, cmx)
        ctx.method, ctx.noise, ctx.philox, ctx.pshape = method, noise, philox, pshape
        return wq, mn, mx

    @staticmethod
    def backward(ctx, g_wq, g_mn, g_mx):
        w, scale, mn, mx, cmn, cmx = ctx.saved_tensors
        w2 = _rows2d(w)
        g_scale = None
        if g_wq is not None:
            L = _Launch(w, scale, mn.view(ctx.pshape), None, None)
            gx, out = _backward_impl(g_wq, w, L, ctx.method, False, ctx.noise, True, ctx.philox)
            g_scale = _reduce_to_param(out[0], scale, L.geo, w.shape)
            g_min = out[1] if g_mn is None else out[1] + g_mn
            gx2 = _rows2d(gx)
        else:
            gx2, g_min = None, g_mn
        if not ctx.needs_input_grad[0]:
            return None, g_scale, None, None, None
        if g_min is None and g_mx is None:
            gw = torch.zeros_like(w) if gx2 is None else _unrows(gx2, w)
        else:
            gw = row_stats_backward(gx2, w2, mn if g_min is not None else None,
                                    cmn if g_min is not None else None, g_min,
                                    mx if g_mx is not None else None,
                                    cmx if g_mx is not None else None, g_mx)
            gw = _unrows(gw, w)
        return gw, (g_scale if ctx.needs_input_grad[1] else None), None, None, None


def weight_fake_quant(w, scale, method="STE", noise=None, philox=None):
    """(wq, row_min, row_max) for a per-channel weight (channel = dim 0); see _WeightFakeQuantFn."""
    _require_cuda(w)
    if scale.numel() != w.shape[0]:
        raise RuntimeError("weight_fake_quant expects one scale per output channel (dim 0)")
    return _WeightFakeQuantFn.apply(w, scale, _method_id(method), noise, philox)


class _ActFakeQuantFn(torch.autograd.Function):
    """NoisyAct.forward's arithmetic (gdnsq_act.py:42-55) as ONE autograd node: the kernels read
    log_act_s / log_act_q / act_b directly (MHAQ_FQ_PARAMS_ACT_LOG) and the finalize returns
    the log-domain gradients, so none of the ~25 tiny exp2/add/sub launches (forward and
    backward) autograd would otherwise run per quantizer exist."""

    @staticmethod
    def forward(ctx, x, log_act_s, log_act_q, act_b, method, noise, philox, funnel=False):
        ctx.set_materialize_grads(False)
        x = _dense(x, None)
        L = _Launch.act_log(x, log_act_s, log_act_q, act_b)
        y, _, _ = _forward_impl(x, L, True, False, False)
        ctx.save_for_backward(x, log_act_s, log_act_q, act_b)
        ctx.L, ctx.method, ctx.noise, ctx.philox = L, method, noise, philox
        if funnel:
            # aliases of the two log parameters as outputs of THIS node: whatever else reads them
            # (PotentialLoss) sends its gradient back here instead of to the leaves
            return y, log_act_s.view_as(log_act_s), log_act_q.view_as(log_act_q)
        return y

    @staticmethod
    def backward(ctx, go, g_las=None, g_laq=None):
        x, log_act_s, log_act_q, act_b = ctx.saved_tensors
        need = ctx.needs_input_grad
        if go is None:          # only the aliases were used: their gradients pass straight through
            return (None, g_las if need[1] else None, g_laq if need[2] else None, None, None, None, None, None)
        acc = None
        if g_las is not None or g_laq is not None:
            c = lambda t: None if t is None else t.contiguous()
            acc = (c(g_las), None, c(g_laq), None)       # kernel outputs: log_act_s, act_b, log_act_q
        gx, out = _backward_impl(go, x, ctx.L, ctx.method, False, ctx.noise, need[0], ctx.philox, acc=acc)
        return (gx if need[0] else None,
                out[0].reshape(log_act_s.shape) if need[1] else None,
                out[2].reshape(log_act_q.shape) if need[2] else None,
                out[1].reshape(act_b.shape) if need[3] else None, None, None, None, None)


def act_fake_quant(x, log_act_s, log_act_q, act_b, method="STE", noise=None, philox=None, funnel=False):
    """Fused NoisyAct: fake_quant(x, s=2^log_act_s, zp=lo=act_b, hi=act_b+2^log_act_q-s).
    funnel=True -> (y, alias of log_act_s, alias of log_act_q): see quantization/gdnsq/_funnel.py."""
    _require_cuda(x)
    return _ActFakeQuantFn.apply(x, log_act_s, log_act_q, act_b, _method_id(method), noise, philox, funnel)


class _WeightLogFakeQuantFn(torch.autograd.Function):
    """_WeightFakeQuantFn with the scale in the log domain (MHAQ_FQ_PARAMS_WEIGHT_LOG):
    (wq, row_min, row_max) from (weight, log_wght_s), d/d log_wght_s straight from the kernel."""

    @staticmethod
    def forward(ctx, w, log_wght_s, method, noise, philox):
        ctx.set_materialize_grads(False)
        w = _dense(w, 0)
        rows = w.shape[0]
        mn, mx, cmn, cmx = row_stats(_rows2d(w))
        L = _Launch.weight_log(w, log_wght_s, mn)
        wq, _, _ = _forward_impl(w, L, True, False, False)
        ctx.save_for_backward(w, log_wght_s, mn, mx, cmn, cmx)
        # (L references `mn`, an OUTPUT of this node: keeping it on ctx would tie the node to its
        # own output — a cycle through C++ that Python's GC cannot see, i.e. a leaked graph whose
        # AccumulateGrad nodes then outlive the step.  It is rebuilt in backward.)
        ctx.method, ctx.noise, ctx.philox = method, noise, philox
        return wq, mn, mx

    @staticmethod
    def backward(ctx, g_wq, g_mn, g_mx):
        w, log_wght_s, mn, mx, cmn, cmx = ctx.saved_tensors
        w2 = _rows2d(w)
        g_log_s = None
        if g_wq is not None:
            L = _Launch.weight_log(w, log_wght_s, mn)
            gx, out = _backward_impl(g_wq, w, L, ctx.method, False, ctx.noise, True, ctx.philox)
            g_log_s = out[0].reshape(log_wght_s.shape)
            g_min = out[1] if g_mn is None else out[1] + g_mn
            gx2 = _rows2d(gx)
        else:
            gx2, g_min = None, g_mn
        if not ctx.needs_input_grad[0]:
            return None, g_log_s, None, None, None
        if g_min is None and g_mx is None:
            gw = torch.zeros_like(w) if gx2 is None else _unrows(gx2, w)
        else:
            gw = row_stats_backward(gx2, w2, mn if g_min is not None else None,
                                    cmn if g_min is not None else None, g_min,
                                    mx if g_mx is not None else None,
                                    cmx if g_mx is not None else None, g_mx)
            gw = _unrows(gw, w)
        return gw, (g_log_s if ctx.needs_input_grad[1] else None), None, None, None


def weight_fake_quant_log(w, log_wght_s, method="STE", noise=None, philox=None):
    """(wq, row_min, row_max) for a per-channel weight from its LOG scale (channel = dim 0)."""
    _require_cuda(w)
    if log_wght_s.numel() != w.shape[0]:
        raise RuntimeError("weight_fake_quant_log expects one log-scale per output channel (dim 0)")
    return _WeightLogFakeQuantFn.apply(w, log_wght_s, _method_id(method), noise, philox)


# ---------------------------------------------------------------------------------------------
# Row-resident fused weight path (include/mhaq_fq.h: mhaq_fq_wrow_*): one launch forward, one
# backward per layer, ModelHelper's log2(max - min + 2^log_s) included.
# ---------------------------------------------------------------------------------------------
WROW_MAX_INNER = 16384       # one CTA per row: conv / linear weight rows, not long tensors


def weight_rows_fusable(w, log_wght_s, method, multi: bool = False) -> bool:
    """Row-resident kernels: one log-scale per row of dim 0, short rows.  A single-tensor launch
    cannot serve AEWGS (its statistics are all-reduced between two passes); the multi-tensor
    form can — statistics kernel, ONE all-reduce for the whole model, apply kernel."""
    rows = w.shape[0] if w.dim() >= 1 else 0
    return (rows > 0 and log_wght_s.numel() == rows and 0 < w.numel() // rows <= WROW_MAX_INNER
            and (multi or _method_id(method) != METHOD_IDS["AEWGS"]))


class _WeightRowFn(torch.autograd.Function):
    """(wq, row_min, row_max, log_range) = f(weight, log_wght_s), channel = dim 0:
        row_min/max = weight.amin/amax over the row           (gdnsq_conv2d.py:80-81)
        wq          = fake_quant(w; 2^log_wght_s, zp=row_min) (gdnsq_conv2d.py:72-98)
        log_range   = log2(row_max - row_min + 2^log_wght_s)  (utils/model_helper.py:24-25,44)
    with the reference's autograd for all of it, in one kernel each way."""

    @staticmethod
    def forward(ctx, w, log_wght_s, method, noise, philox):
        ctx.set_materialize_grads(False)
        w = _dense(w, 0)
        rows = w.shape[0]
        inner = w.numel() // rows
        ls = log_wght_s if log_wght_s.is_contiguous() else log_wght_s.contiguous()
        wq = torch.empty_like(w)
        o = torch.empty(3, rows, dtype=torch.float32, device=w.device)
        check(lib.mhaq_fq_wrow_fwd_f32(_ptr(w), _ptr(wq), _ptr(ls), rows, inner, _ptr(o[0]), _ptr(o[1]),
                                       _ptr(o[2]), _stream()), "mhaq_fq_wrow_fwd_f32")
        mn, mx, lr = o[0], o[1], o[2]
        ctx.save_for_backward(w, log_wght_s, mn, mx)
        ctx.method, ctx.noise, ctx.philox = method, noise, philox
        return wq, mn, mx, lr

    @staticmethod
    def backward(ctx, g_wq, g_mn, g_mx, g_lr):
        w, log_wght_s, mn, mx = ctx.saved_tensors
        rows = w.shape[0]
        inner = w.numel() // rows
        if g_wq is None:            # the quantized weight itself was not used downstream
            g_wq = torch.zeros_like(w)
        g_wq = _like_layout(g_wq, w)
        noise, seed, offset, pdev = _noise_source(w, ctx.method, ctx.noise, ctx.philox)
        c = lambda t: None if t is None else t.contiguous()
        g_mn, g_mx, g_lr = c(g_mn), c(g_mx), c(g_lr)
        ls = log_wght_s if log_wght_s.is_contiguous() else log_wght_s.contiguous()
        gw = torch.empty_like(w) if ctx.needs_input_grad[0] else None
        gls = torch.empty(rows, dtype=torch.float32, device=w.device)
        check(lib.mhaq_fq_wrow_bwd_f32(_ptr(g_wq), _ptr(w), _ptr(ls), _ptr(mn), _ptr(mx), _ptr(g_lr),
                                       _ptr(g_mn), _ptr(g_mx), rows, inner, ctx.method, _ptr(noise),
                                       seed, offset, _ptr(pdev), _ptr(gw), _ptr(gls), _stream()),
              "mhaq_fq_wrow_bwd_f32")
        return (gw, gls.reshape(log_wght_s.shape) if ctx.needs_input_grad[1] else None,
                None, None, None)


def weight_fake_quant_rows(w, log_wght_s, method="STE", noise=None, philox=None):
    """(wq, row_min, row_max, log_range) for a per-channel weight with short rows; see
    _WeightRowFn.  Check `weight_rows_fusable` first."""
    _require_cuda(w)
    if not weight_rows_fusable(w, log_wght_s, method):
        raise RuntimeError("weight_fake_quant_rows: needs one log-scale per row of dim 0, rows of at "
                           f"most {WROW_MAX_INNER} elements and a method other than AEWGS")
    return _WeightRowFn.apply(w, log_wght_s, _method_id(method), noise, philox)


# ---------------------------------------------------------------------------------------------
# Multi-tensor row-resident weight path (include/mhaq_fq.h: mhaq_fq_wrow_multi_*): every
# per-channel weight of a model in ONE launch forward and ONE backward (SURVEY.md §8 row (f)-4).
# ---------------------------------------------------------------------------------------------
def _philox_streams(x, method: int, n: int, philox):
    """(seed, base offset, device state) for `n` consecutive noise streams."""
    if method == METHOD_IDS["LSQ"]:
        return 0, 0, None
    if philox is not None:
        return philox[0], philox[1], None
    pd = _philox_dev.get(x.device.index)
    if pd is not None:
        off = _philox_call[x.device.index]
        _philox_call[x.device.index] = off + n
        return 0, off, pd
    idx = x.device.index if x.device.index is not None else torch.cuda.current_device()
    gen = torch.cuda.default_generators[idx]
    seed, off = gen.initial_seed(), gen.get_offset()
    gen.set_offset(off + 4 * n)
    return seed & 0xFFFFFFFFFFFFFFFF, off // 4, None


class _WeightRowMultiFn(torch.autograd.Function):
    """_WeightRowFn for n tensors at once: inputs (w_0..w_{n-1}, log_s_0..log_s_{n-1}), outputs
    (wq_i, row_min_i, row_max_i, log_range_i) for every i — 4n outputs of one autograd node whose
    backward is one launch too (it runs once the last consumer of any output has run)."""

    @staticmethod
    def forward(ctx, method, noises, philox, n, funnel, *tensors):
        from ._lib import WRowFwdDesc
        ctx.set_materialize_grads(False)
        ws = [_dense(w, 0) for w in tensors[:n]]
        lss = [ls if ls.is_contiguous() else ls.contiguous() for ls in tensors[n:]]
        rows = [w.shape[0] for w in ws]
        dev = ws[0].device
        stats = torch.empty(3, sum(rows), dtype=torch.float32, device=dev)
        descs = (WRowFwdDesc * n)()
        outs, r0 = [], 0
        for i, (w, ls) in enumerate(zip(ws, lss)):
            wq = torch.empty_like(w)
            r1 = r0 + rows[i]
            mn, mx, lr = stats[0, r0:r1], stats[1, r0:r1], stats[2, r0:r1]
            d = descs[i]
            d.w, d.log_scale, d.wq = w.data_ptr(), ls.data_ptr(), wq.data_ptr()
            d.row_min, d.row_max, d.log_range = mn.data_ptr(), mx.data_ptr(), lr.data_ptr()
            d.n_rows, d.n_inner = rows[i], w.numel() // rows[i]
            outs += [wq, mn, mx, lr]
            r0 = r1
        check(lib.mhaq_fq_wrow_multi_fwd_f32(descs, n, _stream()), "mhaq_fq_wrow_multi_fwd_f32")
        ctx.save_for_backward(*ws, *lss, stats)
        ctx.n, ctx.rows, ctx.method, ctx.noises, ctx.philox = n, rows, method, noises, philox
        if funnel:      # + one alias of every log-scale (quantization/gdnsq/_funnel.py)
            outs += [ls.view_as(ls) for ls in tensors[n:]]
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grads):
        from ._lib import WRowBwdDesc
        n, rows = ctx.n, ctx.rows
        saved = ctx.saved_tensors
        ws, lss, stats = saved[:n], saved[n:2 * n], saved[2 * n]
        need = ctx.needs_input_grad
        descs = (WRowBwdDesc * n)()
        keep, gws, glss = [], [], []
        r0 = 0
        c = lambda t: None if t is None else t.contiguous()
        for i in range(n):
            w, ls = ws[i], lss[i]
            g_wq, g_mn, g_mx, g_lr = grads[4 * i: 4 * i + 4]
            g_wq = torch.zeros_like(w) if g_wq is None else _like_layout(g_wq, w)
            g_mn, g_mx, g_lr = c(g_mn), c(g_mx), c(g_lr)
            g_acc = c(grads[4 * n + i]) if len(grads) > 4 * n else None     # through the log-scale alias
            noise = None if ctx.noises is None else ctx.noises[i]
            if noise is not None:
                noise = _like_layout(noise, w)
            gw = torch.empty_like(w) if need[5 + i] else None
            gls = torch.empty(rows[i], dtype=torch.float32, device=w.device) if need[5 + n + i] else None
            r1 = r0 + rows[i]
            d = descs[i]
            d.g_wq, d.w, d.log_scale = g_wq.data_ptr(), w.data_ptr(), ls.data_ptr()
            d.row_min, d.row_max = stats[0, r0:r1].data_ptr(), stats[1, r0:r1].data_ptr()
            d.g_log_range, d.g_row_min, d.g_row_max, d.r = _ptr(g_lr), _ptr(g_mn), _ptr(g_mx), _ptr(noise)
            d.g_w, d.g_log_scale = _ptr(gw), _ptr(gls)
            d.n_rows, d.n_inner = rows[i], w.numel() // rows[i]
            d.g_log_scale_acc = _ptr(g_acc) if gls is not None else None
            keep += [g_wq, g_mn, g_mx, g_lr, noise, g_acc]
            gws.append(gw)
            glss.append(None if gls is None else gls.reshape(ls.shape))
            r0 = r1
        seed, offset, pdev = (0, 0, None) if ctx.noises is not None else _philox_streams(ws[0], ctx.method, n, ctx.philox)
        ae_stats, total_rows = None, 0
        if ctx.method == METHOD_IDS["AEWGS"]:
            # the path's one exchange step, ONCE for the whole model: per-row statistics of every
            # tensor -> one packed [3, total_rows] AVG all-reduce -> apply (gdnsq.py:118-134; the
            # reference issues three all-reduces per weight tensor)
            total_rows = sum(rows)
            ae_stats = torch.empty(3 * total_rows, dtype=torch.float32, device=ws[0].device)
            check(lib.mhaq_fq_wrow_multi_aewgs_stats_f32(descs, n, _ptr(ae_stats), total_rows, _stream()),
                  "mhaq_fq_wrow_multi_aewgs_stats_f32")
            ae_stats = allreduce_packed_stats(ae_stats)
        check(lib.mhaq_fq_wrow_multi_bwd_f32(descs, n, ctx.method, seed, offset, _ptr(pdev), _ptr(ae_stats),
                                             total_rows, _stream()),
              "mhaq_fq_wrow_multi_bwd_f32")
        return (None, None, None, None, None, *gws, *glss)


def weight_fake_quant_rows_multi(weights, log_scales, method="STE", noises=None, philox=None, funnel=False):
    """[(wq, row_min, row_max, log_range), ...] for a list of per-channel weights with short rows
    (each must satisfy `weight_rows_fusable`), one launch each way for the whole list.
    funnel=True appends an alias of the tensor's log-scale to every tuple (quantization/gdnsq/_funnel.py)."""
    n = len(weights)
    if n == 0:
        return []
    mid = _method_id(method)
    for w, ls in zip(weights, log_scales):
        _require_cuda(w)
        if not weight_rows_fusable(w, ls, mid, multi=True):
            raise RuntimeError("weight_fake_quant_rows_multi: every tensor needs one log-scale per row of dim 0 "
                               f"and rows of at most {WROW_MAX_INNER} elements")
    if mid == METHOD_IDS["LSQ"]:
        noises = None
    out = _WeightRowMultiFn.apply(mid, noises, philox, n, bool(funnel), *weights, *log_scales)
    if funnel:
        return [tuple(out[4 * i: 4 * i + 4]) + (out[4 * n + i],) for i in range(n)]
    return [tuple(out[4 * i: 4 * i + 4]) for i in range(n)]


# ---------------------------------------------------------------------------------------------
# PotentialLoss's constraint arithmetic (include/mhaq_fq.h: mhaq_fq_potential_loss_*): one
# launch forward, one backward, instead of ~30 tiny elementwise / reduction launches per step.
# ---------------------------------------------------------------------------------------------
PLOSS_NOUT = 14


class _PotentialLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, base_loss, las, laq, lws, lwq, loss_sum, cnt, wt, at, eps, t, lossless, training):
        c = lambda v: v if v.is_contiguous() else v.contiguous()
        las, laq, lws, lwq = c(las), c(laq), c(lws), c(lwq)
        out = torch.empty(PLOSS_NOUT, dtype=torch.float32, device=lws.device)
        check(lib.mhaq_fq_potential_loss_fwd_f32(_ptr(las), _ptr(laq), las.numel(), _ptr(lws), _ptr(lwq),
                                                 lws.numel(), _ptr(base_loss), _ptr(loss_sum), _ptr(cnt),
                                                 float(wt), float(at), float(eps), float(t), int(lossless),
                                                 int(training), _ptr(out), _stream()),
              "mhaq_fq_potential_loss_fwd_f32")
        ctx.save_for_backward(las, laq, lws, lwq, out)
        ctx.cfg = (float(wt), float(at), float(eps))
        ctx.mark_non_differentiable(out)
        return out[0], out

    @staticmethod
    def backward(ctx, g, _g_out):
        las, laq, lws, lwq, out = ctx.saved_tensors
        need = ctx.needs_input_grad
        g = g.contiguous()
        mk = lambda t, n: torch.empty_like(t) if n else None
        g_base = torch.empty((), dtype=torch.float32, device=lws.device) if need[0] else None
        g_las, g_laq, g_lws, g_lwq = mk(las, need[1]), mk(laq, need[2]), mk(lws, need[3]), mk(lwq, need[4])
        wt, at, eps = ctx.cfg
        check(lib.mhaq_fq_potential_loss_bwd_f32(_ptr(las), _ptr(laq), las.numel(), _ptr(lws), _ptr(lwq),
                                                 lws.numel(), _ptr(out), _ptr(g), wt, at, eps, _ptr(g_las),
                                                 _ptr(g_laq), _ptr(g_lws), _ptr(g_lwq), _ptr(g_base), _stream()),
              "mhaq_fq_potential_loss_bwd_f32")
        return (g_base, g_las, g_laq, g_lws, g_lwq) + (None,) * 8


def potential_loss(base_loss, las, laq, lws, lwq, loss_sum, cnt, wt, at, eps, t, lossless, training):
    """(ploss, record) — see include/mhaq_fq.h; `loss_sum` / `cnt` are 1-element fp32 CUDA tensors
    updated in place when `training`.  `record` holds the logged terms (non-differentiable)."""
    for v in (base_loss, las, laq, lws, lwq, loss_sum, cnt):
        _require_cuda(v)
    return _PotentialLossFn.apply(base_loss.reshape(()), las, laq, lws, lwq, loss_sum, cnt, wt, at, eps, t,
                                  lossless, training)


# ---------------------------------------------------------------------------------------------
# Packed integer codes (include/mhaq_fq.h: "Packed codes", mhaq_fq_pack_f32 / mhaq_fq_unpack_f32):
# the codes the forward computes, stored at 1, 2, 4, 8 or 16 bits with the scale and zero point
# that turn them back into the fake-quantized tensor.
# ---------------------------------------------------------------------------------------------
PACK_BITS = (1, 2, 4, 8, 16)


@dataclass
class PackedCodes:
    """Codes of one tensor in the packed format of include/mhaq_fq.h.

    ``data`` is uint8 ``[n_rows, row_stride]`` over the ``[n_rows][n_inner]`` storage-order view
    (row r quantized with channel r % n_ch); ``shape`` / ``stride`` are those of the packed tensor,
    so ``unpack_codes`` returns the same layout.  ``scale`` / ``zero_point`` are the flattened
    operands the codes were made with, interpreted by parameter mode ``mode`` (log-domain for the
    layer forms).  ``n_out_of_range`` is a device counter of the codes that had to be saturated."""
    data: torch.Tensor
    bits: int
    shape: Tuple[int, ...]
    stride: Tuple[int, ...]
    n_rows: int
    n_inner: int
    n_ch: int
    scale: torch.Tensor
    zero_point: torch.Tensor
    n_out_of_range: torch.Tensor
    mode: int = PARAMS_LINEAR


def packed_row_bytes(n_inner: int, bits: int) -> int:
    """Bytes per packed row: round_up(ceil(n_inner * bits / 8), 16)."""
    n = int(lib.mhaq_fq_packed_row_bytes(n_inner, bits))
    if n < 0:
        raise ValueError(f"packed codes: bits must be one of {PACK_BITS}, got {bits}")
    return n


def _smallest_bits(x, L: _Launch) -> int:
    """Width for the codes' range, from the statistics-only forward (one host read)."""
    _, _, mm = _forward_impl(x, L, want_y=False, want_codes=False, want_minmax=True)
    cmin, cmax, bad = mm[:3].tolist()
    if bad != 0 or cmin < 0:
        raise ValueError(f"packed codes: codes span [{cmin}, {cmax}]; no unsigned width holds them")
    for b in PACK_BITS:
        if cmax <= (1 << b) - 1:
            return b
    raise ValueError(f"packed codes: the largest code {cmax:.0f} needs more than 16 bits")


def _pack(x, L: _Launch, bits, check_range: bool) -> PackedCodes:
    geo = L.geo
    if bits is None:
        bits = _smallest_bits(x, L) if x.numel() else PACK_BITS[0]
    row = packed_row_bytes(geo.n_inner, bits)
    data = torch.empty(geo.n_rows, row, dtype=torch.uint8, device=x.device)
    n_bad = torch.zeros(1, dtype=torch.int64, device=x.device)      # unsigned long long counter
    if x.numel():
        check(lib.mhaq_fq_pack_f32(_ptr(x), _ptr(data), bits, *L.params(), geo.n_rows, geo.n_inner,
                                   geo.n_ch, _ptr(n_bad), _stream()), "mhaq_fq_pack_f32")
    p = PackedCodes(data, bits, tuple(x.shape), tuple(x.stride()), geo.n_rows, geo.n_inner, geo.n_ch,
                    L.scale, L.zp, n_bad, L.mode)
    if check_range:
        n = int(n_bad.item())
        if n:
            raise ValueError(f"packed codes: {n} code(s) outside [0, {(1 << bits) - 1}] (NaN included)")
    return p


def pack_codes(x, scale, zero_point, min_val=None, max_val=None, bits=None, check=True) -> PackedCodes:
    """The codes ``quantize_codes`` returns, packed at ``bits`` (1, 2, 4, 8 or 16) per code.

    Parameters are interpreted exactly as ``fake_quant`` interprets them.  ``bits=None`` picks the
    smallest width that holds [min code, max code] (one statistics pass and one host read; raises
    if no width fits).  ``check=True`` reads the out-of-range counter once and raises ValueError if
    any code had to be saturated; ``check=False`` synchronises nothing (CUDA-graph capture, which
    also needs an explicit ``bits``)."""
    x = x.detach()
    L = _Launch(x, scale, zero_point, min_val, max_val)
    return _pack(_dense(x, L.geo.axis), L, bits, check)


def pack_act_codes(x, log_act_s, log_act_q, act_b, bits=None, check=True) -> PackedCodes:
    """``pack_codes`` with NoisyAct's parameters (s = 2^log_act_s, zero point = min_val = act_b,
    max_val = (act_b + 2^log_act_q) - s, formed in the kernel as the layer's forward forms them)."""
    x = x.detach()
    L = _Launch.act_log(x, log_act_s, log_act_q, act_b)
    return _pack(_dense(x, None), L, bits, check)


def pack_weight_codes(w, log_wght_s, row_min, bits=None, check=True) -> PackedCodes:
    """``pack_codes`` for a per-channel (dim 0) weight from its log scale and row minimum, as the
    layers' fused weight path forms them (s = 2^log_wght_s[row], zero point = row_min[row])."""
    w = _dense(w.detach(), 0)
    L = _Launch.weight_log(w, log_wght_s, row_min)
    return _pack(w, L, bits, check)


def unpack_codes(p: PackedCodes) -> torch.Tensor:
    """code * s + zero_point for every element of ``p``, fp32 with ``p``'s shape and strides: for
    every code that was in range, bit for bit the output of the forward the codes came from."""
    y = torch.empty_strided(p.shape, p.stride, dtype=torch.float32, device=p.data.device)
    if y.numel():
        ss = 0 if p.scale.numel() == 1 else 1
        zs = 0 if p.zero_point.numel() == 1 else 1
        check(lib.mhaq_fq_unpack_f32(_ptr(p.data), p.bits, _ptr(y), _ptr(p.scale), _ptr(p.zero_point), ss, zs,
                                     p.mode, p.n_rows, p.n_inner, p.n_ch, _stream()), "mhaq_fq_unpack_f32")
    return y


# ---------------------------------------------------------------------------------------------
# Integer layers (include/mhaq_fq.h "Integer layers", DESIGN §3): a quantized convolution or
# linear layer evaluated on the activation and weight codes with the int8 tensor cores,
#   y[m][n] = alpha[n] * S[m][n] + beta[n] * SA[m] + ctab[p(m)][n].
# ---------------------------------------------------------------------------------------------
def code_channels(c: int) -> int:
    """Channels of an activation-code row: C rounded up to 16 (the MMA K granularity is 32 bytes
    per instruction and every 16-byte chunk of K must lie within one tap)."""
    return (c + 15) // 16 * 16


def act_codes(x, scale, zero_point, max_val, check=False):
    """uint8 codes of an eval-mode ``NoisyAct`` with operands (scale, zero_point = min_val,
    max_val), each one element: the forward's own codes, saturated to [0, 255] (NaN -> 0).

    ``x`` is a 4-D tensor (taken channels_last; other layouts are copied) or a ``[B, in]``
    matrix.  Returns ``(codes, n_out_of_range)``: codes ``[B, H, W, Cp]`` resp. ``[B, Cp]``,
    Cp = ``code_channels(C)``, padding channels 0, and a device counter of saturated codes.
    ``check=True`` reads the counter (one host synchronisation) and raises ValueError if it is
    not zero."""
    x = x.detach()
    _require_cuda(x)
    if x.dim() == 4:
        x = x.contiguous(memory_format=torch.channels_last)
        b, c, h, w = x.shape
        lead = (b, h, w)
    elif x.dim() == 2:
        x = x.contiguous()
        (b, c), lead = x.shape, (x.shape[0],)
    else:
        raise ValueError(f"act_codes: expected a 4-D or 2-D input, got shape {tuple(x.shape)}")
    cp = code_channels(c)
    codes = torch.empty(*lead, cp, dtype=torch.uint8, device=x.device)
    n_bad = torch.zeros(1, dtype=torch.int64, device=x.device)      # unsigned long long counter
    prm = [_prep_param(p, x, n)[0] for p, n in ((scale, "scale"), (zero_point, "zp"), (max_val, "hi_param"))]
    if any(p.numel() != 1 for p in prm):
        raise ValueError("act_codes: scale, zero_point and max_val must have one element each")
    n_pix = x.numel() // c if c else 0
    _check_rc(lib.mhaq_fq_act_codes_f32(_ptr(x), _ptr(codes), *(_ptr(p) for p in prm), n_pix, c, cp,
                                        _ptr(n_bad), _stream()), "mhaq_fq_act_codes_f32")
    if check:
        n = int(n_bad.item())
        if n:
            raise ValueError(f"act_codes: {n} code(s) outside [0, 255] (NaN included)")
    return codes, n_bad


def iconv_layout(n_out: int, k_bytes: int):
    """(bytes, n_tiles, tile_n, tile_out, k_stages) of the weight operand (mhaq_fq_iconv_weight_bytes)."""
    nt, tn, to, ks = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int64()
    n = int(lib.mhaq_fq_iconv_weight_bytes(n_out, k_bytes, ctypes.byref(nt), ctypes.byref(tn),
                                           ctypes.byref(to), ctypes.byref(ks)))
    if n < 0:
        raise ValueError(f"iconv_layout: bad sizes n_out={n_out}, k_bytes={k_bytes}")
    return n, nt.value, tn.value, to.value, ks.value


def iconv_weight_operand(cw: torch.Tensor) -> torch.Tensor:
    """The weight operand of mhaq_fq_iconv_u8 from integer weight codes ``cw [N, C, kh, kw]``:
    flat uint8, rows (kh, kw, Cp) with zero padding channels, an all-ones row after each tile's
    output channels, every (tile, stage) block in the kernel's shared-memory order."""
    n, c, kh, kw = cw.shape
    cp = code_channels(c)
    k = kh * kw * cp
    nbytes, nt, tn, to, ks = iconv_layout(n, k)
    w = torch.zeros(n, kh, kw, cp, dtype=torch.uint8, device=cw.device)
    w[..., :c] = cw.permute(0, 2, 3, 1).to(torch.uint8)
    w = w.reshape(n, k)
    rows = torch.zeros(nt, tn, ks * 128, dtype=torch.uint8, device=cw.device)
    for t in range(nt):
        lo, hi = t * to, min(n, (t + 1) * to)
        rows[t, :hi - lo, :k] = w[lo:hi]
        rows[t, to, :] = 1
    # [tile][row group][row % 8][stage][chunk][byte] -> [tile][stage][row group][chunk][row % 8][byte]
    out = rows.view(nt, tn // 8, 8, ks, 8, 16).permute(0, 3, 1, 4, 2, 5).reshape(-1)
    assert out.numel() == nbytes
    return out


def iconv_grouped_layout(n_in: int, n_out: int, kh: int, kw: int, groups: int):
    """(bytes, n_tiles, tile_n, tile_out, groups_per_tile, tiles_per_group, k_stages) of the weight
    operand of a grouped layer (mhaq_fq_iconv_grouped_weight_bytes); n_tiles = 0 for a depthwise one."""
    g = _lib.IConvGeometry(kh, kw, 1, 1, 0, 0, 1, 1, groups)
    ints = [ctypes.c_int() for _ in range(5)]
    ks = ctypes.c_int64()
    n = int(lib.mhaq_fq_iconv_grouped_weight_bytes(n_in, n_out, ctypes.byref(g), *(ctypes.byref(v) for v in ints),
                                                   ctypes.byref(ks)))
    if n < 0:
        raise ValueError(f"iconv_grouped_layout: bad geometry n_in={n_in}, n_out={n_out}, groups={groups}")
    return (n, *(v.value for v in ints), ks.value)


def grouped_tile(t: int, groups: int, cin_g: int, cout_g: int, tile_out: int, gpt: int, parts: int):
    """(n_base, n_here, first group, groups, first 16-channel chunk, chunks) of N tile ``t`` of a
    grouped weight operand (the kernel's igroup_tile)."""
    if parts == 1:
        g_lo = t * gpt
        g_hi = min(groups, g_lo + gpt)
        n_base, n_end = g_lo * cout_g, g_hi * cout_g
    else:
        g_lo = t // parts
        g_hi = g_lo + 1
        n_base = g_lo * cout_g + (t % parts) * tile_out
        n_end = min(n_base + tile_out, g_hi * cout_g)
    c_lo = g_lo * cin_g // 16
    return n_base, n_end - n_base, g_lo, g_hi - g_lo, c_lo, (g_hi * cin_g + 15) // 16 - c_lo


def iconv_grouped_weight_operand(cw: torch.Tensor, groups: int) -> torch.Tensor:
    """The weight operand of mhaq_fq_iconv_grouped_u8 from grouped weight codes
    ``cw [N, C / groups, kh, kw]``: for a depthwise layer (groups == C == N) u8 ``[kh * kw][Cp]``,
    otherwise block-diagonal N tiles (include/mhaq_fq.h), flat uint8."""
    n, cin_g, kh, kw = cw.shape
    cin, taps = cin_g * groups, kh * kw
    cp = code_channels(cin)
    nbytes, nt, tn, to, gpt, parts, ks = iconv_grouped_layout(cin, n, kh, kw, groups)
    if nt == 0:
        w = torch.zeros(taps, cp, dtype=torch.uint8, device=cw.device)
        w[:, :cin] = cw[:, 0].reshape(n, taps).t().to(torch.uint8)
        return w.reshape(-1)
    cout_g = n // groups
    cwt = cw.permute(0, 2, 3, 1).reshape(n, taps, cin_g).to(torch.uint8)
    rows = torch.zeros(nt, tn, ks * 128, dtype=torch.uint8, device=cw.device)
    for t in range(nt):
        n_base, n_here, g_lo, n_grp, c_lo, kc = grouped_tile(t, groups, cin_g, cout_g, to, gpt, parts)
        blk = torch.zeros(tn, taps, kc * 16, dtype=torch.uint8, device=cw.device)
        for i in range(n_grp):
            g = g_lo + i
            lo = g * cin_g - c_lo * 16                       # the group's first K column of a tap
            n0, n1 = max(n_base, g * cout_g), min(n_base + n_here, (g + 1) * cout_g)
            blk[n0 - n_base:n1 - n_base, :, lo:lo + cin_g] = cwt[n0:n1]
            blk[to + i, :, lo:lo + cin_g] = 1
        rows[t, :, :taps * kc * 16] = blk.reshape(tn, -1)
    out = rows.view(nt, tn // 8, 8, ks, 8, 16).permute(0, 3, 1, 4, 2, 5).reshape(-1)
    assert out.numel() == nbytes
    return out


def tap_classes(size: int, k: int, stride: int, pad: int, dilation: int = 1):
    """Tap-validity classes along one axis: (class of each output position (int32 [out]),
    valid taps of each class (bool [n_classes, k])).  Tap t of output o reads position
    o * stride - pad + t * dilation."""
    out = (size + 2 * pad - dilation * (k - 1) - 1) // stride + 1
    pos = torch.arange(out)[:, None] * stride - pad + torch.arange(k)[None, :] * dilation
    valid = ((pos >= 0) & (pos < size)).to(torch.uint8)
    uniq, inv = torch.unique(valid, dim=0, return_inverse=True)
    return inv.to(torch.int32), uniq.bool()


@dataclass
class IntLayerOperands:
    """Device operands of one integer layer (``int_layer_operands``).  ``weight``, ``alpha`` and
    ``beta`` are fixed; the pattern tables depend on the input size and are built on first use
    of each (H, W, stride, padding) and cached."""
    weight: torch.Tensor          # uint8 operand (iconv_weight_operand)
    alpha: torch.Tensor           # fp32 [N]: sa * sw
    beta: torch.Tensor            # fp32 [N]: sa * zpw
    n_out: int
    cin: int
    kh: int
    kw: int
    a_top: int                    # largest activation code
    w_top: int                    # largest weight code
    tap_sums: torch.Tensor        # fp64 [N, kh, kw]: sum over the channels of cw
    sw: torch.Tensor              # fp64 [N]
    zpw: torch.Tensor             # fp64 [N]
    zpa: float
    bias: Optional[torch.Tensor]  # fp64 [N] or None
    tables: dict
    sa: float                     # activation scale
    groups: int = 1               # weight: [N, cin / groups, kh, kw]
    dilation: Tuple[int, int] = (1, 1)

    @property
    def cp(self) -> int:
        return code_channels(self.cin)

    @property
    def dense(self) -> bool:
        """An ungrouped, undilated layer: mhaq_fq_iconv_u8 and its weight operand."""
        return self.groups == 1 and tuple(self.dilation) == (1, 1)

    def out_size(self, h: int, w: int, stride, padding) -> Tuple[int, int]:
        return ((h + 2 * padding[0] - self.dilation[0] * (self.kh - 1) - 1) // stride[0] + 1,
                (w + 2 * padding[1] - self.dilation[1] * (self.kw - 1) - 1) // stride[1] + 1)

    def fold_affine(self, k, shift) -> "IntLayerOperands":
        """Operands of ``k * y + shift`` (``k``, ``shift``: ``[N]``, taken in fp64), e.g. an eval
        BatchNorm after the layer: sw, zpw and bias become ``k * sw``, ``k * zpw`` and
        ``k * bias + shift`` in fp64, so alpha = RN32(sa * k * sw), beta = RN32(sa * k * zpw) and
        every constant-table entry RN32(k * C64 + shift) are formed from the fp64 terms and rounded
        once (DESIGN §3, "Fused epilogue").  Shares the weight operand; the pattern tables are
        rebuilt on first use."""
        f64 = dict(dtype=torch.float64, device=self.sw.device)
        k = torch.as_tensor(k).to(**f64).reshape(-1).expand(self.n_out)
        shift = torch.as_tensor(shift).to(**f64).reshape(-1).expand(self.n_out)
        sw, zpw = k * self.sw, k * self.zpw
        bias = shift.clone() if self.bias is None else k * self.bias + shift
        return dataclasses.replace(self, alpha=(self.sa * sw).float(), beta=(self.sa * zpw).float(), sw=sw,
                                   zpw=zpw, bias=bias, tables={})

    def constant_table(self, hvalid: torch.Tensor, wvalid: torch.Tensor) -> torch.Tensor:
        """fp64 ctab [n_h_classes * n_w_classes][N]: zpa * (sw * sum_{k in p} cw + zpw * |p|) + bias,
        |p| = valid taps x input channels per group."""
        mask = (hvalid[:, None, :, None] & wvalid[None, :, None, :]).to(torch.float64)
        mask = mask.to(self.tap_sums.device)
        wsum = torch.einsum("hwab,nab->hwn", mask, self.tap_sums)
        cnt = mask.sum((2, 3))[..., None] * (self.cin // self.groups)
        c = self.zpa * (self.sw * wsum + self.zpw * cnt)
        if self.bias is not None:
            c = c + self.bias
        return c.reshape(-1, self.n_out)

    def pattern_tables(self, h: int, w: int, stride, padding):
        """(h_class int32 [Ho], w_class int32 [Wo], n_w_classes, ctab fp32) on the operands' device."""
        key = (h, w, tuple(stride), tuple(padding))
        t = self.tables.get(key)
        if t is None:
            hc, hv = tap_classes(h, self.kh, stride[0], padding[0], self.dilation[0])
            wc, wv = tap_classes(w, self.kw, stride[1], padding[1], self.dilation[1])
            dev = self.weight.device
            t = self.tables[key] = (hc.to(dev), wc.to(dev), wv.shape[0],
                                    self.constant_table(hv, wv).to(device=dev, dtype=torch.float32).contiguous())
        return t


def int32_bound_ok(k_bytes: int, a_top: int, w_top: int) -> bool:
    """The int32 accumulator holds every sum: K * a_top * w_top < 2^31 (K counts padding channels)."""
    return k_bytes * a_top * w_top < (1 << 31)


def int_layer_operands(cw, sw, zpw, sa, zpa, bias, a_top: int, w_top: int, groups: int = 1,
                       dilation=1) -> IntLayerOperands:
    """Operands of an integer layer on ``cw``'s device from the weight codes ``cw [N, C / groups, kh,
    kw]`` (integers in [0, w_top]), the weight scale / zero point (``[N]`` or one element), the
    activation scale / zero point (floats) and the layer's bias (``[N]`` or None).  alpha and beta
    are formed in fp64 and rounded once to fp32.  A grouped or dilated layer gets the weight operand
    of mhaq_fq_iconv_grouped_u8 (``iconv_grouped_weight_operand``)."""
    n, c_g, kh, kw = cw.shape
    dilation = _pair(dilation)
    c = c_g * groups
    if groups < 1 or n % groups or min(dilation) < 1:
        raise ValueError(f"integer layer: groups={groups} must divide the {n} output channels and the "
                         f"dilation {dilation} be at least 1")
    if not (1 <= a_top <= 255 and 1 <= w_top <= 255):
        raise ValueError(f"integer layer: code bounds must lie in [1, 255], got {a_top} and {w_top}")
    dense = groups == 1 and dilation == (1, 1)
    # a grouped / dilated channel sums kh * kw * C / groups products (no padding channels)
    if not int32_bound_ok(kh * kw * (code_channels(c) if dense else c_g), a_top, w_top):
        raise ValueError("integer layer: K * (n_levels - 1) * (2^bits - 1) >= 2^31 would overflow the "
                         "int32 accumulator")
    dev = cw.device
    f64 = dict(dtype=torch.float64, device=dev)
    sw = torch.as_tensor(sw).to(**f64).reshape(-1).expand(n).contiguous()
    zpw = torch.as_tensor(zpw).to(**f64).reshape(-1).expand(n).contiguous()
    sa, zpa = float(sa), float(zpa)
    return IntLayerOperands(
        weight=iconv_weight_operand(cw) if dense else iconv_grouped_weight_operand(cw, groups),
        alpha=(sa * sw).float(), beta=(sa * zpw).float(),
        n_out=n, cin=c, kh=kh, kw=kw, a_top=a_top, w_top=w_top,
        tap_sums=cw.to(**f64).sum(1), sw=sw, zpw=zpw, zpa=zpa,
        bias=None if bias is None else torch.as_tensor(bias).to(**f64).reshape(n),
        tables={}, sa=sa, groups=groups, dilation=dilation)


def batchnorm_foldable(bn) -> bool:
    """An eval-mode ``BatchNorm2d`` that normalizes with its running statistics."""
    return (isinstance(bn, torch.nn.BatchNorm2d) and not bn.training and bn.track_running_stats
            and bn.running_mean is not None and bn.running_var is not None)


def fold_batchnorm(L: IntLayerOperands, bn) -> IntLayerOperands:
    """``L`` followed by the eval BatchNorm ``bn``: ``IntLayerOperands.fold_affine`` with
    k = gamma / sqrt(running_var + eps) and shift = beta - k * running_mean, all in fp64
    (``affine=False``: gamma = 1, beta = 0).  A BatchNorm without running statistics (or in
    training mode) normalizes with the batch's statistics and cannot be folded: ValueError."""
    if not batchnorm_foldable(bn):
        raise ValueError("fold_batchnorm: only an eval-mode BatchNorm2d with running statistics can be folded")
    if bn.num_features != L.n_out:
        raise ValueError(f"fold_batchnorm: {bn.num_features} BatchNorm features for {L.n_out} output channels")
    f64 = dict(dtype=torch.float64, device=L.sw.device)
    var, mean = bn.running_var.detach().to(**f64), bn.running_mean.detach().to(**f64)
    gamma = bn.weight.detach().to(**f64) if bn.affine else torch.ones_like(var)
    b = bn.bias.detach().to(**f64) if bn.affine else torch.zeros_like(var)
    k = gamma / torch.sqrt(var + float(bn.eps))
    return L.fold_affine(k, b - k * mean)


def _iconv(codes, L: IntLayerOperands, y, b, h, w, stride, padding):
    hc, wc, nwc, ctab = L.pattern_tables(h, w, stride, padding)
    if codes.shape[-1] != L.cp or codes.dtype != torch.uint8 or not codes.is_contiguous():
        raise ValueError(f"integer layer: expected contiguous uint8 codes with {L.cp} channels, "
                         f"got {codes.dtype} {tuple(codes.shape)}")
    if y.numel():
        _check_rc(lib.mhaq_fq_iconv_u8(_ptr(codes), _ptr(L.weight), _ptr(L.alpha), _ptr(L.beta), _ptr(ctab),
                                       _ptr(hc), _ptr(wc), nwc, _ptr(y), b, h, w, L.cp, L.n_out, L.kh, L.kw,
                                       stride[0], stride[1], padding[0], padding[1], L.a_top, L.w_top,
                                       _stream()), "mhaq_fq_iconv_u8")
    return y


def _pair(v):
    return (int(v), int(v)) if isinstance(v, int) else (int(v[0]), int(v[1]))


def _check_geometry(L: IntLayerOperands, dilation, groups):
    if dilation is not None and _pair(dilation) != tuple(L.dilation):
        raise ValueError(f"integer layer: dilation {_pair(dilation)} differs from the operands' {tuple(L.dilation)}")
    if groups is not None and int(groups) != L.groups:
        raise ValueError(f"integer layer: groups={groups} differs from the operands' {L.groups}")


def int_conv2d(codes, L: IntLayerOperands, stride=1, padding=0, dilation=None, groups=None) -> torch.Tensor:
    """fp32 convolution of activation codes ``[B, H, W, Cp]`` (``act_codes``) with the layer's
    operands: a channels_last ``[B, N, Ho, Wo]`` tensor.  ``dilation`` and ``groups`` are those of
    ``L`` (None: as given there; another value raises).  A grouped or dilated layer runs
    mhaq_fq_iconv_grouped_u8 (depthwise on the CUDA cores, the rest on the tensor cores)."""
    _check_geometry(L, dilation, groups)
    if not L.dense:
        return int_conv2d_fused(codes, L, stride, padding)[0]
    b, h, w, _ = codes.shape
    stride, padding = _pair(stride), _pair(padding)
    ho = (h + 2 * padding[0] - L.kh) // stride[0] + 1
    wo = (w + 2 * padding[1] - L.kw) // stride[1] + 1
    y = torch.empty((b, L.n_out, ho, wo), dtype=torch.float32, device=codes.device,
                    memory_format=torch.channels_last)
    return _iconv(codes, L, y, b, h, w, stride, padding)


ACTIVATIONS = {None: _lib.ACT_NONE, "relu": _lib.ACT_RELU, "leaky_relu": _lib.ACT_LEAKY_RELU}


def int_conv2d_fused(codes, L: IntLayerOperands, stride=1, padding=0, dilation=None, groups=None, *,
                     residual=None, activation=None, negative_slope=None, out_fp32=True, code_params=None):
    """``int_conv2d`` with its epilogue extended (mhaq_fq_iconv_fused_u8): t = the convolution
    (with whatever ``fold_batchnorm`` folded into ``L``), then ``t + residual`` (fp32, the output's
    shape; made channels_last-contiguous, which copies an NCHW tensor), then ``activation``
    (None, "relu" or "leaky_relu" with ``negative_slope``, default 0.01), one launch.  Returns
    ``(y, codes)``: y the channels_last fp32 ``[B, N, Ho, Wo]`` if ``out_fp32``, codes the uint8
    ``[B, Ho, Wo, code_channels(N)]`` of the next ``NoisyAct`` if ``code_params`` = (scale,
    zero_point, max_val) is given (as ``act_codes`` would make them from y), else None.
    ``dilation`` and ``groups`` as in ``int_conv2d``."""
    _check_geometry(L, dilation, groups)
    if activation not in ACTIVATIONS:
        raise ValueError(f"int_conv2d_fused: unknown activation {activation!r}")
    if not out_fp32 and code_params is None:
        raise ValueError("int_conv2d_fused: no output requested")
    b, h, w, _ = codes.shape
    stride, padding = _pair(stride), _pair(padding)
    ho, wo = L.out_size(h, w, stride, padding)
    dev = codes.device
    y = torch.empty((b, L.n_out, ho, wo), dtype=torch.float32, device=dev,
                    memory_format=torch.channels_last) if out_fp32 else None
    out_codes, prm = None, (None, None, None)
    if code_params is not None:
        out_codes = torch.empty((b, ho, wo, code_channels(L.n_out)), dtype=torch.uint8, device=dev)
        prm = tuple(torch.as_tensor(p).to(device=dev, dtype=torch.float32).reshape(1).contiguous()
                    for p in code_params)
        if len(prm) != 3:
            raise ValueError("int_conv2d_fused: code_params is (scale, zero_point, max_val)")
    if residual is not None:
        if (residual.dtype != torch.float32 or tuple(residual.shape) != (b, L.n_out, ho, wo)
                or residual.device != dev):
            raise ValueError(f"int_conv2d_fused: the residual must be fp32 {(b, L.n_out, ho, wo)} on {dev}, "
                             f"got {residual.dtype} {tuple(residual.shape)} on {residual.device}")
        residual = residual.detach().contiguous(memory_format=torch.channels_last)
    hc, wc, nwc, ctab = L.pattern_tables(h, w, stride, padding)
    if codes.shape[-1] != L.cp or codes.dtype != torch.uint8 or not codes.is_contiguous():
        raise ValueError(f"integer layer: expected contiguous uint8 codes with {L.cp} channels, "
                         f"got {codes.dtype} {tuple(codes.shape)}")
    if b * ho * wo:
        slope = 0.01 if negative_slope is None else float(negative_slope)
        epi = _lib.IConvEpilogue(_ptr(residual), ACTIVATIONS[activation], slope, _ptr(y), _ptr(out_codes),
                                 *(_ptr(p) for p in prm))
        if not L.dense:
            geo = _lib.IConvGeometry(L.kh, L.kw, stride[0], stride[1], padding[0], padding[1], L.dilation[0],
                                     L.dilation[1], L.groups)
            _check_rc(lib.mhaq_fq_iconv_grouped_u8(_ptr(codes), _ptr(L.weight), _ptr(L.alpha), _ptr(L.beta),
                                                   _ptr(ctab), _ptr(hc), _ptr(wc), nwc, b, h, w, L.cin, L.n_out,
                                                   ctypes.byref(geo), L.a_top, L.w_top, ctypes.byref(epi),
                                                   _stream()), "mhaq_fq_iconv_grouped_u8")
            return y, out_codes
        _check_rc(lib.mhaq_fq_iconv_fused_u8(_ptr(codes), _ptr(L.weight), _ptr(L.alpha), _ptr(L.beta), _ptr(ctab),
                                             _ptr(hc), _ptr(wc), nwc, b, h, w, L.cp, L.n_out, L.kh, L.kw,
                                             stride[0], stride[1], padding[0], padding[1], L.a_top, L.w_top,
                                             ctypes.byref(epi), _stream()), "mhaq_fq_iconv_fused_u8")
    return y, out_codes


def int_linear(codes, L: IntLayerOperands) -> torch.Tensor:
    """fp32 ``[B, N]`` linear layer on activation codes ``[B, Cp]`` (``act_codes``)."""
    if L.kh != 1 or L.kw != 1:
        raise ValueError("int_linear: the operands are those of a convolution")
    b = codes.shape[0]
    y = torch.empty((b, L.n_out), dtype=torch.float32, device=codes.device)
    return _iconv(codes, L, y, b, 1, 1, (1, 1), (0, 0))
