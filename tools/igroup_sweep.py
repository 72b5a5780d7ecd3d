"""Grouped, depthwise and dilated integer convolutions against NoisyAct + cuDNN.

Per quantized convolution shape of MobileNetV2, ResNeXt-50 32x4d and the dilated ResNet-50 (the
3x3 layers the quantizer quantizes, stems excluded) at batch 256 and 224^2 input, W4A4 codes:
  int    ops.int_conv2d on uint8 codes (depthwise: fq_idw_kernel on the CUDA cores; other grouped or
         dilated layers: fq_iconv_kernel<true, true> on the tensor cores; plain layers:
         fq_iconv_kernel<false>)
  tf32   NoisyAct (fp32 fake-quant) + F.conv2d channels_last, TF32 allowed
  bf16   NoisyAct + F.conv2d channels_last on bf16 copies of its output and the weight
and the integer kernel's share of its roofline: the least time from the bytes it must move (codes
in, weight operand, fp32 out, at 7.7 TB/s) and, for the tensor-core kernel, from its int8 MACs at
4.5 POPS dense; "hbm" or "mma" names the larger.  The depthwise kernel has no tensor-core bound: its
row is the HBM bound alone.  Codes inputs rotate over > 2x the 126 MB L2.

Then whole networks at batch 256, 224^2, eval forward: img/s of the fake-quant model (TF32), the
integer model (build_integer_model(..., allow_groups_and_dilation=True)) and the fused one.

CUDA-event timing after warm-up.  Usage: python tools/igroup_sweep.py [--out profiles/r05_igroup_sweep.txt]
"""
import argparse
import collections
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mhaq_b200 import harness, ops  # noqa: E402
from mhaq_b200.quantization.gdnsq.export import (build_integer_model, export_quantized,  # noqa: E402
                                                 fuse_integer_model)
from mhaq_b200.quantization.gdnsq.layers.gdnsq_act import NoisyAct  # noqa: E402

L2 = 126 << 20
HBM = 7.7e12
MMA_I8 = 4.5e15
DEV = torch.device("cuda")
MODELS = ("mobilenet_v2", "resnext50_32x4d", "resnet50_dilated")


def timed(fn, n_bufs, reps=None, warm=3):
    for i in range(warm):
        fn(i % n_bufs)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = reps or max(20, n_bufs)
    e0.record()
    for i in range(reps):
        fn(i % n_bufs)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def layer_shapes(name, hw):
    """Counter of (cin, cout, k, stride, pad, dilation, groups, H, W) over the model's quantized
    convolutions (not 1x1, not excluded), from forward hooks on the fp32 model."""
    model = harness.build_model(name).eval()
    excl = set(harness.EXCLUDED[name])
    shapes = collections.Counter()
    hooks = []
    for n, m in model.named_modules():
        if isinstance(m, torch.nn.Conv2d) and m.kernel_size != (1, 1) and n not in excl:
            hooks.append(m.register_forward_hook(lambda mod, inp, out: shapes.update(
                [(mod.in_channels, mod.out_channels, mod.kernel_size[0], mod.stride[0], mod.padding[0],
                  mod.dilation[0], mod.groups, inp[0].shape[2], inp[0].shape[3])])))
    with torch.no_grad():
        model(torch.zeros(1, 3, hw, hw))
    for h in hooks:
        h.remove()
    return shapes


def shape_row(name, shape, count, b, log):
    cin, cout, k, s, p, d, g, h, w = shape
    levels, w_bits = 16, 4
    sa, zpa = 2.0 ** -4, -0.5
    cw = torch.randint(0, 1 << w_bits, (cout, cin // g, k, k), device=DEV)
    L = ops.int_layer_operands(cw, torch.full((cout,), 2.0 ** -6, device=DEV), torch.full((cout,), -0.1, device=DEV),
                               sa, zpa, None, a_top=levels - 1, w_top=(1 << w_bits) - 1, groups=g, dilation=d)
    cp = L.cp
    c_bytes = b * h * w * cp
    n_bufs = max(1, min(32, -(-2 * L2 // c_bytes)))
    codes = [torch.randint(0, levels, (b, h, w, cp), dtype=torch.uint8, device=DEV) for _ in range(n_bufs)]
    for t in codes:
        t[..., cin:] = 0
    ho, wo = L.out_size(h, w, (s, s), (p, p))
    y_bytes = b * ho * wo * cout * 4
    by = c_bytes + L.weight.numel() + y_bytes
    macs = b * ho * wo * cout * k * k * (cin // g)
    dw = g == cin == cout
    t_hbm, t_mma = by / HBM, (0.0 if dw else macs / MMA_I8)
    bound, which = (t_hbm, "hbm") if t_hbm >= t_mma else (t_mma, "mma")
    act = NoisyAct(signed=True).to(DEV).eval()
    with torch.no_grad():
        act.log_act_s.fill_(-4.0)
        act.log_act_q.fill_(4.0)
        act.act_b.fill_(-0.5)
    x = torch.randn(b, cin, h, w, device=DEV).contiguous(memory_format=torch.channels_last)
    wt = torch.randn(cout, cin // g, k, k, device=DEV).contiguous(memory_format=torch.channels_last)
    wb = wt.bfloat16()
    conv = dict(stride=s, padding=p, dilation=d, groups=g)
    with torch.no_grad():
        t_int = timed(lambda i: ops.int_conv2d(codes[i], L, s, p), n_bufs)
        torch.backends.cudnn.allow_tf32 = True
        t_tf32 = timed(lambda i: F.conv2d(act(x), wt, **conv), 1)
        torch.backends.cudnn.allow_tf32 = False
        t_bf16 = timed(lambda i: F.conv2d(act(x).bfloat16(), wb, **conv), 1)
    kind = "dw" if dw else (f"g{g}" if g > 1 else f"d{d}")
    log(f"{name:<17} {kind:>5} {count:>3} {cin:>5} {cout:>5} {k}x{k} s{s} d{d} {h:>4}x{w:<4} {t_int * 1e6:10.1f} "
        f"{by / t_int / 1e9:8.0f} {bound / t_int * 100:6.1f}% {which:>4} {t_tf32 * 1e6:10.1f} {t_bf16 * 1e6:10.1f} "
        f"{t_tf32 / t_int:6.2f} {t_bf16 / t_int:6.2f}")
    del codes, x
    return count * t_int, count * t_tf32, count * t_bf16


def network(name, batch, hw, log):
    torch.manual_seed(0)
    q = harness.build_qat(name, DEV, qnmethod="STE", act_bit=4, weight_bit=4, distillation=False,
                          calib_batch=torch.randn(16, 3, hw, hw, device=DEV), calib_bits=4)
    q.model.to(memory_format=torch.channels_last)
    q.eval()
    qi = build_integer_model(q, export_quantized(q), allow_groups_and_dilation=True)
    gm = fuse_integer_model(qi)
    x = torch.randn(batch, 3, hw, hw, device=DEV).contiguous(memory_format=torch.channels_last)
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    with torch.no_grad():
        t_fq = timed(lambda i: q(x), 1, reps=10)
        t_int = timed(lambda i: qi(x), 1, reps=10)
        t_fu = timed(lambda i: gm(x), 1, reps=10)
        agree = float((gm(x).argmax(1) == q(x).argmax(1)).float().mean())
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    log(f"{name:<17} b{batch} {hw}x{hw} img/s: fake-quant {batch / t_fq:8.0f}   integer {batch / t_int:8.0f}   "
        f"fused {batch / t_fu:8.0f}   integer/fake-quant {t_fq / t_int:5.2f}x   fused/fake-quant {t_fq / t_fu:5.2f}x   "
        f"argmax agreement fused vs fake-quant {agree:.3f} (untrained, calibrated)")
    del q, qi, gm


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--hw", type=int, default=224)
    args = ap.parse_args()
    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)
    if not torch.cuda.is_available():
        raise SystemExit("igroup_sweep: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    log(f"# device: {torch.cuda.get_device_name()} | nvidia-smi name, power limit, max SM clock: "
        f"{smi[torch.cuda.current_device()] if smi else 'n/a'}")
    log(f"# CUDA events after warm-up; W4A4; batch {args.batch}, {args.hw}^2 input; codes rotated over > 2x L2")
    log("# per quantized layer shape: n = layers of that shape; int_us / GB/s / roof% / bound of ops.int_conv2d;"
        " NoisyAct + cuDNN channels_last in TF32 and bf16; x = their time over int's")
    log(f"{'model':<17} {'kind':>5} {'n':>3} {'cin':>5} {'cout':>5} {'geom':<11} {'HxW':>9} {'int_us':>10} "
        f"{'GB/s':>8} {'roof':>7} {'bnd':>4} {'tf32_us':>10} {'bf16_us':>10} {'x_tf32':>6} {'x_bf16':>6}")
    for name in MODELS:
        tot = [0.0, 0.0, 0.0]
        for shape, count in sorted(layer_shapes(name, args.hw).items(), key=lambda kv: (-kv[0][7], kv[0][1])):
            for i, v in enumerate(shape_row(name, shape, count, args.batch, log)):
                tot[i] += v
        log(f"{name:<17} sum over its quantized layers: int {tot[0] * 1e3:.3f} ms, tf32 {tot[1] * 1e3:.3f} ms, "
            f"bf16 {tot[2] * 1e3:.3f} ms")
        torch.cuda.empty_cache()
    log("")
    log("# whole networks, eval forward")
    for name in MODELS:
        network(name, args.batch, args.hw, log)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
