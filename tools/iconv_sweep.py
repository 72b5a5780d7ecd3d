"""Integer layers against the fake-quant layers they replace, per layer shape and per network.

Per shape (every quantized layer of ResNet-20 at batch 256, the 3x3 layers of ResNet-18 at 224^2
and batch 256, the quantized RFDN layers at 256x256 LR patches and batch 16, as BASELINE configs[4]
trains):
  - fq_act_codes_kernel: bytes/s at 4 B read + 1 B written per input element (padding not counted);
  - fq_iconv_kernel: time, TOPS = 2*M*N*K_valid / t, bytes/s (codes read + u8 weights + fp32 out),
    and its share of the roofline: max(ops / 4,500 TOPS, bytes / 7.7 TB/s) / t, naming the bound;
  - the layer as the fake-quant model runs it: NoisyAct eval forward + cuDNN channels_last conv on
    the fake-quantized weight, once in TF32 and once under bf16 autocast.
Whole networks: eval forward img/s at batch 256, integer model vs fake-quant model.

CUDA-event timing after warm-up; every timed loop rotates over enough input copies to exceed
the 126 MB L2.  Usage: python tools/iconv_sweep.py [--out profiles/r03_iconv_sweep.txt]
"""
import argparse
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mhaq_b200 import harness, ops  # noqa: E402
from mhaq_b200.quantization.gdnsq.export import build_integer_model, export_quantized  # noqa: E402
from mhaq_b200.quantization.gdnsq.layers.gdnsq_conv2d import NoisyConv2d  # noqa: E402

PEAK_OPS, PEAK_BW, L2 = 4500e12, 7.7e12, 126 << 20
DEV = torch.device("cuda")


def timed(fn, n_bufs, reps=None, warm=3):
    for i in range(warm):
        fn(i % n_bufs)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # at least ~20 calls, and at least a full rotation through the buffers
    reps = reps or max(20, n_bufs)
    e0.record()
    for i in range(reps):
        fn(i % n_bufs)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def layer_shapes(name, batch, hw, only3x3=False):
    """(name, B, C, H, W, N, k, stride, pad) of every quantized conv / linear, from hooks on the model."""
    q = harness.build_qat(name, DEV, act_bit=4, weight_bit=4, distillation=False)
    out = []
    hooks = []
    for n, m in q.model.named_modules():
        if isinstance(m, NoisyConv2d):
            def hook(mod, inp, _out, n=n):
                x = inp[0]
                out.append((n, batch, x.shape[1], x.shape[2], x.shape[3], mod.out_channels, mod.kernel_size[0],
                            mod.stride[0], mod.padding[0]))
            hooks.append(m.register_forward_hook(hook))
    q.eval()
    with torch.no_grad():
        q.model(torch.randn(1, 3, hw, hw, device=DEV))
    for h in hooks:
        h.remove()
    if only3x3:
        out = [o for o in out if o[6] == 3]
    return out


def sweep_shape(tag, b, c, h, w, n, k, stride, pad, log):
    levels, w_bits = 16, 4
    sa, zpa = 2.0 ** -4, -0.5
    s_t, b_t = torch.tensor([sa], device=DEV), torch.tensor([zpa], device=DEV)
    hi_t = b_t + (levels - 1) * s_t
    cw = torch.randint(0, 1 << w_bits, (n, c, k, k), device=DEV)
    sw, zpw = torch.full((n,), 2.0 ** -6, device=DEV), torch.full((n,), -0.1, device=DEV)
    L = ops.int_layer_operands(cw, sw, zpw, sa, zpa, None, a_top=levels - 1, w_top=(1 << w_bits) - 1)
    wq = (cw.float() * 2.0 ** -6 - 0.1).contiguous(memory_format=torch.channels_last)
    x_bytes = b * c * h * w * 4
    n_bufs = max(1, min(64, -(-2 * L2 // x_bytes)))
    xs = [(torch.randn(b, c, h, w, device=DEV) * 0.5).contiguous(memory_format=torch.channels_last)
          for _ in range(n_bufs)]
    # the codes are a quarter of the fp32 bytes: their own rotation, also over > 2x L2
    c_bytes = b * h * w * L.cp
    n_cbufs = max(1, min(512, -(-2 * L2 // c_bytes)))
    codes = [ops.act_codes(xs[i % n_bufs], s_t, b_t, hi_t)[0] for i in range(n_cbufs)]
    ho, wo = (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1
    m = b * ho * wo
    # valid MACs: count valid taps per output position along each axis
    vh = sum(min(h, o * stride - pad + k) - max(0, o * stride - pad) for o in range(ho))
    vw = sum(min(w, o * stride - pad + k) - max(0, o * stride - pad) for o in range(wo))
    ops_valid = 2 * b * vh * vw * c * n

    t_q = timed(lambda i: ops.act_codes(xs[i], s_t, b_t, hi_t), n_bufs)
    t_i = timed(lambda i: ops.int_conv2d(codes[i], L, stride, pad), n_cbufs)
    i_bytes = b * h * w * L.cp + L.weight.numel() + m * n * 4
    bound_t = max(ops_valid / PEAK_OPS, i_bytes / PEAK_BW)
    which = "compute" if ops_valid / PEAK_OPS > i_bytes / PEAK_BW else "memory"

    def fq_pair(i, dtype=None):
        xq = ops.quantize_eval(xs[i], s_t, b_t, b_t, hi_t)[0]
        if dtype is None:
            return F.conv2d(xq, wq, None, stride, pad)
        with torch.autocast("cuda", dtype=dtype):
            return F.conv2d(xq, wq, None, stride, pad)
    torch.backends.cudnn.allow_tf32 = True
    t_tf32 = timed(lambda i: fq_pair(i), n_bufs)
    t_bf16 = timed(lambda i: fq_pair(i, torch.bfloat16), n_bufs)
    t_int = t_q + t_i
    log(f"{tag:<34} {b:>4} {c:>4} {h:>4}x{w:<4} {n:>4} {k}/{stride}/{pad}  "
        f"{x_bytes * 1.25 / t_q / 1e12:6.2f}  {t_i * 1e6:9.1f} {ops_valid / t_i / 1e12:7.1f} "
        f"{i_bytes / t_i / 1e12:6.2f} {bound_t / t_i:5.2f} {which:<7}  "
        f"{t_int * 1e6:9.1f} {t_tf32 * 1e6:9.1f} {t_bf16 * 1e6:9.1f}  {t_tf32 / t_int:5.2f} {t_bf16 / t_int:5.2f}")
    del xs, codes
    return t_int, t_tf32


def network(name, batch, hw, log):
    calib = torch.randn(16, 3, hw, hw, device=DEV)
    q = harness.build_qat(name, DEV, act_bit=4, weight_bit=4, distillation=False, calib_batch=calib, calib_bits=4)
    q.eval()
    qi = build_integer_model(q, export_quantized(q))
    x = torch.randn(batch, 3, hw, hw, device=DEV)
    torch.backends.cudnn.allow_tf32 = True
    with torch.no_grad():
        t_fq = timed(lambda i: q(x), 1, reps=20)
        t_int = timed(lambda i: qi(x), 1, reps=20)
        d = float((qi(x) - q(x)).abs().max())
    log(f"{name:<10} b{batch} {hw}x{hw}: fake-quant {batch / t_fq:10.0f} img/s   integer {batch / t_int:10.0f} img/s"
        f"   ({t_fq / t_int:.2f}x)   max |dlogit| {d:.3e}")


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)
    if not torch.cuda.is_available():
        raise SystemExit("iconv_sweep: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    log(f"# device: {torch.cuda.get_device_name()} | nvidia-smi name, power limit, max SM clock: "
        f"{smi[torch.cuda.current_device()] if smi else 'n/a'}")
    log("# W4A4 codes (16 activation levels, 4-bit weights); CUDA events, warm-up; fp32 inputs and uint8 codes "
        "each rotated over > 2x L2")
    log("# quant = act-codes GB/s as TB/s (5 B/elem); iconv: us, TOPS (valid MACs x2), TB/s, share of roofline "
        "(max(ops/4500T, bytes/7.7T) / t) and its bound; int = quant + iconv; fq = NoisyAct eval + cuDNN "
        "channels_last conv (TF32 / bf16 autocast); last two columns: speed-up of int over fq")
    log(f"{'layer':<34} {'B':>4} {'C':>4} {'HxW':>9} {'N':>4} k/s/p  {'quant':>6}  {'iconv_us':>9} {'TOPS':>7} "
        f"{'TB/s':>6} {'roof':>5} {'bound':<7}  {'int_us':>9} {'tf32_us':>9} {'bf16_us':>9}  {'xTF32':>5} {'xBF16':>5}")
    slower, sums = [], {}
    for model, batch, hw, only3 in (("resnet20", 256, 32, False), ("resnet18", 256, 224, True), ("rfdn", 16, 256, False)):
        seen = {}
        for (n, b, c, h, w, o, k, s, p) in layer_shapes(model, batch, hw, only3):
            key = (b, c, h, w, o, k, s, p)
            if key not in seen:
                seen[key] = sweep_shape(f"{model}:{n}", b, c, h, w, o, k, s, p, log)
                if model != "rfdn" and seen[key][0] >= seen[key][1]:
                    slower.append(f"{model}:{n}")
            t_int, t_tf32 = seen[key]
            acc = sums.setdefault(model, [0.0, 0.0])
            acc[0] += t_int
            acc[1] += t_tf32
    log("")
    log(f"# ResNet shapes where the integer layer is not faster than the TF32 fake-quant pair: {slower or 'none'}")
    for model, (t_int, t_tf32) in sums.items():
        log(f"# {model}: sum over its {'3x3 ' if model == 'resnet18' else ''}quantized layers (each shape timed once, "
            f"counted per layer): integer pairs {t_int * 1e3:.3f} ms, TF32 fake-quant pairs {t_tf32 * 1e3:.3f} ms")
    log("")
    for name, hw in (("resnet20", 32), ("resnet18", 224)):
        network(name, 256, hw, log)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
