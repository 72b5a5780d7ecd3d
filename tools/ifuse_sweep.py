"""Fused integer epilogues (fuse_integer_model) against the unfused integer model and the fake-quant model.

Per network (ResNet-20 and ResNet-18 STE W4A4 at b256 32^2 / 224^2; RFDN LSQ W2A2 on b16 256^2 LR
patches, as BASELINE configs[4] trains it): eval-forward img/s of the fake-quant model (TF32), the integer model
(build_integer_model) and the fused integer model, and CUDA kernel launches per forward counted
with torch.profiler in a separate run.

Per ResNet-18 block shape (the second block of layers 1-4, W4A4 codes): the fused convolution
(ops.int_conv2d_fused) against what the integer model runs for the same chain,
  conv1: int_conv2d + BatchNorm + ReLU + act_codes            -> fused: codes only
  conv2: int_conv2d + BatchNorm + add + ReLU + act_codes      -> fused: fp32 and codes
with the bytes each moves, counted from the shapes: codes in (B*H*W*Cp) + weight operand, then
per output element 4 (conv out) + 8 (BN) + 12 (add) + 8 (ReLU) + 5 (act_codes) unfused against
1 (codes) or 4 + 4 + 1 (residual in, fp32 out, codes) fused.

CUDA-event timing after warm-up; the per-shape loops rotate codes and residuals over > 2x the
126 MB L2.  Usage: python tools/ifuse_sweep.py [--out profiles/r04_ifuse_sweep.txt]
"""
import argparse
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mhaq_b200 import harness, ops  # noqa: E402
from mhaq_b200.quantization.gdnsq.export import (build_integer_model, export_quantized,  # noqa: E402
                                                 fuse_integer_model)

L2 = 126 << 20
DEV = torch.device("cuda")


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


def kernel_launches(fn):
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    kern = [n for n in names if "memcpy" not in n.lower() and "memset" not in n.lower()]
    return len(kern), sum("fq_act_codes_kernel" in n for n in kern), sum("fq_iconv_kernel" in n for n in kern)


def block_shape(tag, b, c, hw, log):
    levels, w_bits = 16, 4
    sa, zpa = 2.0 ** -4, -0.5
    s_t, b_t = torch.tensor([sa], device=DEV), torch.tensor([zpa], device=DEV)
    hi_t = b_t + (levels - 1) * s_t
    cw = torch.randint(0, 1 << w_bits, (c, c, 3, 3), device=DEV)
    L = ops.int_layer_operands(cw, torch.full((c,), 2.0 ** -6, device=DEV), torch.full((c,), -0.1, device=DEV),
                               sa, zpa, None, a_top=levels - 1, w_top=(1 << w_bits) - 1)
    bn = torch.nn.BatchNorm2d(c).to(DEV).eval()
    with torch.no_grad():
        bn.running_var.uniform_(0.5, 2.0)
        bn.running_mean.normal_(0, 0.1)
    Lf = ops.fold_batchnorm(L, bn)
    cp = L.cp
    c_bytes = b * hw * hw * cp
    n_cbufs = max(1, min(256, -(-2 * L2 // c_bytes)))
    codes = [torch.randint(0, levels, (b, hw, hw, cp), dtype=torch.uint8, device=DEV) for _ in range(n_cbufs)]
    for t in codes:
        t[..., c:] = 0
    r_bytes = b * c * hw * hw * 4
    n_rbufs = max(1, min(64, -(-2 * L2 // r_bytes)))
    res = [torch.randn(b, c, hw, hw, device=DEV).contiguous(memory_format=torch.channels_last) for _ in range(n_rbufs)]
    n = max(n_cbufs, n_rbufs)
    cpar = (s_t, b_t, hi_t)
    out = b * c * hw * hw
    base = c_bytes + L.weight.numel()
    with torch.no_grad():
        def unf1(i):
            return ops.act_codes(F.relu(bn(ops.int_conv2d(codes[i % n_cbufs], L, 1, 1))), *cpar)

        def unf2(i):
            return ops.act_codes(F.relu(bn(ops.int_conv2d(codes[i % n_cbufs], L, 1, 1)) + res[i % n_rbufs]), *cpar)
        t_u1 = timed(unf1, n)
        t_f1 = timed(lambda i: ops.int_conv2d_fused(codes[i % n_cbufs], Lf, 1, 1, activation="relu", out_fp32=False,
                                                    code_params=cpar), n)
        t_u2 = timed(unf2, n)
        t_f2 = timed(lambda i: ops.int_conv2d_fused(codes[i % n_cbufs], Lf, 1, 1, residual=res[i % n_rbufs],
                                                    activation="relu", code_params=cpar), n)
    by_u1, by_f1 = base + out * (4 + 8 + 8 + 5), base + out * 1
    by_u2, by_f2 = base + out * (4 + 8 + 12 + 8 + 5), base + out * (4 + 4 + 1)
    for kind, tu, tf, bu, bf in (("conv1 BN ReLU codes", t_u1, t_f1, by_u1, by_f1),
                                 ("conv2 BN add ReLU fp32+codes", t_u2, t_f2, by_u2, by_f2)):
        log(f"{tag:<10} {kind:<30} {b:>4} {c:>4} {hw:>4}x{hw:<4} {tu * 1e6:10.1f} {bu / 1e6:9.1f} "
            f"{tf * 1e6:10.1f} {bf / 1e6:9.1f} {tu / tf:6.2f}")
    del codes, res
    return t_u1 + t_u2 - t_f1 - t_f2


def network(name, batch, hw, method, bits, log):
    torch.manual_seed(0)
    calib = (torch.rand if name == "rfdn" else torch.randn)(16 if name != "rfdn" else 4, 3, hw, hw, device=DEV)
    q = harness.build_qat(name, DEV, qnmethod=method, act_bit=bits, weight_bit=bits, distillation=False,
                          calib_batch=calib, calib_bits=bits)
    q.eval()
    qi = build_integer_model(q, export_quantized(q))
    gm = fuse_integer_model(qi)
    x = (torch.rand if name == "rfdn" else torch.randn)(batch, 3, hw, hw, device=DEV)
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    with torch.no_grad():
        t_fq = timed(lambda i: q(x), 1, reps=20)
        t_int = timed(lambda i: qi(x), 1, reps=20)
        t_fu = timed(lambda i: gm(x), 1, reps=20)
        t_int2 = timed(lambda i: qi(x), 1, reps=20)      # again, after the fused run: drift check
        y_int, y_fu = qi(x), gm(x)
        d = float((y_fu - y_int).abs().max())
        agree = float((y_fu.argmax(1) == y_int.argmax(1)).float().mean()) if name != "rfdn" else float("nan")
        launches = [kernel_launches(lambda: m(x)) for m in (q, qi, gm)]
    log(f"{name:<9} {method} W{bits}A{bits} b{batch:<4} {hw}x{hw:<4} img/s: fake-quant {batch / t_fq:9.0f}   "
        f"integer {batch / t_int:9.0f} (again {batch / t_int2:9.0f})   fused {batch / t_fu:9.0f}   fused/integer {t_int / t_fu:5.2f}x   "
        f"ms/forward {t_fq * 1e3:.3f} / {t_int * 1e3:.3f} / {t_fu * 1e3:.3f}")
    log(f"{'':<9} kernel launches per forward (all / act_codes / iconv): fake-quant {launches[0][0]}, "
        f"integer {launches[1]}, fused {launches[2]};  max |fused - integer| {d:.3e}"
        + ("" if name == "rfdn" else f", argmax agreement {agree:.3f}"))
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def log(s=""):
        print(s, flush=True)
        lines.append(s)
    if not torch.cuda.is_available():
        raise SystemExit("ifuse_sweep: no CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    log(f"# device: {torch.cuda.get_device_name()} | nvidia-smi name, power limit, max SM clock: "
        f"{smi[torch.cuda.current_device()] if smi else 'n/a'}")
    log("# CUDA events after warm-up")
    log("")
    log("# whole networks, eval forward; launches counted with torch.profiler in a separate run")
    for name, batch, hw, method, bits in (("resnet20", 256, 32, "STE", 4), ("resnet18", 256, 224, "STE", 4),
                                          ("rfdn", 16, 256, "LSQ", 2)):
        network(name, batch, hw, method, bits, log)
    log("")
    log("# ResNet-18 block chains (second block of each layer), W4A4, b256 224^2 input; codes and residuals rotated "
        "over > 2x L2; MB counted from the shapes (see the tool's docstring)")
    log(f"{'layer':<10} {'chain':<30} {'B':>4} {'C':>4} {'HxW':>9} {'unf_us':>10} {'unf_MB':>9} {'fused_us':>10} "
        f"{'fused_MB':>9} {'x':>6}")
    saved = 0.0
    for tag, c, hw in (("layer1.1", 64, 56), ("layer2.1", 128, 28), ("layer3.1", 256, 14), ("layer4.1", 512, 7)):
        saved += block_shape(tag, 256, c, hw, log)
    log(f"# one block of each layer: fused saves {saved * 1e3:.3f} ms per batch-256 forward over the unfused chains")
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
