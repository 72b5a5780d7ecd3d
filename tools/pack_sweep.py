"""Device time of packing (ops.pack_codes) and unpacking (ops.unpack_codes) against size-matched
torch conversions, N = 2^20 ... 2^30 elements, per-tensor and per-channel [C, N/C] with
C in {64, 512, 4096}, widths b in {1, 2, 4, 8}.

Rates are on the algorithmic bytes: pack reads 4 B and writes b/8 B per element, unpack reads
b/8 B and writes 4 B.  The ceilings are the torch conversions with the same shape of traffic:
fp32 -> uint8 (`x.to(torch.uint8)`, 5 B/element) for pack and uint8 -> fp32 (`u8.to(torch.float32)`,
5 B/element) for unpack.  On torch 2.11 those conversions are not bandwidth-bound, so an fp32
elementwise kernel of the same N (`torch.neg(x, out=y)`, 8 B/element; a same-dtype `copy_` becomes a
copy-engine memcpy node in a graph, which is slower from 2^27 elements) is printed as well, and each
kernel's rate as a fraction of it.
Each measurement captures K calls on K rotating input sets (footprint
> 2x the 126 MB L2, so every call sees cold inputs) into one CUDA graph and times its replays
with CUDA events, like tools/midsize_graph.py.  Pack runs the clamped activation form (codes in
range, no host synchronisation: check=False).

    python tools/pack_sweep.py [--out FILE] [--min-log2 20] [--max-log2 30]

The table goes to stdout and, with --out, to FILE.
"""
import argparse
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mhaq_b200 import ops  # noqa: E402

dev = torch.device("cuda")
L2_BYTES = 126 << 20


def graph_time(body, K, reps=20):
    """body(i) for i in range(K) captured once; returns ms per call over `reps` replays."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in range(K):
            body(i)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(K):
            body(i)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    del g
    return e0.elapsed_time(e1) / (reps * K)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the name from torch is still recorded
        q = f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable: {e})"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the table to this file")
    ap.add_argument("--min-log2", type=int, default=20)
    ap.add_argument("--max-log2", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pack_sweep needs a CUDA device")
    lines = [f"# pack / unpack sweep on {gpu_info()} (name, power limit, max SM clock)",
             "# GB/s on algorithmic bytes: pack 4 + b/8 B/elem, unpack b/8 + 4 B/elem; ceiling = torch "
             "fp32->uint8 (pack) / uint8->fp32 (unpack), 5 B/elem; ratio = kernel GB/s / ceiling GB/s; "
             "of copy = kernel GB/s / fp32 torch.neg GB/s (8 B/elem)",
             "# pack calls include the zero-fill of their 8-byte out-of-range counter (one memset node)",
             f"{'log2N':>5} {'layout':>8} {'b':>2} {'pack us':>9} {'GB/s':>7} {'ceil GB/s':>9} {'ratio':>6}"
             f" {'of copy':>7} {'unpack us':>9} {'GB/s':>7} {'ceil GB/s':>9} {'ratio':>6} {'of copy':>7} {'copy GB/s':>9}"]
    print("\n".join(lines), flush=True)
    gen = torch.Generator(device=dev).manual_seed(0)
    for lg in range(args.min_log2, args.max_log2 + 1):
        n = 1 << lg
        K = max(1, math.ceil(2 * L2_BYTES / (5 * n)))
        xs = [torch.randn(n, generator=gen, device=dev) * 3 for _ in range(K)]
        u8 = [torch.empty(n, dtype=torch.uint8, device=dev) for _ in range(K)]
        f32 = [torch.empty(n, dtype=torch.float32, device=dev) for _ in range(K)]
        t_cp = graph_time(lambda i: torch.neg(xs[i], out=f32[i]), K)     # fp32 1R:1W kernel: the HBM yardstick
        t_c8 = graph_time(lambda i: u8[i].copy_(xs[i]), K)                # x.to(torch.uint8)
        t_cf = graph_time(lambda i: f32[i].copy_(u8[i]), K)               # u8.to(torch.float32)
        ceil_pack = 5 * n / t_c8 / 1e6
        ceil_unpack = 5 * n / t_cf / 1e6
        copy = 8 * n / t_cp / 1e6
        for layout in ("tensor", "64", "512", "4096"):
            C = 1 if layout == "tensor" else int(layout)
            xv = [x.view(C, n // C) if C > 1 else x for x in xs]
            for b in (1, 2, 4, 8):
                top = (1 << b) - 1
                shape = (C, 1) if C > 1 else (1,)
                s = torch.full(shape, 6.0 / top, device=dev) * (1 + 0.01 * torch.rand(shape, device=dev))
                zp = torch.full(shape, -3.0, device=dev)
                hi = zp + top * s
                packs = [ops.pack_codes(x, s, zp, zp, hi, bits=b) for x in xv]

                def pack(i):
                    ops.pack_codes(xv[i], s, zp, zp, hi, bits=b, check=False)

                def unpack(i):
                    ops.unpack_codes(packs[i])

                t_p = graph_time(pack, K)
                t_u = graph_time(unpack, K)
                gp = (4 + b / 8) * n / t_p / 1e6
                gu = (b / 8 + 4) * n / t_u / 1e6
                row = (f"{lg:>5} {layout:>8} {b:>2} {t_p * 1e3:>9.1f} {gp:>7.0f} {ceil_pack:>9.0f} "
                       f"{gp / ceil_pack:>6.3f} {gp / copy:>7.3f} {t_u * 1e3:>9.1f} {gu:>7.0f} {ceil_unpack:>9.0f} "
                       f"{gu / ceil_unpack:>6.3f} {gu / copy:>7.3f} {copy:>9.0f}")
                lines.append(row)
                print(row, flush=True)
                del packs
        del xs, u8, f32, xv
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
