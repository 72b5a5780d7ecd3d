"""Two ranks over NCCL on two GPUs: the ONE exchange step on the path — AEWGS's per-channel
statistics all-reduce (reference gdnsq.py:126-129: three `all_reduce(AVG)`; here one packed
[3, O] all-reduce between the statistics kernel and the apply kernel).

The CUDA path (mhaq_fq_aewgs_stats_f32 -> NCCL all-reduce -> mhaq_fq_bwd_f32, and the layer
wrapper NoisyConv2d built on it) is compared with the LIVE reference (oracle/_ref) run in the same
two processes on the same process group: replicated weights, a different upstream gradient per
rank (different batch shards), so the averaged statistics differ from either rank's own.

Needs 2 GPUs: skipped on a 1-GPU box (run with `gpurun --gpus 2`; the result of that run is kept
in profiles/r02_dist_nccl.txt).
"""
import math
import os
import socket
import sys
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    res = {"rank": rank}
    try:
        sys.path.insert(0, ROOT)
        import mhaq_b200
        from oracle import ref_loader, ref_port
        ref = ref_loader.load_ops() if ref_loader.available() else ref_port.load()
        orig_randint_like = torch.randint_like

        def run_case(shape, per_channel, tag):
            g = torch.Generator().manual_seed(7)                       # replicated weights
            w = (torch.randn(shape, generator=g) * 0.3).to(dev)
            gr = torch.Generator().manual_seed(50 + rank)              # this rank's shard
            go = torch.randn(shape, generator=gr).to(dev)
            r = (torch.randint(0, 2, shape, generator=gr).float() - 0.5).to(dev)
            if per_channel:
                pshape = (shape[0],) + (1,) * (len(shape) - 1)
                dims = tuple(range(1, len(shape)))
                mn, mx = w.amin(dims, keepdim=True), w.amax(dims, keepdim=True)
                scale = ((mx - mn) / 3.0).reshape(pshape)
            else:
                mn, mx = w.amin().reshape(1), w.amax().reshape(1)
                scale = (mx - mn) / 3.0
            # --- live reference (its three all_reduce calls run on this NCCL group)
            wr = w.clone().requires_grad_(True)
            sr = scale.clone().requires_grad_(True)
            zr = mn.clone().requires_grad_(True)
            Q = ref.Quantizer(types.SimpleNamespace(training=True), sr, zr, -math.inf, math.inf,
                              qnmethod=ref.QNMethod.AEWGS)
            torch.randint_like = lambda t, high, **kw: (r + 0.5).to(t.dtype)
            try:
                y_r = Q.dequantize(Q.quantize(wr))
                y_r.backward(go)
            finally:
                torch.randint_like = orig_randint_like
            # --- CUDA path
            wo = w.clone().requires_grad_(True)
            so = scale.clone().requires_grad_(True)
            zo = mn.clone().requires_grad_(True)
            y_o = mhaq_b200.fake_quant(wo, so, zo, -math.inf, math.inf, method="AEWGS", noise=r)
            y_o.backward(go)
            torch.cuda.synchronize()

            def rel(a, b, floor):
                return float(((a - b).abs() / (b.abs() * 1e-5 + floor)).max())
            res[tag] = {
                "y_bit_exact": bool(torch.equal(y_o, y_r)),
                "gx_err_over_tol": rel(wo.grad, wr.grad, 1e-7),          # tol = 1e-5 * |ref| + 1e-7
                "g_scale_err_over_tol": rel(so.grad, sr.grad, 2e-5),
                "g_zp_err_over_tol": rel(zo.grad, zr.grad, 2e-5),
                # the averaged statistics must differ from a single rank's (else the test is vacuous)
                "gx_checksum": float(wo.grad.double().sum()),
            }

        run_case((64, 32, 3, 3), True, "per_channel")
        run_case((48, 50, 3, 3), True, "per_channel_ragged_rows")
        run_case((16, 24, 3, 3), False, "per_tensor_dim0_quirk")

        # --- the layer wrapper under DDP-style use: NoisyConv2d(AEWGS) vs the reference's layer
        from mhaq_b200.aux.types import QScheme
        from mhaq_b200.quantization.gdnsq.gdnsq_utils import QNMethod
        from mhaq_b200.quantization.gdnsq.layers.gdnsq_conv2d import NoisyConv2d
        from mhaq_b200 import ops
        torch.manual_seed(3)                                           # same init on both ranks
        ours = NoisyConv2d(8, 16, 3, padding=1, bias=False, qscheme=QScheme.PER_CHANNEL, qnmethod=QNMethod.AEWGS).to(dev)
        theirs = ref.NoisyConv2d(8, 16, 3, padding=1, bias=False, qscheme=ref.QScheme.PER_CHANNEL,
                                 qnmethod=ref.QNMethod.AEWGS).to(dev)
        with torch.no_grad():
            theirs.weight.copy_(ours.weight)
            ours.log_wght_s.fill_(-4.0); theirs.log_wght_s.fill_(-4.0)
        xg = torch.Generator().manual_seed(900 + rank)
        x = torch.randn(4, 8, 10, 10, generator=xg).to(dev)
        go = torch.randn(4, 16, 10, 10, generator=xg).to(dev)
        rw = (torch.randint(0, 2, tuple(ours.weight.shape), generator=xg).float() - 0.5).to(dev)
        tf32 = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        torch.randint_like = lambda t, high, **kw: (rw + 0.5).to(t.dtype)
        try:
            theirs.train()
            theirs(x).backward(go)
        finally:
            torch.randint_like = orig_randint_like
        real = ops.weight_fake_quant_log
        ops.weight_fake_quant_log = lambda w, ls, method="STE", noise=None, philox=None: real(w, ls, method=method, noise=rw)
        try:
            ours.train()
            ours(x).backward(go)
        finally:
            ops.weight_fake_quant_log = real
            torch.backends.cudnn.allow_tf32 = tf32
        torch.cuda.synchronize()
        gw_o, gw_r = ours.weight.grad, theirs.weight.grad
        gs_o, gs_r = ours.log_wght_s.grad, theirs.log_wght_s.grad
        res["layer"] = {
            "g_weight_err_over_tol": float(((gw_o - gw_r).abs() / (gw_r.abs() * 1e-5 + 1e-5 * float(gw_r.abs().max()))).max()),
            "g_log_wght_s_err_over_tol": float(((gs_o - gs_r).abs() / (gs_r.abs() * 1e-5 + 2e-5)).max()),
        }
        # --- model-wide form: statistics of EVERY tensor -> ONE all-reduce -> apply, against the
        # per-layer streaming path (pinned against the reference above) on the same two ranks
        gm = torch.Generator().manual_seed(11)
        shapes = [(16, 8, 3, 3), (24, 16, 3, 3), (10, 50)]
        Ws = [(torch.randn(s_, generator=gm) * 0.2).to(dev) for s_ in shapes]
        Ls = [torch.full((s_[0],) + (1,) * (len(s_) - 1), -3.5).to(dev) for s_ in shapes]
        gr2 = torch.Generator().manual_seed(70 + rank)
        Gs = [torch.randn(s_, generator=gr2).to(dev) for s_ in shapes]
        Ns = [(torch.randint(0, 2, s_, generator=gr2).float() - 0.5).to(dev) for s_ in shapes]
        per_layer = []
        for w_, l_, g_, n_ in zip(Ws, Ls, Gs, Ns):
            wl, ll = w_.clone().requires_grad_(True), l_.clone().requires_grad_(True)
            wq_, _, _ = ops.weight_fake_quant_log(wl, ll, method="AEWGS", noise=n_)
            wq_.backward(g_)
            per_layer.append((wl.grad, ll.grad))
        Wm = [w_.clone().requires_grad_(True) for w_ in Ws]
        Lm = [l_.clone().requires_grad_(True) for l_ in Ls]
        outs = ops.weight_fake_quant_rows_multi(Wm, Lm, method="AEWGS", noises=Ns)
        sum((o[0] * g_).sum() for o, g_ in zip(outs, Gs)).backward()
        torch.cuda.synchronize()
        worst = 0.0
        for (gw_r2, gl_r2), wm, lm in zip(per_layer, Wm, Lm):
            worst = max(worst, float(((wm.grad - gw_r2).abs() / (gw_r2.abs() * 1e-5 + 2e-5)).max()),
                        float(((lm.grad - gl_r2).abs() / (gl_r2.abs() * 1e-5 + 2e-5)).max()))
        res["multi_tensor_vs_per_layer_err_over_tol"] = worst
        q.put(res)
    except Exception as exc:       # surface the failure in the parent instead of a silent hang
        import traceback
        res["error"] = f"{type(exc).__name__}: {exc}\n{traceback.format_exc()[-1500:]}"
        q.put(res)
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs (gpurun --gpus 2)")
def test_two_rank_nccl_aewgs_cuda_path_matches_the_live_reference():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    out.sort(key=lambda d: d["rank"])
    import json
    report = json.dumps(out, indent=1)
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    with open(os.path.join(ROOT, "gpurun_out", "dist_nccl_aewgs.json"), "w") as f:
        f.write(report)
    for d in out:
        assert "error" not in d, d["error"]
        for tag in ("per_channel", "per_channel_ragged_rows", "per_tensor_dim0_quirk"):
            c = d[tag]
            assert c["y_bit_exact"], (d["rank"], tag)
            assert c["gx_err_over_tol"] <= 1.0, (d["rank"], tag, c)
            assert c["g_scale_err_over_tol"] <= 1.0, (d["rank"], tag, c)
            assert c["g_zp_err_over_tol"] <= 1.0, (d["rank"], tag, c)
        assert d["layer"]["g_weight_err_over_tol"] <= 1.0, d
        assert d["layer"]["g_log_wght_s_err_over_tol"] <= 1.0, d
        assert d["multi_tensor_vs_per_layer_err_over_tol"] <= 1.0, d
    # different shards -> different per-rank gradients (the exchange really mixed two ranks' data)
    assert out[0]["per_channel"]["gx_checksum"] != out[1]["per_channel"]["gx_checksum"]
