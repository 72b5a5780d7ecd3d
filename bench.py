#!/usr/bin/env python
"""bench.py — fake-quant fwd+bwd throughput (BASELINE.json metric) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W]           # our sm_100a path
    python bench.py --impl reference [...]                        # the LIVE reference's CPU path (oracle/_ref)
    python bench.py --dump-outputs DIR [...]                      # + the last timed step's outputs as DIR/*.npy

A "step" is one pass of the hot path over one batch of synthetic input: one
fake-quant forward + one backward (incl. the in-kernel deterministic reduction) over a
[C, N/C] fp32 tensor.  Default workload = BASELINE.json configs[1] headline
point: per-channel (C=512) N=2^28 elements, GDNSQ/STE estimator with fused
Philox noise, 4 bits.  GB/s = 20 B/element (8 fwd + 12 bwd, SURVEY.md §8d) x N / t.

Prints ONE JSON line (rank 0).  See DESIGN.md §Measurement.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

BYTES_FWD, BYTES_BWD = 8, 12          # algorithmic bytes / element (fp32)
METRIC = "fake-quant fwd+bwd GB/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2n", type=int, default=28)
    ap.add_argument("--channels", type=int, default=512, help="0 = per-tensor activation style")
    ap.add_argument("--bits", type=int, default=4)
    ap.add_argument("--method", default="STE", choices=["STE", "LSQ", "AEWGS", "EWGS"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sweep", action="store_true", help="also run the config-2 sweep -> gpurun_out/")
    ap.add_argument("--cpu-log2n", type=int, default=26,
                    help="elements per step of the CPU reference sample (SURVEY.md §8d: N capped at 2^26)")
    ap.add_argument("--no-resnet", action="store_true", help="skip the QAT legs (configs[2..4])")
    ap.add_argument("--qat-legs", default="resnet18,resnet20,rfdn",
                    help="which QAT legs the default line carries: resnet18 = configs[3] STE W4A4 b256, "
                         "resnet20 = configs[2] AEWGS W1A1 b256, rfdn = configs[4] LSQ W2A2 b16")
    ap.add_argument("--no-graph-microbench", action="store_true",
                    help="launch the microbench step from Python instead of replaying its CUDA graph")
    ap.add_argument("--resnet-batch", type=int, default=None, help="override the per-GPU batch of the QAT legs")
    ap.add_argument("--resnet-steps", type=int, default=12)
    ap.add_argument("--qat-model", default=None, choices=["resnet18", "resnet20", "rfdn"],
                    help="run ONE custom QAT leg instead of --qat-legs (combine with --qat-method / --qat-bits)")
    ap.add_argument("--qat-method", default=None, choices=["STE", "LSQ", "AEWGS", "EWGS"])
    ap.add_argument("--qat-bits", type=int, default=None)
    ap.add_argument("--ddp-reference-flags", action="store_true",
                    help="N > 1: run the main QAT legs with the reference Trainer's flags (SyncBatchNorm, "
                         "find_unused_parameters=True, buffer broadcast; training/trainer.py:88-97,166), eagerly "
                         "launched, instead of the lean graph-captured wrapping.  (The default N > 1 line carries "
                         "one such ResNet-18 row beside the lean one.)")
    ap.add_argument("--graph", action="store_true", default=True, help=argparse.SUPPRESS)
    ap.add_argument("--no-graph", dest="graph", action="store_false",
                    help="QAT leg: launch the training step eagerly from Python.  Default: the whole step "
                         "(teacher+student forward, loss, backward, DDP all-reduces, RAdam) is captured "
                         "once in a CUDA graph and replayed")
    ap.add_argument("--nchw", dest="channels_last", action="store_false",
                    help="QAT leg: keep model and batch in row-major NCHW (the reference Trainer's layout). "
                         "Default is torch.channels_last (NHWC): cuDNN's Blackwell convolution / batch-norm "
                         "kernels are NHWC-native (NCHW costs ~8 ms of layout transposes and 2x slower BN per "
                         "step), and the fake-quant kernels walk dense NHWC storage directly, no copies")
    ap.add_argument("--no-eager-ref", action="store_true",
                    help="skip timing the reference's ATen chain on the GPU (second denominator)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed microbench steps, write what the last one returned (y, grad_x, grad_scale) "
                         "as DIR/<name>.npy; an output above 2^22 elements is cut to a fixed seeded sample, "
                         "saved flat")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs dumps the outputs of our timed path; it does not apply to --impl reference")
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def workload_name(a):
    lay = f"per-channel [C={a.channels}, N/C]" if a.channels else "per-tensor"
    return (f"configs[1] quantizer microbench: {lay} fp32 N=2^{a.log2n}, {a.method}"
            f"{' (GDNSQ, fused Philox noise)' if a.method == 'STE' else ''}, {a.bits} bits, fwd+bwd")


def make_inputs(a, device, log2n=None):
    """x~N(0,1) seed 0, go~N(0,1) seed 1 (SURVEY.md §8d)."""
    n = 1 << (log2n if log2n is not None else a.log2n)
    gx = torch.Generator(device=device).manual_seed(0)
    gg = torch.Generator(device=device).manual_seed(1)
    if a.channels:
        shape = (a.channels, n // a.channels)
    else:
        shape = (n,)
    x = torch.randn(shape, device=device, generator=gx)
    go = torch.randn(shape, device=device, generator=gg)
    if a.channels:
        mn = x.amin(1, keepdim=True)
        mx = x.amax(1, keepdim=True)
        scale = (mx - mn) / (2 ** a.bits - 1)        # calibration formula, minmaxobserver.py:82
        zp, lo, hi = mn, None, None
    else:
        b = torch.tensor([-2.0], device=device)
        scale = torch.exp2(torch.tensor([2.0 - a.bits], device=device))
        zp, lo, hi = b, b, b + 4.0 - scale
    return x, go, scale, zp, lo, hi


DUMP_SAMPLE = 1 << 22      # elements kept of a larger output: 16 MB of fp32 per output


def dump_outputs(out_dir, arrays):
    """Write each tensor as <out_dir>/<name>.npy in fp32.  One with more than DUMP_SAMPLE elements is
    cut to the flat indices drawn by a CPU generator seeded 0, so that runs with the same arguments,
    and different builds, write the same elements."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(0, t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0))
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


# ---------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons around the timed region (one sample every 20 ms, each
    stamped on arrival; `summary` keeps those from 0.15 s before the region to its end)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def wait_ready(self, timeout=2.0):
        """Block (GPU idle) until the first sample has arrived, so the burst that follows is seen."""
        t = time.perf_counter()
        while self.proc and not self.rows and time.perf_counter() - t < timeout:
            time.sleep(0.01)

    def mark_start(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.1)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        rows = self.rows
        if self.t0 is not None and self.t1 is not None:
            near = [r for r in rows if self.t0 - 0.15 <= r[0] <= self.t1 + 0.06]
            rows = near or rows
        sm, mx, reasons = [], [], set()
        for _, r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


def time_region(fn, steps, sync_dist, per_rank=None):
    """K steps between barrier+synchronize on both sides, CUDA events on the launching stream;
    returns the MAX over ranks (ms for the K steps).  `per_rank`: list that receives every rank's
    own time."""
    import torch.distributed as dist
    torch.cuda.synchronize()
    if sync_dist:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if sync_dist:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if sync_dist:
        t = torch.tensor([ms], device="cuda")
        if per_rank is not None:
            allt = [torch.zeros_like(t) for _ in range(dist.get_world_size())]
            dist.all_gather(allt, t)
            per_rank.extend(float(v.item()) for v in allt)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    elif per_rank is not None:
        per_rank.append(ms)
    return ms


def bench_config(a):
    """The workload description — IDENTICAL in both arms (`--impl ours` / `--impl reference`)."""
    n = 1 << a.log2n
    return {"workload": workload_name(a), "elements_per_gpu": n,
            "layout": [a.channels, n // a.channels] if a.channels else [n],
            "method": a.method, "bits": a.bits, "bytes_per_element": 20,
            "l2": "inputs (1 GiB each at N=2^28) far exceed the 126 MB L2; no flush needed",
            "multi_gpu": "replicas only (independent tensors per GPU, no data-path collective)"}


# ---------------------------------------------------------------------------
QAT_LEGS = {
    "resnet18": dict(model="resnet18", method="STE", bits=4, batch=256, key="resnet18_w4a4_qat"),
    "resnet20": dict(model="resnet20", method="AEWGS", bits=1, batch=256, key="resnet20_aewgs_w1a1_qat"),
    "rfdn": dict(model="rfdn", method="LSQ", bits=2, batch=16, key="rfdn_lsq_w2a2_qat"),
}


def qat_specs(a):
    if a.qat_model:
        spec = dict(QAT_LEGS[a.qat_model])
        names = [a.qat_model]
        QATS = {a.qat_model: spec}
    else:
        names = [n for n in a.qat_legs.split(",") if n]
        QATS = {n: dict(QAT_LEGS[n]) for n in names}
    out = []
    for n in names:
        s = QATS[n]
        if a.qat_method:
            s["method"] = a.qat_method
        if a.qat_bits:
            s["bits"] = a.qat_bits
        if a.resnet_batch:
            s["batch"] = a.resnet_batch
        if (s["model"], s["method"], s["bits"]) != tuple(QAT_LEGS[n][k] for k in ("model", "method", "bits")):
            s["key"] = f"{s['model']}_{s['method'].lower()}_w{s['bits']}a{s['bits']}_qat"
        out.append(s)
    return out


def qat_leg(a, dev, world, rank, use_dist, spec, ref_flags=False, profile_share=True):
    """One QAT leg (BASELINE configs[2..4]) through Quantizer(config)().quantize(lmodel) and the
    patched training_step: synthetic batch per GPU, RAdam, fp32 + TF32 convolutions, DDP over NCCL
    for N > 1.  configs[3]: torchvision ResNet-18, 224x224, GDNSQ/STE W4A4 per-channel, Symmetrical-KL
    distillation from a frozen FP copy.  configs[2]: CIFAR ResNet-20 (100 classes), AEWGS W1A1 (the
    config with a data-path collective: AEWGS's in-backward statistics all-reduce).  configs[4]: RFDN
    x4 on 256x256 LR patches, LSQ W2A2, L1, no teacher.  `ref_flags`: the reference Trainer's DDP
    flags (SyncBatchNorm, find_unused_parameters=True, buffer broadcast), eagerly launched."""
    from mhaq_b200 import harness, ops
    torch.backends.cudnn.benchmark = True
    torch.set_float32_matmul_precision("high")
    model_name, method, bits, B = spec["model"], spec["method"], spec["bits"], spec["batch"]
    graph = a.graph and not ref_flags
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    sr = model_name == "rfdn"
    if sr:      # LR patch in [0,1] (denormalised x255 inside the module), HR target x4
        x = torch.rand(B, 3, 256, 256, device=dev, generator=g)
        t = torch.rand(B, 3, 1024, 1024, device=dev, generator=g)
        q = harness.build_qat("rfdn", dev, qnmethod=method, act_bit=bits, weight_bit=bits,
                              distillation=False, lr=5e-4, calib_batch=x[: min(B, 4)], calib_bits=bits)
    else:
        side, classes = (224, 1000) if model_name == "resnet18" else (32, 100)
        x = torch.randn(B, 3, side, side, device=dev, generator=g)
        t = torch.randint(0, classes, (B,), device=dev, generator=g)
        q = harness.build_qat(model_name, dev, qnmethod=method, act_bit=bits, weight_bit=bits,
                              distillation=True, num_classes=classes, calib_batch=x[: min(B, 64)])
    if a.channels_last:
        q.model.to(memory_format=torch.channels_last)
        if getattr(q, "tmodel", None) is not None:
            q.tmodel.to(memory_format=torch.channels_last)
        x = x.contiguous(memory_format=torch.channels_last)
    if use_dist:
        if ref_flags:      # training/trainer.py:88,166 (sync_batchnorm=True) and :92-97
            q.model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(q.model)
            if a.channels_last:
                q.model.to(memory_format=torch.channels_last)
        wrap = harness.ddp_side_stream if graph else harness.wrap_ddp
        q.model = wrap(q.model, dev, lean=not ref_flags)
    q.train(); q.wrapped_criterion.train()
    if getattr(q, "tmodel", None) is not None:
        q.tmodel.eval()
    opt = q.configure_optimizers()

    def eager_step(batch=None):
        loss = q.training_step(batch or (x, t), 0)
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss.detach()

    res = {}
    k = a.resnet_steps
    if use_dist and method == "AEWGS":
        # the ONE data-path collective (gdnsq.py:126-129, here one packed all-reduce per weight
        # tensor): its GPU time per step, CUDA events around every call over 3 eager DDP steps
        evs, orig = [], ops.allreduce_packed_stats

        def timed_allreduce(stats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = orig(stats)
            e1.record()
            evs.append((e0, e1))
            return out

        for _ in range(2):
            eager_step()
        ops.allreduce_packed_stats = timed_allreduce
        try:
            for _ in range(3):
                eager_step()
            torch.cuda.synchronize()
        finally:
            ops.allreduce_packed_stats = orig
        tot = sum(e0.elapsed_time(e1) for e0, e1 in evs)
        res["aewgs_stats_allreduce"] = {"calls_per_step": len(evs) // 3, "ms_per_step": round(tot / 3, 3),
                                        "what": "the path's one collective: packed [3, rows] AVG all-reduce between the "
                                                "statistics and the apply kernel — ONE per step for all conv weights of the "
                                                "model (the reference: 3 per weight tensor).  Stream time between CUDA events "
                                                "recorded right before and after the call in eager DDP steps: NCCL launch + "
                                                "transfer + waiting for the slowest rank to reach this point of its backward"}

    # The headline (graph-replayed step) is measured FIRST, on a GPU that has not yet been pushed
    # into its power cap by the eager / profiler passes below (sustained load lowers the SM clock).
    graphed = None
    if graph:
        # capture; if it fails on ANY rank every rank falls back to eager launches (the bench
        # line must not depend on a capture succeeding) and says so
        note = None
        try:
            graphed = harness.GraphedTrainStep(q, (x, t), seed=1234 + rank)
        except Exception as exc:
            note = f"{type(exc).__name__}: {str(exc)[:160]}"
        ok = torch.tensor([0 if graphed is None else 1], device=dev)
        if use_dist:
            import torch.distributed as dist
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            if graphed is not None:
                graphed.close()
            graphed = None
            ops.set_device_philox_state(None)
            torch.cuda.synchronize()
            opt = q.configure_optimizers()
            res["graph_capture_failed"] = note or "capture failed on another rank"
    step = graphed if graphed is not None else eager_step

    # end to end: every step's batch comes from pinned host memory (H2D inside the timed region,
    # double-buffered on a copy stream so the copy of batch k+1 overlaps step k) and the step's
    # loss is read back to the host
    hx = x.cpu().pin_memory(); ht = t.cpu().pin_memory()      # (keeps x's memory format)
    hloss = torch.empty((), dtype=torch.float32).pin_memory()
    feed = harness.BatchPrefetcher((x, t))
    feed.put((hx, ht))

    def step_e2e():
        batch = feed.get()
        feed.put((hx, ht))                  # next step's copy, in flight while this step computes
        hloss.copy_(step(batch), non_blocking=True)
        feed.release()

    for _ in range(4):
        step()
    ranks_ms = []
    ms = time_region(step, k, use_dist, per_rank=ranks_ms) / k
    ke = max(3, k // 2)
    step_e2e()
    ms_e = time_region(step_e2e, ke, use_dist) / ke
    if graphed is not None:
        graphed.close()
        graphed = None
        graph_was_used = True
        torch.cuda.synchronize()
        opt = q.configure_optimizers()
    else:
        graph_was_used = False
    if graph and not use_dist:
        # the same step launched eagerly from Python first: its time, and (CUPTI) which share of
        # the GPU time the fake-quant kernels take — a graph replay hides kernel names from CUPTI
        for _ in range(4):
            eager_step()
        res["eager_ms_per_step"] = round(time_region(eager_step, k, False) / k, 2)
    if rank == 0 and not use_dist and profile_share:   # (a rank-local DDP step would dead-lock the other ranks)
        try:
            from torch.profiler import profile, ProfilerActivity
            eager_step()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                eager_step(); eager_step()
                torch.cuda.synchronize()
            tot = fq = 0.0
            nl = nfq = 0
            for ev in prof.key_averages():
                dt = getattr(ev, "device_time_total", 0.0) or getattr(ev, "cuda_time_total", 0.0)
                if dt <= 0:
                    continue                 # host-side runtime-API records: not GPU work
                tot += dt
                nl += ev.count
                if "fq_" in ev.key:
                    fq += dt
                    nfq += ev.count
            if tot > 0:
                res["fake_quant_kernel_share"] = round(fq / tot, 4)
                res["fake_quant_ms_per_step"] = round(fq / 2 / 1e3, 3)
                res["gpu_kernel_ms_per_step"] = round(tot / 2 / 1e3, 2)   # rest of an eager step = GPU idle
                res["launches_per_step"] = nl // 2
                res["fake_quant_launches_per_step"] = nfq // 2
        except Exception as exc:   # profiler unavailable: the throughput numbers stand alone
            res["fake_quant_kernel_share"] = None
            res["profiler_error"] = str(exc)[:80]
    cfg = {"resnet18": "configs[3] ResNet-18 224x224", "resnet20": "configs[2] ResNet-20 32x32 (CIFAR-100 shaped)",
           "rfdn": "configs[4] RFDN x4 SR, 256x256 LR patches, L1"}[model_name]
    par = "single GPU"
    if use_dist:
        par = f"DDP dp{world}" + (", reference Trainer flags: SyncBatchNorm + find_unused_parameters=True + buffer "
                                  "broadcast" if ref_flags else ", lean wrapping (log_b_s ignored, no buffer broadcast)")
    res = {"workload": f"{cfg} {method} W{bits}A{bits} QAT, {'no teacher' if sr else 'distillation'}, RAdam, fp32/TF32, "
                       f"batch {B}/GPU, {'channels_last' if a.channels_last else 'NCHW'}, {par}, "
                       f"{'whole step (NCCL all-reduces included) replayed from a CUDA graph' if graph_was_used else 'eager launches'}",
           "img_per_s": round(world * B / (ms * 1e-3), 1), "ms_per_step": round(ms, 2),
           "e2e_img_per_s": round(world * B / (ms_e * 1e-3), 1),
           "e2e_h2d_bytes_per_step": hx.numel() * hx.element_size() + ht.numel() * ht.element_size(),
           "n_gpus": world,
           "quantized_act_elems_per_step": {"resnet18": 1680896, "resnet20": 184320, "rfdn": 59093392}[model_name] * B,
           **res}
    if use_dist:   # replicas must hold identical parameters after the DDP steps
        import torch.distributed as dist
        rm = sorted(v / k for v in ranks_ms)
        res["per_rank_ms_per_step"] = {"min": round(rm[0], 3), "median": round(rm[len(rm) // 2], 3), "max": round(rm[-1], 3)}
        chk = torch.stack([p.detach().double().sum() for p in q.model.parameters()]).sum().reshape(1)
        lo_, hi_ = chk.clone(), chk.clone()
        dist.all_reduce(lo_, op=dist.ReduceOp.MIN); dist.all_reduce(hi_, op=dist.ReduceOp.MAX)
        res["ddp_replicas_in_sync"] = bool((lo_ == hi_).item())
    del q, graphed, step, feed
    torch.cuda.empty_cache()
    return res


def host_link_probe(dev, use_dist):
    """What bounds the host-buffer e2e leg: pinned-host <-> device copy bandwidth of THIS rank with every
    rank copying at the same time (H2D alone, D2H alone, both directions at once) and a plain host
    memcpy, 256 MiB buffers."""
    n = 64 << 20
    h_in = torch.empty(n, dtype=torch.float32).pin_memory()
    h_out = torch.empty(n, dtype=torch.float32).pin_memory()
    d_in, d_out = torch.empty(n, device=dev), torch.empty(n, device=dev)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    by = 4 * n

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        if use_dist:
            import torch.distributed as dist
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps

    def both():
        with torch.cuda.stream(s1):
            d_in.copy_(h_in, non_blocking=True)
        with torch.cuda.stream(s2):
            h_out.copy_(d_out, non_blocking=True)

    t_h2d = timed(lambda: d_in.copy_(h_in, non_blocking=True))
    t_d2h = timed(lambda: h_out.copy_(d_out, non_blocking=True))
    t_both = timed(both)
    t0 = time.perf_counter()
    for _ in range(2):
        h_out.copy_(h_in)
    t_mem = (time.perf_counter() - t0) / 2
    return {"h2d_GBps": round(by / t_h2d / 1e9, 1), "d2h_GBps": round(by / t_d2h / 1e9, 1),
            "duplex_each_way_GBps": round(by / t_both / 1e9, 1), "host_memcpy_GBps": round(2 * by / t_mem / 1e9, 1),
            "what": "this rank's pinned-host<->device copies with all ranks copying concurrently; host_memcpy = "
                    "one thread's read+write bytes/s"}


# ---------------------------------------------------------------------------
def run_ours(a):
    import mhaq_b200
    from mhaq_b200 import ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    use_dist = world > 1
    if use_dist:
        import torch.distributed as dist
        import datetime
        if a.graph:   # torch's recipe for capturing DDP's NCCL all-reduces in a CUDA graph
            os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    n = 1 << a.log2n
    x, go, scale, zp, lo, hi = make_inputs(a, dev)
    lo_ = -math.inf if lo is None else lo
    hi_ = math.inf if hi is None else hi
    scale_p = scale.clone().requires_grad_(True)
    launches = {"n": 0}
    # launches of OUR kernels per step: forward + backward (+ finalize when it is a separate launch)
    # (+ AEWGS statistics kernel and its finalize)
    per_step_launches = ops.launches_per_fwd_bwd(x, scale, zp, lo_, hi_, a.method)
    keep = {}

    def eager_body():
        xs = x.detach().requires_grad_(True)
        scale_p.grad = None
        y = mhaq_b200.fake_quant(xs, scale_p, zp, lo_, hi_, method=a.method)
        y.backward(go)
        keep["out"] = (y, xs.grad, scale_p.grad)

    # The step is captured ONCE in a CUDA graph and replayed: with 8 processes on one host the
    # Python launch path of a 0.8 ms step is exposed to host jitter (round 1: one straggler rank
    # cost 6.5 % at N=8 in a 16 ms timed window); a replay is one cudaGraphLaunch per step.
    # The in-kernel noise reads a device-resident Philox state advanced inside the graph, so every
    # replay draws fresh noise, exactly like the eager step does from torch's generator.
    # clocks / throttle reasons: the sampler (nvidia-smi needs ~0.1 s to start) runs from before the
    # capture to the end of the timed region; the summary keeps the samples around the timed region.
    # The timed region is a BURST — W warm-up replays, then K timed ones, ~20 ms in all: the same regime
    # as MEASURED_PEAKS.json's `hbm_gbs` (best of 10 copies).  Seconds of back-to-back replays run into
    # the 1 kW power cap (sw_power_cap, SM clock ~1.65 GHz) and lose ~3 %.
    with ClockSampler(local) as cs:
        cs.wait_ready()
        graph_note = None
        graph = None
        if not a.no_graph_microbench:
            try:
                state = torch.tensor([1234 + rank, 0], dtype=torch.int64, device=dev)
                ops.set_device_philox_state(state)

                def graph_body():
                    ops.reset_philox_call_counter()
                    state[1] += 16
                    eager_body()

                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for _ in range(3):
                        graph_body()
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                keep.clear()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    graph_body()
            except Exception as exc:
                graph, graph_note = None, f"{type(exc).__name__}: {str(exc)[:120]}"
                ops.set_device_philox_state(None)
                torch.cuda.synchronize()

        def step():
            if graph is not None:
                graph.replay()
            else:
                eager_body()
            launches["n"] += per_step_launches

        n_warm = 0
        for _ in range(max(a.warmup, 3)):
            step()
            n_warm += 1
        launches["n"] = 0                   # gpu_launches counts the timed region only
        ranks_ms = []
        cs.mark_start()
        ms = time_region(step, a.steps, use_dist, per_rank=ranks_ms)
        cs.mark_end()
    clocks = cs.summary()
    clocks["window"] = f"from 0.15 s before the timed region ({n_warm} warm-up steps) to its end"
    n_l = launches["n"]
    per_step = ms / a.steps
    gbs = world * (BYTES_FWD + BYTES_BWD) * n / (per_step * 1e-3) / 1e9
    if a.dump_outputs and rank == 0:
        # the last timed step's outputs (a replayed graph rewrites the tensors its capture kept)
        y, gx, gs = keep["out"]
        dump_outputs(a.dump_outputs, {"y": y, "grad_x": gx, "grad_scale": gs})
    if graph is not None:
        del graph
        ops.set_device_philox_state(None)
    keep.clear()

    out = None
    if rank == 0:
        peak, peak_src = peaks()
        # ---- per-kernel roofline, measured live with CUDA events on the launch stream ----
        L = ops._Launch(x.detach(), scale, zp, lo_, hi_)
        xd = x.detach()

        def fwd_only():
            ops._forward_impl(xd, L, True, False, False)

        def bwd_only():
            ops._backward_impl(go, xd, L, ops._method_id(a.method), False, None, True, philox=(1, 2))

        for f in (fwd_only, bwd_only):
            for _ in range(3):
                f()
        k = max(a.steps, 10)
        t_f = time_region(fwd_only, k, False) / k
        t_b = time_region(bwd_only, k, False) / k
        bwd_bytes = BYTES_BWD + (8 if a.method == "AEWGS" else 0)
        ach_b = bwd_bytes * n / (t_b * 1e-3) / 1e9
        ach_f = BYTES_FWD * n / (t_f * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("fq_bwd_kernel_bytes_per_launch")
            except Exception:
                traffic = None
        roofline = {"bound": "hbm", "kernel": "fq_bwd_kernel (+ deterministic finalize)", "achieved": round(ach_b, 1),
                    "peak": peak, "unit": "GB/s", "frac": round(ach_b / peak, 4), "traffic": traffic,
                    "peak_source": peak_src, "frac_of_8TBps_nominal": round(ach_b / 8000.0, 4),
                    "bytes_per_elem": bwd_bytes, "ms_per_launch": round(t_b, 4),
                    "fwd_kernel": {"achieved": round(ach_f, 1), "frac": round(ach_f / peak, 4),
                                   "bytes_per_elem": BYTES_FWD, "ms_per_launch": round(t_f, 4)}}
        rm = sorted(v / a.steps for v in ranks_ms)
        out = {"metric": METRIC, "value": round(gbs, 1), "unit": "GB/s", "n_gpus": world,
               "steps": a.steps, "warmup": max(a.warmup, 3), "warmup_actual": n_warm,
               "ms_per_step": round(per_step, 4),
               "per_rank_ms_per_step": {"min": round(rm[0], 4), "median": round(rm[len(rm) // 2], 4),
                                        "max": round(rm[-1], 4)},
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
               "data": "synthetic", "impl": "ours",
               "config": bench_config(a),
               "launch": ("step captured once in a CUDA graph and replayed (one cudaGraphLaunch per step; noise from a "
                          "device-resident Philox state advanced inside the graph)" if graph_note is None and
                          not a.no_graph_microbench else f"eager Python launches ({graph_note or '--no-graph-microbench'})"),
               "frac_of_hbm_peak": round(gbs / world / peak, 4),
               "roofline": roofline, "clocks": clocks, "gpu_launches": n_l}

    # ---- end to end through the public API with HOST buffers -------------------------
    if not a.no_e2e:
        try:
            from mhaq_b200.host import fake_quant_fwd_bwd_host
            hx = torch.empty(x.shape, dtype=torch.float32).pin_memory()
            hg = torch.empty(x.shape, dtype=torch.float32).pin_memory()
            hx.copy_(x.detach()); hg.copy_(go)
            hy = torch.empty(x.shape, dtype=torch.float32).pin_memory()
            hgx = torch.empty(x.shape, dtype=torch.float32).pin_memory()
            hgs = torch.empty(scale.shape, dtype=torch.float32).pin_memory()
            del x, go                       # the e2e leg owns its (staged) device memory
            torch.cuda.empty_cache()

            def e2e_step():
                _, _, grads = fake_quant_fwd_bwd_host(hx, hg, scale, zp, lo, hi, method=a.method,
                                                      y_host=hy, gx_host=hgx, chunks=16)
                hgs.copy_(grads["scale"], non_blocking=True)

            ke = max(3, min(a.steps, 5))
            for _ in range(2):
                e2e_step()
            ms_e = time_region(e2e_step, ke, use_dist) / ke
            link = host_link_probe(dev, use_dist)
            if rank == 0:
                by_way = 2 * 4 * n
                floor_ms = by_way / (link["duplex_each_way_GBps"] * 1e9) * 1e3
                out["e2e"] = {"value": round(world * 20 * n / (ms_e * 1e-3) / 1e9, 2), "unit": "GB/s",
                              "h2d_bytes_per_step": by_way, "d2h_bytes_per_step": by_way + 4 * scale.numel(),
                              "ms_per_step": round(ms_e, 3), "steps": ke,
                              "api": "mhaq_b200.host.fake_quant_fwd_bwd_host: pinned host x/go in, y/gx/g_scale out, "
                                     "16 row chunks pipelined over full-duplex PCIe (copies inside the timed region)",
                              "host_link": link,
                              "bound": f"host link, not the GPU: {by_way / 2**30:.0f} GiB each way per step per rank at the measured "
                                       f"{link['duplex_each_way_GBps']} GB/s each way (all {world} rank(s) copying at once) = "
                                       f"{floor_ms:.1f} ms of copies vs {ms_e:.1f} ms measured; the kernels need "
                                       f"{per_step:.2f} ms.  All ranks share one host's DRAM / PCIe root complexes, so the "
                                       "aggregate does not scale with the GPU count"}
            del hx, hg, hy, hgx
        except Exception as exc:       # e.g. the box refuses 4 GiB of pinned host memory
            if use_dist:
                raise
            if rank == 0:
                out["e2e"] = {"value": None, "unit": "GB/s", "error": f"{type(exc).__name__}: {str(exc)[:200]}"}

    x = go = None
    torch.cuda.empty_cache()
    if not a.no_resnet:
        for spec in qat_specs(a):
            try:
                rn = qat_leg(a, dev, world, rank, use_dist, spec, ref_flags=a.ddp_reference_flags)
            except Exception as exc:       # a QAT leg must never take the headline line down with it
                if use_dist:
                    raise
                rn = {"error": f"{type(exc).__name__}: {str(exc)[:200]}"}
                torch.cuda.empty_cache()
            if rank == 0:
                out[spec["key"]] = rn
        if use_dist and not a.ddp_reference_flags and not a.qat_model and "resnet18" in a.qat_legs:
            # the same ResNet-18 step the way the reference's Trainer wraps it (trainer.py:88-97,166)
            rn = qat_leg(a, dev, world, rank, use_dist, dict(QAT_LEGS["resnet18"]), ref_flags=True)
            if rank == 0:
                out["resnet18_w4a4_qat_reference_trainer_flags"] = rn
    if rank == 0:
        if not a.no_eager_ref:
            # the honest speed-up denominators: the LIVE reference run eagerly on this GPU
            try:
                from oracle import ref_bench
                b = argparse.Namespace(**vars(a))
                b.log2n = min(a.log2n, 26)
                out["reference_eager_gpu"] = ref_bench.eager_gpu_microbench(make_inputs(b, dev), a.method, b.log2n)
                torch.cuda.empty_cache()
                if not a.no_resnet and not use_dist and any(s["model"] == "resnet18" for s in qat_specs(a)):
                    B = a.resnet_batch or 256
                    for cl in ((False, True) if a.channels_last else (False,)):
                        key = "resnet18_w4a4_qat" + ("_channels_last" if cl else "")
                        try:
                            out["reference_eager_gpu"][key] = ref_bench.eager_gpu_resnet18_step(B, cl)
                        except Exception as exc:
                            out["reference_eager_gpu"][key] = {"error": f"{type(exc).__name__}: {str(exc)[:200]}"}
                            torch.cuda.empty_cache()
            except Exception as exc:
                out["reference_eager_gpu"] = {"error": f"{type(exc).__name__}: {str(exc)[:200]}"}
        if not a.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(a, steps=5, warmup=2)
        if a.sweep:
            sweep(a, dev)
        emit(out)
    if use_dist:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------
def cpu_baseline(a, steps, warmup):
    """The reference's CPU quantizer path on the host cores: the LIVE reference (oracle/_ref)
    when staged, else the oracle port (`kind` says which)."""
    from oracle import ref_bench
    log2n = min(a.cpu_log2n, a.log2n)
    return ref_bench.cpu_microbench(make_inputs(a, "cpu", log2n), a.method, steps, warmup, log2n, a.log2n)


def run_reference(a):
    """`--impl reference`: the reference's own CPU implementation of the path, all host threads,
    same metric / config / steps / warm-up as our arm; each step is a bounded sample (N = 2^26 of
    the workload's 2^28 elements, SURVEY.md §8d) so the run ends within a few minutes.  This
    process never imports mhaq_b200 (nothing of the product is loaded)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_bench
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cb = cpu_baseline(a, steps=max(1, a.steps), warmup=max(0, a.warmup))
    out = {"metric": METRIC, "value": cb["value"], "unit": "GB/s", "n_gpus": world, "steps": a.steps,
           "warmup": a.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
           "config": bench_config(a),
           "note": "GB/s is size-normalised (20 B/element x elements / time); see cpu_baseline.sample for the sample",
           "cpu_baseline": cb,
           "e2e": {"value": cb["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "product_modules_loaded": sorted(m for m in sys.modules if m.startswith("mhaq_b200"))}
    if not a.no_resnet:
        try:
            out["cpu_config0_step"] = ref_bench.config0_step()
        except Exception as exc:   # never let the extra leg break the contract line
            out["cpu_config0_step"] = {"error": f"{type(exc).__name__}: {str(exc)[:160]}"}
    emit(out)


# ---------------------------------------------------------------------------
def sweep(a, dev):
    """BASELINE config 2: N in 2^20..2^30, layouts, methods, bits.  Writes gpurun_out/sweep.json."""
    import mhaq_b200
    from mhaq_b200 import ops
    peak, _ = peaks()
    rows = []
    for log2n in (20, 22, 24, 26, 28, 30):
        for ch in (0, 64, 512, 4096):
            for method in ("STE", "LSQ", "AEWGS"):
                if method == "AEWGS" and ch == 0:
                    continue
                for bits in ((4,) if log2n != 28 else (1, 2, 4, 8)):
                    b = argparse.Namespace(**vars(a))
                    b.log2n, b.channels, b.method, b.bits = log2n, ch, method, bits
                    try:
                        x, go, scale, zp, lo, hi = make_inputs(b, dev)
                    except torch.OutOfMemoryError:
                        continue
                    n = 1 << log2n
                    lo_ = -math.inf if lo is None else lo
                    hi_ = math.inf if hi is None else hi
                    L = ops._Launch(x, scale, zp, lo_, hi_)
                    mid = ops._method_id(method)
                    f = lambda: ops._forward_impl(x, L, True, False, False)
                    g = lambda: ops._backward_impl(go, x, L, mid, False, None, True, philox=(1, 2))
                    reps = 20 if log2n <= 28 else 5
                    res = {}
                    # tensors that fit the 126 MB L2 are evicted between iterations by a 256 MB
                    # write; its own time is measured the same way and subtracted.  Launches are
                    # enqueued back to back so the figure is GPU time, not host launch latency.
                    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev) if log2n <= 24 else None

                    def timed(body):
                        for _ in range(3):
                            body()
                        torch.cuda.synchronize()
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        if log2n <= 24:
                            # short kernels: `reps` calls captured into ONE CUDA graph, so the figure is
                            # what a graph-captured training step pays — no Python launch latency in it
                            side = torch.cuda.Stream()
                            side.wait_stream(torch.cuda.current_stream())
                            with torch.cuda.stream(side):
                                body()
                            torch.cuda.current_stream().wait_stream(side)
                            gr = torch.cuda.CUDAGraph()
                            with torch.cuda.graph(gr):
                                for _ in range(reps):
                                    body()
                            gr.replay()
                            torch.cuda.synchronize()
                            ts = []
                            for _ in range(5):
                                e0.record()
                                gr.replay()
                                e1.record()
                                torch.cuda.synchronize()
                                ts.append(e0.elapsed_time(e1) / reps)
                            del gr
                            return sorted(ts)[len(ts) // 2]
                        e0.record()
                        for _ in range(reps):
                            body()
                        e1.record()
                        torch.cuda.synchronize()
                        return e0.elapsed_time(e1) / reps

                    ev = lambda: ops._forward_impl(x, L, True, False, True)      # eval: + code / input min-max
                    t_flush = timed(lambda: flush.zero_()) if flush is not None else 0.0
                    for nm, fn, by in (("fwd", f, 8), ("eval", ev, 8), ("bwd", g, 12 + (8 if method == "AEWGS" else 0))):
                        if flush is not None:
                            med = max(timed(lambda: (flush.zero_(), fn())) - t_flush, 1e-6)
                        else:
                            med = timed(fn)
                        res[nm] = {"ms_median": round(med, 5), "GBps": round(by * n / med / 1e6, 1),
                                   "frac": round(by * n / med / 1e6 / peak, 4)}
                    tot = res["fwd"]["ms_median"] + res["bwd"]["ms_median"]
                    by = 20 + (8 if method == "AEWGS" else 0)
                    rows.append({"log2n": log2n, "channels": ch, "method": method, "bits": bits, **res,
                                 "fwd_bwd_GBps": round(by * n / tot / 1e6, 1),
                                 "fwd_bwd_frac": round(by * n / tot / 1e6 / peak, 4)})
                    print("sweep", json.dumps(rows[-1]), file=sys.stderr, flush=True)
                    del x, go, L
                    torch.cuda.empty_cache()
    os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
    json.dump({"peak_GBps": peak, "rows": rows}, open(os.path.join(ROOT, "gpurun_out", "sweep.json"), "w"), indent=1)


_JSON_FD = None


def _claim_stdout():
    """ONE JSON line on stdout: NCCL (NCCL_DEBUG=VERSION/INFO) and other native libraries print
    to fd 1; keep a private copy of the real stdout for the JSON line and point fd 1 at stderr."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, line)


def main():
    a = parse_args()
    _claim_stdout()
    if a.impl == "reference":
        run_reference(a)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                             "(use --impl reference for the CPU baseline)")
        run_ours(a)


if __name__ == "__main__":
    main()
