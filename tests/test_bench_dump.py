"""bench.py --dump-outputs: the last timed step's outputs as .npy files, the same from run to run, so
that two builds can be compared output for output."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_keeps_small_outputs_and_samples_large_ones_alike(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    big, small = torch.randn(40, 100), torch.randn(40, 1)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small})
    a = np.load(tmp_path / "a" / "big.npy")
    assert a.shape == (1000,) and a.dtype == np.float32
    assert np.isin(a, big.numpy()).all()
    assert np.array_equal(a, np.load(tmp_path / "b" / "big.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "small.npy"), small.numpy())


def _bench(tmp_path, tag, *extra):
    d = tmp_path / tag
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--warmup", "2",
                          "--log2n", "16", "--channels", "64", "--no-e2e", "--no-cpu-baseline", "--no-resnet",
                          "--no-eager-ref", *extra, "--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert out.returncode == 0, out.stderr[-2000:]
    json.loads(out.stdout.strip().splitlines()[-1])
    return {n: np.load(d / f"{n}.npy") for n in ("y", "grad_x", "grad_scale")}


@pytest.mark.gpu
def test_bench_dumps_what_its_last_timed_step_computed(tmp_path):
    import mhaq_b200
    from oracle import checks as C
    from oracle import fq_oracle as O
    from tests.test_gpu_live_reference import _exact_per_channel, _exact_per_channel_aewgs
    ste = [_bench(tmp_path, f"ste{k}", "--steps", "3") for k in range(2)]
    for n in ste[0]:
        assert np.array_equal(ste[0][n], ste[1][n]), n
    aewgs = _bench(tmp_path, "aewgs", "--steps", "5", "--method", "AEWGS")
    x, go, scale, zp, _, _ = bench.make_inputs(argparse.Namespace(log2n=16, channels=64, bits=4), "cuda")
    n_inner = x.shape[1]
    for method, steps, got in (("STE", 3, ste[0]), ("AEWGS", 5, aewgs)):
        # the replayed step draws its noise from the device state (seed 1234, stream base advanced by
        # 16 per step): 3 runs before the capture, max(--warmup, 3) warm-up replays, then the timed
        # ones — so the last timed step's stream tells how many steps ran
        r = mhaq_b200.philox_noise(x, scale, seed=1234, offset=16 * (3 + 3 + steps))
        xs, sp = x.clone().requires_grad_(True), scale.clone().requires_grad_(True)
        y = O.fake_quant(xs, sp, zp, method=method, noise=r)
        y.backward(go)
        assert np.array_equal(got["y"], y.detach().cpu().numpy()), method
        gx, gs = torch.from_numpy(got["grad_x"]), torch.from_numpy(got["grad_scale"])
        if method == "AEWGS":
            C.assert_close_rel(gx, xs.grad, 1e-5, "grad_x AEWGS", abs_floor=1e-7)
            exact, floor = _exact_per_channel_aewgs(x, go, scale, zp, r)[0], 2.0 ** -20 * n_inner ** 0.5
        else:
            C.assert_bit_exact(gx, xs.grad, "grad_x STE")
            exact, floor = _exact_per_channel(x, go, scale, zp, method, r)[0], 4e-7 * n_inner ** 0.5
        C.assert_param_grad(gs, sp.grad, exact, 1e-5, f"grad_scale {method}", floor)
