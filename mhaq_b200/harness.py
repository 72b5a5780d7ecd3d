"""Minimal stand-in for the Lightning side of the reference, used by the benchmarks and tests.

Lightning, torchmetrics and pytorchcv are absent from this image (and the GPU box has no
network), so ``Trainer.fit`` cannot run here.  This module mirrors only what the hot path
needs from it, in the same order Lightning executes it:

* ``LModule``  — the attributes/methods ``GDNSQQuant.quantize`` touches on a
  ``LVisionCls`` (reference src/models/compose/vision/vision_cls_module.py:10-93);
* ``make_config`` — the ``config.quantization`` tree of the YAML configs;
* ``calibrate`` — the effect of ``Trainer.calibrate`` (training/trainer.py:187-223,
  calib/minmaxobserver.py:39-88) from one batch;
* ``fit_steps`` — forward → loss → backward → optimizer step, optionally under
  ``DistributedDataParallel`` (one process per GPU, NCCL), the strategy the reference's
  ``Trainer`` picks (training/trainer.py:92-97).

With Lightning installed the real ``Trainer.fit`` drives the same quantized module.
"""
from __future__ import annotations

from types import SimpleNamespace
from typing import Callable, Dict, List, Optional

import torch
import torch.nn.functional as F
from torch import nn



class LModule(nn.Module):
    """Duck-typed LightningModule: model + criterion + optimizer factory + log sink."""

    def __init__(self, model: nn.Module, criterion: Callable, optimizer=torch.optim.RAdam,
                 lr: float = 3e-4):
        super().__init__()
        self.model = model
        self.criterion = criterion
        self.optimizer = optimizer
        self.lr = lr
        self.metrics: List = []
        self.logged: Dict[str, object] = {}
        self.trainer = SimpleNamespace(logged_metrics={})

    # Lightning's self.log(..., sync_dist=True) all-reduces one scalar per call; here the
    # values are kept on the device and never synchronised inside the step (SURVEY.md §2c).
    def log(self, name, value, **kw):
        self.logged[name] = value.detach() if torch.is_tensor(value) else value

    def configure_optimizers(self):
        return self.optimizer([p for p in self.parameters() if p.requires_grad], self.lr)

    def forward(self, inputs):
        return self.model(inputs)

    def training_step(self, batch, batch_idx):
        inputs, target = batch
        loss = self.criterion(self.model(inputs), target)
        self.log("loss", loss)
        return loss

    def validation_step(self, batch, batch_idx):
        inputs, target = batch
        return self.criterion(self.forward(inputs), target)

    def test_step(self, batch, batch_idx):
        return self.validation_step(batch, batch_idx)

    def predict_step(self, batch, batch_idx=0):
        inputs = batch[0] if isinstance(batch, (tuple, list)) else batch
        return self.forward(inputs)


def make_config(act_bit=4, weight_bit=4, qscheme=1, qnmethod="STE", excluded_layers=(),
                distillation=False, distillation_loss="Symmetrical KL", quantize_bias=False,
                freeze_batchnorm=False, fuse_batchnorm=False, name="GDNSQQuant"):
    """`config.quantization` as the YAML loader would build it (config/*.yaml:49-66)."""
    params = SimpleNamespace(distillation=distillation, distillation_loss=distillation_loss,
                             distillation_teacher=None, qnmethod=qnmethod)
    quant = SimpleNamespace(name=name, qscheme=qscheme, act_bit=act_bit, weight_bit=weight_bit,
                            freeze_batchnorm=freeze_batchnorm, fuse_batchnorm=fuse_batchnorm,
                            quantize_bias=quantize_bias, excluded_layers=list(excluded_layers),
                            calibration=SimpleNamespace(act_bit=10, weight_bit=10), params=params)
    return SimpleNamespace(quantization=quant)


# ------------------------------------------------------------------ models
class _CifarBlock(nn.Module):
    """3x3-3x3 residual block with the parameter-free (option A) shortcut."""

    def __init__(self, cin, cout, stride):
        super().__init__()
        self.conv1 = nn.Conv2d(cin, cout, 3, stride, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(cout)
        self.conv2 = nn.Conv2d(cout, cout, 3, 1, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(cout)
        self.pad = (cout - cin) // 2 if (stride != 1 or cin != cout) else None

    def forward(self, x):
        out = F.relu(self.bn1(self.conv1(x)))
        out = self.bn2(self.conv2(out))
        sc = x if self.pad is None else F.pad(x[:, :, ::2, ::2], (0, 0, 0, 0, self.pad, self.pad))
        return F.relu(out + sc)


class CifarResNet(nn.Module):
    """ResNet-20/32/.. for 32x32 inputs (He et al. 2015, 6n+2 layers, 16/32/64 channels) —
    same topology and module names (conv1, layer1..3, linear) as the reference's in-tree
    src/models/cls/resnet/resnet_cifar.py:99-136, so the configs' excluded_layers apply."""

    def __init__(self, n=3, num_classes=10):
        super().__init__()
        self.conv1 = nn.Conv2d(3, 16, 3, 1, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(16)
        cin, layers = 16, []
        for i, (c, s) in enumerate(((16, 1), (32, 2), (64, 2))):
            blocks = []
            for b in range(n):
                blocks.append(_CifarBlock(cin, c, s if b == 0 else 1))
                cin = c
            layers.append(nn.Sequential(*blocks))
        self.layer1, self.layer2, self.layer3 = layers
        self.linear = nn.Linear(64, num_classes)
        for m in self.modules():
            if isinstance(m, (nn.Conv2d, nn.Linear)):
                nn.init.kaiming_normal_(m.weight)

    def forward(self, x):
        out = F.relu(self.bn1(self.conv1(x)))
        out = self.layer3(self.layer2(self.layer1(out)))
        out = F.adaptive_avg_pool2d(out, 1).flatten(1)
        return self.linear(out)


class _Esa(nn.Module):
    """Enhanced spatial attention of RFDN: 1x1 squeeze to n/4 channels, a strided 3x3 + 7x7/3
    max-pool pyramid of three 3x3 convolutions, bilinear upsampling, sigmoid gate."""

    def __init__(self, n):
        super().__init__()
        f = n // 4
        self.conv1 = nn.Conv2d(n, f, 1)
        self.conv_f = nn.Conv2d(f, f, 1)
        self.conv_max = nn.Conv2d(f, f, 3, padding=1)
        self.conv2 = nn.Conv2d(f, f, 3, stride=2, padding=0)
        self.conv3 = nn.Conv2d(f, f, 3, padding=1)
        self.conv3_ = nn.Conv2d(f, f, 3, padding=1)
        self.conv4 = nn.Conv2d(f, n, 1)

    def forward(self, x):
        c1 = self.conv1(x)
        v = F.max_pool2d(self.conv2(c1), kernel_size=7, stride=3)
        v = F.relu(self.conv_max(v))
        v = self.conv3_(F.relu(self.conv3(v)))
        v = F.interpolate(v, (x.size(2), x.size(3)), mode="bilinear", align_corners=False)
        return x * torch.sigmoid(self.conv4(v + self.conv_f(c1)))


class _Rfdb(nn.Module):
    """Residual feature distillation block: three (1x1 distil | 3x3 refine + skip) stages, a
    final 3x3 distil, 1x1 fusion of the four distilled halves, ESA."""

    def __init__(self, n):
        super().__init__()
        d = n // 2
        self.c1_d, self.c1_r = nn.Conv2d(n, d, 1), nn.Conv2d(n, n, 3, padding=1)
        self.c2_d, self.c2_r = nn.Conv2d(n, d, 1), nn.Conv2d(n, n, 3, padding=1)
        self.c3_d, self.c3_r = nn.Conv2d(n, d, 1), nn.Conv2d(n, n, 3, padding=1)
        self.c4 = nn.Conv2d(n, d, 3, padding=1)
        self.c5 = nn.Conv2d(4 * d, n, 1)
        self.esa = _Esa(n)

    def forward(self, x):
        act = lambda t: F.leaky_relu(t, 0.05)
        d1, r = act(self.c1_d(x)), act(self.c1_r(x) + x)
        d2, r2 = act(self.c2_d(r)), act(self.c2_r(r) + r)
        d3, r3 = act(self.c3_d(r2)), act(self.c3_r(r2) + r2)
        d4 = act(self.c4(r3))
        return self.esa(self.c5(torch.cat([d1, d2, d3, d4], dim=1)))


class Rfdn(nn.Module):
    """RFDN super-resolution network (Liu et al., "Residual Feature Distillation Network for
    Lightweight Image Super-Resolution", 2020): 50 features, 4 RFDBs, x4 pixel-shuffle — BASELINE
    configs[4].  Module names (fea_conv, B1..B4, c, LR_conv, upsampler) follow the reference's
    src/models/sr/rfdn/rfdn.py:11-42 so the YAML's excluded_layers
    (`fea_conv`, `upsampler.0`) apply; 33 of its 3x3 convolutions get quantized, the 29 1x1
    convolutions do not (reference quirk 2)."""

    def __init__(self, in_nc=3, nf=50, num_modules=4, out_nc=3, scale=4):
        super().__init__()
        self.fea_conv = nn.Conv2d(in_nc, nf, 3, padding=1)
        self.B1, self.B2, self.B3, self.B4 = (_Rfdb(nf) for _ in range(4))
        self.c = nn.Sequential(nn.Conv2d(nf * num_modules, nf, 1), nn.LeakyReLU(0.05, inplace=True))
        self.LR_conv = nn.Conv2d(nf, nf, 3, padding=1)
        self.upsampler = nn.Sequential(nn.Conv2d(nf, out_nc * scale * scale, 3, padding=1),
                                       nn.PixelShuffle(scale))

    def forward(self, x):
        fea = self.fea_conv(x)
        b1 = self.B1(fea)
        b2 = self.B2(b1)
        b3 = self.B3(b2)
        b4 = self.B4(b3)
        out = self.LR_conv(self.c(torch.cat([b1, b2, b3, b4], dim=1))) + fea
        return self.upsampler(out)


class SRModule(LModule):
    """LVisionSR's forward (vision_sr_module.py:49-53): the network sees 0..255 inputs."""

    def forward(self, inputs):
        return self.model(inputs * 255).div(255)

    def training_step(self, batch, batch_idx):
        inputs, target = batch
        loss = self.criterion(self.forward(inputs), target)
        self.log("loss", loss)
        return loss


def build_model(name: str, num_classes: Optional[int] = None) -> nn.Module:
    if name == "resnet18":
        import torchvision
        return torchvision.models.resnet18(num_classes=num_classes or 1000)
    if name == "resnet20":
        return CifarResNet(3, num_classes or 10)
    if name == "rfdn":
        return Rfdn(scale=4)
    # grouped, depthwise and dilated networks (random weights; nothing is downloaded)
    if name == "mobilenet_v2":
        import torchvision
        return torchvision.models.mobilenet_v2(num_classes=num_classes or 1000)
    if name == "resnext50_32x4d":
        import torchvision
        return torchvision.models.resnext50_32x4d(num_classes=num_classes or 1000)
    if name == "resnet50_dilated":      # the DeepLab backbone: layer3 / layer4 at dilation 2 / 4
        import torchvision
        return torchvision.models.resnet50(num_classes=num_classes or 1000,
                                           replace_stride_with_dilation=[False, True, True])
    raise ValueError(name)


EXCLUDED = {"resnet18": ("conv1", "fc"), "resnet20": ("conv1", "linear"),
            "rfdn": ("fea_conv", "upsampler.0"),
            "mobilenet_v2": ("features.0.0", "classifier.1"),
            "resnext50_32x4d": ("conv1", "fc"), "resnet50_dilated": ("conv1", "fc")}


# ------------------------------------------------------------------ calibration
@torch.no_grad()
def calibrate(qmodel: LModule, batch, act_bits=10, weight_bits=10):
    """`Trainer.calibrate` (training/trainer.py:187-223) on one batch: weight scales via
    apply_quantile_weights_s, activation ranges via MinMaxObserver forward hooks on every
    NoisyAct during an eval forward, then apply_mean_stats_activations."""
    from .quantization.gdnsq.calib.hooks import register_lightning_activation_forward_hook
    from .quantization.gdnsq.calib.minmaxobserver import (MinMaxObserver, apply_mean_stats_activations,
                                                          apply_quantile_weights_s)
    model = qmodel.model
    if weight_bits:
        apply_quantile_weights_s(model, wbits=weight_bits)
    if act_bits:
        handles = register_lightning_activation_forward_hook(model, MinMaxObserver())
        was_training = model.training
        model.eval()
        qmodel(batch)          # through the module's own forward (LVisionSR denormalises)
        model.train(was_training)
        for h in handles:
            h.remove()
        apply_mean_stats_activations(model, abits=act_bits)


# ------------------------------------------------------------------ build + fit
def build_qat(model_name="resnet18", device="cuda", qnmethod="STE", act_bit=4, weight_bit=4,
              distillation=True, num_classes=None, lr=3e-4, calib_batch=None, calib_bits=10):
    """FP model → LModule → Quantizer(config)().quantize(lm) → calibrated, on `device`."""
    from .quantization.quantizer import Quantizer
    model = build_model(model_name, num_classes).to(device)
    if model_name == "rfdn":      # config/gdnsq_config_rfdn_lsq_w2a2.yaml: L1, no teacher
        lm = SRModule(model, nn.L1Loss(), torch.optim.RAdam, lr)
    else:
        lm = LModule(model, nn.CrossEntropyLoss(), torch.optim.RAdam, lr)
    cfg = make_config(act_bit=act_bit, weight_bit=weight_bit, qscheme=1, qnmethod=qnmethod,
                      excluded_layers=EXCLUDED[model_name], distillation=distillation)
    qmodel = Quantizer(cfg)().quantize(lm, in_place=True)
    qmodel.to(device)
    if calib_batch is not None:
        calibrate(qmodel, calib_batch, act_bits=calib_bits, weight_bits=calib_bits)
    return qmodel


def wrap_ddp(model: nn.Module, device, lean: bool = True):
    """DistributedDataParallel around the quantized model.

    The reference's Trainer passes ``find_unused_parameters=True`` (training/trainer.py:93-95)
    only because every per-channel ``NoisyConv2d`` owns a trainable ``log_b_s`` that is never
    used (SURVEY.md quirk 5); that flag makes DDP walk the autograd graph on every step.
    ``lean=True`` instead tells DDP to ignore exactly those parameters, and skips the per-step
    broadcast of BatchNorm running statistics (they do not enter the training arithmetic).
    ``lean=False`` reproduces the reference's flags."""
    from torch.nn.parallel import DistributedDataParallel as DDP
    ids = [device.index] if device is not None and device.type == "cuda" else None
    if not lean:
        return DDP(model, device_ids=ids, find_unused_parameters=True, gradient_as_bucket_view=True)
    ignore = [n for n, _ in model.named_parameters() if n.endswith("log_b_s")]
    DDP._set_params_and_buffers_to_ignore_for_model(model, ignore)
    return DDP(model, device_ids=ids, find_unused_parameters=False, broadcast_buffers=False,
               gradient_as_bucket_view=True)


def ddp_side_stream(model: nn.Module, device, lean: bool = True):
    """`wrap_ddp` executed on a side stream — what torch requires of a DDP module whose backward
    (bucket all-reduces included) is later captured into a CUDA graph."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        wrapped = wrap_ddp(model, device, lean=lean)
    torch.cuda.current_stream().wait_stream(side)
    return wrapped


def fit_steps(qmodel: LModule, batches, ddp: bool = False, device=None, on_step=None,
              sync_bn: bool = False):
    """Run the training steps in Lightning's order.  `batches`: iterable of (inputs, target).
    Under DDP the quantized model is wrapped like Lightning's DDPStrategy does
    (find_unused_parameters=True: the reference's never-used `log_b_s`, trainer.py:93-95)."""
    if ddp:
        if sync_bn:
            qmodel.model = nn.SyncBatchNorm.convert_sync_batchnorm(qmodel.model)
        qmodel.model = wrap_ddp(qmodel.model, device, lean=False)
    opt = qmodel.configure_optimizers()
    qmodel.train()
    if hasattr(qmodel, "wrapped_criterion"):
        qmodel.wrapped_criterion.train()
    for i, batch in enumerate(batches):
        loss = qmodel.training_step(batch, i)
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        if on_step is not None:
            on_step(i, loss)
    return qmodel


class BatchPrefetcher:
    """Double-buffered host->device staging of training batches on a copy stream, so the PCIe
    copy of batch k+1 overlaps the GPU work of step k (what a DataLoader with pinned memory and
    `non_blocking` copies gives the reference's Trainer).  put() enqueues a copy into the free
    slot; get() makes the current stream wait for the oldest filled slot and returns its device
    tensors; release() marks that slot reusable once the current stream's work so far is done."""

    def __init__(self, example_batch, depth: int = 2):
        self.slots = [tuple(torch.empty_like(t) for t in example_batch) for _ in range(depth)]
        self.stream = torch.cuda.Stream()
        self.ready = [torch.cuda.Event() for _ in range(depth)]
        self.free = [torch.cuda.Event() for _ in range(depth)]
        for ev in self.free:
            ev.record()
        self.head = self.tail = self.count = 0

    def put(self, host_batch):
        if self.count == len(self.slots):
            raise RuntimeError("BatchPrefetcher: all slots are in flight")
        i = self.head
        self.head = (i + 1) % len(self.slots)
        self.count += 1
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(self.free[i])
            for d, h in zip(self.slots[i], host_batch):
                d.copy_(h, non_blocking=True)
            self.ready[i].record(self.stream)

    def get(self):
        if self.count == 0:
            raise RuntimeError("BatchPrefetcher: nothing in flight")
        torch.cuda.current_stream().wait_event(self.ready[self.tail])
        return self.slots[self.tail]

    def release(self):
        self.free[self.tail].record()
        self.tail = (self.tail + 1) % len(self.slots)
        self.count -= 1


class GraphedTrainStep:
    """One QAT training step (teacher + student forward, loss, backward, optimizer) captured
    in a CUDA graph and replayed — SURVEY.md §8 row (f)-4.  CIFAR-sized models are bound by
    host launch overhead (ResNet-20, batch 256: ~19 ms of Python/launch time for ~9 ms of GPU
    work); a replay has none.  The in-kernel noise reads a device-resident Philox state that is
    advanced inside the graph, so every replay draws fresh noise.  Under DDP (one process per
    GPU) the bucketed gradient all-reduces — and AEWGS's packed statistics all-reduce — are
    NCCL kernels captured into the same graph with their stream dependencies: wrap the model
    with `wrap_ddp` on a side stream first (`ddp_side_stream`), the warm-up then runs the >= 11
    eager DDP iterations torch asks for before a whole-backward capture.  Host-side schedules (`wrapped_criterion.t`, learning-rate callbacks) are
    frozen at capture time — re-capture after changing them."""

    STRIDE = 4096        # > number of quantizer backward calls per step

    def __init__(self, qmodel: LModule, example_batch, seed: int = 0, warmup: Optional[int] = None):
        from . import ops
        import torch.distributed as dist
        self.distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
        if warmup is None:
            warmup = 11 if self.distributed else 3
        x, t = example_batch
        self.ops, self.qmodel = ops, qmodel
        self.x, self.t = x.clone(), t.clone()
        dev = x.device
        self.state = torch.tensor([seed, 0], dtype=torch.int64, device=dev)
        ops.set_device_philox_state(self.state)
        params = [p for p in qmodel.parameters() if p.requires_grad]
        self.opt = qmodel.optimizer(params, lr=torch.tensor(float(qmodel.lr), device=dev),
                                    capturable=True)
        qmodel.train()
        if hasattr(qmodel, "wrapped_criterion"):
            qmodel.wrapped_criterion.train()
            qmodel.wrapped_criterion.make_capturable(dev)
        self._release_autograd_state(qmodel)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self._body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self._release_autograd_state(qmodel)      # (the warm-up's graph lives on the side stream)
        self.graph = torch.cuda.CUDAGraph()
        self.opt.zero_grad(set_to_none=True)
        # (thread_local: NCCL's watchdog thread may query events while this thread captures)
        with torch.cuda.graph(self.graph, capture_error_mode="thread_local" if self.distributed else "global"):
            self.loss = self._body()

    @staticmethod
    def _release_autograd_state(qmodel):
        """Drop whatever still references the autograd graph of an earlier eager step: the
        criterion keeps its last loss terms for logging (gdnsq_loss.py:60-66) and a layer may hold
        a quantized weight whose backward never ran.  A live graph keeps its AccumulateGrad nodes —
        bound to the stream of that eager step — and a captured backward may not synchronise
        with a stream outside the capture."""
        crit = getattr(qmodel, "wrapped_criterion", None)
        if crit is not None:
            for k, v in list(vars(crit).items()):
                if torch.is_tensor(v) and v.grad_fn is not None:
                    setattr(crit, k, v.detach())
        for m in qmodel.modules():
            cache = getattr(m, "_wq_cache", None)
            if cache is not None:
                cache.clear()
            # the layers leave their last operands on the Quantizer (gdnsq_conv2d.py:80-84:
            # `self.Q.zero_point = weight.amin(...)` carries that step's graph)
            for name in ("Q", "Q_b"):
                qz = m.__dict__.get(name)
                if qz is not None and hasattr(qz, "_resolve"):
                    qz._resolve()
                    for attr in ("_scale", "_zero_point", "_min_val", "_max_val"):
                        v = getattr(qz, attr, None)
                        if torch.is_tensor(v) and v.grad_fn is not None:
                            setattr(qz, attr, v.detach())

    def _body(self):
        self.ops.reset_philox_call_counter()
        self.state[1] += self.STRIDE
        loss = self.qmodel.training_step((self.x, self.t), 0)
        loss.backward()
        self.opt.step()
        self.opt.zero_grad(set_to_none=True)
        return loss.detach()

    def __call__(self, batch=None):
        if batch is not None:
            self.x.copy_(batch[0], non_blocking=True)
            self.t.copy_(batch[1], non_blocking=True)
        self.graph.replay()
        return self.loss

    def close(self):
        self.ops.set_device_philox_state(None)
