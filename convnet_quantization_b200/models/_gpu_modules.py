"""``nn.Module`` shells around the CUDA engines, shaped so the reference's drivers can use them unchanged
(``utils/inference_benchmark.py:19-28`` calls ``eval()/to(device)/model(data)``; ``utils/model_evaluator.py:19-33``
calls ``eval()/cpu()/model(cpu_images)`` and ``outputs.topk`` on the result):

* ``forward`` accepts fp32 NCHW ``[B,3,32,32]`` on CPU **or** CUDA and returns fp32 logits ``[B,10]`` on the input's
  device (H2D / D2H done here when the caller hands CPU tensors);
* ``.cpu()`` / ``.to('cpu')`` never tear the GPU engine down (the arithmetic has no CPU fallback);
* ``.to('cuda:N')`` re-homes the engine; everything mutates in place because the driver discards ``.to()``'s result;
* ``forward`` on a CUDA input synchronises the stream before returning (``sync_on_forward``, default on): the
  reference's benchmark reads ``time.time()`` right after ``model(data)`` without a device synchronize
  (``utils/inference_benchmark.py:93-100``), so an asynchronous return would make it time the launch, not the work.
  Pipelines that manage their own streams call ``engine.forward`` (never synchronises) or clear the flag.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import _lib, ops
from ..engine import StaticEngine, eval_result


def _default_device() -> torch.device:
    if not torch.cuda.is_available():
        raise _lib.B200QError("no CUDA device: the quantized forward has no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


class _GpuResident(nn.Module):
    """Common device handling: the engine lives on ``self.engine_device`` regardless of ``.cpu()``."""

    quantized = True  # sniffed by utils/model_evaluator.py:25,66
    sync_on_forward = True

    def __init__(self, device=None):
        super().__init__()
        if isinstance(device, int):
            device = torch.device("cuda", device)
        self.engine_device = torch.device(device) if device is not None else _default_device()
        if self.engine_device.type != "cuda":
            raise _lib.B200QError("engine device must be CUDA")
        if self.engine_device.index is None:
            self.engine_device = torch.device("cuda", torch.cuda.current_device())

    def _rehome(self, device: torch.device):  # overridden
        raise NotImplementedError

    def to(self, *args, **kwargs):
        device = kwargs.get("device", args[0] if args else None)
        if isinstance(device, bool):
            device = None
        elif isinstance(device, int):  # model.to(1) == model.to("cuda:1"), as torch.nn.Module.to reads it
            device = torch.device("cuda", device)
        elif isinstance(device, str):
            device = torch.device(device)
        if isinstance(device, torch.device) and device.type == "cuda":
            if device.index is None:
                device = torch.device("cuda", torch.cuda.current_device())
            if device != self.engine_device:
                self._rehome(device)
        return self  # 'cpu' (or dtype-only) requests: nothing to move, the engine stays on its GPU

    def cpu(self):
        return self

    def cuda(self, device=None):
        return self.to(torch.device("cuda", device) if isinstance(device, int) else (device or "cuda"))

    def _run(self, x: torch.Tensor, fn):
        if x.dtype != torch.float32:
            x = x.float()
        if x.is_cuda and x.device == self.engine_device:
            y = fn(x.contiguous())
            if self.sync_on_forward:
                torch.cuda.current_stream(self.engine_device).synchronize()
            return y
        y = fn(x.to(self.engine_device, non_blocking=True).contiguous())
        return y.to(x.device)  # device -> host (or peer) copy: synchronises by itself


class _HostPipelined(_GpuResident):
    """Host inputs (what ``utils/model_evaluator.py`` hands over, and ``utils/inference_benchmark.py`` with
    ``device='cpu'``) are processed in chunks on two CUDA streams, so the host->device copy of chunk i+1 overlaps
    the kernels of chunk i; logits come back through a pinned staging buffer.  Only for nets whose result for an image
    does not depend on the rest of the batch (the int8 static and sandwich nets; NOT the dynamic one, whose activation
    qparams come from the whole batch).  Subclasses provide ``_chunk_forward(xin, yout, u8)``."""

    # images per pipelined chunk (B200Q_HOST_CHUNK overrides, for tuning).  The pipeline is bound by the host->device
    # copy (12 KiB of fp32 per image over PCIe), so what the chunk size controls is the un-overlapped tail: the kernels
    # of the LAST chunk.  2048 images = 24 MiB per copy, still far above the size where PCIe copies lose efficiency.
    HOST_CHUNK = int(os.environ.get("B200Q_HOST_CHUNK", "2048"))
    TAIL_MIN = int(os.environ.get("B200Q_TAIL_MIN", "256"))
    # uint8 route: 3 KiB per image crosses PCIe at ~17 M images/s, the kernels run at ~7.6 M images/s, so that pipeline
    # is COMPUTE-bound and what is exposed is the copy of the FIRST chunk.  Chunks therefore ramp up: a smaller first one
    # (fast fill), the next ones twice the size (their copies still finish inside the kernels of the chunk before).
    # The cap keeps the doubling short: on a host whose links are shared by eight GPUs the copy rate per GPU falls to
    # about the compute rate, and every doubling then stalls the kernels for one chunk.  Measured (first, cap) at
    # N = 1 / N = 8 ranks, M images/s: (8192, 8192) 6.3-6.5 / 45.6, (1024, 8192) 7.0-7.1 / 42.1, (2048, 4096) 7.0 / 47.1
    # (profiles/r02_e2e_timeline.txt, r02_u8_plan_n8.txt).
    U8_FIRST_CHUNK = int(os.environ.get("B200Q_U8_FIRST_CHUNK", "2048"))
    U8_MAX_CHUNK = int(os.environ.get("B200Q_U8_MAX_CHUNK", "4096"))

    _pipe = None

    def _pipeline(self):
        if self._pipe is None:
            dev = self.engine_device
            self._pipe = {
                "streams": [torch.cuda.Stream(dev), torch.cuda.Stream(dev)],
                "x": [torch.empty((self.HOST_CHUNK, 3, 32, 32), dtype=torch.float32, device=dev) for _ in range(2)],
                "xu8": None,  # uint8 NHWC staging buffers, allocated on first use of forward_uint8
                "y": [torch.empty((self.HOST_CHUNK, 10), dtype=torch.float32, device=dev) for _ in range(2)],
                "out": None,
            }
        return self._pipe

    def _chunks(self, b: int, chunk: int | None = None):
        """(offset, size) of the pipelined chunks.  The copies run back to back, so the un-overlapped part of a call is
        the kernels of the LAST chunk; the final ``HOST_CHUNK`` images are therefore split 3/4 + 1/4 (one extra chunk:
        every chunk costs ~30 us of fixed overhead, and chunks much smaller than 512 images take longer to compute than
        to copy - measured, scripts/gpu_e2e_chunks.sh)."""
        chunk = chunk or self.HOST_CHUNK
        lo = 0
        while b - lo > chunk:
            yield lo, chunk
            lo += chunk
        rest = b - lo
        tail = rest // 4
        if tail >= self.TAIL_MIN:
            yield lo, rest - tail
            lo += rest - tail
        yield lo, b - lo

    def _chunks_ramp(self, b: int, first: int, cap: int):
        """(offset, size) for the compute-bound uint8 pipeline: ``first``, 2*first, 4*first ... capped at ``cap``."""
        lo, n = 0, max(1, first)
        while b - lo > n:
            yield lo, n
            lo += n
            n = min(2 * n, cap)
        yield lo, b - lo

    def _pipelined(self, x: torch.Tensor, u8: bool, run_chunk) -> None:
        """Host ``x`` through the two-stream chunk plan: copies each chunk into its stream's staging buffer and calls
        ``run_chunk(xin, k, lo, n)`` on that stream (``k``: stream index; ``[lo, lo+n)``: the chunk's images).  Returns
        once both streams have finished."""
        b = x.shape[0]
        x = x.contiguous()
        pipe = self._pipeline()
        chunk = self.U8_MAX_CHUNK if u8 else self.HOST_CHUNK
        if u8 and pipe["xu8"] is None:
            pipe["xu8"] = [torch.empty((chunk, 32, 32, 3), dtype=torch.uint8, device=self.engine_device) for _ in range(2)]
            pipe["yu8"] = [torch.empty((chunk, 10), dtype=torch.float32, device=self.engine_device) for _ in range(2)]
        cur = torch.cuda.current_stream(self.engine_device)
        for s in pipe["streams"]:
            s.wait_stream(cur)
        plan = self._chunks_ramp(b, self.U8_FIRST_CHUNK, chunk) if u8 else self._chunks(b, chunk)
        for i, (lo, n) in enumerate(plan):
            k = i & 1
            with torch.cuda.stream(pipe["streams"][k]):  # per-stream buffers: reuse is ordered by the stream itself
                xin = (pipe["xu8"] if u8 else pipe["x"])[k][:n]
                xin.copy_(x[lo:lo + n], non_blocking=True)
                run_chunk(xin, k, lo, n)
        for s in pipe["streams"]:
            s.synchronize()

    def _forward_host(self, x: torch.Tensor, u8: bool = False) -> torch.Tensor:
        b = x.shape[0]
        pipe = self._pipeline()
        if pipe["out"] is None or pipe["out"].shape[0] < b:
            pipe["out"] = torch.empty((max(b, self.HOST_CHUNK), 10), dtype=torch.float32).pin_memory()
        out = pipe["out"][:b]

        def run_chunk(xin, k, lo, n):
            yout = (pipe["yu8"] if u8 else pipe["y"])[k][:n]
            self._chunk_forward(xin, yout, u8)
            out[lo:lo + n].copy_(yout, non_blocking=True)

        self._pipelined(x, u8, run_chunk)
        return out.clone()  # the pinned staging buffer is reused by the next call


class B200StaticQuantizedNet(_HostPipelined):
    """True static-PTQ int8 ``SimpleConvNet`` (all eight layers int8, fbgemm-exact requantisation) on a B200."""

    def __init__(self, qparams: dict, device=None):
        super().__init__(device)
        self.qparams = qparams
        self.engine = StaticEngine(qparams, self.engine_device)
        self._pipe = None

    def _rehome(self, device):
        self.engine = StaticEngine(self.qparams, device)
        self.engine_device = device
        self._pipe = None

    def _chunk_forward(self, xin, yout, u8):
        if u8:
            self.engine.forward_u8(xin, out=yout)
        else:
            self.engine.forward(xin, out=yout)

    @torch.no_grad()
    def forward(self, x):
        if x.is_cuda:
            if x.dtype is torch.float32 and x.device == self.engine_device:  # the driver's loop: no conversions to make
                y = self.engine.forward(x)
                if self.sync_on_forward:
                    torch.cuda.current_stream(self.engine_device).synchronize()
                return y
        elif x.dim() == 4 and x.shape[0] > 0:
            return self._forward_host(x.float())
        return self._run(x, self.engine.forward)

    @torch.no_grad()
    def forward_uint8(self, pixels: torch.Tensor) -> torch.Tensor:
        """uint8 data path (SURVEY 8f rank 4): raw pixels, uint8 NHWC ``[B,32,32,3]`` as ``torchvision``'s CIFAR-10
        ``.data`` holds them, CPU or CUDA -> fp32 logits on the input's device.  Bit-identical to
        ``forward(Normalize(ToTensor(pixels)))``; a quarter of the bytes cross PCIe."""
        if pixels.dtype != torch.uint8 or pixels.dim() != 4 or tuple(pixels.shape[1:]) != (32, 32, 3):
            raise _lib.B200QError(f"forward_uint8 expects uint8 NHWC [B,32,32,3], got {pixels.dtype} {tuple(pixels.shape)}")
        if not pixels.is_cuda and pixels.shape[0] > 0:
            return self._forward_host(pixels, u8=True)
        if not pixels.is_cuda:
            return torch.empty((0, 10), dtype=torch.float32)
        y = self.engine.forward_u8(pixels)
        if self.sync_on_forward:
            torch.cuda.current_stream(self.engine_device).synchronize()
        return y

    @torch.no_grad()
    def eval_counters(self, images: torch.Tensor, labels: torch.Tensor, u8: bool = False) -> torch.Tensor:
        """int64 ``[5]`` counters (``_lib.EVAL_COUNTER_NAMES``) on the engine's device, not synchronised: ``evaluate``
        without the read-back, for callers that reduce them further (``sharding.evaluate_sharded``).  Host images go
        through the chunk pipeline of ``forward`` / ``forward_uint8``; the labels are copied to the device once."""
        shape, dtype = ((32, 32, 3), torch.uint8) if u8 else ((3, 32, 32), torch.float32)
        if images.dim() != 4 or tuple(images.shape[1:]) != shape or (u8 and images.dtype != torch.uint8):
            raise _lib.B200QError(f"evaluate{'_uint8' if u8 else ''} expects {dtype} [B,{','.join(map(str, shape))}], "
                                  f"got {images.dtype} {tuple(images.shape)}")
        if labels.dtype != torch.int64 or tuple(labels.shape) != (images.shape[0],):
            raise _lib.B200QError(f"labels must be int64 [{images.shape[0]}], got {labels.dtype} {tuple(labels.shape)}")
        dev = self.engine_device
        with torch.cuda.device(dev):
            counters = torch.zeros(_lib.EVAL_COUNTERS, dtype=torch.int64, device=dev)
            labels = labels.to(dev).contiguous()
            run = self.engine.evaluate_u8 if u8 else self.engine.evaluate
            if images.is_cuda:
                run(images.to(dev, dtype), labels, counters)
            elif images.shape[0] > 0:  # integer counts: chunking and the two streams change no total
                self._pipelined(images.to(dtype), u8, lambda xin, k, lo, n: run(xin, labels[lo:lo + n], counters))
        return counters

    @torch.no_grad()
    def evaluate(self, images: torch.Tensor, labels: torch.Tensor) -> dict:
        """Top-1 / top-5 accuracy over fp32 NCHW ``images`` (CPU or CUDA) and int64 ``labels``, counted inside the
        classifier-head kernel (tie rule: ``include/b200q.h``): ``{"top1", "top5", "images", "top1_tied",
        "top5_tied", "top1_pct", "top5_pct"}``.  The ``*_tied`` counts bound how far a ``topk``-based count of the
        same logits can differ.  Only the 40 bytes of counters come back to the host."""
        return eval_result(self.eval_counters(images, labels))

    @torch.no_grad()
    def evaluate_uint8(self, pixels: torch.Tensor, labels: torch.Tensor) -> dict:
        """``evaluate`` from raw uint8 NHWC pixels ``[B,32,32,3]`` (the input of ``forward_uint8``)."""
        return eval_result(self.eval_counters(pixels, labels, u8=True))

    @torch.no_grad()
    def forward_with_taps(self, x):
        """(logits, {layer: uint8 NHWC activations}) — parity-test hook."""
        return self.engine.forward(x.to(self.engine_device).float().contiguous(), taps=True)

    def state_dict(self, *args, **kwargs):
        """int8 weights + fp32 scales/bias, so ``get_model_size`` (torch.save of the state_dict,
        ``models/static_ptq_model.py:36-43``) reports the quantized size."""
        sd = {"quant.scale": torch.tensor(self.qparams["in_scale"]), "quant.zero_point": torch.tensor(self.qparams["in_zp"])}
        for name, L in self.qparams.items():
            if isinstance(L, dict):
                sd[f"{name}.weight"] = L["w_int8"]
                sd[f"{name}.weight_scales"] = L["w_scales"].float()
                sd[f"{name}.bias"] = L["bias"]
                sd[f"{name}.scale"] = torch.tensor(L["out_scale"])
                sd[f"{name}.zero_point"] = torch.tensor(L["out_zp"])
        return sd


class B200DynamicQuantizedNet(_GpuResident):
    """The reference's dynamic-PTQ net *as written* (SURVEY F3): ``quantize_dynamic`` only swaps ``fc1``/``fc2`` for
    ``DynamicQuantizedLinear``; the six BN-folded convs stay fp32.  Here the convs run as fp32 ATen/cuDNN ops (TF32 off;
    this is the tolerance path, not the product) and both linears run ``b200q_linear_dynamic`` (device-side min/max ->
    qparams -> quantize -> int8 GEMM -> fp32)."""

    def __init__(self, fused_fp32: nn.Module, fc_weights: dict, device=None, bn_after_fc1: nn.Module | None = None):
        """``bn_after_fc1``: eval-mode BatchNorm1d applied to fc1's output when fc1 was quantised WITHOUT the
        batch-norm folded in (``StaticPTQModel`` as written quantises the unfused net: fc1 -> bn7 -> relu)."""
        super().__init__(device)
        self._fused_cpu = fused_fp32
        self._fc_cpu = fc_weights  # name -> (w_int8, w_scale, bias)
        self._bn_cpu = None
        if bn_after_fc1 is not None:
            bn = bn_after_fc1
            scale = (bn.weight / torch.sqrt(bn.running_var + bn.eps)).detach().float()
            self._bn_cpu = (scale, (bn.bias - bn.running_mean * scale).detach().float())
        self._build(self.engine_device)

    def _build(self, device):
        self.convs = [(getattr(self._fused_cpu, f"conv{i}").weight.detach().to(device),
                       getattr(self._fused_cpu, f"conv{i}").bias.detach().to(device)) for i in range(1, 7)]
        self.fc = {n: ops.DynamicLinearWeights(w, s, b, device) for n, (w, s, b) in self._fc_cpu.items()}
        self.bn = None if self._bn_cpu is None else tuple(t.to(device) for t in self._bn_cpu)

    def _rehome(self, device):
        self._build(device)
        self.engine_device = device

    @torch.no_grad()
    def features(self, x):
        """fp32 conv stack (BN folded) -> ``[B,4096]`` in the reference's NCHW flatten order."""
        with torch.backends.cudnn.flags(enabled=True, allow_tf32=False):
            for i, (w, b) in enumerate(self.convs, start=1):
                x = F.relu(F.conv2d(x, w, b, padding=1))
                if i % 2 == 0:
                    x = F.max_pool2d(x, 2, 2)
        return x.reshape(x.shape[0], -1).contiguous()

    def _forward_dev(self, x):
        if x.shape[0] == 0:
            return torch.empty((0, 10), dtype=torch.float32, device=x.device)
        x = self.features(x)
        if self.bn is None:
            x = ops.linear_dynamic(x, self.fc["fc1"], relu=True)
        else:  # unfused fc1: batch-norm, then ReLU, in fp32 (tolerance path)
            x = F.relu(ops.linear_dynamic(x, self.fc["fc1"], relu=False) * self.bn[0] + self.bn[1]).contiguous()
        return ops.linear_dynamic(x, self.fc["fc2"], relu=False)

    @torch.no_grad()
    def forward(self, x):
        return self._run(x, self._forward_dev)

    def state_dict(self, *args, **kwargs):
        sd = {k: v for k, v in self._fused_cpu.state_dict().items() if not k.startswith(("fc1", "fc2"))}
        for n, (w, s, b) in self._fc_cpu.items():
            sd[f"{n}.weight"], sd[f"{n}.scale"], sd[f"{n}.bias"] = w, torch.tensor(s), b
        return sd


class B200SandwichQuantizedNet(_HostPipelined):
    """The custom variant *as intended* (``models/custom_quantization_model.py:34-58, 202-261``; SURVEY 8f rank 3):
    each conv and ``fc1`` is QuantStub -> int8 layer -> DeQuantStub, ReLU / max-pool run in fp32 between the
    sandwiches, ``fc2`` is fp32.  On the GPU the fp32 detours collapse without changing a bit:

    * the int8 layers are the tensor-core kernels of the static net with ReLU fusion OFF (the sandwich's conv output
      observer sees pre-ReLU values) and the 2x2 max-pool still fused into conv2/4/6;
    * DeQuantStub -> fp32 ReLU (-> fp32 max-pool) -> next QuantStub is a monotone uint8 -> uint8 map, applied as a
      256-entry table (``b200q_lut_u8``) that ``ptq.sandwich_boundary_lut`` evaluates with the reference's own torch
      ops; being monotone it commutes with the max-pool, so it runs on the pooled (4x smaller) tensor;
    * ``fc1``'s uint8 output is ReLU'd and dequantised (``b200q_relu_q`` + ``b200q_dequantize`` == fp32 ReLU of the
      dequantised tensor), then ``fc2`` is an fp32 ATen GEMM (the tolerance part of this variant)."""

    is_custom_quantized = True

    def __init__(self, sparams: dict, device=None):
        super().__init__(device)
        self.sparams = sparams
        self._build(self.engine_device)

    def _build(self, device):
        from .. import ptq
        from ..packing import PackedConv, PackedLinear
        sp = self.sparams
        names = ptq.SANDWICH_LAYERS
        with torch.cuda.device(device):
            self.convs = [PackedConv(n, sp[n], sp[n]["in_scale"], sp[n]["in_zp"], device, relu=False) for n in names[:6]]
            self.fc1 = PackedLinear("fc1", sp["fc1"], sp["fc1"]["in_scale"], sp["fc1"]["in_zp"], device, relu=False,
                                    nhwc_from=(256, 4, 4))
            self.fc2_w = sp["fc2"]["weight"].to(device)
            self.fc2_b = sp["fc2"]["bias"].to(device)
        # boundary tables: output qparams of layer i -> input qparams of layer i+1 (host uint8 [256])
        self.luts = [ptq.sandwich_boundary_lut(sp[a]["out_scale"], sp[a]["out_zp"], sp[b]["in_scale"], sp[b]["in_zp"])
                     for a, b in zip(names[:-1], names[1:])]

    def _rehome(self, device):
        self._build(device)
        self.engine_device = device
        self._pipe = None

    def _chunk_forward(self, xin, yout, u8):
        yout.copy_(self._forward_dev(xin))

    @torch.no_grad()
    def _forward_dev(self, x, taps: dict | None = None):
        sp = self.sparams
        a = ops.quantize_conv2d_first(x, sp["conv1"]["in_scale"], self.convs[0])
        if taps is not None:
            taps["conv1"] = a
        for i in range(1, 6):
            a = ops.lut_u8(a, self.luts[i - 1])
            a = ops.conv2d_q(a, self.convs[i], pool2x2=(i % 2 == 1) and taps is None)
            if taps is not None:
                taps[f"conv{i + 1}"] = a
                if i % 2 == 1:
                    a = ops.max_pool2d_q(a)
        a = ops.lut_u8(a, self.luts[5]).reshape(a.shape[0], -1)  # NHWC [B,4,4,256]; fc1's columns are permuted to match
        h = ops.linear_q(a, self.fc1)
        if taps is not None:
            taps["fc1"] = h
        h = ops.dequantize(ops.relu_q(h, sp["fc1"]["out_zp"]), sp["fc1"]["out_scale"], sp["fc1"]["out_zp"])
        return torch.addmm(self.fc2_b, h, self.fc2_w.t())

    @torch.no_grad()
    def forward(self, x):
        if x.shape[0] == 0:
            return torch.empty((0, 10), dtype=torch.float32, device=x.device)
        if not x.is_cuda and x.dim() == 4:  # per-image arithmetic: chunking changes no bit of the int8 layers
            return self._forward_host(x.float())
        return self._run(x, self._forward_dev)

    @torch.no_grad()
    def forward_with_taps(self, x):
        """(logits, {layer: uint8 NHWC output of the sandwich's int8 layer, before ReLU}) - parity-test hook."""
        taps: dict = {}
        logits = self._forward_dev(x.to(self.engine_device).float().contiguous(), taps)
        return logits, taps

    def state_dict(self, *args, **kwargs):
        sd = {}
        for name, L in self.sparams.items():
            if name == "fc2":
                sd["fc2.weight"], sd["fc2.bias"] = L["weight"], L["bias"]
                continue
            sd[f"{name}.quant.scale"], sd[f"{name}.quant.zero_point"] = torch.tensor(L["in_scale"]), torch.tensor(L["in_zp"])
            sd[f"{name}.weight"], sd[f"{name}.weight_scales"], sd[f"{name}.bias"] = L["w_int8"], L["w_scales"].float(), L["bias"]
            sd[f"{name}.scale"], sd[f"{name}.zero_point"] = torch.tensor(L["out_scale"]), torch.tensor(L["out_zp"])
        return sd
