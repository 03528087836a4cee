"""Device engine for the static-PTQ SimpleConvNet: packed weights + workspace + the single C-ABI forward call."""
from __future__ import annotations

import contextlib
import ctypes as C
from collections import OrderedDict

import torch

from . import _lib
from .packing import PackedSandwichNet, PackedStaticNet

TAP_NAMES = ("quant", "conv1", "conv2", "pool1", "conv3", "conv4", "pool2", "conv5", "conv6", "pool3", "fc1", "fc2")
TAP_SHAPES = {  # per image, NHWC (quant is NHWC4: channel 3 is padding)
    "quant": (32, 32, 4), "conv1": (32, 32, 64), "conv2": (32, 32, 64), "pool1": (16, 16, 64),
    "conv3": (16, 16, 128), "conv4": (16, 16, 128), "pool2": (8, 8, 128), "conv5": (8, 8, 256),
    "conv6": (8, 8, 256), "pool3": (4, 4, 256), "fc1": (512,), "fc2": (10,),
}


SANDWICH_TAP_NAMES = ("conv1", "conv2", "conv3", "conv4", "conv5", "conv6", "fc1")  # int8 layer outputs, before ReLU

_NULL_CTX = contextlib.nullcontext()

# The current stream's raw handle without building a torch.cuda.Stream object (1.5 us -> 0.2 us on the batch-1 path).
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _current_stream_handle(device_index: int) -> int:
    if _raw_stream is not None:
        return _raw_stream(device_index)
    return torch.cuda.current_stream(device_index).cuda_stream


def eval_result(counters: torch.Tensor) -> dict:
    """The five counters of ``StaticEngine.evaluate`` as ints by name, plus ``top1_pct`` / ``top5_pct`` (of
    ``images``).  Copies to the host (synchronises)."""
    r = dict(zip(_lib.EVAL_COUNTER_NAMES, (int(v) for v in counters.tolist())))
    r["top1_pct"] = 100.0 * r["top1"] / max(r["images"], 1)
    r["top5_pct"] = 100.0 * r["top5"] / max(r["images"], 1)
    return r


class _Graph:
    """One captured forward (``b200q_*graph_create*``): fixed batch, fixed input / logits buffers, private workspace.
    ``u8``: ``x`` holds uint8 NHWC pixels (``b200q_graph_create_u8``), else fp32 NCHW images."""

    def __init__(self, engine, x: torch.Tensor, logits: torch.Tensor, pdl: bool, u8: bool = False):
        lib = engine.lib
        b = x.shape[0]
        self.x, self.logits = x, logits  # keeps the captured buffers alive
        self.ws = torch.empty(int(lib.b200q_static_workspace_bytes(b)), dtype=torch.uint8, device=engine.device)
        self.handle = C.c_void_p()
        self.lib = lib
        cur = torch.cuda.current_stream(engine.device)
        side = engine._capture_stream()
        side.wait_stream(cur)
        flags = _lib.GRAPH_PDL if pdl else 0
        engine._create_graph(x, logits, self.ws, flags, side.cuda_stream, C.byref(self.handle), u8)
        cur.wait_stream(side)

    def launch(self, stream: int):
        _lib.check(self.lib.b200q_graph_launch(self.handle, stream), "graph_launch")

    def __del__(self):
        try:  # may run during interpreter shutdown, after the library or the CUDA context is gone
            if getattr(self, "handle", None):
                self.lib.b200q_graph_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class _NetEngine:
    """What the whole-network engines share: eager workspaces (one per CUDA stream, LRU) and the whole-network executor
    (SURVEY 8f rank 1).  Batches of at most ``GRAPH_MAX_BATCH`` images - the latency-bound regime the reference's own
    driver measures (``utils/inference_benchmark.py:126-138``: batch 1 and 32) - are replayed from a CUDA graph
    captured on the caller's input buffer, with programmatic dependent launch between the layer kernels.  A graph is
    captured the second time the same (input kind, batch, input buffer[, output buffer]) is seen and ``GRAPH_CACHE`` of
    them are kept (least recently used evicted).  Subclasses provide ``_create_graph``."""

    GRAPH_MAX_BATCH = 1024
    GRAPH_CACHE = 8
    WORKSPACE_CACHE = 4  # eager workspaces kept, one per CUDA stream that called forward (LRU)

    def __init__(self, device, use_graphs: bool, pdl: bool):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.B200QError(f"{type(self).__name__} needs a CUDA device (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.lib = _lib.load()
        self.use_graphs, self.pdl = use_graphs, pdl
        self._ws = OrderedDict()      # CUDA stream handle -> workspace (forwards on different streams must not share one)
        self._graphs = OrderedDict()  # (uint8 input?, batch, x ptr, out ptr or 0) -> _Graph
        self._seen = OrderedDict()    # keys seen once (capture on the second sighting)
        self._side = None

    def _create_graph(self, x, logits, ws, flags: int, stream: int, handle_ref, u8: bool) -> None:
        raise NotImplementedError

    def _capture_stream(self):
        if self._side is None:
            self._side = torch.cuda.Stream(self.device)
        return self._side

    def release(self):
        """Drop cached workspaces and captured graphs (device memory goes back to torch's allocator)."""
        self._ws.clear()
        self._graphs.clear()
        self._seen.clear()

    def _workspace(self, b: int) -> torch.Tensor:
        need = int(self.lib.b200q_static_workspace_bytes(b))
        key = torch.cuda.current_stream(self.device).cuda_stream
        ws = self._ws.pop(key, None)
        if ws is None or ws.numel() < need:
            ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        self._ws[key] = ws
        while len(self._ws) > self.WORKSPACE_CACHE:  # short-lived streams must not pin memory for ever
            self._ws.popitem(last=False)
        return ws

    def _check_input(self, x: torch.Tensor, shape, dtype, what: str):
        if not x.is_cuda or x.device != self.device:
            raise _lib.B200QError(f"{what}: expected a tensor on {self.device}, got {x.device}")
        if x.dtype != dtype:
            raise _lib.B200QError(f"{what}: expected {dtype}, got {x.dtype}")
        if x.dim() != 4 or tuple(x.shape[1:]) != shape:
            raise _lib.B200QError(f"{what}: expected [B,{','.join(map(str, shape))}] input, got {tuple(x.shape)}")

    def _check_out(self, out, b: int):
        if out is None:
            return
        if (not out.is_cuda or out.device != self.device or out.dtype != torch.float32 or tuple(out.shape) != (b, 10)
                or not out.is_contiguous()):
            raise _lib.B200QError(f"out must be a contiguous fp32 [{b},10] tensor on {self.device}, got "
                                  f"{out.dtype} {tuple(out.shape)} on {out.device}")

    def _graph_for(self, x: torch.Tensor, out, u8: bool = False):
        """The captured graph for this (input kind, batch, input buffer, output buffer), or None (not yet / not
        eligible)."""
        key = (u8, x.shape[0], x.data_ptr(), 0 if out is None else out.data_ptr())
        g = self._graphs.get(key)
        if g is not None:
            self._graphs.move_to_end(key)
            return g
        if key not in self._seen:  # one-off buffers (an evaluation sweep over fresh tensors) are not worth a capture
            self._seen[key] = True
            while len(self._seen) > 64:
                self._seen.popitem(last=False)
            return None
        del self._seen[key]
        logits = out if out is not None else torch.empty((x.shape[0], 10), dtype=torch.float32, device=self.device)
        g = _Graph(self, x, logits, self.pdl, u8)
        self._graphs[key] = g
        while len(self._graphs) > self.GRAPH_CACHE:
            self._graphs.popitem(last=False)
        return g

    def _replay(self, x: torch.Tensor, out, graph, u8: bool = False):
        """Logits from a graph replay on the current stream when the policy (or ``graph=True``) says so, else None."""
        use_graph = self.use_graphs and x.shape[0] <= self.GRAPH_MAX_BATCH if graph is None else graph
        if not use_graph:
            return None
        g = self._graph_for(x, out, u8)
        if g is None and graph:  # forced: capture right away
            g = self._graph_for(x, out, u8)
        if g is None:
            return None
        g.launch(_current_stream_handle(self.device.index))
        return out if out is not None else g.logits.clone()

    def _tap_buffers(self, b: int, names, shapes):
        """uint8 NHWC tap tensors by name and the C array of their pointers."""
        arr = (C.c_void_p * len(names))()
        tensors = {}
        for i, name in enumerate(names):
            t = torch.empty((b,) + shapes[name], dtype=torch.uint8, device=self.device)
            tensors[name] = t
            arr[i] = t.data_ptr()
        return tensors, arr


class StaticEngine(_NetEngine):
    """Runs ``b200q_static_forward`` on one CUDA device.  fp32 NCHW ``[B,3,32,32]`` (CUDA) -> fp32 logits ``[B,10]``.
    Small batches run on the whole-network executor (``_NetEngine``).  ``forward_u8`` (raw uint8 pixels) follows the
    same policy; its graphs share the cache, keyed apart by the input kind."""

    def __init__(self, qparams: dict, device="cuda", use_graphs: bool = True, pdl: bool = True):
        super().__init__(device, use_graphs, pdl)
        self.qparams = qparams
        with torch.cuda.device(self.device):
            self.packed = PackedStaticNet(qparams, self.device)

    def _create_graph(self, x, logits, ws, flags, stream, handle_ref, u8):
        if u8:
            rc = self.lib.b200q_graph_create_u8(self.packed.ptr(), x.data_ptr(), self.packed.input_lut.data_ptr(),
                                                logits.data_ptr(), x.shape[0], ws.data_ptr(), ws.numel(), flags, stream,
                                                handle_ref)
        else:
            rc = self.lib.b200q_graph_create(self.packed.ptr(), x.data_ptr(), logits.data_ptr(), x.shape[0],
                                             ws.data_ptr(), ws.numel(), flags, stream, handle_ref)
        _lib.check(rc, "graph_create_u8" if u8 else "graph_create")

    @torch.no_grad()
    def forward(self, x: torch.Tensor, taps: bool = False, out: torch.Tensor | None = None, graph: bool | None = None):
        """``out`` (optional): preallocated fp32 ``[B,10]`` CUDA tensor to receive the logits.  ``graph``: force
        (True) or forbid (False) the CUDA-graph executor; default: use it for small batches."""
        if x.is_cuda and x.dtype != torch.float32:
            x = x.float()
        x = x.contiguous()
        self._check_input(x, (3, 32, 32), torch.float32, "StaticEngine.forward")
        b = x.shape[0]
        self._check_out(out, b)
        # small batches are latency-bound down to the Python level: skip the device context manager when the engine's
        # device is already current (the common, single-GPU-per-process case)
        ctx = _NULL_CTX if torch.cuda.current_device() == self.device.index else torch.cuda.device(self.device)
        with ctx:
            if b == 0:
                logits = out if out is not None else torch.empty((0, 10), dtype=torch.float32, device=self.device)
                return (logits, {}) if taps else logits
            if not taps:
                y = self._replay(x, out, graph)
                if y is not None:
                    return y
            logits = out if out is not None else torch.empty((b, 10), dtype=torch.float32, device=self.device)
            ws = self._workspace(b)
            tap_ptrs = None
            tap_tensors = {}
            if taps:
                tap_tensors, tap_ptrs = self._tap_buffers(b, TAP_NAMES, TAP_SHAPES)
            rc = self.lib.b200q_static_forward(self.packed.ptr(), x.data_ptr(), logits.data_ptr(), b, ws.data_ptr(),
                                               ws.numel(), tap_ptrs, torch.cuda.current_stream().cuda_stream)
            _lib.check(rc, "static_forward")
        return (logits, tap_tensors) if taps else logits

    __call__ = forward

    @torch.no_grad()
    def forward_u8(self, x_u8: torch.Tensor, out: torch.Tensor | None = None, graph: bool | None = None) -> torch.Tensor:
        """uint8 data path: raw pixels, uint8 NHWC ``[B,32,32,3]`` (CUDA) -> fp32 logits ``[B,10]``; bit-identical to
        ``forward(synth.normalize(pixels))`` (``packing.input_lut``).  ``out`` and ``graph`` as for ``forward``."""
        x_u8 = x_u8.contiguous()
        self._check_input(x_u8, (32, 32, 3), torch.uint8, "StaticEngine.forward_u8")
        b = x_u8.shape[0]
        self._check_out(out, b)
        ctx = _NULL_CTX if torch.cuda.current_device() == self.device.index else torch.cuda.device(self.device)
        with ctx:
            if b == 0:
                return out if out is not None else torch.empty((0, 10), dtype=torch.float32, device=self.device)
            y = self._replay(x_u8, out, graph, u8=True)
            if y is not None:
                return y
            logits = out if out is not None else torch.empty((b, 10), dtype=torch.float32, device=self.device)
            ws = self._workspace(b)
            rc = self.lib.b200q_static_forward_u8(self.packed.ptr(), x_u8.data_ptr(), self.packed.input_lut.data_ptr(),
                                                  logits.data_ptr(), b, ws.data_ptr(), ws.numel(),
                                                  torch.cuda.current_stream().cuda_stream)
            _lib.check(rc, "static_forward_u8")
        return logits

    def _check_eval_args(self, b: int, labels, counters, pred):
        def bad(t, dtype, shape):
            return (not torch.is_tensor(t) or not t.is_cuda or t.device != self.device or t.dtype != dtype
                    or tuple(t.shape) != shape or not t.is_contiguous())
        for name, t, dtype, shape in (("counters", counters, torch.int64, (_lib.EVAL_COUNTERS,)),
                                      ("pred", pred, torch.int32, (b,)),
                                      ("labels", labels, torch.int64, (b,))):
            if (t is not None or name == "labels") and bad(t, dtype, shape):
                got = f"{t.dtype} {tuple(t.shape)} on {t.device}" if torch.is_tensor(t) else type(t).__name__
                raise _lib.B200QError(f"{name} must be a contiguous {dtype} {list(shape)} tensor on {self.device}, "
                                      f"got {got}")

    @torch.no_grad()
    def _evaluate(self, x, labels, counters, pred, logits, u8: bool) -> torch.Tensor:
        b = x.shape[0]
        self._check_eval_args(b, labels, counters, pred)
        self._check_out(logits, b)
        ctx = _NULL_CTX if torch.cuda.current_device() == self.device.index else torch.cuda.device(self.device)
        with ctx:
            if counters is None:
                counters = torch.zeros(_lib.EVAL_COUNTERS, dtype=torch.int64, device=self.device)
            if b == 0:
                return counters
            ws = self._workspace(b)
            ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
            stream = torch.cuda.current_stream().cuda_stream
            if u8:
                rc = self.lib.b200q_static_evaluate_u8(self.packed.ptr(), x.data_ptr(), self.packed.input_lut.data_ptr(),
                                                       labels.data_ptr(), b, counters.data_ptr(), ptr(pred), ptr(logits),
                                                       ws.data_ptr(), ws.numel(), stream)
            else:
                rc = self.lib.b200q_static_evaluate(self.packed.ptr(), x.data_ptr(), labels.data_ptr(), b,
                                                    counters.data_ptr(), ptr(pred), ptr(logits), ws.data_ptr(),
                                                    ws.numel(), stream)
            _lib.check(rc, "static_evaluate_u8" if u8 else "static_evaluate")
        return counters

    def evaluate(self, x: torch.Tensor, labels: torch.Tensor, counters: torch.Tensor | None = None,
                 pred: torch.Tensor | None = None, logits: torch.Tensor | None = None) -> torch.Tensor:
        """Top-1 / top-5 counting inside the classifier head (``b200q_static_evaluate``; the tie rule is in
        ``include/b200q.h``).  ``x``: fp32 NCHW ``[B,3,32,32]``, ``labels``: int64 ``[B]``, both on this device.
        Returns the int64 ``[5]`` counters ``_lib.EVAL_COUNTER_NAMES`` - ``counters`` when given (ACCUMULATED into),
        else a fresh zeroed tensor.  Optional outputs: ``pred`` int32 ``[B]`` (rank-0 class) and ``logits`` fp32
        ``[B,10]`` (what ``forward`` returns).  Runs eagerly on the current stream (no CUDA graph) and never
        synchronises: read the counters when the stream has got there."""
        x = x.contiguous()
        self._check_input(x, (3, 32, 32), torch.float32, "StaticEngine.evaluate")
        return self._evaluate(x, labels, counters, pred, logits, u8=False)

    def evaluate_u8(self, x_u8: torch.Tensor, labels: torch.Tensor, counters: torch.Tensor | None = None,
                    pred: torch.Tensor | None = None, logits: torch.Tensor | None = None) -> torch.Tensor:
        """``evaluate`` from raw pixels, uint8 NHWC ``[B,32,32,3]`` (the input of ``forward_u8``)."""
        x_u8 = x_u8.contiguous()
        self._check_input(x_u8, (32, 32, 3), torch.uint8, "StaticEngine.evaluate_u8")
        return self._evaluate(x_u8, labels, counters, pred, logits, u8=True)

    def stage_names(self):
        return [self.lib.b200q_static_stage_name(i).decode() for i in range(self.lib.b200q_static_num_stages())]

    @torch.no_grad()
    def forward_profiled(self, x: torch.Tensor):
        """(logits, {stage: ms}) — one forward with a CUDA event between kernels (measurement hook; synchronises)."""
        x = x.contiguous().float()
        self._check_input(x, (3, 32, 32), torch.float32, "StaticEngine.forward_profiled")
        b = x.shape[0]
        n = self.lib.b200q_static_num_stages()
        ms = (C.c_float * n)()
        with torch.cuda.device(self.device):
            logits = torch.empty((b, 10), dtype=torch.float32, device=self.device)
            ws = self._workspace(b)
            rc = self.lib.b200q_static_forward_profiled(self.packed.ptr(), x.data_ptr(), logits.data_ptr(), b,
                                                        ws.data_ptr(), ws.numel(), ms,
                                                        torch.cuda.current_stream().cuda_stream)
            _lib.check(rc, "static_forward_profiled")
        return logits, dict(zip(self.stage_names(), (float(v) for v in ms)))


class SandwichEngine(_NetEngine):
    """Runs ``b200q_sandwich_forward`` (the per-layer sandwich net, ``ptq.calibrate_sandwich`` parameters) on one CUDA
    device: fp32 NCHW ``[B,3,32,32]`` (CUDA) -> fp32 logits ``[B,10]``, with the executor policy of ``_NetEngine``.
    The logits of an image do not depend on the batch it comes in, nor on eager / graph / PDL: the fp32 head has one
    fixed summation order (``include/b200q.h``, restated in numpy by ``tests/test_gpu_sandwich_forward.py``)."""

    def __init__(self, sparams: dict, device="cuda", use_graphs: bool = True, pdl: bool = True):
        super().__init__(device, use_graphs, pdl)
        self.sparams = sparams
        with torch.cuda.device(self.device):
            self.packed = PackedSandwichNet(sparams, self.device)

    def _create_graph(self, x, logits, ws, flags, stream, handle_ref, u8):
        rc = self.lib.b200q_sandwich_graph_create(self.packed.ptr(), x.data_ptr(), logits.data_ptr(), x.shape[0],
                                                  ws.data_ptr(), ws.numel(), flags, stream, handle_ref)
        _lib.check(rc, "sandwich_graph_create")

    @torch.no_grad()
    def forward(self, x: torch.Tensor, taps: bool = False, out: torch.Tensor | None = None, graph: bool | None = None):
        """``taps``: also return ``{layer: uint8 NHWC output}`` of conv1..conv6 (un-pooled) and fc1 (``[B,512]``), the
        int8 layers' outputs before ReLU.  ``out`` and ``graph`` as for ``StaticEngine.forward``."""
        if x.is_cuda and x.dtype != torch.float32:
            x = x.float()
        x = x.contiguous()
        self._check_input(x, (3, 32, 32), torch.float32, "SandwichEngine.forward")
        b = x.shape[0]
        self._check_out(out, b)
        ctx = _NULL_CTX if torch.cuda.current_device() == self.device.index else torch.cuda.device(self.device)
        with ctx:
            if b == 0:
                logits = out if out is not None else torch.empty((0, 10), dtype=torch.float32, device=self.device)
                return (logits, {}) if taps else logits
            if not taps:
                y = self._replay(x, out, graph)
                if y is not None:
                    return y
            logits = out if out is not None else torch.empty((b, 10), dtype=torch.float32, device=self.device)
            ws = self._workspace(b)
            tap_tensors, tap_ptrs = self._tap_buffers(b, SANDWICH_TAP_NAMES, TAP_SHAPES) if taps else ({}, None)
            rc = self.lib.b200q_sandwich_forward(self.packed.ptr(), x.data_ptr(), logits.data_ptr(), b, ws.data_ptr(),
                                                 ws.numel(), tap_ptrs, _current_stream_handle(self.device.index))
            _lib.check(rc, "sandwich_forward")
        return (logits, tap_tensors) if taps else logits

    __call__ = forward
