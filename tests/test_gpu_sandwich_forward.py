"""The sandwich net's native forward (``b200q_sandwich_forward``), its CUDA-graph executor
(``b200q_sandwich_graph_create``) and the fixed-order fp32 head, through ``engine.SandwichEngine`` and
``CustomQuantizationModel(mode="sandwich")``.

The head's summation order is part of the interface (``include/b200q.h``), so the logits are compared EXACTLY with a
numpy restatement: the int8 layers of ``oracle.int_ops.sandwich_forward`` followed by ``head_fixed_order`` below.
The CPU-only tests at the end check the C-ABI surface, the struct layout and the argument checks without a device."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# 1, 2: tiny conv kernels; 3 / 31-33 / 37 / 38 / 74 / 75 / 148 / 149 / 445: either side of the small-batch head (32 | 33)
# and of the conv kernel switches on 148 SMs; 2 305: fc1's wide tile; 4 099: many persistent rounds
LOGIT_SIZES = (1, 2, 3, 31, 32, 33, 37, 38, 74, 75, 148, 149, 445, 2305, 4099)
GRAPH_SIZES = (1, 2, 7, 32, 33, 128, 1024)
SAMPLE = 48
GUARD = 8192
SENTINEL = 0xA5


class Guarded:
    """A device buffer inside a larger allocation pre-filled with a sentinel (stray stores show in the bands)."""

    def __init__(self, shape, dtype):
        self.nbytes = int(torch.empty(shape, dtype=dtype).numel() * torch.empty((), dtype=dtype).element_size())
        self.raw = torch.full((2 * GUARD + self.nbytes,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.view = self.raw[GUARD:GUARD + self.nbytes].view(dtype).view(shape)

    def intact(self) -> bool:
        torch.cuda.synchronize()
        front, back = self.raw[:GUARD], self.raw[GUARD + self.nbytes:]
        return bool((front == SENTINEL).all()) and bool((back == SENTINEL).all())


@pytest.fixture(scope="module")
def sp(fp32_net):
    from convnet_quantization_b200 import ptq, synth
    return ptq.calibrate_sandwich(fp32_net, synth.calibration_batches())


@pytest.fixture(scope="module")
def sp_np(sp):
    from tests.conftest import qparams_to_numpy
    return qparams_to_numpy(sp)


@pytest.fixture(scope="module")
def engines(sp):
    """SandwichEngine with PDL on and off (module scope: their graph caches persist across the tests)."""
    from convnet_quantization_b200.engine import SandwichEngine
    return {True: SandwichEngine(sp, "cuda", pdl=True), False: SandwichEngine(sp, "cuda", pdl=False)}


def _images(b: int, seed: int) -> torch.Tensor:
    """Synthetic images x 3: conv1's QuantStub saturates at both ends."""
    from convnet_quantization_b200 import synth
    return synth.images_f32(b, seed=seed) * 3


def _sample(b: int, seed: int) -> np.ndarray:
    if b <= SAMPLE:
        return np.arange(b)
    idx = {0, 1, 31, 32, 33, b - 2, b - 1} & set(range(b))
    rest = np.setdiff1d(np.arange(b), np.fromiter(idx, dtype=np.int64))
    fill = np.random.default_rng(seed).choice(rest, size=SAMPLE - len(idx), replace=False)
    return np.sort(np.concatenate([np.fromiter(idx, dtype=np.int64), fill]))


def head_fixed_order(h_u8: np.ndarray, zp: int, scale: float, w: np.ndarray, b: np.ndarray) -> np.ndarray:
    """The sandwich net's fp32 head in the summation order ``b200q_sandwich_forward`` defines (``include/b200q.h``):
    ``h = f32(max(q, zp) - zp) * scale`` (fc1's ReLU + DeQuantStub); per output n, 32 partial sums over k = 16l..16l+15
    in increasing k; the partials added by an XOR butterfly at distances 16, 8, 4, 2, 1; then the bias.  numpy float32
    rounds after every operation and never fuses a multiply with an add, which is the arithmetic wanted.
    h_u8 uint8 [B, 512], w [10, 512], b [10] -> float32 [B, 10]."""
    f32 = np.float32
    q = np.asarray(h_u8).astype(np.int32)
    h = (np.maximum(q, int(zp)) - int(zp)).astype(f32) * f32(scale)                  # [B, 512]
    w = np.asarray(w, dtype=f32)
    prod = (h[:, None, :] * w[None, :, :]).reshape(h.shape[0], w.shape[0], 32, 16)   # [B, N, lane, j], rounded products
    p = prod[..., 0]
    for j in range(1, 16):
        p = p + prod[..., j]
    lanes = np.arange(32)
    for d in (16, 8, 4, 2, 1):
        p = p + p[..., lanes ^ d]
    return p[..., 0] + np.asarray(b, dtype=f32)


def _restated(x: np.ndarray, sp_np: dict):
    """(logits, taps) of the numpy restatement: the oracle's int8 layers, then the fixed-order fp32 head."""
    from oracle import int_ops as IO
    taps = {}
    IO.sandwich_forward(x, sp_np, taps)
    L, fc2 = sp_np["fc1"], sp_np["fc2"]
    return head_fixed_order(taps["fc1"], L["out_zp"], L["out_scale"], fc2["weight"], fc2["bias"]), taps


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------------------------ exactness
@gpu
@pytest.mark.parametrize("b", LOGIT_SIZES)
def test_sandwich_logits_and_taps_bit_exact_against_restatement(engines, sp_np, b):
    """Production route (eager) and taps route: logits bit-exact against the restatement, the seven taps bit-exact
    against the integer oracle, on a sample of the batch."""
    eng = engines[True]
    x = _images(b, seed=600 + b)
    xd = x.cuda()
    logits = eng.forward(xd, graph=False)
    tl, taps = eng.forward(xd, taps=True)
    idx = _sample(b, seed=b)
    want, want_taps = _restated(x[idx].numpy(), sp_np)
    assert set(taps) == set(want_taps)
    for n, t in taps.items():
        got = t[idx].cpu().numpy()
        assert np.array_equal(got, want_taps[n]), f"{n} tap, b={b}: {int((got != want_taps[n]).sum())} bytes differ"
    assert (want_taps["fc1"] < sp_np["fc1"]["out_zp"]).any() and (want_taps["fc1"] > sp_np["fc1"]["out_zp"]).any()
    assert np.array_equal(logits[idx].cpu().numpy(), want), f"b={b}: production logits differ from the restatement"
    assert torch.equal(tl, logits), f"b={b}: taps route logits differ from the production route"


@gpu
def test_sandwich_logits_against_golden(golden, fp32_net):
    """With the activation qparams pinned to ``sandwich_golden.npz`` (the reference's own wrapper class): logits within
    1e-3 of the golden's fp32 GEMM, the same argmax, and bit-exact against the restatement."""
    from convnet_quantization_b200 import ptq, synth
    from convnet_quantization_b200.engine import SandwichEngine
    from oracle import torch_oracle as TO
    from tests.conftest import qparams_to_numpy
    g = np.load(os.path.join(ROOT, "tests", "golden", "sandwich_golden.npz"))
    sp = ptq.calibrate_sandwich(fp32_net, synth.calibration_batches())
    for n in TO.SANDWICH_LAYERS:
        sp[n]["in_scale"], sp[n]["in_zp"] = float(g[f"{n}_qparams"][0]), int(g[f"{n}_qparams"][1])
        sp[n]["out_scale"], sp[n]["out_zp"] = float(g[f"{n}_qparams"][2]), int(g[f"{n}_qparams"][3])
    x = synth.normalize(torch.from_numpy(golden["x_u8"])).contiguous()
    got = SandwichEngine(sp, "cuda").forward(x.cuda(), graph=False).cpu().numpy()
    want = g["sandwich_logits"]
    np.testing.assert_allclose(got, want, rtol=1e-3, atol=1e-3 * np.abs(want).max())
    assert np.array_equal(got.argmax(1), want.argmax(1))
    assert np.array_equal(got, _restated(x.numpy(), qparams_to_numpy(sp))[0])


@gpu
def test_sandwich_logits_do_not_depend_on_the_batch(sp, engines):
    """The same image gives the same bytes alone, inside batches of 33 and 2 305, through the host chunk pipeline (two
    full chunks and a split tail), eagerly, and from graphs with and without PDL."""
    from convnet_quantization_b200.models._gpu_modules import B200SandwichQuantizedNet
    net = B200SandwichQuantizedNet(sp, "cuda")
    b = 2 * net.HOST_CHUNK + 4 * net.TAIL_MIN + 7
    chunks = list(net._chunks(b))
    assert len(chunks) == 4 and chunks[3][1] < chunks[2][1] < net.HOST_CHUNK, chunks
    x = _images(b, seed=5)
    want = engines[True].forward(x.cuda(), graph=False)
    assert torch.equal(net(x), want.cpu())  # host input
    assert torch.equal(net(x.cuda()), want)
    for lo, n in ((0, 1), (2047, 1), (b - 1, 1), (0, 33), (2040, 33), (1000, 2305)):
        xs = x[lo:lo + n].cuda()
        assert torch.equal(engines[True].forward(xs, graph=False), want[lo:lo + n]), (lo, n)
        if n <= 1024:
            for pdl in (True, False):
                assert torch.equal(engines[pdl].forward(xs, graph=True), want[lo:lo + n]), (lo, n, pdl)
                assert torch.equal(engines[pdl].forward(xs, graph=True), want[lo:lo + n]), (lo, n, pdl)  # replay


# ------------------------------------------------------------------------------------------------ executor
@gpu
@pytest.mark.parametrize("pdl", [True, False], ids=["pdl", "no_pdl"])
@pytest.mark.parametrize("b", GRAPH_SIZES)
def test_sandwich_graph_replay_equals_eager(engines, b, pdl):
    """Replays read the captured input buffer: rewriting it between replays gives the eager logits of the new input."""
    eng = engines[pdl]
    xbuf = _images(b, seed=700 + b).cuda()
    out = torch.empty((b, 10), device="cuda")
    eng.forward(xbuf, out=out, graph=True)  # capture (and one replay)
    for seed in (1, 2):
        xbuf.copy_(_images(b, seed=700 + b + seed))
        want = eng.forward(xbuf, graph=False)
        out.zero_()
        assert eng.forward(xbuf, out=out, graph=True) is out
        assert torch.equal(out, want), f"b={b} pdl={pdl}"


def _plain(name: str) -> str:
    return name.replace(" ", "").replace("(int)", "").replace("(bool)0", "false").replace("(bool)1", "true")


@gpu
def test_sandwich_launch_accounting_and_kernel_order(sp):
    """b200q_launch_count rises by 14 per eager forward (13 up to 32 images); a replay counts the kernels it stands for;
    the profiler lists the expected kernels in order, and nothing else (no library GEMM)."""
    from torch.profiler import ProfilerActivity, profile
    from convnet_quantization_b200 import _lib
    from convnet_quantization_b200.engine import SandwichEngine
    lib = _lib.load()
    eng = SandwichEngine(sp, "cuda")
    xs = {b: _images(b, seed=b).cuda() for b in (1, 32, 33, 300)}
    for b, x in xs.items():
        n0 = lib.b200q_launch_count()
        eng.forward(x, graph=False)
        assert lib.b200q_launch_count() - n0 == (13 if b <= 32 else 14), b
    for b in (1, 33):
        eng.forward(xs[b], graph=True)  # capture
        n0 = lib.b200q_launch_count()
        for _ in range(3):
            eng.forward(xs[b], graph=True)
        assert lib.b200q_launch_count() - n0 == 3 * (13 if b <= 32 else 14), b
    torch.cuda.synchronize()
    for b in (1, 300):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.forward(xs[b], graph=False)
            torch.cuda.synchronize()
        names = [_plain(e.name) for e in sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                                                 and not e.name.startswith(("Memcpy", "Memset"))),
                                                key=lambda e: e.time_range.start)]
        assert len(names) == (13 if b <= 32 else 14), names
        assert "conv1" in names[0]
        assert all("lut_u8_kernel" in names[i] for i in (1, 3, 5, 7, 9, 11)), names
        assert not any("lut_u8_kernel" in names[i] for i in (2, 4, 6, 8, 10)), names
        if b <= 32:
            assert "fc_head_small_kernel<false,true>" in names[12], names
        else:
            assert "igemm_tc_kernel<0,4096,512" in names[12] and "sandwich_head_kernel" in names[13], names


@gpu
@pytest.mark.parametrize("b", [1, 32, 33, 149, 2305])
def test_sandwich_forward_writes_only_its_outputs(engines, b):
    """Logits and an exactly-sized workspace between sentinel bands, eager (and graph up to 1 024 images): the bands
    stay untouched and the payload equals an ordinary call."""
    from convnet_quantization_b200 import _lib
    lib = _lib.load()
    eng = engines[True]
    x = _images(b, seed=800 + b).cuda()
    want = eng.forward(x, graph=False)
    ws_bytes = int(lib.b200q_static_workspace_bytes(b))
    ws = Guarded((ws_bytes,), torch.uint8)
    out = Guarded((b, 10), torch.float32)
    _lib.check(lib.b200q_sandwich_forward(eng.packed.ptr(), x.data_ptr(), out.view.data_ptr(), b, ws.view.data_ptr(),
                                          ws_bytes, None, _stream()), "sandwich_forward")
    assert ws.intact(), f"b={b}: wrote outside the workspace"
    assert out.intact(), f"b={b}: wrote outside the logits"
    assert torch.equal(out.view, want)
    if b > 1024:
        return
    out.view.zero_()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    gh = C.c_void_p()
    with torch.cuda.stream(side):
        _lib.check(lib.b200q_sandwich_graph_create(eng.packed.ptr(), x.data_ptr(), out.view.data_ptr(), b,
                                                   ws.view.data_ptr(), ws_bytes, _lib.GRAPH_PDL, side.cuda_stream,
                                                   C.byref(gh)), "sandwich_graph_create")
        try:
            for _ in range(3):
                _lib.check(lib.b200q_graph_launch(gh, side.cuda_stream), "graph_launch")
            side.synchronize()
            assert ws.intact() and out.intact(), f"b={b}: graph wrote outside its buffers"
            assert torch.equal(out.view, want)
        finally:
            side.synchronize()
            _lib.check(lib.b200q_graph_destroy(gh), "graph_destroy")


@gpu
def test_sandwich_graph_concurrent_with_eager_on_another_stream(engines):
    """One engine: graph replays on one stream while a 4 096-image eager forward runs on another == each run alone."""
    eng = engines[True]
    xs = _images(32, seed=77).cuda()
    xl = _images(4096, seed=78).cuda()
    want_s = eng.forward(xs, graph=False)
    want_l = eng.forward(xl, graph=False)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    out_s = torch.empty((32, 10), device="cuda")
    out_l = torch.empty((4096, 10), device="cuda")
    for s in (s1, s2):
        s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s1):
        eng.forward(xs, out=out_s, graph=True)  # capture
    s1.synchronize()
    results = []
    for _ in range(3):
        out_s.zero_()
        with torch.cuda.stream(s2):
            eng.forward(xl, out=out_l, graph=False)
        with torch.cuda.stream(s1):
            for _ in range(4):
                eng.forward(xs, out=out_s, graph=True)
        s1.synchronize()
        s2.synchronize()
        results.append((out_s.clone(), out_l.clone()))
    for o_s, o_l in results:
        assert torch.equal(o_s, want_s)
        assert torch.equal(o_l, want_l)


# ------------------------------------------------------------------------------------------------ model class
@gpu
def test_custom_sandwich_model_runs_on_the_engine():
    """``CustomQuantizationModel(mode="sandwich")``: CUDA and host inputs equal ``engine.forward`` bit for bit, and the
    reference's ``compare_models`` driver runs it."""
    from convnet_quantization_b200 import drivers, synth
    from convnet_quantization_b200.models.custom_quantization_model import CustomQuantizationModel
    cm = CustomQuantizationModel(mode="sandwich")
    cm.load_state_dict(synth.make_state_dict(0))
    q = cm.quantize()
    x = _images(37, seed=9)
    want = q.engine.forward(x.cuda(), graph=False)
    assert torch.equal(cm(x.cuda()), want)
    got = cm(x)
    assert not got.is_cuda and torch.equal(got, want.cpu())
    _, taps = q.forward_with_taps(x)
    assert tuple(taps["conv2"].shape) == (37, 32, 32, 64) and tuple(taps["fc1"].shape) == (37, 512)
    loader = synth.SyntheticLoader(64, 32, seed=5)
    res = drivers.InferenceBenchmark(loader, device="cuda").compare_models({"custom sandwich (B200)": q}, batch_size=32,
                                                                           num_iterations=5, verbose=False)
    assert res["custom sandwich (B200)"] > 0


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_custom_sandwich_model_rehomes_to_another_gpu():
    from convnet_quantization_b200 import synth
    from convnet_quantization_b200.models.custom_quantization_model import CustomQuantizationModel
    cm = CustomQuantizationModel(mode="sandwich")
    cm.load_state_dict(synth.make_state_dict(0))
    q = cm.quantize()
    x = _images(33, seed=10)
    want = q(x.cuda()).cpu()
    q.to("cuda:1")
    assert q.engine.device == torch.device("cuda", 1)
    got = q(x.to("cuda:1"))
    assert got.device == torch.device("cuda", 1) and torch.equal(got.cpu(), want)
    assert torch.equal(q(x), want)


# ------------------------------------------------------------------------------------------------ CPU only
def test_header_declares_the_sandwich_entries_and_binding_matches():
    from convnet_quantization_b200 import _lib
    text = open(os.path.join(ROOT, "include", "b200q.h")).read()
    for name, n in (("b200q_sandwich_forward", 8), ("b200q_sandwich_graph_create", 9)):
        m = re.search(rf"int {name}\(([^)]*)\);", text)
        assert m, f"include/b200q.h must declare {name}"
        assert len(m.group(1).split(",")) == n == len(_lib._SIGNATURES[name])
        assert name in _lib.EXPORTS
    assert "const b200q_sandwich_net* net" in text


_LAYOUT_C = r"""
#include <stddef.h>
#include <stdio.h>
#include "b200q.h"
#define F(m) printf("%s %zu\n", #m, offsetof(b200q_sandwich_net, m));
int main(void) {
  printf("sizeof %zu\n", sizeof(b200q_sandwich_net));
  F(in_inv_scale) F(conv) F(fc1) F(lut_host) F(fc1_scale) F(fc2_w) F(fc2_b)
  printf("conv_stride %zu\n", sizeof(b200q_conv3x3));
  return 0;
}
"""


@pytest.mark.skipif(shutil.which("cc") is None and shutil.which("gcc") is None, reason="no host C compiler")
def test_sandwich_struct_layout_matches_ctypes(tmp_path):
    """sizeof / offsetof of every b200q_sandwich_net field, as the host compiler lays it out, equal the ctypes struct."""
    from convnet_quantization_b200 import _lib
    src, exe = tmp_path / "layout.c", tmp_path / "layout"
    src.write_text(_LAYOUT_C)
    cc = shutil.which("cc") or shutil.which("gcc")
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True,
                                                        check=True).stdout.splitlines())
    S = _lib.SandwichNet
    assert int(got["sizeof"]) == C.sizeof(S)
    for f, _ in S._fields_:
        assert int(got[f]) == getattr(S, f).offset, f
    assert int(got["conv_stride"]) == C.sizeof(_lib.Conv3x3)


def _valid_net():
    """A struct with the net's geometry and dangling (never dereferenced) device pointers."""
    from convnet_quantization_b200 import _lib
    net = _lib.SandwichNet()
    for i, (cin, cout, img) in enumerate(((4, 64, 32), (64, 64, 32), (64, 128, 16), (128, 128, 16), (128, 256, 8),
                                          (256, 256, 8))):
        net.conv[i].cin, net.conv[i].cout, net.conv[i].img = cin, cout, img
    net.fc1.k, net.fc1.n = 4096, 512
    net.fc2_w, net.fc2_b = 1 << 20, 1 << 20
    return net


def test_sandwich_forward_rejects_bad_arguments_before_any_cuda_call(lib):
    """Each call below fails its argument check before touching the device (the pointers are never dereferenced)."""
    fake = 1 << 20
    ws_ok = int(lib.b200q_static_workspace_bytes(4))

    def call(net, b=4, ws_bytes=ws_ok, x=fake):
        return lib.b200q_sandwich_forward(None if net is None else C.byref(net), x, fake, b, fake, ws_bytes, None, fake)

    def refused(net, what, **kw):
        assert call(net, **kw) == -1, what
        assert what.encode() in lib.b200q_last_error(), (what, lib.b200q_last_error())

    refused(None, "null net")
    refused(_valid_net(), "negative batch", b=-1)
    refused(_valid_net(), "null pointer", x=None)
    refused(_valid_net(), "workspace too small", ws_bytes=ws_ok - 1)
    for i, field in ((0, "cin"), (2, "cout"), (5, "img")):
        net = _valid_net()
        setattr(net.conv[i], field, getattr(net.conv[i], field) * 2)
        refused(net, f"conv{i + 1} geometry")
    for k, n in ((2048, 512), (4096, 256)):
        net = _valid_net()
        net.fc1.k, net.fc1.n = k, n
        refused(net, "fc1 must be 4096 -> 512")
    for field, value in (("fc2_w", None), ("fc2_b", None), ("fc2_w", (1 << 20) + 4), ("fc2_b", (1 << 20) + 2)):
        net = _valid_net()
        setattr(net, field, value)
        refused(net, "fc2")
    assert call(_valid_net(), b=0, x=None) == 0  # an empty batch enqueues nothing


def test_sandwich_graph_create_rejects_bad_arguments_before_any_cuda_call(lib):
    fake = 1 << 20
    ws_ok = int(lib.b200q_static_workspace_bytes(4))
    h = C.c_void_p()

    def call(net, out=C.byref(h), stream=fake, b=4, ws_bytes=ws_ok):
        return lib.b200q_sandwich_graph_create(None if net is None else C.byref(net), fake, fake, b, fake, ws_bytes, 0,
                                               stream, out)

    assert call(_valid_net(), out=None) == -1 and b"null out" in lib.b200q_last_error()
    assert call(None) == -1 and h.value is None
    assert call(_valid_net(), b=0) == -1 and b"empty batch" in lib.b200q_last_error()
    assert call(_valid_net(), stream=None) == -1 and b"legacy default stream" in lib.b200q_last_error()
    assert call(_valid_net(), ws_bytes=ws_ok - 1) == -1 and b"workspace too small" in lib.b200q_last_error()
    net = _valid_net()
    net.fc1.n = 10
    assert call(net) == -1 and b"fc1" in lib.b200q_last_error()


def test_fixed_order_head_is_close_to_float64():
    """The restatement of the fp32 head is a summation order, not another result: within 1e-6 relative of fc2 in
    float64 on the same dequantised inputs, and it depends on each row alone."""
    rng = np.random.default_rng(0)
    q = rng.integers(0, 256, (257, 512), dtype=np.uint8)
    q[0] = 255
    w = (rng.standard_normal((10, 512)) * 0.05).astype(np.float32)
    b = rng.standard_normal(10).astype(np.float32)
    zp, scale = 97, 0.0421
    got = head_fixed_order(q, zp, scale, w, b)
    assert got.dtype == np.float32 and got.shape == (257, 10)
    h = (np.maximum(q.astype(np.int32), zp) - zp).astype(np.float32) * np.float32(scale)
    ref = h.astype(np.float64) @ w.astype(np.float64).T + b.astype(np.float64)
    assert np.abs(got - ref).max() <= 1e-6 * np.abs(ref).max()
    assert np.array_equal(head_fixed_order(q[100:101], zp, scale, w, b), got[100:101])
