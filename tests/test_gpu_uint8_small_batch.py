"""uint8 pixel input at every batch size: the CUDA-core table-lookup conv1 (a few images, and layers the tensor-core
kernel refuses), the CUDA-graph executor for ``forward_u8`` (``b200q_graph_create_u8``), and their bookkeeping.

Every comparison is exact: the fp32 route on ``synth.normalize(pixels)`` and the torch/fbgemm CPU oracle are the
references.  The CPU-only tests at the end check the C-ABI surface and its argument checks without a device."""
import copy
import ctypes as C
import os
import re

import pytest
import torch

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

GUARD = 8192  # bytes either side; a multiple of every alignment the kernels ask for
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


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _pixels(b: int, seed: int, extreme: bool = False) -> torch.Tensor:
    """uint8 NHWC [b,32,32,3] on the host; ``extreme``: blocks of 0 and of 255 (saturated first-layer inputs)."""
    pix = torch.randint(0, 256, (b, 32, 32, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(seed))
    if extreme:
        pix[:, :8] = 0
        pix[:, 8:16] = 255
        pix[0] = 255
        pix[-1, :, 16:] = 0
    return pix


def _normalized(pix: torch.Tensor) -> torch.Tensor:
    from convnet_quantization_b200 import synth
    return synth.normalize(pix.permute(0, 3, 1, 2)).contiguous()


def _references(eng, oracle, pix):
    """(fp32-route logits on the device, CPU-oracle logits) for host pixels; asserts the two agree."""
    from oracle import torch_oracle as TO
    x = _normalized(pix)
    want = eng.forward(x.cuda(), graph=False)
    ref, _ = TO.run_static_oracle(oracle, x)
    assert torch.equal(want.cpu(), ref)
    return want, ref


def _conv1(qparams):
    from convnet_quantization_b200.packing import PackedConv, input_lut
    s, zp = qparams["in_scale"], qparams["in_zp"]
    return PackedConv("conv1", qparams["conv1"], s, zp, "cuda"), s, input_lut(s, zp)


@pytest.fixture(scope="module")
def unbounded(qparams, fp32_net):
    """Product qparams and a matching CPU oracle with conv1's output scale divided by 400: requantisation multipliers
    above 0.5, so conv1 is not B200Q_RQ_BOUNDED and the tensor-core first layer refuses it."""
    from convnet_quantization_b200 import synth
    from oracle import torch_oracle as TO
    qp = copy.deepcopy(qparams)
    qp["conv1"]["out_scale"] = float(qp["conv1"]["out_scale"]) / 400.0
    act = {"in": (qp["in_scale"], qp["in_zp"])}
    for n in ("conv1", "conv2", "conv3", "conv4", "conv5", "conv6", "fc1", "fc2"):
        act[n] = (float(qp[n]["out_scale"]), int(qp[n]["out_zp"]))
    oracle = TO.override_activation_qparams(TO.build_static_oracle(fp32_net, synth.calibration_batches()), act)
    return qp, oracle


def _drop_conv1_host_mirrors(packed):
    c = packed.c.conv[0]  # shares memory with the net struct the forward reads
    c.corr_host = None
    c.rq.mult_host = None
    c.rq.bdiv_host = None


# ------------------------------------------------------------------------------------------------ whole network
@gpu
@pytest.mark.parametrize("b", [1, 2, 3, 7, 31, 32, 33, 64, 128, 500, 1024, 1025])
@pytest.mark.parametrize("pdl", [True, False])
def test_uint8_forward_eager_and_graph_bit_exact(qparams, oracle_model, b, pdl):
    """forward_u8 eager and as a CUDA graph (with / without programmatic dependent launch) == fp32 route == CPU oracle,
    with different pixels in the captured buffer before every replay (one with all-0 / all-255 blocks), replays issued
    back to back, and a graph that writes straight into the caller's ``out``."""
    from convnet_quantization_b200.engine import StaticEngine
    eng = StaticEngine(qparams, "cuda", pdl=pdl)
    buf = torch.empty((b, 32, 32, 3), dtype=torch.uint8, device="cuda")
    out = torch.empty((b, 10), device="cuda")
    last = None
    for rep in range(3):
        pix = _pixels(b, 70 * b + rep, extreme=(rep == 1))
        buf.copy_(pix)
        want, ref = _references(eng, oracle_model, pix)
        assert torch.equal(eng.forward_u8(buf, graph=False), want), (b, rep, "eager")
        y = eng.forward_u8(buf, graph=True)  # rep 0: capture, then replays of the same graph
        assert torch.equal(y.cpu(), ref), (b, rep, "graph")
        assert eng.forward_u8(buf, out=out, graph=True) is out
        assert torch.equal(out, want), (b, rep, "graph out=")
        last = want
    assert len(eng._graphs) == 2  # (buffer) and (buffer, out): one capture each, reused across the replays
    ys = [eng.forward_u8(buf, graph=True) for _ in range(10)]
    torch.cuda.synchronize()
    assert all(torch.equal(y, last) for y in ys)


@gpu
@pytest.mark.parametrize("b", [1, 2, 31, 32, 33, 200])
def test_uint8_conv1_layer_equals_fp32_route(qparams, b):
    """b200q_u8_conv3x3_first output bytes == b200q_quantize_conv3x3_first on the normalised pixels, either side of the
    CUDA-core | tensor-core cut (32 | 33 images)."""
    from convnet_quantization_b200 import _lib, ops
    lib = _lib.load()
    pc, s, lut = _conv1(qparams)
    pix = _pixels(b, 500 + b, extreme=(b % 2 == 1))
    x = _normalized(pix).cuda()
    want = torch.empty((b, 32, 32, 64), dtype=torch.uint8, device="cuda")
    _lib.check(lib.b200q_quantize_conv3x3_first(x.data_ptr(), want.data_ptr(), b, ops._inv_scale(s), pc.ptr(), _stream()),
               "quantize_conv3x3_first")
    got = torch.empty_like(want)
    xu8 = pix.cuda()
    _lib.check(lib.b200q_u8_conv3x3_first(xu8.data_ptr(), got.data_ptr(), b, lut.data_ptr(), pc.ptr(), _stream()),
               "u8_conv3x3_first")
    torch.cuda.synchronize()
    assert torch.equal(got, want)


@gpu
@pytest.mark.parametrize("case", ["not_bounded", "no_host_mirrors"])
@pytest.mark.parametrize("b", [1, 33, 300])
def test_uint8_route_serves_layers_the_tensor_core_kernel_refuses(qparams, oracle_model, unbounded, case, b):
    """conv1 without B200Q_RQ_BOUNDED, or without host mirrors of its constants: the tensor-core first layer refuses
    it, the CUDA-core table-lookup kernel serves it; forward_u8 / forward_uint8 == fp32 route == CPU oracle."""
    from convnet_quantization_b200 import _lib
    from convnet_quantization_b200.engine import StaticEngine
    from convnet_quantization_b200.models._gpu_modules import B200StaticQuantizedNet
    qp, oracle = unbounded if case == "not_bounded" else (qparams, oracle_model)
    eng = StaticEngine(qp, "cuda")
    net = B200StaticQuantizedNet(qp, "cuda")
    if case == "not_bounded":
        assert not (eng.packed.c.conv[0].rq.flags & _lib.RQ_BOUNDED)
    else:
        _drop_conv1_host_mirrors(eng.packed)
        _drop_conv1_host_mirrors(net.engine.packed)
    pix = _pixels(b, 900 + b, extreme=True)
    want, ref = _references(eng, oracle, pix)
    assert len(torch.unique(ref)) >= 3  # not a constant output
    xu8 = pix.cuda()
    assert torch.equal(eng.forward_u8(xu8, graph=False), want)
    assert torch.equal(eng.forward_u8(xu8, graph=True), want)
    lib = _lib.load()
    pc_out = torch.empty((b, 32, 32, 64), dtype=torch.uint8, device="cuda")
    rc = lib.b200q_u8_conv3x3_first(xu8.data_ptr(), pc_out.data_ptr(), b, eng.packed.input_lut.data_ptr(),
                                    C.byref(eng.packed.c.conv[0]), _stream())
    assert rc == 0, lib.b200q_last_error()
    assert torch.equal(net.forward_uint8(xu8).cpu(), ref)
    assert torch.equal(net.forward_uint8(pix), ref)  # host input: chunked pipeline through the staging buffers


# ------------------------------------------------------------------------------------------------ bookkeeping
@gpu
def test_uint8_graph_launch_accounting_cache_and_release(qparams):
    from convnet_quantization_b200 import _lib, synth
    from convnet_quantization_b200.engine import StaticEngine
    lib = _lib.load()
    eng = StaticEngine(qparams, "cuda")
    pix = _pixels(8, 1).cuda()
    n0 = lib.b200q_launch_count()
    eng.forward_u8(pix, graph=False)
    per_forward = lib.b200q_launch_count() - n0
    assert per_forward in (7, 8)
    eng.forward_u8(pix)  # first sighting: eager
    eng.forward_u8(pix)  # second: capture
    assert any(k[0] for k in eng._graphs)
    n0 = lib.b200q_launch_count()
    for _ in range(5):
        eng.forward_u8(pix)
    assert lib.b200q_launch_count() - n0 == 5 * per_forward  # replays are counted like the launches they stand for
    for i in range(StaticEngine.GRAPH_CACHE + 3):  # both kinds through one LRU: no growth
        xi = _pixels(3, 10 + i).cuda() if i % 2 else synth.images_f32(3, seed=i).cuda()
        fwd = eng.forward_u8 if i % 2 else eng.forward
        fwd(xi)
        fwd(xi)
    assert len(eng._graphs) == StaticEngine.GRAPH_CACHE
    assert {k[0] for k in eng._graphs} == {True, False}
    big = _pixels(StaticEngine.GRAPH_MAX_BATCH + 1, 3).cuda()
    eng.forward_u8(big)
    eng.forward_u8(big)
    assert all(k[1] <= StaticEngine.GRAPH_MAX_BATCH for k in eng._graphs)
    eng.release()
    assert not eng._graphs and not eng._ws and not eng._seen


@gpu
@pytest.mark.parametrize("b", [1, 2, 32, 33, 37])
def test_uint8_conv1_and_graph_write_only_their_outputs(qparams, b):
    """The uint8 conv1 output, and the logits and exact-size workspace of b200q_graph_create_u8, between sentinel bands:
    the bands stay untouched and the payloads equal the unguarded results."""
    from convnet_quantization_b200 import _lib, ops
    from convnet_quantization_b200.engine import StaticEngine
    lib = _lib.load()
    pc, s, lut = _conv1(qparams)
    pix = _pixels(b, 300 + b, extreme=True)
    xu8 = pix.cuda()
    g = Guarded((b, 32, 32, 64), torch.uint8)
    _lib.check(lib.b200q_u8_conv3x3_first(xu8.data_ptr(), g.view.data_ptr(), b, lut.data_ptr(), pc.ptr(), _stream()),
               "u8_conv3x3_first")
    assert g.intact(), f"b={b}: conv1 wrote outside its output"
    assert torch.equal(g.view, ops.quantize_conv2d_first(_normalized(pix).cuda(), s, pc))

    eng = StaticEngine(qparams, "cuda", use_graphs=False)
    want = eng.forward_u8(xu8)
    ws_bytes = int(lib.b200q_static_workspace_bytes(b))
    ws = Guarded((ws_bytes,), torch.uint8)
    ws.view.zero_()
    out = Guarded((b, 10), torch.float32)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    gh = C.c_void_p()
    with torch.cuda.stream(side):
        rc = lib.b200q_graph_create_u8(eng.packed.ptr(), xu8.data_ptr(), eng.packed.input_lut.data_ptr(),
                                       out.view.data_ptr(), b, ws.view.data_ptr(), ws_bytes, _lib.GRAPH_PDL,
                                       side.cuda_stream, C.byref(gh))
        _lib.check(rc, "graph_create_u8")
        for _ in range(3):
            _lib.check(lib.b200q_graph_launch(gh, side.cuda_stream), "graph_launch")
    side.synchronize()
    try:
        assert ws.intact(), f"b={b}: wrote outside the workspace"
        assert out.intact(), f"b={b}: wrote outside the logits"
        assert torch.equal(out.view, want)
    finally:
        _lib.check(lib.b200q_graph_destroy(gh), "graph_destroy")


@gpu
def test_uint8_graph_concurrent_with_fp32_eager_on_another_stream(qparams):
    """One engine: uint8 graph replays on one stream while a large fp32 eager forward runs on another == the same
    calls made one after the other."""
    from convnet_quantization_b200 import synth
    from convnet_quantization_b200.engine import StaticEngine
    eng = StaticEngine(qparams, "cuda")
    pix = _pixels(32, 77, extreme=True).cuda()
    x = synth.images_f32(4096, seed=78).cuda()
    want8 = eng.forward_u8(pix, graph=False)
    want32 = eng.forward(x, graph=False)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    out8 = torch.empty((32, 10), device="cuda")
    out32 = torch.empty((4096, 10), device="cuda")
    for s in (s1, s2):
        s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s1):
        eng.forward_u8(pix, out=out8, graph=True)  # capture (and one replay)
    s1.synchronize()
    out8.zero_()
    results = []
    for _ in range(3):
        with torch.cuda.stream(s2):
            eng.forward(x, out=out32, graph=False)
        with torch.cuda.stream(s1):
            for _ in range(4):
                eng.forward_u8(pix, out=out8, graph=True)
        s1.synchronize()
        s2.synchronize()
        results.append((out8.clone(), out32.clone()))
    assert len(eng._graphs) == 1
    for o8, o32 in results:
        assert torch.equal(o8, want8)
        assert torch.equal(o32, want32)


# ------------------------------------------------------------------------------------------------ CPU only
def test_header_declares_graph_create_u8_and_binding_matches():
    from convnet_quantization_b200 import _lib
    text = open(os.path.join(ROOT, "include", "b200q.h")).read()
    m = re.search(r"int b200q_graph_create_u8\(([^)]*)\);", text)
    assert m, "include/b200q.h must declare b200q_graph_create_u8"
    params = [p.strip() for p in m.group(1).split(",")]
    assert len(params) == 10 and params[2] == "const uint8_t* lut_host"
    assert "b200q_graph_create_u8" in _lib.EXPORTS
    assert len(_lib._SIGNATURES["b200q_graph_create_u8"]) == 10


def test_graph_create_u8_rejects_bad_arguments_before_any_cuda_call(lib):
    """NULL lut_host, NULL out and the legacy default stream are refused up front (no device is needed to see it)."""
    from convnet_quantization_b200 import _lib
    net = _lib.StaticNet()
    fake = 1 << 20  # never dereferenced: each call fails its argument check first
    h = C.c_void_p()
    args = dict(x=fake, lut=fake, logits=fake, b=4, ws=fake, ws_bytes=1 << 30, stream=fake)

    def call(out=C.byref(h), **kw):
        a = {**args, **kw}
        return lib.b200q_graph_create_u8(C.byref(net), a["x"], a["lut"], a["logits"], a["b"], a["ws"], a["ws_bytes"], 0,
                                         a["stream"], out)

    assert call(lut=None) == -1 and b"null" in lib.b200q_last_error()
    assert h.value is None
    assert call(out=None) == -1 and b"null out" in lib.b200q_last_error()
    assert call(stream=None) == -1 and b"legacy default stream" in lib.b200q_last_error()
    assert call(x=None) == -1
    assert lib.b200q_u8_conv3x3_first(fake, fake, 4, None, None, fake) == -1
