"""Accuracy counting inside the classifier head: ``b200q_static_evaluate`` / ``_u8``, ``StaticEngine.evaluate`` /
``evaluate_u8``, ``B200StaticQuantizedNet.evaluate`` / ``evaluate_uint8`` and ``sharding.evaluate_sharded``.

The reference for every count is ``sharding.rank_rule_hits``, the torch restatement of the rule in ``b200q.h``, applied
to the logits ``forward`` returns; the restatement itself is checked against ``torch.sort(stable=True)`` on the CPU.
The uint8 logits of this net tie often (a few percent of images at top-1 and at the 5th/6th place), so the tie rule is
exercised by ordinary inputs."""
import ctypes as C
import os
import re
import socket

import pytest
import torch

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

GUARD = 8192
SENTINEL = 0xA5
BATCHES = [1, 2, 7, 32, 33, 64, 128, 1000, 4096, 16384]


class Guarded:
    """A device buffer inside a larger allocation pre-filled with a sentinel (stray stores show in the bands)."""

    def __init__(self, shape, dtype, fill=None):
        self.nbytes = int(torch.empty(shape, dtype=dtype).numel() * torch.empty((), dtype=dtype).element_size())
        self.raw = torch.full((2 * GUARD + self.nbytes,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.view = self.raw[GUARD:GUARD + self.nbytes].view(dtype).view(shape)
        if fill is not None:
            self.view.fill_(fill)

    def intact(self) -> bool:
        torch.cuda.synchronize()
        front, back = self.raw[:GUARD], self.raw[GUARD + self.nbytes:]
        return bool((front == SENTINEL).all()) and bool((back == SENTINEL).all())


def _pixels(b: int, seed: int) -> torch.Tensor:
    """uint8 NHWC [b,32,32,3] on the host."""
    return torch.randint(0, 256, (b, 32, 32, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(seed))


def _images(b: int, seed: int, u8: bool) -> torch.Tensor:
    from convnet_quantization_b200 import synth
    return _pixels(b, seed) if u8 else synth.images_f32(b, seed=seed)


def _label_sets(logits: torch.Tensor, seed: int) -> dict:
    """random labels, labels = argmax, and labels with out-of-range entries (-1, 10, 2^40) among valid ones."""
    b = logits.shape[0]
    g = torch.Generator().manual_seed(seed)
    rnd = torch.randint(0, 10, (b,), generator=g)
    oor = rnd.clone()
    bad = torch.tensor([-1, 10, 1 << 40], dtype=torch.int64)
    oor[::3] = bad[torch.arange(0, b, 3) % 3]
    return {"random": rnd, "argmax": logits.argmax(1).cpu(), "out_of_range": oor}


@pytest.fixture(scope="module")
def engine(qparams):
    from convnet_quantization_b200.engine import StaticEngine
    return StaticEngine(qparams, "cuda")


@pytest.fixture(scope="module")
def model(qparams):
    from convnet_quantization_b200.models._gpu_modules import B200StaticQuantizedNet
    return B200StaticQuantizedNet(qparams, "cuda")


def _forward(engine, x, u8):
    return engine.forward_u8(x, graph=False) if u8 else engine.forward(x, graph=False)


def _evaluate(engine, x, labels, u8, **kw):
    return engine.evaluate_u8(x, labels, **kw) if u8 else engine.evaluate(x, labels, **kw)


# ------------------------------------------------------------------------------------------------ GPU
@gpu
@pytest.mark.parametrize("u8", [False, True], ids=["fp32", "uint8"])
@pytest.mark.parametrize("b", BATCHES)
def test_counters_equal_the_rule_on_forward_logits(engine, b, u8):
    from convnet_quantization_b200 import sharding
    x = _images(b, 1000 + b, u8).cuda()
    logits = _forward(engine, x, u8)
    for kind, labels in _label_sets(logits, b).items():
        lab = labels.cuda()
        got = _evaluate(engine, x, lab, u8)
        want = sharding.rank_rule_counts(logits, lab)
        assert torch.equal(got, want), (b, kind, got.tolist(), want.tolist())
        if kind == "argmax":
            assert int(got[0]) == b  # the first maximal index is the rank-0 class
    if b >= 1000:  # the sample really contains ties at the top and across the 5th / 6th place
        s = logits.sort(1, descending=True).values
        assert int((s[:, 0] == s[:, 1]).sum()) > 0 and int((s[:, 4] == s[:, 5]).sum()) > 0
        argmax_counts = _evaluate(engine, x, logits.argmax(1), u8)
        assert int(argmax_counts[3]) > 0  # top-1 tied
    if b >= 4096:
        assert int(_evaluate(engine, x, _label_sets(logits, b)["random"].cuda(), u8)[4]) > 0  # top-5 tied


@gpu
@pytest.mark.parametrize("u8", [False, True], ids=["fp32", "uint8"])
@pytest.mark.parametrize("b", [1, 7, 32, 33, 1000, 4096])
def test_pred_is_argmax_and_logits_equal_forward(engine, b, u8):
    x = _images(b, 2000 + b, u8).cuda()
    want = _forward(engine, x, u8)
    labels = torch.randint(0, 10, (b,), generator=torch.Generator().manual_seed(b)).cuda()
    pred = torch.full((b,), -7, dtype=torch.int32, device="cuda")
    logits = torch.full((b, 10), float("nan"), device="cuda")
    _evaluate(engine, x, labels, u8, pred=pred, logits=logits)
    assert torch.equal(logits, want)
    assert torch.equal(pred.long(), want.argmax(1))


@gpu
@pytest.mark.parametrize("u8", [False, True], ids=["fp32", "uint8"])
@pytest.mark.parametrize("b", [5, 33, 3000])
def test_counters_accumulate_and_empty_batch_changes_nothing(engine, b, u8):
    from convnet_quantization_b200 import sharding
    x = _images(b, 3000 + b, u8).cuda()
    logits = _forward(engine, x, u8)
    labels = torch.randint(0, 10, (b,), generator=torch.Generator().manual_seed(b)).cuda()
    one = sharding.rank_rule_counts(logits, labels)
    counters = torch.full((5,), 1000, dtype=torch.int64, device="cuda")
    assert _evaluate(engine, x, labels, u8, counters=counters) is counters
    _evaluate(engine, x, labels, u8, counters=counters)
    assert torch.equal(counters, 1000 + 2 * one)
    empty = x[:0]
    assert _evaluate(engine, empty, labels[:0], u8, counters=counters) is counters
    assert torch.equal(counters, 1000 + 2 * one)
    assert torch.equal(_evaluate(engine, empty, labels[:0], u8), torch.zeros(5, dtype=torch.int64, device="cuda"))


@gpu
@pytest.mark.parametrize("u8", [False, True], ids=["fp32", "uint8"])
@pytest.mark.parametrize("b", [1, 2047, 2048, 2049, 10000])
def test_host_input_equals_device_input(model, b, u8):
    from convnet_quantization_b200.engine import eval_result
    x = _images(b, 4000 + b, u8)
    labels = torch.randint(-1, 11, (b,), generator=torch.Generator().manual_seed(b))
    run = model.evaluate_uint8 if u8 else model.evaluate
    host = run(x, labels)
    dev = run(x.cuda(), labels.cuda())
    direct = eval_result(_evaluate(model.engine, x.cuda(), labels.cuda(), u8))
    assert host == dev == direct
    assert host["images"] == b and 0 <= host["top1"] <= host["top5"] <= b
    assert host["top1_pct"] == pytest.approx(100.0 * host["top1"] / b)


@gpu
def test_counts_equal_the_rule_on_the_cpu_oracle(engine, oracle_model):
    from convnet_quantization_b200 import sharding, synth
    from oracle import torch_oracle as TO
    b = 1024
    x = synth.images_f32(b, seed=0)
    ref, _ = TO.run_static_oracle(oracle_model, x)
    for kind, labels in _label_sets(ref, 77).items():
        want = sharding.rank_rule_counts(ref, labels)
        got = engine.evaluate(x.cuda(), labels.cuda()).cpu()
        assert torch.equal(got, want), (kind, got.tolist(), want.tolist())
    assert int(sharding.rank_rule_counts(ref, ref.argmax(1))[3]) > 0


@gpu
@pytest.mark.parametrize("b", [1, 32, 4096])
def test_evaluate_launches_as_many_kernels_as_forward(engine, b):
    from convnet_quantization_b200 import _lib
    lib = _lib.load()
    x = _images(b, 5000 + b, False).cuda()
    labels = torch.zeros(b, dtype=torch.int64, device="cuda")
    for u8, xx in ((False, x), (True, _images(b, 5000 + b, True).cuda())):
        n0 = lib.b200q_launch_count()
        _forward(engine, xx, u8)
        fwd = lib.b200q_launch_count() - n0
        n0 = lib.b200q_launch_count()
        _evaluate(engine, xx, labels, u8)
        assert lib.b200q_launch_count() - n0 == fwd, (b, u8)


@gpu
@pytest.mark.parametrize("b", [1, 7, 32, 33, 1000])
def test_evaluate_writes_only_its_outputs(engine, b):
    """pred, counters, logits and the exact-size workspace between sentinel bands: the bands stay untouched."""
    from convnet_quantization_b200 import _lib, sharding
    lib = _lib.load()
    pix = _pixels(b, 6000 + b).cuda()
    want = engine.forward_u8(pix, graph=False)
    labels = torch.randint(0, 10, (b,), generator=torch.Generator().manual_seed(b)).cuda()
    ws_bytes = int(lib.b200q_static_workspace_bytes(b))
    ws = Guarded((ws_bytes,), torch.uint8, fill=0)
    counters = Guarded((5,), torch.int64, fill=0)
    pred = Guarded((b,), torch.int32, fill=-1)
    out = Guarded((b, 10), torch.float32, fill=0)
    stream = torch.cuda.current_stream().cuda_stream
    rc = lib.b200q_static_evaluate_u8(engine.packed.ptr(), pix.data_ptr(), engine.packed.input_lut.data_ptr(),
                                      labels.data_ptr(), b, counters.view.data_ptr(), pred.view.data_ptr(),
                                      out.view.data_ptr(), ws.view.data_ptr(), ws_bytes, stream)
    _lib.check(rc, "static_evaluate_u8")
    assert ws.intact() and counters.intact() and pred.intact() and out.intact()
    assert torch.equal(out.view, want) and torch.equal(pred.view.long(), want.argmax(1))
    assert torch.equal(counters.view, sharding.rank_rule_counts(want, labels))
    x = _images(b, 6000 + b, False).cuda()
    counters2 = Guarded((5,), torch.int64, fill=0)
    pred2 = Guarded((b,), torch.int32, fill=-1)
    rc = lib.b200q_static_evaluate(engine.packed.ptr(), x.data_ptr(), labels.data_ptr(), b, counters2.view.data_ptr(),
                                   pred2.view.data_ptr(), None, ws.view.data_ptr(), ws_bytes, stream)
    _lib.check(rc, "static_evaluate")
    assert ws.intact() and counters2.intact() and pred2.intact()
    want2 = engine.forward(x, graph=False)
    assert torch.equal(counters2.view, sharding.rank_rule_counts(want2, labels))


@gpu
def test_evaluate_on_a_side_stream_concurrent_with_forward(engine):
    from convnet_quantization_b200 import sharding
    pix = _pixels(8192, 7001).cuda()
    x = _images(4096, 7002, False).cuda()
    labels = torch.randint(0, 10, (8192,), generator=torch.Generator().manual_seed(3)).cuda()
    want = sharding.rank_rule_counts(engine.forward_u8(pix, graph=False), labels)
    want_logits = engine.forward(x, graph=False)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for s in (s1, s2):
        s.wait_stream(torch.cuda.current_stream())
    out = torch.empty((4096, 10), device="cuda")
    results = []
    for _ in range(3):
        with torch.cuda.stream(s1):
            c = engine.evaluate_u8(pix, labels)
        with torch.cuda.stream(s2):
            engine.forward(x, out=out, graph=False)
        s1.synchronize()
        s2.synchronize()
        results.append((c.clone(), out.clone()))
    for c, o in results:
        assert torch.equal(c, want)
        assert torch.equal(o, want_logits)


@gpu
@pytest.mark.parametrize("u8", [False, True], ids=["fp32", "uint8"])
def test_bad_labels_counters_and_pred_are_rejected(engine, u8):
    from convnet_quantization_b200 import _lib
    b = 4
    x = _images(b, 1, u8).cuda()
    good = torch.zeros(b, dtype=torch.int64, device="cuda")
    for bad in (good.int(), good.cpu(), good[:3], torch.zeros(2 * b, dtype=torch.int64, device="cuda")[::2]):
        with pytest.raises(_lib.B200QError, match="labels"):
            _evaluate(engine, x, bad, u8)
    for bad in (torch.zeros(5, dtype=torch.int32, device="cuda"), torch.zeros(5, dtype=torch.int64),
                torch.zeros(6, dtype=torch.int64, device="cuda")):
        with pytest.raises(_lib.B200QError, match="counters"):
            _evaluate(engine, x, good, u8, counters=bad)
    with pytest.raises(_lib.B200QError, match="pred"):
        _evaluate(engine, x, good, u8, pred=torch.zeros(b, dtype=torch.int64, device="cuda"))
    with pytest.raises(_lib.B200QError, match="out must be"):
        _evaluate(engine, x, good, u8, logits=torch.zeros(b, 9, device="cuda"))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, n, u8, out):
    import torch.distributed as dist
    from convnet_quantization_b200 import ptq, sharding, synth
    from convnet_quantization_b200.models._gpu_modules import B200StaticQuantizedNet
    from convnet_quantization_b200.models.baseline_model import SimpleConvNet
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        net = SimpleConvNet()
        net.load_state_dict(synth.make_state_dict(0))
        model = B200StaticQuantizedNet(ptq.calibrate_static(net.eval(), synth.calibration_batches()), rank)
        x = _images(n, 8000, u8)
        labels = torch.randint(0, 10, (n,), generator=torch.Generator().manual_seed(8001))
        out[rank] = sharding.evaluate_sharded(model, x, labels, rank, world, u8=u8)
    finally:
        dist.destroy_process_group()


@gpu
@pytest.mark.parametrize("u8", [False, True], ids=["fp32", "uint8"])
def test_evaluate_sharded_over_two_gpus_equals_one_process(model, u8):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    from convnet_quantization_b200 import sharding
    n = 5001
    with mp.Manager() as m:
        out = m.dict()
        mp.spawn(_nccl_worker, args=(2, _free_port(), n, u8, out), nprocs=2, join=True)
        got = [out[r] for r in range(2)]
    x = _images(n, 8000, u8)
    labels = torch.randint(0, 10, (n,), generator=torch.Generator().manual_seed(8001))
    want = sharding.evaluate_sharded(model, x, labels, 0, 1, u8=u8)
    assert got[0] == got[1] == want and want["images"] == n


# ------------------------------------------------------------------------------------------------ CPU only
@pytest.mark.parametrize("n", [1, 3, 5, 6, 10, 32])
def test_rule_restatement_matches_stable_sort(n):
    """rank_rule_hits == the position of the label in torch.sort(descending, stable) on tie-heavy integer logits; the
    tied flags == "the label's tie group straddles position k"."""
    from convnet_quantization_b200 import sharding
    g = torch.Generator().manual_seed(n)
    b = 20000
    logits = torch.randint(0, 4, (b, n), generator=g).float() * 0.25
    labels = torch.randint(-2, n + 2, (b,), generator=g)
    hits = sharding.rank_rule_hits(logits, labels)
    order = torch.sort(logits, dim=1, descending=True, stable=True).indices
    valid = (labels >= 0) & (labels < n)
    pos = torch.where(order == labels.clamp(0, n - 1).view(-1, 1))[1]
    k5 = min(5, n)
    assert torch.equal(hits[:, 0], valid & (pos < 1))
    assert torch.equal(hits[:, 1], valid & (pos < k5))
    assert torch.equal(hits[:, 0], valid & (torch.argmax(logits, 1) == labels))
    v = logits.gather(1, labels.clamp(0, n - 1).view(-1, 1))
    first = (logits > v).sum(1)                    # first position of the label's tie group
    last = first + (logits == v).sum(1) - 1        # last position
    for col, k in ((2, 1), (3, k5)):
        assert torch.equal(hits[:, col], valid & (first < k) & (last >= k))
    assert (int(hits[:, 2].sum()) > 0) == (n > 1)  # one class cannot tie
    assert (int(hits[:, 3].sum()) > 0) == (n > 5)  # k = n: every order keeps the label in the top n
    counts = sharding.rank_rule_counts(logits, labels)
    assert counts.tolist() == [int(hits[:, 0].sum()), int(hits[:, 1].sum()), b, int(hits[:, 2].sum()),
                               int(hits[:, 3].sum())]


def test_header_declares_evaluate_and_binding_matches():
    from convnet_quantization_b200 import _lib
    text = open(os.path.join(ROOT, "include", "b200q.h")).read()
    for name, nparams in (("b200q_static_evaluate", 10), ("b200q_static_evaluate_u8", 11)):
        m = re.search(rf"int {name}\(([^)]*)\);", text)
        assert m, f"include/b200q.h must declare {name}"
        params = [p.strip() for p in m.group(1).split(",")]
        assert len(params) == nparams and "const int64_t* labels" in params and "uint64_t* counters" in params
        assert name in _lib.EXPORTS and len(_lib._SIGNATURES[name]) == nparams
    defines = dict(re.findall(r"#define (B200Q_EVAL_\w+) (\d+)", text))
    assert int(defines["B200Q_EVAL_COUNTERS"]) == _lib.EVAL_COUNTERS == len(_lib.EVAL_COUNTER_NAMES)
    for i, name in enumerate(_lib.EVAL_COUNTER_NAMES):
        assert int(defines[f"B200Q_EVAL_{name.upper()}"]) == i


def test_evaluate_rejects_bad_arguments_before_any_cuda_call(lib):
    """Null labels / counters, a negative batch and misaligned labels / counters / pred are refused up front (no device
    is needed to see it); so is an fc2 the counting head does not cover."""
    from convnet_quantization_b200 import _lib
    net = _lib.StaticNet()
    net.fc2.k, net.fc2.n = 512, 10
    fake = 1 << 20  # never dereferenced: each call fails its argument check first
    args = dict(x=fake, labels=fake, b=4, counters=fake, pred=fake, logits=fake, ws=fake, ws_bytes=1 << 30,
                stream=fake)

    def call(u8, **kw):
        a = {**args, **kw}
        if u8:
            return lib.b200q_static_evaluate_u8(C.byref(net), a["x"], fake, a["labels"], a["b"], a["counters"],
                                                a["pred"], a["logits"], a["ws"], a["ws_bytes"], a["stream"])
        return lib.b200q_static_evaluate(C.byref(net), a["x"], a["labels"], a["b"], a["counters"], a["pred"],
                                         a["logits"], a["ws"], a["ws_bytes"], a["stream"])

    for u8 in (False, True):
        assert call(u8, labels=None) == -1 and b"null labels or counters" in lib.b200q_last_error()
        assert call(u8, counters=None) == -1 and b"null labels or counters" in lib.b200q_last_error()
        assert call(u8, b=-1) == -1 and b"negative batch" in lib.b200q_last_error()
        for k, v in (("labels", fake + 4), ("counters", fake + 4), ("pred", fake + 2)):
            assert call(u8, **{k: v}) == -1 and b"misaligned" in lib.b200q_last_error(), k
    assert lib.b200q_static_evaluate_u8(C.byref(net), fake, None, fake, 4, fake, None, None, fake, 1 << 30, fake) == -1
    net.fc2.n = 12
    assert call(False) == -1 and b"fc2" in lib.b200q_last_error()


def test_engine_wrappers_reject_bad_labels_and_counters_without_a_device():
    """StaticEngine's argument checks run before the library is called: tensors of the wrong device, dtype or shape."""
    from convnet_quantization_b200 import _lib
    from convnet_quantization_b200.engine import StaticEngine
    eng = StaticEngine.__new__(StaticEngine)
    eng.device = torch.device("cuda", 0)
    eng.lib = None  # any library call would fail differently
    good_shape = torch.zeros(4, dtype=torch.int64)
    for name, kw in (("labels", dict(labels=good_shape)), ("labels", dict(labels=good_shape.int())),
                     ("labels", dict(labels=[0, 1, 2, 3])), ("labels", dict(labels=None)),
                     ("counters", dict(counters=torch.zeros(5, dtype=torch.int64))),
                     ("counters", dict(counters=torch.zeros(5))),
                     ("pred", dict(pred=torch.zeros(4, dtype=torch.int32)))):
        with pytest.raises(_lib.B200QError, match=name):
            eng._check_eval_args(4, kw.get("labels"), kw.get("counters"), kw.get("pred"))
