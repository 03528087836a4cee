"""The reference's two drivers (SURVEY 8a row a8 / VERDICT r1 item 6) against this package's models.

The reference's ``utils/inference_benchmark.py`` and ``utils/model_evaluator.py`` are not part of this repository.
``convnet_quantization_b200.drivers`` restates them (same classes, methods, arguments and return values); what the
reference's own files returned on the fixed synthetic loader below is stored here and compared with, and the one
protocol detail the restatement changes on purpose - the reference times CUDA forwards with ``time.time()`` and no
device synchronize (``inference_benchmark.py:95-98``) - is reproduced inline.
"""
import time

import pytest
import torch

# ModelEvaluator(loader).evaluate_accuracy(net) of the reference's own driver file for the fp32 net on ``loader``:
# the labels are this net's own argmax, so every image is a top-1 hit
REFERENCE_FP32_ACCURACY = (100.0, 100.0)


@pytest.fixture(scope="module")
def sd():
    from convnet_quantization_b200 import synth
    return synth.make_state_dict(0)


@pytest.fixture(scope="module")
def loader(sd):
    from convnet_quantization_b200 import synth
    from convnet_quantization_b200.models.baseline_model import SimpleConvNet
    net = SimpleConvNet()
    net.load_state_dict(sd)
    return synth.SyntheticLoader(256, 64, seed=5, label_model=net)


def test_restated_drivers_agree_with_the_reference_drivers_on_cpu(sd, loader, capsys):
    """``convnet_quantization_b200.drivers`` computes what the reference's drivers computed."""
    from convnet_quantization_b200 import drivers
    from convnet_quantization_b200.models.baseline_model import SimpleConvNet
    net = SimpleConvNet()
    net.load_state_dict(sd)
    net.eval()
    assert drivers.ModelEvaluator(loader).evaluate_accuracy(net, verbose=False) == REFERENCE_FP32_ACCURACY
    thr = drivers.InferenceBenchmark(loader, device="cpu").measure_throughput(net, batch_size=32, num_iterations=3)
    assert thr > 0
    capsys.readouterr()


@pytest.mark.gpu
def test_reference_drivers_drive_the_gpu_models_unchanged(sd, loader, oracle_model, capsys):
    """evaluate_accuracy (forces ``model.cpu()`` + CPU images, ``model_evaluator.py:15-55``), measure_throughput and
    compare_models (``inference_benchmark.py:81-157``; ``device='cuda'``) on StaticPTQModel / DynamicPTQModel /
    CustomQuantizationModel of this package, and the reference's unsynchronised wall-clock throughput loop."""
    from convnet_quantization_b200 import _lib, drivers
    from convnet_quantization_b200.models.custom_quantization_model import CustomQuantizationModel
    from convnet_quantization_b200.models.dynamic_ptq_model import DynamicPTQModel
    from convnet_quantization_b200.models.static_ptq_model import StaticPTQModel
    from oracle import torch_oracle as TO
    RefBench, RefEval = drivers.InferenceBenchmark, drivers.ModelEvaluator
    m = StaticPTQModel()
    m.fp32_model.load_state_dict(sd)
    q = m.quantize()
    dyn = DynamicPTQModel()
    dyn.load_state_dict(sd)
    dyn.quantize()
    cus = CustomQuantizationModel(mode="sandwich")
    cus.load_state_dict(sd)
    cus.quantize()

    # accuracy driver: the static net must score exactly what the CPU oracle's logits score
    top1, top5 = RefEval(loader).evaluate_accuracy(q)
    hits1 = hits5 = n = 0
    for images, labels in loader:
        logits, _ = TO.run_static_oracle(oracle_model, images)
        top = logits.topk(5, 1).indices
        hits1 += int((top[:, 0] == labels).sum())
        hits5 += int((top == labels.view(-1, 1)).sum())
        n += labels.numel()
    assert top1 == pytest.approx(100.0 * hits1 / n) and top5 == pytest.approx(100.0 * hits5 / n)
    d1, d5 = RefEval(loader).evaluate_accuracy(dyn)   # DynamicPTQModel: plain class with eval()/cpu()/__call__
    c1, c5 = RefEval(loader).evaluate_accuracy(cus)
    assert d1 > 90.0 and c1 > 60.0 and d5 >= d1 and c5 >= c1

    # throughput driver: launches must be counted inside its timed loop
    lib = _lib.load()
    bench = RefBench(loader, device="cuda")
    bench.warm_up(q)
    n0 = lib.b200q_launch_count()
    assert bench.measure_throughput(q, batch_size=32, num_iterations=50) > 0
    assert lib.b200q_launch_count() - n0 >= 50 * 7
    # the reference's loop reads time.time() around each forward without a device synchronize; that wall clock must
    # cover the work (forward synchronises for CUDA inputs): compare with a device-timed run of the same loop
    x = next(iter(loader))[0][:32].cuda()
    wall = 0.0
    with torch.no_grad():
        for _ in range(50):
            t0 = time.time()
            q(x)
            wall += time.time() - t0
    thr = 32 * 50 / wall
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(50):
        q(x)
    ev1.record()
    torch.cuda.synchronize()
    device_thr = 32 * 50 / (ev0.elapsed_time(ev1) * 1e-3)
    assert thr <= 1.25 * device_thr, (thr, device_thr)  # an asynchronous return would report many times more
    res = bench.compare_models({"static int8 (B200)": q, "dynamic (B200)": dyn, "custom sandwich (B200)": cus},
                               batch_size=32, num_iterations=10)
    assert set(res) == {"static int8 (B200)", "dynamic (B200)", "custom sandwich (B200)"}
    assert all(v > 0 for v in res.values())
    capsys.readouterr()
