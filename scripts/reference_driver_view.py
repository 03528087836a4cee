"""The drop-in view (SURVEY 8d): the reference's OWN, unmodified `utils/inference_benchmark.py` timing this package's
models on the GPU (`device='cuda'`) next to the torch/fbgemm CPU oracle model on the host (`device='cpu'`), at the
driver's own operating points (batch 1 and batch 32, `inference_benchmark.py:126-138`).
    python scripts/reference_driver_view.py REFERENCE_CHECKOUT > profiles/r02_reference_driver_view.json
REFERENCE_CHECKOUT is a checkout of the reference project (the driver is imported from its `utils/`)."""
import contextlib, io, json, os, sys, warnings
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")
import torch

ref_root = sys.argv[1] if len(sys.argv) > 1 else ""
if not os.path.isfile(os.path.join(ref_root, "utils", "inference_benchmark.py")):
    raise SystemExit("usage: reference_driver_view.py REFERENCE_CHECKOUT (no utils/inference_benchmark.py there)")
sys.path.insert(0, ref_root)
from utils.inference_benchmark import InferenceBenchmark  # noqa: E402  (the reference's file, unmodified)

from convnet_quantization_b200 import synth  # noqa: E402
from convnet_quantization_b200.models.baseline_model import SimpleConvNet  # noqa: E402
from convnet_quantization_b200.models.custom_quantization_model import CustomQuantizationModel  # noqa: E402
from convnet_quantization_b200.models.dynamic_ptq_model import DynamicPTQModel  # noqa: E402
from convnet_quantization_b200.models.static_ptq_model import StaticPTQModel  # noqa: E402
from oracle import torch_oracle  # noqa: E402

sd = synth.make_state_dict(0)
net = SimpleConvNet()
net.load_state_dict(sd)
net.eval()
loader = synth.SyntheticLoader(256, 64, seed=5, label_model=net)
m = StaticPTQModel(); m.fp32_model.load_state_dict(sd); static = m.quantize()
d = DynamicPTQModel(); d.load_state_dict(sd); d.quantize()
c = CustomQuantizationModel(mode="sandwich"); c.load_state_dict(sd); c.quantize()
oracle = torch_oracle.build_static_oracle(net, synth.calibration_batches())


class _CpuOracle(torch.nn.Module):  # the driver calls .eval() / .to(device) / model(data)
    def forward(self, x):
        return oracle(x)


out = {"what": "reference utils/inference_benchmark.py (unmodified) measure_throughput, 200 iterations, wall clock as the "
               "driver reads it; GPU models synchronise before returning", "driver": os.path.join(ref_root, "utils/inference_benchmark.py"),
       "host_cpus": os.cpu_count(), "rows": []}
with contextlib.redirect_stdout(io.StringIO()):
    gpu = InferenceBenchmark(loader, device="cuda")
    cpu = InferenceBenchmark(loader, device="cpu")
    for name, model, bench in (("static int8 (B200)", static, gpu), ("dynamic (B200)", d, gpu), ("custom sandwich (B200)", c, gpu),
                               ("static int8 fbgemm (host CPU oracle)", _CpuOracle(), cpu)):
        bench.warm_up(model)
        row = {"model": name}
        for bs in (1, 32):
            bench.measure_throughput(model, batch_size=bs, num_iterations=20, verbose=False)
            row[f"throughput_{bs}"] = bench.measure_throughput(model, batch_size=bs, num_iterations=200, verbose=False)
        out["rows"].append(row)
json.dump(out, sys.stdout, indent=1)
