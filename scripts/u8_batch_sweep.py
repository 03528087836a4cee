"""uint8 pixel route at small and medium batches (device-resident input): fp32 graph + PDL against uint8 graph + PDL and
uint8 eager launches, plus, in the same process, uint8 eager on the development library with B200Q_CONV1_TINY_MAX_B=0
(conv1 always on the tensor-core kernel: the uint8 route before it had a CUDA-core small-batch shape).
    python scripts/u8_batch_sweep.py [--batches 1,2,...] > profiles/r03_u8_batch_sweep.json
Each variant is timed as the best of 3 loops, the variants alternating within each repeat; every row's logits are
checked bit for bit against the plain fp32 forward of the normalised pixels."""
import argparse, json, os, subprocess, sys, warnings
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
warnings.filterwarnings("ignore")
os.environ["B200Q_CONV1_TINY_MAX_B"] = "0"  # read by the development library only
import torch
from convnet_quantization_b200 import _lib, synth
from convnet_quantization_b200.engine import StaticEngine, _Graph
from convnet_quantization_b200.models.static_ptq_model import StaticPTQModel

ap = argparse.ArgumentParser()
ap.add_argument("--batches", default="1,2,8,32,128,512,1024")
a = ap.parse_args()
dev = torch.device("cuda", 0)
model = StaticPTQModel(device=dev)
model.fp32_model.load_state_dict(synth.make_state_dict(0))
engine = model.quantize().engine
before = StaticEngine(engine.qparams, dev, use_graphs=False)
before.lib = _lib.load_dev()
smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
stream = torch.cuda.current_stream().cuda_stream
rows = []
for b in (int(v) for v in a.batches.split(",")):
    g = torch.Generator(device=dev).manual_seed(b)
    pix = torch.randint(0, 256, (b, 32, 32, 3), dtype=torch.uint8, device=dev, generator=g)
    x = synth.normalize(pix.permute(0, 3, 1, 2)).contiguous()
    out = torch.empty((b, 10), dtype=torch.float32, device=dev)
    ref = engine.forward(x, graph=False)
    iters = max(20, min(1000, int(4e6 / max(b, 1000))))
    g32 = _Graph(engine, x, out, True)
    g8 = _Graph(engine, pix, out, True, u8=True)
    variants = {
        "fp32_graph_pdl": lambda: g32.launch(stream),
        "u8_graph_pdl": lambda: g8.launch(stream),
        "u8_eager": lambda: engine.forward_u8(pix, out=out, graph=False),
        "u8_eager_before": lambda: before.forward_u8(pix, out=out, graph=False),
    }
    best = {}
    for rep in range(3):
        for name, fn in variants.items():
            for _ in range(5):
                fn()
            torch.cuda.synchronize()
            out.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                fn()
            e1.record()
            torch.cuda.synchronize()
            assert torch.equal(out, ref), f"{name} differs from the plain fp32 forward at batch {b}"
            us = e0.elapsed_time(e1) / iters * 1e3
            best[name] = min(best.get(name, us), us)
    del g32, g8
    row = {"batch": b, "iters": iters}
    for name, us in best.items():
        row[f"us_{name}"] = round(us, 2)
        row[f"images_per_s_{name}"] = round(b / us * 1e6)
    rows.append(row)
    print(f"batch {b:5d}: " + "  ".join(f"{k} {v:8.1f} us" for k, v in best.items()), file=sys.stderr)
json.dump({"what": "static-PTQ forward from device-resident input, one GPU; uint8 NHWC pixels vs fp32 NCHW images; "
                   "best of 3 timed loops per variant, variants alternating (CUDA events); inputs fit in L2",
           "gpu": smi, "torch_device_name": torch.cuda.get_device_name(dev),
           "before": "u8_eager_before = development library, B200Q_CONV1_TINY_MAX_B=0 (conv1 on the tensor-core kernel "
                     "at every batch)",
           "rows": rows}, sys.stdout, indent=1)
