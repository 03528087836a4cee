"""The per-layer sandwich net (``CustomQuantizationModel(mode="sandwich")``) from device-resident input, three ways:
    ops_chain   the forward as it was composed in Python before ``b200q_sandwich_forward``: ``ops.*`` per layer (six
                convs, six boundary tables, fc1, ``relu_q``, ``dequantize``, each with its own torch allocation) and a
                cuBLAS ``torch.addmm`` for fc2;
    eager       ``SandwichEngine.forward(graph=False)``: the native forward, one C-ABI call;
    graph_pdl   a captured graph of it with programmatic dependent launch (batches <= 1024, the executor's range).
Then the package's port of the reference driver (``drivers.InferenceBenchmark.measure_throughput``) at batch 1 and
32 for the sandwich and the static model, as the reference measures them.
    python scripts/sandwich_batch_sweep.py > profiles/r05_sandwich_batch_sweep.json
Each variant is timed as 3 loops (CUDA events), the variants alternating within each repeat; all three loop times are
kept (the spread) and the best is reported.  Every row asserts that eager and graph logits are equal and that the
ops chain agrees with them to fp32 rounding (its fc2 is cuBLAS)."""
import argparse, contextlib, io, json, os, subprocess, sys, warnings
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
warnings.filterwarnings("ignore")
import torch
from convnet_quantization_b200 import drivers, ops, synth
from convnet_quantization_b200.engine import _Graph
from convnet_quantization_b200.models.baseline_model import SimpleConvNet
from convnet_quantization_b200.models.custom_quantization_model import CustomQuantizationModel
from convnet_quantization_b200.models.static_ptq_model import StaticPTQModel

ap = argparse.ArgumentParser()
ap.add_argument("--batches", default="1,2,8,32,33,128,512,1024,4096,16384")
a = ap.parse_args()
dev = torch.device("cuda", 0)
sd = synth.make_state_dict(0)
cm = CustomQuantizationModel(mode="sandwich", device=dev)
cm.load_state_dict(sd)
model = cm.quantize()
engine = model.engine
p = engine.packed
sp = engine.sparams
smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
stream = torch.cuda.current_stream().cuda_stream


def ops_chain(x):
    """The Python composition the native forward replaces (fused pools, tables on the pooled tensors)."""
    t = ops.quantize_conv2d_first(x, sp["conv1"]["in_scale"], p.convs[0])
    for i in range(1, 6):
        t = ops.lut_u8(t, p.luts[i - 1])
        t = ops.conv2d_q(t, p.convs[i], pool2x2=(i % 2 == 1))
    t = ops.lut_u8(t, p.luts[5]).reshape(t.shape[0], -1)
    h = ops.linear_q(t, p.fc1)
    h = ops.dequantize(ops.relu_q(h, p.fc1_zp), p.fc1_scale, p.fc1_zp)
    return torch.addmm(p.fc2_b, h, p.fc2_w.t())


rows = []
for b in (int(v) for v in a.batches.split(",")):
    x = synth.images_f32(b, seed=b).to(dev) * 3
    out = torch.empty((b, 10), dtype=torch.float32, device=dev)
    ref = engine.forward(x, graph=False)
    chain = ops_chain(x)
    chain_err = float((chain - ref).abs().max() / ref.abs().max())
    assert chain_err < 1e-5, f"ops chain differs from the native forward by {chain_err} at batch {b}"
    iters = max(20, min(1000, int(4e6 / max(b, 1000))))
    variants = {"ops_chain": lambda: out.copy_(ops_chain(x)),
                "eager": lambda: engine.forward(x, out=out, graph=False)}
    g = None
    if b <= engine.GRAPH_MAX_BATCH:
        g = _Graph(engine, x, out, True)
        variants["graph_pdl"] = lambda: g.launch(stream)
    times = {name: [] for name in variants}
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
            if name == "ops_chain":
                assert torch.equal(out, chain), f"ops chain not repeatable at batch {b}"
            else:
                assert torch.equal(out, ref), f"{name} logits differ from the eager forward at batch {b}"
            times[name].append(e0.elapsed_time(e1) / iters * 1e3)
    del g
    row = {"batch": b, "iters": iters, "ops_chain_max_abs_err_over_logit_range": chain_err}
    for name, ts in times.items():
        row[f"us_{name}"] = round(min(ts), 2)
        row[f"us_{name}_loops"] = [round(t, 2) for t in ts]
        row[f"images_per_s_{name}"] = round(b / min(ts) * 1e6)
    rows.append(row)
    print(f"batch {b:5d}: " + "  ".join(f"{k} {min(v):9.1f} us" for k, v in times.items()), file=sys.stderr)

# the reference's driver protocol (utils/inference_benchmark.py:126-138: batch 1 and 32; wall clock, model(data) returns
# after a device synchronise), through the package's port of it
net = SimpleConvNet()
net.load_state_dict(sd)
loader = synth.SyntheticLoader(256, 64, seed=5, label_model=net.eval())
sm = StaticPTQModel(device=dev)
sm.fp32_model.load_state_dict(sd)
static = sm.quantize()
driver = {"what": "drivers.InferenceBenchmark(device='cuda').measure_throughput, 200 iterations after a warm-up and a "
                  "20-iteration pass; images/s as the driver reads the wall clock", "rows": []}
with contextlib.redirect_stdout(io.StringIO()):
    bench = drivers.InferenceBenchmark(loader, device="cuda")
    for name, m in (("custom sandwich (B200)", model), ("static int8 (B200)", static)):
        bench.warm_up(m)
        row = {"model": name}
        for bs in (1, 32):
            bench.measure_throughput(m, batch_size=bs, num_iterations=20, verbose=False)
            row[f"throughput_{bs}"] = round(bench.measure_throughput(m, batch_size=bs, num_iterations=200, verbose=False))
        driver["rows"].append(row)
print(json.dumps(driver["rows"]), file=sys.stderr)

json.dump({"what": "sandwich net forward from device-resident input, one GPU: the old Python ops chain against the native "
                   "forward (eager, and graph + PDL up to 1024 images); 3 timed loops per variant, variants alternating "
                   "(CUDA events), best reported, all three kept; input = synthetic images x 3",
           "gpu": smi, "torch_device_name": torch.cuda.get_device_name(dev), "rows": rows, "driver_protocol": driver},
          sys.stdout, indent=1)
