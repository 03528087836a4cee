#!/usr/bin/env python
"""Headline benchmark: images/sec of the static-PTQ int8 SimpleConvNet forward (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]

``--dump-outputs DIR`` writes the logits of the last timed step as ``DIR/logits.npy`` (float32; ``logits_rank<r>.npy``
for ranks > 0), so two builds of the project can be compared output for output: inputs and weights are generated from
fixed seeds, so the same arguments give the same inputs on every run.

* ours (default): one process per GPU (torchrun for N>1).  A step = one ``b200q_static_forward`` over a batch of
  B synthetic images resident in HBM (fp32 NCHW, the reference's input contract).  ``value`` = all ranks' images /
  max-over-ranks CUDA-event time.  ``e2e`` = the same through the reference-facing model object
  (``StaticPTQModel().quantize()`` -> ``model(x_cpu)``) with pinned HOST input and HOST logits, copies in the timed
  region.  ``roofline`` = the dominant kernel's achieved int8 TOP/s (or GB/s) from per-kernel CUDA events of the same
  forward, against MEASURED_PEAKS.json.  ``cpu_baseline`` = torch/fbgemm CPU oracle on this box's host cores
  (rank 0, N=1, bounded sample).
* ``--impl reference``: the reference's CPU implementation of the path — torch's fbgemm quantized ops applied to
  the reference's fused SimpleConvNet (``oracle/torch_oracle.py``; the reference has no native code of its own) —
  on all host threads, batch 64 (BASELINE config 1), each step a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

import torch  # noqa: E402

METRIC = "int8 ConvNet images/sec (static-PTQ SimpleConvNet forward)"
UNIT = "images/s"
OPS_PER_IMAGE = 309_733_376  # SURVEY.md 8(d): 154 866 688 MACs x 2

# Algorithmic work per image and stage (SURVEY.md 8(d)); "tensor" stages in int8 ops, "hbm" stages in bytes (in+out).
STAGE_WORK = {
    "quant_conv1": ("hbm", 12288 + 65536),
    "conv2": ("tensor", 75_497_472),
    "pool1": ("hbm", 81_920),
    "conv3": ("tensor", 37_748_736),
    "conv4": ("tensor", 75_497_472),
    "pool2": ("hbm", 40_960),
    "conv5": ("tensor", 37_748_736),
    "conv6": ("tensor", 75_497_472),
    "pool3": ("hbm", 20_480),
    "fc1": ("tensor", 4_194_304),
    "fc2_dequant": ("hbm", 512 + 40),
    # fused variants (pool folded into the producing conv): same ops, fewer bytes
    "conv2_pool": ("tensor", 75_497_472),
    "conv1_conv2_pool": ("tensor", 3_538_944 + 75_497_472),  # conv1 + conv2 in one kernel (conv12_fused.cu)
    "conv4_pool": ("tensor", 75_497_472),
    "conv6_pool": ("tensor", 75_497_472),
}


def load_peaks():
    """HBM GB/s and dense bf16 TFLOP/s from MEASURED_PEAKS.json (driver-written) or the profiling recipe's fallback, plus
    the int8 tensor-pipe rate this repo measured with tools/int8_peak.cu (profiles/r02_int8_peak.json).  int8 peaks:
    ``int8_burst`` / ``int8_sustained`` = 2 x the bf16 figures (tcgen05 kind::i8 issues K=32 per instruction against 16
    for bf16), ``int8_pipe`` = the measured tcgen05.mma.kind::i8 rate with all SMs issuing back to back."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        out = {"hbm_gbs": float(p["hbm_gbs"]), "bf16_burst": float(p["bf16_tflops"]),
               "bf16_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "MEASURED_PEAKS.json"}
    else:
        out = {"hbm_gbs": 6650.0, "bf16_burst": 1590.0, "bf16_sustained": 1400.0, "source": "B200_PROFILING.md fallback"}
    out["int8_burst"], out["int8_sustained"] = 2.0 * out["bf16_burst"], 2.0 * out["bf16_sustained"]
    out["int8_pipe"] = None
    try:
        with open(os.path.join(ROOT, "profiles", "r02_int8_peak.json")) as f:
            d = json.load(f)
        out["int8_pipe"] = max(float(r["tops"]) for r in d["burst"])
        out["int8_pipe_sustained"] = max(float(r["tops"]) for r in d["sustained"])
    except (OSError, KeyError, ValueError, TypeError):
        pass
    return out


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled through NVML (what nvidia-smi prints) every 5 ms while running."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, device_index: int):
        self.samples, self.mask, self.max_mhz, self.ok = [], 0, None, False
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                uuid = str(torch.cuda.get_device_properties(device_index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:  # pragma: no cover
            self.err = repr(e)
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
            except Exception:
                pass
            time.sleep(0.005)

    def __enter__(self):
        if self.ok:
            self.t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self.ok:
            self.t.join()

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": int(statistics.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": [n for bit, n in self.REASONS.items() if self.mask & bit], "samples": len(self.samples)}


# ----------------------------------------------------------------------------------------------- CPU (reference) leg
def build_cpu_oracle():
    from convnet_quantization_b200 import synth
    from convnet_quantization_b200.models.baseline_model import SimpleConvNet
    from oracle import torch_oracle
    net = SimpleConvNet()
    net.load_state_dict(synth.make_state_dict(0))
    return torch_oracle.build_static_oracle(net.eval(), synth.calibration_batches())


def time_cpu_oracle(q, batch: int, batches_per_step: int, steps: int, warmup: int):
    """images/s of the torch/fbgemm CPU static-PTQ forward: ``steps`` timed steps of ``batches_per_step`` x ``batch``."""
    from convnet_quantization_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.backends.quantized.engine = "fbgemm"
    x = synth.images_f32(batch, seed=11)
    with torch.no_grad():
        for _ in range(max(1, warmup)):
            y = q(x)
        t0 = time.perf_counter()
        for _ in range(steps):
            for _ in range(batches_per_step):
                y = q(x)
        dt = time.perf_counter() - t0
    return batch * batches_per_step * steps / dt, dt, cores, y


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    q = build_cpu_oracle()
    batch, per_step = 64, 16  # BASELINE config 1: batch 64 on CPU; a step = 16 such batches (1024 images)
    ips, dt, cores, y = time_cpu_oracle(q, batch, per_step, args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": y})
    sample = f"{args.steps} steps x {per_step} batches x {batch} images (torch {torch.__version__} fbgemm, {cores} threads)"
    line = {
        "impl": "reference", "metric": METRIC, "value": ips, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "static-PTQ int8 SimpleConvNet forward, CIFAR-10 shape fp32 [B,3,32,32] -> logits [B,10]",
                   "batch": batch, "images_per_step": batch * per_step, "device": "host CPU"},
        "cpu_baseline": {"value": ips, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": ips, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


_REAL_STDOUT = None


def emit_line(obj) -> None:
    """Write the one JSON line to the process's original stdout (see run_ours)."""
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def ncu_traffic(stage: str, batch: int):
    """DRAM bytes (read + written) per launch of `stage`, from the committed `ncu --set full` capture of one forward
    at the same batch (profiles/r01_ncu_net.json, written by scripts/ncu_summary.py); None when no capture matches."""
    for name in ("r02_ncu_net.json", "r01_ncu_net.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            if int(d["batch"]) == int(batch):
                return float(d["stages"][stage]["dram_bytes"])
        except (OSError, KeyError, ValueError, TypeError):
            continue
    return None


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Write each tensor of ``arrays`` as ``out_dir/<name>.npy`` (float32 or float64).  A tensor larger than 64 MB is
    cut to a fixed, seeded sample of its rows, kept in their original order."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu()
        if a.dtype not in (torch.float32, torch.float64):
            a = a.float()
        nbytes = a.numel() * a.element_size()
        if nbytes > DUMP_MAX_BYTES:
            keep = DUMP_MAX_BYTES * a.shape[0] // nbytes
            a = a[torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values]
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a.numpy()))


def oracle_sample_indices(n: int, count: int = 1024):
    """>= ``count`` image indices of a batch of ``n``: the first and last 128 plus a stride over the whole batch."""
    idx = torch.cat([torch.arange(min(128, n)), torch.arange(max(n - 128, 0), n), torch.arange(0, n, max(1, n // count))])
    return torch.unique(idx)


# ----------------------------------------------------------------------------------------------- GPU leg
def run_ours(args):
    import torch.distributed as dist
    from convnet_quantization_b200 import _lib, synth
    from convnet_quantization_b200.models.static_ptq_model import StaticPTQModel

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the quantized forward has no CPU fallback; use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one process per GPU: pin this rank to the CPUs next to its GPU before any pinned staging buffer is allocated
    from convnet_quantization_b200 import sharding as _sh
    host_binding = _sh.gpu_numa_info(local) if args.no_bind else _sh.bind_to_gpu_numa(local)
    # The contract is ONE JSON line on stdout.  NCCL prints its version banner on the C-level stdout when the first
    # communicator is created, so everything but that line is routed to stderr: fd 1 is pointed at fd 2 for the whole
    # run and the line is written to a private duplicate of the original stdout at the end (emit_line).
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    lib = _lib.load()
    model = StaticPTQModel(device=dev)
    model.fp32_model.load_state_dict(synth.make_state_dict(0))
    qmodel = model.quantize()  # fixed synthetic calibration set
    engine = qmodel.engine
    B = args.batch

    # synthetic shard of this rank, generated on the device (SURVEY 8(d)): uint8 pixels -> /255 -> CIFAR normalise
    g = torch.Generator(device=dev).manual_seed(rank)
    x_u8 = torch.randint(0, 256, (B, 3, 32, 32), dtype=torch.uint8, device=dev, generator=g)
    x = synth.normalize(x_u8).contiguous()
    labels = torch.randint(0, 10, (B,), device=dev, generator=g)
    del x_u8

    for _ in range(max(args.warmup, 3)):
        logits = engine.forward(x)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = lib.b200q_launch_count()
    with ClockSampler(local) as clocks:
        barrier()
        ev0.record()
        for _ in range(args.steps):
            logits = engine.forward(x)
        ev1.record()
        barrier()
    launches = int(lib.b200q_launch_count() - n0)
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    value = world * B * args.steps / (ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits" if rank == 0 else f"logits_rank{rank}": logits})

    # ---- per-kernel durations of the same forward (CUDA events between kernels, on the launching stream)
    prof_steps = max(3, min(args.steps, 20))
    acc = {}
    for i in range(prof_steps + 2):
        _, stage_ms = engine.forward_profiled(x)
        if i >= 2:
            for k, v in stage_ms.items():
                acc[k] = acc.get(k, 0.0) + v / prof_steps
    peaks = load_peaks()
    # Roofline denominator: the timed region is args.steps x ~2 ms, far below 1 s, so the BURST figure applies (a kernel
    # timed alone); the sustained one and the measured tensor-pipe rate are reported beside it for every tensor stage.
    timed_s = ms * 1e-3
    int8_peak = peaks["int8_burst"] if timed_s < 1.0 else peaks["int8_sustained"]
    stages = {}
    for k, v in acc.items():
        bound, work = STAGE_WORK[k]
        if bound == "tensor":
            ach = work * B / (v * 1e-3) / 1e12
            stages[k] = {"ms": v, "bound": "tensor", "achieved": ach, "unit": "TOP/s", "frac": ach / int8_peak,
                         "frac_of": {"2x_bf16_burst": ach / peaks["int8_burst"],
                                     "2x_bf16_sustained": ach / peaks["int8_sustained"],
                                     "measured_i8_pipe": (ach / peaks["int8_pipe"]) if peaks["int8_pipe"] else None}}
        else:
            ach = work * B / (v * 1e-3) / 1e9
            stages[k] = {"ms": v, "bound": "hbm", "achieved": ach, "unit": "GB/s", "frac": ach / peaks["hbm_gbs"]}
    total_stage_ms = sum(acc.values())
    dom = max(acc, key=acc.get)
    d = stages[dom]
    net_tops = OPS_PER_IMAGE * B / (total_stage_ms * 1e-3) / 1e12
    roofline = {"kernel": dom, "bound": d["bound"], "achieved": d["achieved"],
                "peak": int8_peak if d["bound"] == "tensor" else peaks["hbm_gbs"], "unit": d["unit"], "frac": d["frac"],
                "traffic": ncu_traffic(dom, B), "share_of_step": acc[dom] / total_stage_ms,
                "peak_source": (f"{peaks['source']}: 2 x bf16_tflops ({'burst' if timed_s < 1.0 else 'sustained'}; timed "
                                f"window {timed_s:.3f} s; tcgen05 kind::i8 issues K=32 per MMA against 16 for bf16)"
                                if d["bound"] == "tensor" else f"{peaks['source']}: hbm_gbs"),
                "peaks": {"hbm_gbs": peaks["hbm_gbs"], "int8_2x_bf16_burst": peaks["int8_burst"],
                          "int8_2x_bf16_sustained": peaks["int8_sustained"], "int8_measured_pipe": peaks["int8_pipe"],
                          "int8_measured_pipe_source": "profiles/r02_int8_peak.json (tools/int8_peak.cu)"},
                "net_int8_tops": net_tops,
                "net_frac_of": {"2x_bf16_burst": net_tops / peaks["int8_burst"],
                                "2x_bf16_sustained": net_tops / peaks["int8_sustained"],
                                "measured_i8_pipe": (net_tops / peaks["int8_pipe"]) if peaks["int8_pipe"] else None},
                "stages": stages}

    if args.stages_only:  # kernel-timing experiments (scripts/gpu_debug_modes.sh): no e2e leg, no parity assertion
        if rank == 0:
            emit_line({"value": value, "ms_per_step": ms / args.steps, "roofline": roofline})
        return 0

    # ---- end to end through the reference-facing model object: pinned host input -> host logits
    x_host = x.cpu().pin_memory()
    e2e_steps = max(3, min(args.steps, 20))
    for _ in range(2):
        out_host = qmodel(x_host)
    barrier()
    ev0.record()
    for _ in range(e2e_steps):
        out_host = qmodel(x_host)
    ev1.record()
    barrier()
    e2e_ms = max_over_ranks(ev0.elapsed_time(ev1))
    e2e = {"value": world * B * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "steps": e2e_steps,
           "h2d_bytes_per_step": x_host.numel() * x_host.element_size(),
           "d2h_bytes_per_step": out_host.numel() * out_host.element_size(),
           "api": "StaticPTQModel().quantize() -> model(x_cpu_pinned) -> cpu logits"}
    assert torch.equal(out_host, logits.cpu()), "e2e logits differ from the device-resident run"

    # ---- the same call on the uint8 data path (SURVEY 8f rank 4; extra key, NOT the contract's e2e): raw uint8 NHWC
    #      pixels from pinned host memory -> host logits; a quarter of the bytes cross PCIe.  Its inputs are other images
    #      (the fp32 batch above was normalised on the device), so only determinism is checked here; bit-identity with
    #      the fp32 route is a parity test (tests/test_gpu_net.py).
    pix_host = torch.randint(0, 256, (B, 32, 32, 3), dtype=torch.uint8,
                             generator=torch.Generator().manual_seed(1000 + rank)).pin_memory()
    for _ in range(2):
        out_u8 = qmodel.forward_uint8(pix_host)
    barrier()
    ev0.record()
    for _ in range(e2e_steps):
        out_u8_2 = qmodel.forward_uint8(pix_host)
    ev1.record()
    barrier()
    u8_ms = max_over_ranks(ev0.elapsed_time(ev1))
    assert torch.equal(out_u8, out_u8_2)
    e2e_u8 = {"value": world * B * e2e_steps / (u8_ms * 1e-3), "unit": UNIT, "steps": e2e_steps,
              "h2d_bytes_per_step": pix_host.numel(), "d2h_bytes_per_step": out_u8.numel() * out_u8.element_size(),
              "api": "model.forward_uint8(pixels_cpu_pinned uint8 NHWC) -> cpu logits"}

    # ---- sustained: the same loop for >= args.sustain_s seconds of device time (power cap / thermals in force), clocks
    #      sampled throughout; `value` above is the contract's K-step number, this is what a long job sees
    sustained = None
    if args.sustain_s > 0:
        n_sus = max(args.steps, int(args.sustain_s / (ms * 1e-3 / args.steps)) + 1)
        with ClockSampler(local) as sclk:
            barrier()
            ev0.record()
            for _ in range(n_sus):
                logits = engine.forward(x)
            ev1.record()
            barrier()
        sus_ms = max_over_ranks(ev0.elapsed_time(ev1))
        sustained = {"value": world * B * n_sus / (sus_ms * 1e-3), "unit": UNIT, "steps": n_sus, "seconds": sus_ms * 1e-3,
                     "ms_per_step": sus_ms / n_sus, "clocks": sclk.summary(),
                     "net_int8_tops": OPS_PER_IMAGE * B * n_sus / (sus_ms * 1e-3) / 1e12 ,
                     "net_frac_of_2x_bf16_sustained": OPS_PER_IMAGE * B * n_sus / (sus_ms * 1e-3) / 1e12 / peaks["int8_sustained"]}

    # ---- parity gate in the same run (BASELINE.md 4): >= 1 024 images of the TIMED batch - first, last, strided -
    #      through the torch/fbgemm CPU oracle; the logits of the timed loop must equal them bit for bit
    parity = None
    if rank == 0 and not args.no_parity:
        from oracle import torch_oracle
        q_oracle = build_cpu_oracle()
        idx = oracle_sample_indices(B)
        x_s = x[idx.to(dev)].cpu()
        want, _ = torch_oracle.run_static_oracle(q_oracle, x_s)
        got = logits[idx.to(dev)].cpu()
        ok = bool(torch.equal(got, want)) and bool(torch.equal(out_host[idx], want))
        parity = {"images": int(idx.numel()), "of_batch": B, "bit_exact": ok,
                  "oracle": f"torch {torch.__version__} fbgemm static-PTQ CPU ops (oracle/torch_oracle.py)",
                  "checked": "logits of the timed device-resident loop and of the e2e host-input call",
                  "mismatching_logits": int((got != want).sum())}
        assert ok, f"bench parity gate failed: {parity}"

    # ---- correct-count: the only collective, off the hot path (one NCCL all-reduce of 3 int64)
    from convnet_quantization_b200 import sharding
    counts = [int(v) for v in sharding.allreduce_counts(sharding.topk_counts(logits, labels)).tolist()]

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        q = q_oracle if parity is not None else build_cpu_oracle()
        # bounded sample: ~10-20 s of CPU work at batch 64 (BASELINE config 1)
        ips0, _, cores, _ = time_cpu_oracle(q, 64, 8, 2, 1)
        steps_cpu = max(2, int(12.0 * ips0 / (64 * 16)))
        ips, dt, cores, _ = time_cpu_oracle(q, 64, 16, steps_cpu, 1)
        cpu_baseline = {"value": ips, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"{steps_cpu * 16} batches x 64 images in {dt:.1f} s, torch {torch.__version__} "
                                  f"fbgemm static-PTQ oracle, {cores} threads"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic",
            "config": {"workload": "static-PTQ int8 SimpleConvNet forward, CIFAR-10 shape fp32 [B,3,32,32] -> logits [B,10]",
                       "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"batch-sharded x{world}",
                       "l2": f"input {x.numel() * 4 / 2**20:.0f} MiB + activations > 126 MiB L2 (no flush needed)",
                       "host_binding_rank0": host_binding},
            "clocks": clocks.summary(), "e2e": e2e, "e2e_u8": e2e_u8, "gpu_launches": launches, "roofline": roofline,
            "sustained": sustained, "parity": parity, "cpu_baseline": cpu_baseline,
            "eval": {"top1": counts[0], "top5": counts[1], "total": counts[2], "labels": "random (collective exercise only)"},
        }
        emit_line(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


# ----------------------------------------------------------------------------------------------- BASELINE configs 3-4
def run_variant(args):
    """``--variant dynamic|fp32|custom|custom_sandwich`` (BASELINE.json configs 3 and 4) on ONE B200: images/s of the
    drop-in model class with the batch resident in HBM, the same call from pinned host memory (e2e), the CPU counterpart
    (what the reference's class computes, built by oracle/torch_oracle.py) timed beside it at batch 64, and the logits
    of a sample compared with that counterpart (tolerance variants: max error relative to the logit range + argmax)."""
    from convnet_quantization_b200 import _lib, ops, synth
    from convnet_quantization_b200.models.baseline_model import SimpleConvNet
    from convnet_quantization_b200.models.custom_quantization_model import CustomQuantizationModel
    from convnet_quantization_b200.models.dynamic_ptq_model import DynamicPTQModel
    from oracle import torch_oracle

    if int(os.environ.get("WORLD_SIZE", "1")) != 1:
        raise SystemExit("--variant legs are single-GPU measurements (BASELINE configs 3-4)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (no CPU fallback; use --impl reference)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    sd = synth.make_state_dict(0)
    net = SimpleConvNet()
    net.load_state_dict(sd)
    net.eval()
    v = args.variant
    B = args.batch if args.batch != 16384 else 4096
    if v == "dynamic":
        m = DynamicPTQModel(device=dev)
        m.load_state_dict(sd)
        model = m.quantize()
        cpu_model, kind = torch_oracle.build_dynamic_oracle(net), "reference DynamicPTQModel: BN-folded fp32 convs + quantize_dynamic fc1/fc2"
    elif v == "fp32":
        model = SimpleConvNet()
        model.load_state_dict(sd)
        model = model.eval().to(dev)
        cpu_model, kind = net, "reference SimpleConvNet fp32 (MKL-DNN)"
    else:
        m = CustomQuantizationModel(mode="sandwich" if v == "custom_sandwich" else "as_written", device=dev)
        m.load_state_dict(sd)
        model = m.quantize()
        if v == "custom":
            model = model.to(dev)
            from torch.ao.quantization import fuse_modules
            import copy
            cpu_model = fuse_modules(copy.deepcopy(net), torch_oracle.FUSE_LIST, inplace=False).eval()
            kind = "reference CustomQuantizationModel as written: BN-folded fp32 net, identity stubs"
        else:
            q = torch_oracle.build_sandwich_oracle(net, synth.calibration_batches())
            cpu_model, kind = (lambda t: q(t)), "custom variant as intended: converted per-layer sandwiches (torch fbgemm)"
    if hasattr(model, "sync_on_forward"):
        model.sync_on_forward = False  # timed with CUDA events below

    g = torch.Generator(device=dev).manual_seed(0)
    x = synth.normalize(torch.randint(0, 256, (B, 3, 32, 32), dtype=torch.uint8, device=dev, generator=g)).contiguous()
    ctx = torch.backends.cudnn.flags(enabled=True, allow_tf32=False)
    with torch.no_grad(), ctx:
        for _ in range(max(args.warmup, 3)):
            y = model(x)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = lib.b200q_launch_count()
        with ClockSampler(0) as clocks:
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(args.steps):
                y = model(x)
            ev1.record()
            torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        launches = int(lib.b200q_launch_count() - n0)
        value = B * args.steps / (ms * 1e-3)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"logits": y})

        x_host = x.cpu().pin_memory()
        e2e_steps = max(3, min(args.steps, 20))
        for _ in range(2):
            out_host = model(x_host.to(dev, non_blocking=True)).cpu() if v in ("fp32", "custom") else model(x_host)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(e2e_steps):
            out_host = model(x_host.to(dev, non_blocking=True)).cpu() if v in ("fp32", "custom") else model(x_host)
        ev1.record()
        torch.cuda.synchronize()
        e2e_ms = ev0.elapsed_time(ev1)
        e2e = {"value": B * e2e_steps / (e2e_ms * 1e-3), "unit": UNIT, "steps": e2e_steps,
               "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": out_host.numel() * 4,
               "api": "model(x_cpu_pinned) -> cpu logits (fp32 / custom-as-written: plain nn.Module, .to(device) by the caller)"}

        # ---- the int8 kernel of the dynamic variant against the HBM roofline (fc1: fp32 [B,4096] read twice - min/max pass
        #      and GEMM producer - plus the fp32 [B,512] result)
        roofline = None
        peaks = load_peaks()
        if v == "dynamic":
            feats = model.features(x)
            for _ in range(3):
                ops.linear_dynamic(feats, model.fc["fc1"], relu=True)
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(20):
                ops.linear_dynamic(feats, model.fc["fc1"], relu=True)
            ev1.record()
            torch.cuda.synchronize()
            t = ev0.elapsed_time(ev1) / 20 * 1e-3
            bytes_alg = B * 4096 * 4 * 2 + B * 512 * 4 + 4096 * 512
            roofline = {"kernel": "linear_dynamic fc1 (minmax_kernel + linear_dynamic_tc_kernel<512>)", "bound": "hbm",
                        "achieved": bytes_alg / t / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": bytes_alg / t / 1e9 / peaks["hbm_gbs"], "traffic": None, "ms": t * 1e3,
                        "algorithmic_bytes": bytes_alg, "peak_source": f"{peaks['source']}: hbm_gbs"}

        # ---- tolerance check against the CPU counterpart (batch 64: dynamic quantisation is per batch tensor)
        xs = x[:64].cpu()
        torch.set_num_threads(os.cpu_count() or 1)
        want = cpu_model(xs)
        got = model(x[:64].contiguous()).cpu()
    scale = float(want.abs().max())
    err = (got - want).abs()
    parity = {"images": 64, "max_abs_err_over_logit_range": float(err.max()) / scale,
              "frac_within_1e-3": float((err <= 1e-3 * scale).float().mean()),
              "argmax_agree": float((got.argmax(1) == want.argmax(1)).float().mean()), "against": kind}

    # ---- CPU baseline: bounded sample at batch 64 (BASELINE config 1 protocol)
    cpu_baseline = None
    if not args.no_cpu_baseline:
        xb = synth.images_f32(64, seed=11)
        with torch.no_grad():
            cpu_model(xb)
            t0 = time.perf_counter()
            n = 0
            while time.perf_counter() - t0 < 8.0:
                cpu_model(xb)
                n += 1
            dt = time.perf_counter() - t0
        cpu_baseline = {"value": 64 * n / dt, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                        "sample": f"{n} batches x 64 images in {dt:.1f} s; {kind}"}
    line = {"metric": METRIC.replace("static-PTQ", v), "variant": v, "value": value, "unit": UNIT, "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32" if v in ("fp32", "custom") else "u8", "data": "synthetic",
            "config": {"workload": f"{v} SimpleConvNet forward (BASELINE config {'3' if v in ('dynamic', 'fp32') else '4'}), "
                                   "CIFAR-10 shape fp32 [B,3,32,32] -> logits [B,10]", "batch_per_gpu": B,
                       "l2": f"input {x.numel() * 4 / 2**20:.0f} MiB + activations exceed the 126 MiB L2"},
            "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": launches,
            "gpu_launches_note": "kernels of libb200q.so only; fp32 convolutions of this variant are ATen/cuDNN (tolerance path)",
            "roofline": roofline, "parity": parity, "cpu_baseline": cpu_baseline}
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=16384, help="images per GPU per step")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bind", action="store_true", help="do not pin the rank to its GPU's NUMA-local CPUs")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run oracle comparison (timing experiments)")
    ap.add_argument("--sustain-s", type=float, default=2.0, help="seconds of the extra sustained loop (0: skip)")
    ap.add_argument("--variant", default="static", choices=["static", "dynamic", "fp32", "custom", "custom_sandwich"],
                    help="static = the headline (BASELINE config 2/5); the others are BASELINE configs 3-4")
    ap.add_argument("--stages-only", action="store_true", help="print only the per-kernel table (timing experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the logits of the last timed step to DIR/logits.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "ours" and world != args.gpus and args.gpus > 1:
        raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args) if args.variant == "static" else run_variant(args)


if __name__ == "__main__":
    sys.exit(main())
