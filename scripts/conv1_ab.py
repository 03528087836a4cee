"""Interleaved A-B timing of two builds of the product library on one GPU: ``bench.py --stages-only`` pairs plus one full
``bench.py`` per build (with ``--dump-outputs``, whose logits must be byte-identical), alternating builds.

    python scripts/conv1_ab.py --base-lib convnet_quantization_b200/build/libb200q_base.so --out OUT.json

``--base-lib`` is a ``libb200q.so`` built from the parent commit; the current tree's library is the other side.  The
card's name and power limit are read in the same run and stored beside the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(lib, extra):
    env = dict(os.environ)
    env.pop("B200Q_LIB", None)
    if lib:
        env["B200Q_LIB"] = lib
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", *extra], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    if r.returncode != 0:
        raise RuntimeError(f"bench.py {extra} failed:\n{r.stderr[-3000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])


def _stages(d):
    return {k: v["ms"] for k, v in d["roofline"]["stages"].items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base-lib", required=True)
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    sides = {"base": os.path.abspath(args.base_lib), "new": None}
    res = {"gpu": smi[0] if smi else None, "pairs": [], "full": {}}
    steps = ["--steps", str(args.steps), "--warmup", str(args.warmup)]
    for p in range(args.pairs):
        pair = {}
        for name in (("base", "new") if p % 2 == 0 else ("new", "base")):
            d = _bench(sides[name], steps + ["--stages-only"])
            pair[name] = {"ms_per_step": d["ms_per_step"], "stages": _stages(d)}
            print(name, "stages-only", json.dumps(pair[name]), flush=True)
        res["pairs"].append(pair)
    with tempfile.TemporaryDirectory() as tmp:
        for name in ("base", "new"):
            dump = os.path.join(tmp, name)
            d = _bench(sides[name], steps + ["--dump-outputs", dump])
            res["full"][name] = {"value": d["value"], "ms_per_step": d["ms_per_step"], "stages": _stages(d),
                                 "e2e": d.get("e2e", {}).get("value"), "e2e_u8": d.get("e2e_u8", {}).get("value"),
                                 "parity": d.get("parity")}
            print(name, "full", json.dumps(res["full"][name]), flush=True)
        a, b = (open(os.path.join(tmp, n, "logits.npy"), "rb").read() for n in ("base", "new"))
        res["logits_byte_identical"] = a == b
        res["logits_shape"] = list(np.load(os.path.join(tmp, "new", "logits.npy")).shape)
    c1 = {n: [p[n]["stages"]["quant_conv1"] for p in res["pairs"]] for n in sides}
    step = {n: [p[n]["ms_per_step"] for p in res["pairs"]] for n in sides}
    res["summary"] = {
        "quant_conv1_ms": c1, "ms_per_step": step,
        "quant_conv1_gain_per_pair": [1 - b / a for a, b in zip(c1["base"], c1["new"])],
        "step_gain_per_pair": [1 - b / a for a, b in zip(step["base"], step["new"])],
        "step_gain_mean": 1 - statistics.mean(step["new"]) / statistics.mean(step["base"]),
        "step_spread_same_build": {n: max(v) - min(v) for n, v in step.items()},
        "step_diff_of_means_ms": statistics.mean(step["base"]) - statistics.mean(step["new"]),
    }
    print(json.dumps(res["summary"], indent=1))
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
