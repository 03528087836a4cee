"""Sharded accuracy sweep over a host-resident labelled dataset (BASELINE config 5 / SURVEY 8(e)): one process per GPU,
NCCL, each rank's shard through ``B200StaticQuantizedNet.evaluate`` / ``evaluate_uint8`` (counting in the head kernel),
one all-reduce of the five counters.
    python scripts/eval_sweep.py --gpus N --images 1048576 --input u8|fp32 [--out profiles/r04_eval_sweep.json]
The dataset is synthetic: uint8 pixels and labels generated in fixed blocks of BLOCK images, each seeded by its block
index, so every N sees the same images (the fp32 input is the normalised pixels: both inputs give the same counts).
Each rank's shard is pinned host memory.  Timed, alternating, best of REPS: the evaluate sweep (barrier -> counters
all-reduced) and the plain host-input forward of the same shard (``forward`` / ``forward_uint8``, logits to the host).
On the first ``--sample`` images of every shard the script also compares the old ``topk`` counting
(``sharding.topk_counts`` arithmetic on the same logits) with the counts, image by image.
The result is merged into ``--out`` under the key ``"<input>_n<N>"``; the card's name and power limit are read in the
run."""
import argparse, json, os, socket, subprocess, sys, time, warnings
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
warnings.filterwarnings("ignore")
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

BLOCK = 16384
REPS = 3


def _block(i: int):
    from convnet_quantization_b200 import synth
    pix = synth.images_u8(BLOCK, seed=100_000 + i).permute(0, 2, 3, 1).contiguous()  # NHWC
    labels = torch.randint(0, 10, (BLOCK,), generator=torch.Generator().manual_seed(200_000 + i))
    return pix, labels


def _shard(lo: int, hi: int, u8: bool):
    """Images [lo, hi) of the dataset as pinned host tensors (uint8 NHWC or fp32 NCHW) plus int64 labels."""
    from convnet_quantization_b200 import synth
    n = hi - lo
    x = torch.empty((n, 32, 32, 3) if u8 else (n, 3, 32, 32), dtype=torch.uint8 if u8 else torch.float32).pin_memory()
    labels = torch.empty(n, dtype=torch.int64)
    for blk in range(lo // BLOCK, (hi + BLOCK - 1) // BLOCK):
        pix, lab = _block(blk)
        a, b = max(lo, blk * BLOCK), min(hi, (blk + 1) * BLOCK)
        p = pix[a - blk * BLOCK:b - blk * BLOCK]
        x[a - lo:b - lo] = p if u8 else synth.normalize(p.permute(0, 3, 1, 2))
        labels[a - lo:b - lo] = lab[a - blk * BLOCK:b - blk * BLOCK]
    return x, labels


def _worker(rank, world, port, a, result):
    from convnet_quantization_b200 import ptq, sharding, synth
    from convnet_quantization_b200.models._gpu_modules import B200StaticQuantizedNet
    from convnet_quantization_b200.models.baseline_model import SimpleConvNet
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    sharding.bind_to_gpu_numa(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        u8 = a.input == "u8"
        net = SimpleConvNet()
        net.load_state_dict(synth.make_state_dict(0))
        model = B200StaticQuantizedNet(ptq.calibrate_static(net.eval(), synth.calibration_batches()), dev)
        lo, hi = sharding.shard_range(a.images, rank, world)
        x, labels = _shard(lo, hi, u8)
        fwd = model.forward_uint8 if u8 else model.forward

        def sweep():
            return sharding.allreduce_counts(model.eval_counters(x, labels, u8=u8)).cpu()

        w = min(8192, hi - lo)  # warm-up: every kernel shape and the staging buffers
        model.eval_counters(x[:w], labels[:w], u8=u8)
        fwd(x[:w])
        best = {"evaluate": float("inf"), "forward": float("inf")}
        counts = None
        for _ in range(REPS):
            for name in best:
                dist.barrier()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if name == "evaluate":
                    counts = sweep()
                else:
                    fwd(x)
                    torch.cuda.synchronize()
                dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)  # the sweep ends with its slowest rank
                best[name] = min(best[name], float(dt))

        # old topk counting vs the counts, image by image, on a sample of every shard
        s = min(a.sample, hi - lo)
        xs, ls = x[:s].to(dev), labels[:s].to(dev)
        logits = model.engine.forward_u8(xs, graph=False) if u8 else model.engine.forward(xs, graph=False)
        top5 = logits.topk(min(5, logits.shape[1]), dim=1).indices.eq(ls.view(-1, 1))  # sharding.topk_counts
        rule = sharding.rank_rule_hits(logits, ls)
        disagree = (top5[:, 0] != rule[:, 0]) | (top5.any(1) != rule[:, 1])
        kernel = model.engine.evaluate_u8(xs, ls) if u8 else model.engine.evaluate(xs, ls)
        assert torch.equal(kernel, sharding.rank_rule_counts(logits, ls)), "kernel counts differ from the rule"
        stats = torch.cat([sharding.topk_counts(logits, ls), sharding.rank_rule_counts(logits, ls),
                           torch.stack([disagree.sum(), (top5[:, 0] != rule[:, 0]).sum(),
                                        (top5.any(1) != rule[:, 1]).sum()])]).to(torch.int64)
        dist.all_reduce(stats)
        if rank == 0:
            st = stats.tolist()
            result.update(
                gpus=world, input=a.input, images=a.images,
                eval_s=round(best["evaluate"], 4), forward_s=round(best["forward"], 4),
                eval_images_per_s=round(a.images / best["evaluate"]),
                forward_images_per_s=round(a.images / best["forward"]),
                counters=dict(zip(("top1", "top5", "images", "top1_tied", "top5_tied"), counts.tolist())),
                topk_vs_counts_sample={
                    "images": st[5], "per_shard": s,
                    "topk_counts": dict(zip(("top1", "top5", "images"), st[0:3])),
                    "counts": dict(zip(("top1", "top5", "images", "top1_tied", "top5_tied"), st[3:8])),
                    "images_scored_differently": st[8], "top1_differs": st[9], "top5_differs": st[10]})
    finally:
        dist.destroy_process_group()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--images", type=int, default=1 << 20)
    ap.add_argument("--input", choices=("u8", "fp32"), default="u8")
    ap.add_argument("--sample", type=int, default=16384, help="images per shard compared with the topk counting")
    ap.add_argument("--out", default="profiles/r04_eval_sweep.json")
    a = ap.parse_args()
    if a.gpus > torch.cuda.device_count():
        sys.exit(f"--gpus {a.gpus}: only {torch.cuda.device_count()} CUDA devices")
    smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    with mp.Manager() as m:
        result = m.dict()
        mp.spawn(_worker, args=(a.gpus, _free_port(), a, result), nprocs=a.gpus, join=True)
        row = dict(result)
    row["gpu"] = smi
    doc = {}
    if os.path.exists(a.out):
        with open(a.out) as f:
            doc = json.load(f)
    doc.setdefault("what", "sharded accuracy sweep over a host-resident synthetic labelled dataset (pinned uint8 NHWC or "
                           "fp32 NCHW shards), one process per GPU, NCCL all-reduce of the five counters; eval_s = "
                           "barrier to all-reduced counters on the host, forward_s = the host-input forward of the same "
                           "shards (logits to the host); best of 3, alternating; scripts/eval_sweep.py")
    doc.setdefault("runs", {})[f"{a.input}_n{a.gpus}"] = row
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1, sort_keys=True)
    print(json.dumps(row))


if __name__ == "__main__":
    main()
