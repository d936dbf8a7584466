"""Measures the pooled-row front end of the fused step with the frozen MiniLM backbone and prints one JSON line.

  * build: both pooled banks of the synthetic train split at max_samples=-1 (676,193 pairs, shape Z), query texts
    truncated to 32 tokens and passages to 256; wall time and encoded (unpadded) tokens per second;
  * step: the fused MiniLM step at configs[1] shape (global batch 2048, projection 512) over the banks, batches
    assembled on the device, graph replays, device-timed with CUDA events; no graph capture inside the timed window;
  * epoch: one full epoch through the device feeder, plus the build it needs;
  * reference: the reference-shaped MiniLM step (bench.py's full_backbone recipe: the encoder runs for all three texts
    of every triplet), in the same process, for comparison.

Run:   python scripts/pooled_front_bench.py [--steps 200]
       torchrun --nproc_per_node N scripts/pooled_front_bench.py   (adds the sharded build time on N GPUs)
"""
import argparse
import json
import os
import subprocess
import sys
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def card_info(dev):
    """Card name and power limit, read in this call (the limit is part of every number measured here)."""
    info = {"name": torch.cuda.get_device_name(dev)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i",
                              str(dev.index or 0)], capture_output=True, text=True, timeout=20).stdout.strip()
        name, limit = [s.strip() for s in out.split(",")]
        info.update(smi_name=name, power_limit_w=float(limit))
    except Exception as e:  # noqa: BLE001
        info["power_limit_w"] = f"unavailable ({type(e).__name__})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--proj", type=int, default=512)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    from two_towers_overlords_b200 import TwoTowersModel
    from two_towers_overlords_b200.data import DeviceTripletFeeder, MSMarcoDataset, PooledBank
    from two_towers_overlords_b200.training import FusedTrainer

    Lq, Ld = 32, 256
    ds = MSMarcoDataset("train", max_samples=-1, synthetic=True)
    torch.manual_seed(0)
    model = TwoTowersModel(projection_dim=args.proj, backbone="minilm").to(dev)
    if world > 1:
        for t in model.parameters():
            dist.broadcast(t.data, src=0)

    def tokens(bank, L):
        return int(np.minimum(np.diff(bank.offsets), L).sum())

    # a first small build pays the one-time costs (weight split, kernel attributes) outside the timed build
    PooledBank.encode_rows(model.query_tower, ds.query_bank, Lq, 0, 64)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    build = {}
    t0 = time.perf_counter()
    bq = PooledBank.build(model.query_tower, ds.query_bank, Lq, world_size=world, rank=rank)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    bd = PooledBank.build(model.document_tower, ds.doc_bank, Ld, world_size=world, rank=rank)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    for name, bank, L, dt in (("queries", ds.query_bank, Lq, t1 - t0), ("passages", ds.doc_bank, Ld, t2 - t1)):
        n_tok = tokens(bank, L)
        build[name] = {"texts": len(bank), "tokens": n_tok, "s": dt, "tokens_per_s": n_tok / dt}
    build["total_s"] = t2 - t0
    build["gpus"] = world

    B = args.batch // world
    tr = FusedTrainer(model, 0.3, 1e-4, B, Lq, Ld, token_slots=2, world_size=world, rank=rank, pooled=(bq, bd))
    feeder = DeviceTripletFeeder(ds, args.batch, Lq, Ld, dev, rank=rank, world_size=world, seed=0,
                                 rows_only=True)
    tr.prepare(2)
    feeder.start_epoch()
    n_steps = len(feeder)
    total = min(args.warmup + args.steps, n_steps)
    steps = total - args.warmup
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    feeder.assemble(tr, 0, 0)
    cap0 = None
    for i in range(total):
        if i == args.warmup:
            tr.sync_ranks()
            cap0 = tr.graph_captures
            ev0.record()
        nslot = (i + 1) % 2 if i + 1 < n_steps else None
        if nslot is not None:
            feeder.assemble(tr, nslot, i + 1)
        loss = tr.step(i % 2, nslot)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / steps
    step = {"global_batch": args.batch, "per_gpu": B, "proj": args.proj, "precision": tr.precision,
            "ms_per_step": ms, "triplets_per_s": args.batch / (ms * 1e-3), "steps_timed": steps,
            "graph_captures_in_timed": tr.graph_captures - cap0, "loss": float(loss.item())}

    tr.sync_ranks()
    t0 = time.perf_counter()
    avg = tr.train_epoch_device(feeder)
    torch.cuda.synchronize()
    epoch_s = time.perf_counter() - t0
    epoch = {"steps": n_steps, "s": epoch_s, "s_with_build": epoch_s + build["total_s"], "avg_loss": avg}

    out = {"metric": "pooled_front_minilm", "card": card_info(dev), "world": world, "build": build, "step": step,
           "epoch": epoch}
    if world == 1:
        import bench

        out["reference_step"] = bench.run_backbone_leg(dev, types.SimpleNamespace(precision=None, no_cpu=True))
        out["speedup_vs_reference_triplets_per_s"] = step["triplets_per_s"] / out["reference_step"]["triplets_per_s"]
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        tr.sync_ranks()
        tr.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
