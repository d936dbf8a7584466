"""Measures gradient accumulation in the fused trainer (FusedTrainer(accumulation_steps=a)) and prints one JSON line.

  * fused: configs[1] shape (B = 2048, P = 512, token table, 32 / 256 tokens), device feeder, graph replays, a in
    {1, 2, 4}; ms per micro-step and triplets/s are the median of --epochs full epochs of the synthetic train split after
    one warm-up epoch, each timed with CUDA events; no graph capture may happen in the timed epochs;
  * reference: the reference-shaped train_epoch_optimized (what run_training runs for main.py's defaults with the
    switch off) at the same shape with a = 2, host-tokenised batches, over --ref-batches batches after one warm-up
    batch (synchronised host clock);
  * minilm: the pooled MiniLM trainer (banks of a --minilm-pairs-pair subset of the split) at a = 1 and 2;
  * multi_gpu: "not measured" on a machine with one GPU.

Run:   python scripts/accumulation_bench.py [--epochs 3]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from pooled_front_bench import card_info  # noqa: E402


def time_epochs(tr, feeder, epochs, batch):
    """Median ms per micro-step over `epochs` timed epochs after one warm-up epoch."""
    tr.train_epoch_device(feeder)  # warm-up epoch (also every mode of the window schedule)
    cap0 = tr.graph_captures
    ms, losses = [], []
    for _ in range(epochs):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        losses.append(tr.train_epoch_device(feeder))
        ev1.record()
        torch.cuda.synchronize()
        ms.append(ev0.elapsed_time(ev1) / len(feeder))
    med = statistics.median(ms)
    return {"ms_per_micro_step": med, "ms_per_micro_step_all": ms, "triplets_per_s": batch / (med * 1e-3),
            "micro_steps_per_epoch": len(feeder), "optimizer_steps": int(tr.adam_state[0].item()),
            "graph_captures_in_timed": tr.graph_captures - cap0, "avg_loss_last_epoch": losses[-1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--epochs", type=int, default=3)
    ap.add_argument("--batch", type=int, default=2048)
    ap.add_argument("--proj", type=int, default=512)
    ap.add_argument("--ref-batches", type=int, default=10)
    ap.add_argument("--minilm-pairs", type=int, default=2048 * 40)
    args = ap.parse_args()
    assert args.epochs >= 3, "report a median of at least 3 epochs"
    dev = torch.device("cuda", 0)
    from two_towers_overlords_b200 import TripletLoss, TwoTowersModel
    from two_towers_overlords_b200.data import DeviceTripletFeeder, MSMarcoDataset, PooledBank, TripletDataLoader
    from two_towers_overlords_b200.training import FusedTrainer, train_epoch_optimized

    B, P = args.batch, args.proj
    out = {"metric": "fused_gradient_accumulation", "card": card_info(dev), "batch": B, "proj": P, "fused": {}}
    ds = MSMarcoDataset("train", max_samples=-1, synthetic=True)
    for a in (1, 2, 4):
        torch.manual_seed(0)
        model = TwoTowersModel(projection_dim=P).to(dev)
        tr = FusedTrainer(model, 0.3, 1e-4, B, token_slots=2, in_batch_negatives=True, accumulation_steps=a)
        feeder = DeviceTripletFeeder(ds, B, tr.Lq, tr.Ld, dev, seed=0)
        tr.prepare(2)
        r = time_epochs(tr, feeder, args.epochs, B)
        assert r["graph_captures_in_timed"] == 0, r
        out["fused"][f"a{a}"] = r
        del tr, model, feeder
        torch.cuda.empty_cache()

    # the reference-shaped loop run_training takes for main.py's defaults without the switch
    torch.manual_seed(0)
    model = TwoTowersModel(projection_dim=P).to(dev)
    ref_ds = MSMarcoDataset("train", max_samples=B * (args.ref_batches + 1), synthetic=True)
    model.query_tower.tokenizer = model.document_tower.tokenizer = ref_ds.tokenizer()
    dl = list(TripletDataLoader(ref_ds, batch_size=B, num_workers=0, device=dev))
    opt = torch.optim.Adam(model.parameters(), lr=1e-4)
    scaler = torch.amp.GradScaler("cuda")
    crit = TripletLoss(0.3)
    train_epoch_optimized(model, dl[:2], crit, opt, dev, scaler, accumulation_steps=2, log_wandb=False)  # warm-up
    timed = dl[: args.ref_batches]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    train_epoch_optimized(model, timed, crit, opt, dev, scaler, accumulation_steps=2, log_wandb=False)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3 / len(timed)
    out["reference_train_epoch_optimized_a2"] = {"ms_per_micro_step": ms, "triplets_per_s": B / (ms * 1e-3),
                                                 "batches_timed": len(timed),
                                                 "note": "host-tokenised batches, synchronised host clock"}
    del model, opt, dl
    torch.cuda.empty_cache()

    # the pooled MiniLM trainer
    mds = MSMarcoDataset("train", max_samples=args.minilm_pairs, synthetic=True)
    out["minilm"] = {"pairs": args.minilm_pairs}
    torch.manual_seed(0)
    model = TwoTowersModel(projection_dim=P, backbone="minilm").to(dev)
    banks = (PooledBank.build(model.query_tower, mds.query_bank, 32), PooledBank.build(model.document_tower,
                                                                                       mds.doc_bank, 256))
    for a in (1, 2):
        tr = FusedTrainer(model, 0.3, 1e-4, B, 32, 256, token_slots=2, pooled=banks, accumulation_steps=a)
        feeder = DeviceTripletFeeder(mds, B, 32, 256, dev, seed=0, rows_only=True)
        tr.prepare(2)
        r = time_epochs(tr, feeder, args.epochs, B)
        assert r["graph_captures_in_timed"] == 0, r
        out["minilm"][f"a{a}"] = r
        del tr, feeder
    out["multi_gpu"] = ("not measured: this machine has one GPU" if torch.cuda.device_count() < 2 else
                        "not measured: no torchrun leg in this script")
    print(json.dumps(out))


if __name__ == "__main__":
    main()
