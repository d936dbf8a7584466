"""Measures hard-negative mining (data.HardNegativeMiner) on one GPU and writes one JSON file.

  * refresh: one table refresh at the full synthetic train split (82,463 queries x 676,193 passages, pooled rows of
    the frozen token tables), for projection dims 128 and 512, split into projection, normalise, scan, merge and filter
    by device events; median of --refreshes after one warm-up refresh;
  * epoch: full epochs of the fused trainer through the device feeder at configs[1] shape (batch 2048, projection 512),
    with in-batch negatives and with mined negatives (ratio 0.5, depth 8, the table refreshed once before), for
    - the pooled MiniLM trainer (banks of random unit rows carrying the towers' identity: a step copies rows by index,
      so its time does not depend on their values; encoding 760 k texts is pooled_front_bench.py's subject),
    - the token-table trainer: in-batch negatives reuse the positives' pooled rows (neg_index), mined negatives cannot,
      so that leg pools the negatives' tokens;
    epoch time = device events around train_epoch_device after one warm-up epoch, median of --epochs.

Run:   python scripts/hard_negative_bench.py [--out profiles/r04_hard_negatives_n1.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

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


def timed_epoch(trainer, feeder):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    loss = trainer.train_epoch_device(feeder)
    b.record()
    b.synchronize()
    return a.elapsed_time(b), loss


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_hard_negatives_n1.json"))
    ap.add_argument("--refreshes", type=int, default=5)
    ap.add_argument("--epochs", type=int, default=3)
    args = ap.parse_args()
    import __graft_entry__ as g

    g.build()
    from two_towers_overlords_b200 import TwoTowersModel, data, training

    dev = torch.device("cuda", 0)
    result = {"card": card_info(dev), "refresh": {}, "epoch": {}}
    ds = data.MSMarcoDataset("train", max_samples=-1, synthetic=True)
    Lq, Ld, B = 32, 256, 2048
    result["split"] = {"pairs": len(ds), "queries": len(ds.query_bank), "passages": len(ds.doc_bank)}

    # ---- refresh -------------------------------------------------------------------------------------------------
    for P in (128, 512):
        torch.manual_seed(0)
        model = TwoTowersModel(projection_dim=P).to(dev)
        banks = (data.PooledBank.build(model.query_tower, ds.query_bank, Lq),
                 data.PooledBank.build(model.document_tower, ds.doc_bank, Ld))
        miner = data.HardNegativeMiner(ds, *banks, depth=8, k_scan=32)
        miner.refresh(model)  # warm-up: module loads, scan plan
        runs = [miner.refresh(model) for _ in range(args.refreshes)]
        med = {k: statistics.median(r[k] for r in runs) for k in runs[0]}
        flop = 2.0 * miner.n_rows * miner.n_docs * P
        result["refresh"][f"P{P}"] = {
            "ms": {k[:-2]: round(v * 1e3, 3) for k, v in med.items() if k.endswith("_s")},
            "scan_tflops_bf16_nominal": round(flop / med["scan_s"] / 1e12, 1),
            "mean_count": med["mean_count"], "empty_queries": int(med["empty_queries"]), "refreshes": args.refreshes,
        }
        print(f"refresh P={P}: {result['refresh'][f'P{P}']}", flush=True)
        del miner, banks, model
        torch.cuda.empty_cache()

    # ---- epochs --------------------------------------------------------------------------------------------------
    def run(kind, mined):
        torch.manual_seed(1)
        if kind == "minilm":
            model = TwoTowersModel(projection_dim=512, backbone="minilm").to(dev)
            gen = torch.Generator(device=dev).manual_seed(2)
            banks = tuple(data.PooledBank(torch.nn.functional.normalize(torch.randn(n, 384, generator=gen, device=dev),
                                                                        dim=1), data.backbone_identity(t), L)
                          for n, t, L in ((len(ds.query_bank), model.query_tower, Lq),
                                          (len(ds.doc_bank), model.document_tower, Ld)))
            trainer = training.FusedTrainer(model, 0.3, 1e-4, B, Lq, Ld, token_slots=2, pooled=banks)
        else:
            model = TwoTowersModel(projection_dim=512).to(dev)
            trainer = training.FusedTrainer(model, 0.3, 1e-4, B, Lq, Ld, token_slots=2, in_batch_negatives=not mined)
            banks = (data.PooledBank.build(model.query_tower, ds.query_bank, Lq),
                     data.PooledBank.build(model.document_tower, ds.doc_bank, Ld)) if mined else None
        feeder = data.DeviceTripletFeeder(ds, B, Lq, Ld, dev, seed=3, rows_only=kind == "minilm")
        if mined:
            miner = data.HardNegativeMiner(ds, *banks, depth=8, ratio=0.5)
            miner.refresh(model)
            feeder.hard_negatives = miner
        trainer.prepare(2)
        timed_epoch(trainer, feeder)  # warm-up epoch (graph captures)
        times, losses = zip(*[timed_epoch(trainer, feeder) for _ in range(args.epochs)])
        steps = len(feeder)
        ms = statistics.median(times)
        return {"epoch_ms": round(ms, 2), "steps": steps, "ms_per_step": round(ms / steps, 4),
                "epochs_timed": args.epochs, "last_loss": round(losses[-1], 5)}

    for kind in ("minilm", "table"):
        for mined in (False, True):
            key = f"{kind}_{'mined' if mined else 'in_batch'}"
            result["epoch"][key] = run(kind, mined)
            print(f"epoch {key}: {result['epoch'][key]}", flush=True)
            torch.cuda.empty_cache()
    result["card_after"] = card_info(dev)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
