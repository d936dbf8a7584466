"""Measures the token tables' optimiser in the fused step (FusedTrainer(optimize_tables=True)) and prints one JSON line.

configs[2] shape: B = 4096 triplets, P = 384, 32 / 256-token rows, both 30522 x 384 fp32 tables trainable, bf16x3,
persistent chain kernel, graph replays over 4 rotating token sets.  Timed in one process, alternating, --reps rounds of
--steps steps each (CUDA events, after --warmup steps of every mode):

  (a) grads:   table gradients only (what bench.py's config2 leg times);
  (b) fused:   optimize_tables=True, Adam in the scatter-add's epilogue;
  (c) unfused: (a), then tt_adam_step_dev on each table (gradient written, then a dense Adam pass);
  (d) peer:    (b) through the data-parallel code path at world 1 (tables in a peer segment, tt_dp_reduce_adam).

(b) and (c) run the same steps on the same tokens from the same seed and must leave bit-identical tables and moments.
The table update's bytes (read + write p, m, v: 24 B per element of both tables) over (b) - (a) is compared with the
7.7 TB/s HBM peak.  Under torchrun with N > 1 ranks only (b) runs, data parallel; the script checks that every
replica's tables are bit-identical to rank 0's and reports the table exchange's DpExchange.timing().

Run:   python scripts/table_training_bench.py [--out profiles/r09_table_training_n1.json]
       torchrun --nproc-per-node 8 scripts/table_training_bench.py --out /tmp/r09_table_training_n8.json
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from pooled_front_bench import card_info  # noqa: E402

HBM_PEAK = 7.7e12  # B/s, NVIDIA's data sheet figure for one B200


def tokens(B, Lq, Ld, V, seed):
    g = torch.Generator().manual_seed(seed)
    out = []
    for L in (Lq, Ld, Ld):
        ids = torch.randint(1000, V, (B, L), generator=g, dtype=torch.int64).to(torch.int32)
        n = torch.randint(L // 4, L + 1, (B,), generator=g)
        ids[:, 0] = 101  # [CLS]: a heavy row in every text
        out += [ids, (torch.arange(L)[None, :] < n[:, None]).to(torch.uint8)]
    return tuple(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--proj", type=int, default=384)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_table_training_n1.json"))
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    from two_towers_overlords_b200 import TwoTowersModel, _native as N
    from two_towers_overlords_b200.training import FusedTrainer

    B, P, Lq, Ld, S = args.batch // world, args.proj, 32, 256, 4
    sets = [tokens(B, Lq, Ld, 30522, 1000 * rank + i) for i in range(S)]

    def build(optimize, exchange=None):
        torch.manual_seed(0)
        m = TwoTowersModel(projection_dim=P, train_table=True).to(dev)
        tr = FusedTrainer(m, 0.3, 1e-4, B, Lq, Ld, precision="bf16x3", token_slots=S, world_size=world, rank=rank,
                          optimize_tables=optimize, exchange=exchange)
        for s, t in enumerate(sets):
            tr.load_packed(tr.pack_host_tokens(t, pin=False), s)
        tr.prepare(S)
        return m, tr

    tables = lambda m: (m.query_tower.pretrained_model.table, m.document_tower.pretrained_model.table)  # noqa: E731
    out = {"metric": "table_training", "card": card_info(dev), "world": world, "batch_global": args.batch, "proj": P,
           "vocab": 30522, "hidden": 384, "precision": "bf16x3", "token_sets": S, "steps": args.steps,
           "reps": args.reps}
    V, H = 30522, 384
    update_bytes = 2 * V * H * 24
    modes = {}
    if world == 1:
        modes["grads"] = build(False)
        modes["fused"] = build(True)
        modes["unfused"] = build(False)
        modes["peer"] = build(True, "peer")
        # (c): the unfused table update as one captured graph after each step (own step counters, advanced in lockstep)
        mu, tu = modes["unfused"]
        um = [torch.zeros(V, H, device=dev) for _ in range(4)]
        ust = [torch.zeros(4, dtype=torch.float64, device=dev) for _ in range(2)]

        def unfused_adam():
            for k, (p, g) in enumerate(zip(tables(mu), tu.table_grads)):
                N.check(N.load().tt_adam_step_dev(N.ptr(p.data), N.ptr(g), N.ptr(um[2 * k]), N.ptr(um[2 * k + 1]),
                                                  V * H, tu.lr, tu.betas[0], tu.betas[1], tu.eps, N.ptr(ust[k]), 1.0,
                                                  N.stream()), "tt_adam_step_dev")

        gu = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):  # the capture itself runs nothing
            with torch.cuda.graph(gu, stream=s):
                unfused_adam()
        torch.cuda.current_stream().wait_stream(s)
    else:
        modes["fused"] = build(True)

    def run(name, n, i0):
        m, tr = modes[name]
        for i in range(n):
            tr.step((i0 + i) % S)
            if name == "unfused":
                gu.replay()

    for name in modes:
        run(name, args.warmup, 0)
    torch.cuda.synchronize()
    caps = {k: tr.graph_captures for k, (_, tr) in modes.items()}
    if "peer" in modes:
        modes["peer"][1].txchg.reset_timing()
    times = {k: [] for k in modes}
    for r in range(args.reps):
        for name in modes:
            if world > 1:
                modes[name][1].sync_ranks()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            ev0.record()
            run(name, args.steps, args.warmup + r * args.steps)
            ev1.record()
            torch.cuda.synchronize()
            times[name].append(ev0.elapsed_time(ev1) / args.steps)
    for k, (_, tr) in modes.items():
        assert tr.graph_captures == caps[k], (k, "graph captured inside the timed steps")
        tr.check()
    res = {k: {"ms_per_step": statistics.median(v), "ms_per_step_all": v,
               "triplets_per_s": args.batch / (statistics.median(v) * 1e-3)} for k, v in times.items()}
    out["modes"] = res
    if world == 1:
        added = res["fused"]["ms_per_step"] - res["grads"]["ms_per_step"]
        out["fused_minus_grads_us"] = added * 1e3
        out["unfused_minus_grads_us"] = (res["unfused"]["ms_per_step"] - res["grads"]["ms_per_step"]) * 1e3
        out["table_update_bytes"] = update_bytes
        out["table_update_bytes_per_s_over_added_time"] = update_bytes / (added * 1e-3) if added > 0 else None
        out["share_of_hbm_peak"] = (update_bytes / (added * 1e-3)) / HBM_PEAK if added > 0 else None
        out["hbm_peak_bytes_per_s"] = HBM_PEAK
        mf, tf = modes["fused"]
        ok = all(torch.equal(x, y) for x, y in zip(tables(mf), tables(mu)))
        ok &= all(torch.equal(x, y) for x, y in zip(tf.table_exp_avg + tf.table_exp_avg_sq, um[0::2] + um[1::2]))
        ok &= torch.equal(tf.adam_state, ust[0]) and torch.equal(ust[0], ust[1])
        out["fused_equals_unfused_bitwise"] = bool(ok)
        out["optimizer_steps"] = int(tf.adam_state[0].item())
        mp, tp = modes["peer"]
        out["peer_equals_fused_bitwise"] = bool(all(torch.equal(x, y) for x, y in zip(tables(mp), tables(mf))))
        out["peer_table_exchange_us"] = dict(zip(("until_all_slices", "to_kernel_end", "calls", "own_push"),
                                                 tp.txchg.timing()))
        out["multi_gpu"] = "not measured: one GPU" if torch.cuda.device_count() < 2 else "not measured: run torchrun"
    else:
        import torch.distributed as dist

        mf, tf = modes["fused"]
        same = True
        for t in tables(mf):
            ref = t.detach().clone()
            dist.broadcast(ref, src=0)
            same &= torch.equal(ref, t.detach())
        flag = torch.tensor([int(same)], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        out["replica_tables_bitwise_equal"] = bool(flag.item())
        out["table_exchange_us"] = dict(zip(("until_all_slices", "to_kernel_end", "calls", "own_push"),
                                            tf.txchg.timing()))
    if rank == 0:
        line = json.dumps(out)
        print(line)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    for _, tr in modes.values():
        tr.close()
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
