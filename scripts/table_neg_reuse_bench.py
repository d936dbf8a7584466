"""Measures in-batch negatives by index with trainable token tables (tt_step_args.neg_index + optimize_tables) and prints
one JSON line.

configs[2] shape: B = 4096 triplets, P = 384, 32 / 256-token rows, both 30522 x 384 fp32 tables trained in the step
(FusedTrainer(optimize_tables=True)), bf16x3, persistent chain kernel, graph replays over 4 rotating token sets whose
negatives are a derangement of the positives.  Two trainers from the same seed:

  off: the negatives' own token tensors are gathered and scatter-added like any document (the parent's path);
  on:  in_batch_negatives=True: the negatives' indices are loaded, their token tensors are poisoned (never read), every
       positive is gathered once and each negative's table-gradient row is folded into its positive's.

For token shapes U (full rows) and Z (Zipf ids, log-normal lengths): the first step's loss of both (must be
bit-identical), then --reps alternating rounds of --steps steps each after --warmup steps (CUDA events; no graph capture
inside the timed rounds), then the tables of both compared (the tolerance of tests/test_table_neg_reuse.py's end-to-end
test: no element more than 6 lr apart, at most 1e-3 of the touched elements plus 16 more than 0.02 lr apart, never-touched
rows bit-identical).  A separate eager run under torch.profiler gives the kernel times of the pooled gather, the fold and
the document table's tt_pool_bwd segment (sort + segment sum + Adam) per step.

Run:   python scripts/table_neg_reuse_bench.py [--out profiles/r10_table_neg_reuse_n1.json]
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

from oracle import two_towers_oracle as O  # noqa: E402
from pooled_front_bench import card_info  # noqa: E402

LR = 1e-4
# kernels of one tt_pool_bwd scatter call (csrc/tt_pool_bwd.cu); make_keys_kernel opens each call
SCATTER = ("make_keys_kernel", "radix_hist_kernel", "digit_scan_kernel", "radix_scatter_kernel", "id_offsets_kernel",
           "seg_reduce_kernel", "heavy_chunk_kernel", "heavy_final_kernel")


def token_set(B, Lq, Ld, V, shape, seed):
    """(q_ids, q_mask, p_ids, p_mask) int32 / uint8 padded to Lq / Ld, and a derangement: negative i is positive neg[i]."""
    gen = torch.Generator().manual_seed(seed)
    q_ids, q_mask = O.synth_tokens(B, Lq, shape, gen, "query", V)
    p_ids, p_mask = O.synth_tokens(B, Ld, shape, gen, "doc", V)
    neg = O.derangement(B, gen)
    pad = lambda t, L: torch.nn.functional.pad(t, (0, L - t.shape[1]))  # noqa: E731
    return (pad(q_ids, Lq).to(torch.int32), pad(q_mask, Lq).to(torch.uint8), pad(p_ids, Ld).to(torch.int32),
            pad(p_mask, Ld).to(torch.uint8)), neg


def build(dev, B, P, Lq, Ld, V, sets, reuse, use_graph):
    from two_towers_overlords_b200 import TwoTowersModel
    from two_towers_overlords_b200.training import FusedTrainer

    torch.manual_seed(0)
    m = TwoTowersModel(projection_dim=P, vocab_size=V, train_table=True).to(dev)
    tr = FusedTrainer(m, 0.3, LR, B, Lq, Ld, precision="bf16x3", token_slots=len(sets), use_graph=use_graph,
                      optimize_tables=True, in_batch_negatives=reuse)
    for s, (toks, neg) in enumerate(sets):
        if reuse:
            toks = toks + (torch.full_like(toks[2], V - 1), torch.ones_like(toks[3]))
            tr.load_neg_index(neg, s)
        else:
            toks = toks + (toks[2][neg].clone(), toks[3][neg].clone())
        tr.load_packed(tr.pack_host_tokens(toks, pin=False), s)
    return m, tr


def tables(m):
    return (m.query_tower.pretrained_model.table, m.document_tower.pretrained_model.table)


def compare_tables(m_on, m_off, init, touched):
    out = []
    ok = True
    for k, (a, b, t0) in enumerate(zip(tables(m_on), tables(m_off), init)):
        err = (a - b).detach().abs()
        hot = touched[k].to(a.device)
        n_touched = int(hot.sum()) * a.shape[1]
        n_off = int((err[hot] > 0.02 * LR).sum())
        cold_same = bool(torch.equal(a[~hot], t0[~hot]) and torch.equal(b[~hot], t0[~hot]))
        row_ok = float(err.max()) <= 6 * LR and n_off <= 1e-3 * n_touched + 16 and cold_same
        ok &= row_ok
        out.append({"table": "qd"[k], "max_abs_diff": float(err.max()), "max_abs_diff_over_lr": float(err.max()) / LR,
                    "touched_elements": n_touched, "elements_over_0.02lr": n_off,
                    "never_touched_rows_bit_identical": cold_same})
    return out, bool(ok)


def profile(dev, B, P, Lq, Ld, V, sets, n_steps):
    """Per-step CUDA kernel times (us) of an eager run of each mode under torch.profiler: the pooled gather, g, the
    fold, and the query / document table's tt_pool_bwd scatter (the calls alternate q, d in stream order)."""
    from torch.profiler import ProfilerActivity, profile as tprofile

    res = {}
    for name, reuse in (("off", False), ("on", True)):
        _, tr = build(dev, B, P, Lq, Ld, V, sets, reuse, use_graph=False)
        for i in range(3):
            tr.step(i % len(sets))
        torch.cuda.synchronize()
        with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(n_steps):
                tr.step(i % len(sets))
            torch.cuda.synchronize()
        kernels = sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start)
        acc = {"gather": 0.0, "prep": 0.0, "fold": 0.0, "scatter_q": 0.0, "scatter_d": 0.0}
        calls = -1
        for e in kernels:
            us = e.time_range.elapsed_us()
            if "pool_fwd_kernel" in e.name:
                acc["gather"] += us
            elif "pool_bwd_prep_kernel" in e.name:
                acc["prep"] += us
            elif "pool_bwd_fold_kernel" in e.name:
                acc["fold"] += us
            elif any(k in e.name for k in SCATTER):
                if "make_keys_kernel" in e.name:
                    calls += 1
                acc["scatter_q" if calls % 2 == 0 else "scatter_d"] += us
        assert calls + 1 == 2 * n_steps, ("tt_pool_bwd calls seen", calls + 1)
        res[name] = {k: v / n_steps for k, v in acc.items()}
        tr.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--proj", type=int, default=384)
    ap.add_argument("--profile-steps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_table_neg_reuse_n1.json"))
    args = ap.parse_args()
    os.environ["TT_CHAIN"] = "1"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, P, Lq, Ld, V, H, S = args.batch, args.proj, 32, 256, 30522, 384, 4
    out = {"metric": "table_neg_reuse", "card": card_info(dev), "batch": B, "proj": P, "vocab": V, "hidden": H,
           "Lq": Lq, "Ld": Ld, "precision": "bf16x3", "chain": "persistent", "optimize_tables": True, "lr": LR,
           "token_sets": S, "steps": args.steps, "warmup": args.warmup, "reps": args.reps,
           "table_rows_gathered": {"off": B * (Lq + 2 * Ld), "on": B * (Lq + Ld)},
           "document_scatter_keys": {"off": 2 * B * Ld, "on": B * Ld}, "shapes": {}}
    for shape in ("U", "Z"):
        sets = [token_set(B, Lq, Ld, V, shape, 1000 + 17 * i + (0 if shape == "U" else 500)) for i in range(S)]
        touched = [torch.zeros(V, dtype=torch.bool) for _ in range(2)]
        for toks, _ in sets:
            touched[0][toks[0][toks[1] != 0].long()] = True
            touched[1][toks[2][toks[3] != 0].long()] = True
        modes = {name: build(dev, B, P, Lq, Ld, V, sets, reuse, use_graph=True)
                 for name, reuse in (("off", False), ("on", True))}
        init = [t.detach().clone() for t in tables(modes["off"][0])]
        for _, tr in modes.values():
            tr.prepare(S)
        first = {name: float(tr.step(0).item()) for name, (_, tr) in modes.items()}
        for name, (_, tr) in modes.items():
            for i in range(1, args.warmup):
                tr.step(i % S)
        torch.cuda.synchronize()
        caps = {k: tr.graph_captures for k, (_, tr) in modes.items()}
        times = {k: [] for k in modes}
        for r in range(args.reps):
            for name, (_, tr) in modes.items():
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                ev0.record()
                for i in range(args.steps):
                    tr.step((args.warmup + r * args.steps + i) % S)
                ev1.record()
                torch.cuda.synchronize()
                times[name].append(ev0.elapsed_time(ev1) / args.steps)
        for k, (_, tr) in modes.items():
            assert tr.graph_captures == caps[k], (k, "graph captured inside the timed steps")
            assert int(tr.step_obj.err.item()) == 0, (k, "error flag")
        res = {k: {"ms_per_step": statistics.median(v), "ms_per_step_all": v,
                   "triplets_per_s": B / (statistics.median(v) * 1e-3)} for k, v in times.items()}
        cmp, ok = compare_tables(modes["on"][0], modes["off"][0], init, touched)
        rec = {"modes": res, "speedup_off_over_on": res["off"]["ms_per_step"] / res["on"]["ms_per_step"],
               "first_step_loss": first, "first_step_loss_bit_identical": first["on"] == first["off"],
               "optimizer_steps": int(modes["on"][1].adam_state[0].item()), "tables": cmp,
               "tables_within_tolerance": ok}
        for _, tr in modes.values():
            tr.close()
        del modes
        torch.cuda.empty_cache()
        try:
            rec["kernel_us_per_step_profiled_eager"] = profile(dev, B, P, Lq, Ld, V, sets, args.profile_steps)
        except Exception as e:  # noqa: BLE001  (the timings above stand on their own)
            rec["kernel_us_per_step_profiled_eager"] = f"not measured: {type(e).__name__}: {e}"
        out["shapes"][shape] = rec
        print(json.dumps({shape: rec}), file=sys.stderr)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
