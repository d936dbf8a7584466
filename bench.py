#!/usr/bin/env python
"""
bench.py — the two-tower hot path on B200: train triplets/s (headline) with the pooled-gather roofline, an
end-to-end number through the public API with host buffers, a top-10 corpus-scan figure, and the CPU
baseline (the oracle port of the reference's fp32 step, oracle/two_towers_oracle.py) beside it.

    python bench.py [--gpus N --steps K --warmup W]            # N>1: launched by torch.distributed.run
    python bench.py --impl reference [--steps K --warmup W]    # the reference's CPU path (oracle port)
    python bench.py ... --dump-outputs DIR                     # + the last timed step's results as DIR/<name>.npy

Workload (BASELINE.json configs[1], "heavy GPU run shape"): per-GPU batch 2048 triplets, projection dim 512,
margin 0.3, query length 32 / document length 256 tokens (SURVEY.md §8d shape U: full-length rows, ids
uniform in [999, 30522) — the roofline case), random-init 30522x384 tables, Adam lr 1e-3.  Weak scaling:
every rank processes its own 2048-triplet batch; the one exchange per step is a fused reduce-scatter -> Adam ->
all-gather kernel over NVLink peer memory (TT_DP_EXCHANGE=nccl selects all-reduce + Adam instead).

A "step" = H2D'd tokens -> pooled gather (q,p,n) -> both tower MLPs -> cosine triplet loss -> all gradients
-> [gradient exchange +] Adam.  Steps are software-pipelined: the pooled gather of step i+1 (tokens + frozen tables
only) runs beside the rest of step i; every step still does all of its own work.  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

B_PER_GPU, P_DIM, LQ, LD, MARGIN, LR = 2048, 512, 32, 256, 0.3, 1e-3
VOCAB, HIDDEN = 30522, 384
N_TOKEN_SETS = 48  # rotating input batches: 48 x 3.34 MB (u16 ids + u8 masks) = 160 MB > 126 MB L2
METRIC, UNIT = "train_triplets_per_sec", "triplets/s"


def ncu_traffic(key: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed `ncu --set full` capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
            t = json.load(f)[key]
        return int(t["dram_bytes_read"]) + int(t["dram_bytes_write"])
    except Exception:  # noqa: BLE001
        return None


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1400.0))), "measured"
    except Exception:  # noqa: BLE001
        return 6650.0, 1590.0, "fallback"


# --------------------------------------------------------------------------------------------------
# synthetic inputs (same generator for both arms)
# --------------------------------------------------------------------------------------------------
def token_sets(n_sets: int, B: int, seed: int, ids_dtype, mask_dtype, pin: bool, neg_index: list = None):
    """n_sets x (q_ids,q_mask,p_ids,p_mask,n_ids,n_mask): shape U, negatives = in-batch derangement of the positives
    (neg_index, when given, receives one int32 [B] tensor per set: negative i is positive neg_index[i])."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n_sets):
        q = torch.randint(999, VOCAB, (B, LQ), generator=g, dtype=torch.int64)
        p = torch.randint(999, VOCAB, (B, LD), generator=g, dtype=torch.int64)
        shift = int(torch.randint(1, B, (1,), generator=g)) if B > 1 else 0
        n = torch.roll(p, shift, 0)  # negative_i = positive_{i-shift}: no fixed point
        if neg_index is not None:
            neg_index.append(torch.roll(torch.arange(B, dtype=torch.int32), shift, 0))
        ts = []
        for ids in (q, p, n):
            ts += [ids.to(ids_dtype), torch.ones(ids.shape, dtype=mask_dtype)]
        if pin:
            ts = [t.pin_memory() for t in ts]
        out.append(tuple(ts))
    return out


# --------------------------------------------------------------------------------------------------
# clocks during the timed region (B200_PROFILING.md recipe)
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.thr = [], None, None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50", "-i",
                 str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return None
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        rows = [r for t, r in self.rows if t0 - 0.06 <= t <= t1 + 0.06 and len(r) >= 7] or \
               [r for _, r in self.rows if len(r) >= 7]
        if not rows:
            return None
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows)}


# --------------------------------------------------------------------------------------------------
# CPU arm: the reference's fp32 training step restated in oracle/ (training.py:36-53)
# --------------------------------------------------------------------------------------------------
def cpu_train_throughput(budget_s: float, steps: int | None = None, warmup: int = 1, batch: int | None = None):
    """Times oracle.train_step on the host cores.  Returns (triplets/s, description dict)."""
    from oracle import two_towers_oracle as O

    torch.manual_seed(0)
    try:  # all the host cores this process may use (torchrun exports OMP_NUM_THREADS=1, which would cripple the CPU arm)
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:  # noqa: BLE001
        pass
    threads = torch.get_num_threads()
    model = O.OracleTwoTowers(P_DIM, vocab=VOCAB, hidden=HIDDEN)
    opt = torch.optim.Adam(model.parameters(), lr=LR)
    B = batch or B_PER_GPU
    sets = token_sets(2, B, 1234, torch.int64, torch.int64, pin=False)
    t0 = time.perf_counter()
    O.train_step(model, opt, sets[0], MARGIN)
    t_first = time.perf_counter() - t0
    for _ in range(max(0, warmup - 1)):
        O.train_step(model, opt, sets[1], MARGIN)
    if steps is None:
        steps = max(2, min(16, int(budget_s / max(t_first, 1e-3))))
    t0 = time.perf_counter()
    for i in range(steps):
        O.train_step(model, opt, sets[i % 2], MARGIN)
    dt = time.perf_counter() - t0
    return B * steps / dt, {"cores": threads, "steps": steps, "batch": B, "seconds": round(dt, 2),
                            "ms_per_step": 1e3 * dt / steps}


def cpu_eval_throughput(n_docs_full: int, P: int, budget_s: float = 12.0, n_sample_docs: int = 1_000_000):
    """The reference's eval inner loop (backend/training.py:297-304: per query a CPU cosine_similarity against all
    documents + sklearn-semantics ndcg_score, restated in oracle.retrieval_eval) on a 1 M-document sample with the
    host cores, extrapolated linearly in the document count to the full corpus."""
    from oracle import two_towers_oracle as O

    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:  # noqa: BLE001
        pass
    g = torch.Generator().manual_seed(7)
    n = min(n_sample_docs, n_docs_full)
    De = torch.randn(n, P, generator=g)
    Qe = torch.randn(16, P, generator=g)
    rel = [set(range(i, i + 5)) for i in range(16)]
    t0 = time.perf_counter()
    O.retrieval_eval(Qe[:1], De, rel[:1], k=10)
    t_first = time.perf_counter() - t0
    nq = int(max(2, min(15, budget_s / max(t_first, 1e-3))))
    t0 = time.perf_counter()
    O.retrieval_eval(Qe[1: 1 + nq], De, rel[1: 1 + nq], k=10)
    dt = time.perf_counter() - t0
    qps_sample = nq / dt
    return {"value": qps_sample * n / n_docs_full, "unit": "queries/s", "cores": torch.get_num_threads(), "kind": "port",
            "measured_queries_per_s_on_sample": qps_sample, "seconds_per_query_on_sample": dt / nq,
            "sample": f"{nq} queries x {n} documents x {P}-d in {dt:.1f} s (oracle.retrieval_eval = the reference's "
                      f"per-query cosine_similarity + ndcg_score loop, torch/numpy CPU, {torch.get_num_threads()} "
                      f"threads), extrapolated linearly in the document count to {n_docs_full}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # size the per-step sample so that K steps end within ~2 minutes
    probe, info = cpu_train_throughput(0, steps=1, warmup=1, batch=256)
    B = B_PER_GPU
    while B > 64 and (args.steps + args.warmup) * B / probe > 120.0:
        B //= 2
    value, info = cpu_train_throughput(0, steps=args.steps, warmup=max(1, args.warmup), batch=B)
    sample = (f"{args.steps} fp32 steps of {B} triplets (of the {B_PER_GPU}-triplet batch), oracle port of "
              f"backend/training.py:36-53 with the embedding-only backbone, torch CPU, {info['cores']} threads")
    emit(({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": info["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus), "variant": {"arithmetic": "fp32 torch CPU", "cpu_sample_batch": B},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": info["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def workload_config(world):
    """The workload both arms run (identical dict in both JSON lines); how each arm computes it is in `variant`."""
    return {
        "workload": "configs[1] heavy GPU run shape: triplet training step, batch 2048/GPU, proj-dim 512, "
                    "query 32 / doc 256 tokens (shape U), margin 0.3, Adam lr 1e-3, random-init 30522x384 fp32 tables",
        "global_batch": B_PER_GPU * world, "batch_per_gpu": B_PER_GPU, "projection_dim": P_DIM, "Lq": LQ, "Ld": LD,
        "parallelism": f"dp{world}",
        "l2": f"inputs rotate over {N_TOKEN_SETS} token batches (>= {N_TOKEN_SETS * 3.34:.0f} MB > 126 MB L2); the two "
              "token tables are weights and stay cache-warm across steps as in real training",
    }


# FusedTrainer's parameter order (TwoTowersModel.projection_parameters): Wq1, bq1, Wq2, bq2, Wd1, bd1, Wd2, bd2
PROJECTION_NAMES = [f"{t}.projection.{i}.{k}" for t in ("query_tower", "document_tower") for i in (0, 2)
                    for k in ("weight", "bias")]


def dump_outputs(out_dir: str, trainer):
    """What the last timed step hands its caller, one float32 DIR/<name>.npy each: the loss, the gradients of the 8
    projection tensors (grad.<name>, this rank's) and the parameters after the Adam update (<name>); 7.4 MB at
    configs[1].  The inputs depend on the arguments only (seeded model and token batches), so two builds run with the
    same arguments can be compared file by file."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": trainer.loss_view}
    for name, p, g in zip(PROJECTION_NAMES, trainer.p_views, trainer.g_views):
        arrays[name] = p
        arrays["grad." + name] = g
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().to(torch.float32).cpu().numpy())


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA (sm_100a) device: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # NCCL's version banner goes to stdout: keep stdout to the ONE JSON line
        dist.init_process_group("nccl", device_id=dev)

    from two_towers_overlords_b200 import TwoTowersModel, _native
    from two_towers_overlords_b200.training import FusedTrainer

    lib = _native.load()
    table_dtype = torch.bfloat16 if args.table_dtype == "bf16" else torch.float32
    torch.manual_seed(0)
    model = TwoTowersModel(projection_dim=P_DIM, table_dtype=table_dtype, precision=args.precision).to(dev)
    # token ids travel as uint16 (vocab 30522 < 65536) and masks as uint8: 3 bytes per token over PCIe instead of the
    # 16 bytes of the reference tokenizer's int64 ids + int64 mask (--ids-dtype i32 for 4-byte ids)
    ids_dtype, mask_dtype = (torch.uint16 if args.ids_dtype == "u16" else torch.int32), torch.uint8
    trainer = FusedTrainer(model, MARGIN, LR, B_PER_GPU, LQ, LD, precision=args.precision, world_size=world, rank=rank,
                           use_graph=not args.no_graph, ids_dtype=ids_dtype, mask_dtype=mask_dtype,
                           token_slots=N_TOKEN_SETS)
    host_sets = token_sets(N_TOKEN_SETS, B_PER_GPU, 1234 + rank, ids_dtype, mask_dtype, pin=True)
    h2d_bytes = sum(t.numel() * t.element_size() for t in host_sets[0])
    host_packed = [trainer.pack_host_tokens(hs) for hs in host_sets]  # one pinned buffer per batch: one H2D copy
    h2d_bytes = host_packed[0].numel()
    for slot, hp in enumerate(host_packed):  # inputs resident in HBM for the `value` leg
        trainer.load_packed(hp, slot)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    K, W = args.steps, args.warmup
    NS = N_TOKEN_SETS
    trainer.prepare()  # capture the round-robin step graphs up front
    for i in range(W):
        trainer.step(i % NS, (i + 1) % NS)
    barrier()
    launches_per_step = int(trainer.kernel_launches_per_step or 0)

    # ---- leg 1: device-resident inputs -----------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 and not os.environ.get("TT_BENCH_NO_SAMPLER") else None  # (diagnostic switch)
    time.sleep(0.15 if sampler else 0.0)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if trainer.xchg is not None:
        trainer.xchg.reset_timing()
    t_wall0 = time.time()
    cap0 = trainer.graph_captures
    ev0.record()
    for i in range(K):
        trainer.step((W + i) % NS, (W + i + 1) % NS)  # the next step's pooled gather runs beside this step
    ev1.record()
    barrier()
    t_wall1 = time.time()
    captures_in_timed = {"value_leg": trainer.graph_captures - cap0}
    exchange_us = None
    if trainer.xchg is not None:
        t_wait, t_rest, n_calls, t_push = trainer.xchg.timing()
        exchange_us = {"own_push": round(t_push, 2), "wait_for_all_ranks_gradients": round(t_wait, 2),
                       "reduce_adam_allgather": round(t_rest, 2), "calls": n_calls,
                       "note": "inside tt_dp_reduce_adam (CTA 0 of rank 0) over the timed steps: time until every "
                               "rank's gradient slice has landed (own push + rank skew), then sum + Adam + parameter "
                               "broadcast; wait_per_rank: the rank that waits least arrives last"}
        if world > 1:
            waits = [None] * world
            dist.all_gather_object(waits, round(t_wait, 1))
            exchange_us["wait_per_rank"] = waits
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    loss_after = float(trainer.loss_view[0].item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer)
    value = B_PER_GPU * world * K / (ms_total * 1e-3)

    # ---- leg 2: end to end through the public API, host buffers --------------------------------------
    # every step: pinned host tokens -> H2D (copy stream, two steps ahead at most) -> FusedTrainer.step -> loss D2H
    copy_stream = torch.cuda.Stream()
    main = torch.cuda.current_stream()
    loss_host = torch.zeros(K + W + 1, dtype=torch.float32).pin_memory()
    done = [torch.cuda.Event() for _ in range(4)]
    ready = [torch.cuda.Event() for _ in range(4)]

    def stage(j):  # tokens of step j: pinned host -> its slot, on the copy stream, at most 3 steps ahead
        if j >= 3:
            copy_stream.wait_event(done[(j - 3) % 4])
        with torch.cuda.stream(copy_stream):
            trainer.load_packed(host_packed[j % NS], j % NS)
            ready[j % 4].record(copy_stream)

    def e2e_step(i):
        stage(i + 1)                       # step i launches the pooled gather of step i + 1, so stage one ahead
        main.wait_event(ready[(i + 1) % 4])
        trainer.step(i % NS, (i + 1) % NS)
        trainer.read_loss_async(loss_host[i: i + 1])
        done[i % 4].record(main)

    stage(0)
    main.wait_event(ready[0])
    for i in range(W):
        e2e_step(i)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cap0 = trainer.graph_captures
    ev0.record()
    for i in range(W, W + K):
        e2e_step(i)
    ev1.record()
    barrier()
    captures_in_timed["e2e_leg"] = trainer.graph_captures - cap0
    if not args.no_graph and any(captures_in_timed.values()):
        raise SystemExit(f"a CUDA graph was captured inside a timed region: {captures_in_timed}")
    e2e_ms = max_over_ranks(ev0.elapsed_time(ev1))
    e2e_value = B_PER_GPU * world * K / (e2e_ms * 1e-3)

    # ---- the same step with nothing overlapped (gather, then the chain): the denominator that is comparable with
    # ncu's serialised launch list when quoting the gather's share of a step -------------------------------------
    for i in range(8):
        trainer.step(i % 8, None)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    n_seq = max(16, min(K, 64))
    for i in range(n_seq):
        trainer.step(i % 8, None)
    ev1.record()
    torch.cuda.synchronize()
    seq_ms = ev0.elapsed_time(ev1) / n_seq

    # ---- roofline of the dominant kernel: the pooled gather, timed alone on the launching stream -----
    esz = 2 if table_dtype == torch.bfloat16 else 4
    tok_per_triplet = LQ + 2 * LD
    ids_bytes = 2 if ids_dtype == torch.uint16 else 4
    alg_bytes_per_triplet = tok_per_triplet * HIDDEN * esz + tok_per_triplet * (ids_bytes + 1) + 3 * (HIDDEN * 4 + 8)
    segs = (_native.PoolSeg * 3)()
    xhat = torch.empty(3 * B_PER_GPU, HIDDEN, dtype=torch.float32, device=dev)
    cnt = torch.empty(3 * B_PER_GPU, dtype=torch.float32, device=dev)
    nrm = torch.empty(3 * B_PER_GPU, dtype=torch.float32, device=dev)
    tq = model.query_tower.pretrained_model.table.data
    td = model.document_tower.pretrained_model.table.data

    def pool_only(slot):
        t = trainer.tok_slots[slot]
        for s, (tab, ids, mask, L) in enumerate(((tq, t[0], t[1], LQ), (td, t[2], t[3], LD), (td, t[4], t[5], LD))):
            segs[s].table, segs[s].ids, segs[s].mask = tab.data_ptr(), ids.data_ptr(), mask.data_ptr()
            segs[s].B, segs[s].L, segs[s].row0 = B_PER_GPU, L, s * B_PER_GPU
        _native.check(lib.tt_pool_fwd_multi(segs, 3, _native.dtype_code(tq), VOCAB, HIDDEN, _native.dtype_code(t[0]),
                                            _native.dtype_code(t[1]), xhat.data_ptr(), cnt.data_ptr(), nrm.data_ptr(),
                                            None, _native.stream()), "tt_pool_fwd_multi")

    for i in range(max(3, W)):
        pool_only(i % N_TOKEN_SETS)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(K):
        pool_only(i % N_TOKEN_SETS)
    ev1.record()
    torch.cuda.synchronize()
    pool_ms = ev0.elapsed_time(ev1) / K
    hbm_peak, tensor_peak, peak_kind = peaks()
    achieved = alg_bytes_per_triplet * B_PER_GPU / (pool_ms * 1e-3) / 1e9
    # measured L2 -> SM read ceiling (tt_ubench_l2_read): the gather's tables are cache-resident, so THIS is the
    # bandwidth that bounds it; probed at one table (47 MB) and at both (94 MB), the larger figure is the peak
    l2 = {}
    sink = torch.zeros(4, dtype=torch.int32, device=dev)
    for label, nbytes in (("one_table_47MB", VOCAB * HIDDEN * 4), ("two_tables_94MB", 2 * VOCAB * HIDDEN * 4)):
        probe = torch.empty(nbytes // 4, dtype=torch.float32, device=dev).normal_()
        its = 40
        for _ in range(2):
            _native.check(lib.tt_ubench_l2_read(probe.data_ptr(), nbytes, its, 8, sink.data_ptr(), _native.stream()), "l2")
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        _native.check(lib.tt_ubench_l2_read(probe.data_ptr(), nbytes, its, 8, sink.data_ptr(), _native.stream()), "l2")
        ev1.record()
        torch.cuda.synchronize()
        l2[label] = nbytes * its / (ev0.elapsed_time(ev1) * 1e-3) / 1e9
        del probe
    l2_peak = max(l2.values())
    roofline = {
        "kernel": "pool_fwd_kernel (token-row gather + masked mean + L2 normalise, q|p|n in one launch)",
        "bound": "l2", "achieved": achieved, "peak": l2_peak, "peak_kind": "measured in this run (tt_ubench_l2_read)",
        "unit": "GB/s", "frac": achieved / l2_peak, "l2_probe_gbs": l2,
        "traffic": ncu_traffic("pool_fwd_kernel") if table_dtype == torch.float32 else None,
        "hbm_formula": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "peak_kind": peak_kind, "unit": "GB/s",
                        "frac": achieved / hbm_peak,
                        "note": "the contract's formula (algorithmic bytes / time / HBM copy peak): both 46.9 MB fp32 "
                                "tables fit the 126 MB L2, DRAM traffic is ~7 % of the algorithmic bytes, so this "
                                "fraction exceeds 1 and is not a roofline; the L2 figure above is"},
        "algorithmic_bytes_per_launch": alg_bytes_per_triplet * B_PER_GPU, "us_per_launch": pool_ms * 1e3,
        "share_of_step": pool_ms / (ms_total / K),
        "share_of_serialised_step": pool_ms / seq_ms, "serialised_step_ms": seq_ms,
        "share_note": "timed alone (tables cache-warm); with the per-kernel chain (TT_CHAIN=0) or under data "
                      "parallelism this kernel (for step i+1) runs BESIDE other work of step i; share_of_serialised_step divides by the "
                      "step time with nothing overlapped and is the figure to compare with the ncu launch list",
    }

    # ---- data-parallel parity on real peers (N > 1): replicas bit-identical, and equal (to rounding) to ONE rank
    # running the same global batch ---------------------------------------------------------------------------------
    dp_check = None
    if world > 1:
        dp_check = run_dp_check(dev, world, rank, args, ids_dtype, mask_dtype)

    # ---- CPU baseline beside it (rank 0, N = 1 only) ----------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, info = cpu_train_throughput(args.cpu_budget)
        cpu = {"value": v, "unit": UNIT, "cores": info["cores"], "kind": "port",
               "sample": f"{info['steps']} fp32 steps of {info['batch']} triplets in {info['seconds']} s "
                         f"(oracle/two_towers_oracle.train_step, torch CPU, {info['cores']} threads)"}

    exchange_kind = trainer.exchange
    barrier()
    trainer.close()
    del trainer, model
    torch.cuda.empty_cache()
    chain_variant = run_chain_variant(dev, args, ids_dtype, mask_dtype, host_packed) if (world == 1 and not args.no_chain_variant) else None
    backbone_leg = run_backbone_leg(dev, args) if (world == 1 and not args.no_backbone) else None
    reuse_leg = run_negative_reuse_leg(dev, args, ids_dtype, mask_dtype) if (world == 1 and not args.no_chain_variant) else None
    config2 = run_config2(dev, world, rank, args, l2_peak=l2_peak) if not args.no_config2 else None
    epoch_leg = run_epoch_leg(dev, world, rank, args) if not args.no_epoch else None
    torch.cuda.empty_cache()
    scan = None
    if not args.no_scan:
        scan = run_scan(dev, world, rank, args.scan_docs, args.scan_queries, HIDDEN, args.scan_passes)
        if scan is not None and rank == 0 and world == 1 and not args.no_cpu:
            scan["cpu_baseline"] = cpu_eval_throughput(args.scan_docs, HIDDEN, args.cpu_budget)

    if rank == 0:
        emit(({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else f"f32 ({args.precision} tensor-core projection)",
            "data": "synthetic", "config": workload_config(world),
            "variant": {"projection_precision": args.precision, "table_dtype": args.table_dtype,
                        "dp_exchange": exchange_kind, "token_dtypes": f"ids {args.ids_dtype}, mask u8"},
            "graph_captures_in_timed_region": captures_in_timed, "dp_check": dp_check, "config2": config2,
            "epoch_leg": epoch_leg, "projection_chain": chain_variant, "full_backbone": backbone_leg,
            "in_batch_negative_reuse": reuse_leg,
            "dp_exchange_us": exchange_us,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms / K},
            "gpu_launches": launches_per_step * K, "gpu_launches_per_step": launches_per_step,
            "cuda_graph": not args.no_graph, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "loss_after": loss_after, "scan": scan,
        }))
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------
# the reference's actual backbone (frozen MiniLM-L6) in front of the same pool / projection / loss
# --------------------------------------------------------------------------------------------------
def run_backbone_leg(dev, args, B=256, steps=6):
    """SURVEY.md section 8f rank 2: the reference-shaped training step (3 tower calls -> TripletLoss -> backward ->
    torch.optim.Adam, backend/training.py:37-51) with `backbone="minilm"`: the frozen 6-layer encoder runs forward-only
    on the device (tt_encoder_fwd), then the same masked-mean pool, projection and loss kernels.  Random-init weights
    of the MiniLM-L6 shape, full-length tokens (32 / 256).  CPU beside it: transformers' BertModel forward for the same
    token counts on a small sample (this is >99 % of the true reference's step, SURVEY.md section 0 D1)."""
    from two_towers_overlords_b200 import TripletLoss, TwoTowersModel

    torch.manual_seed(0)
    model = TwoTowersModel(projection_dim=P_DIM, backbone="minilm", precision=args.precision).to(dev)
    crit = TripletLoss(MARGIN)
    opt = torch.optim.Adam([p for p in model.parameters() if p.requires_grad], lr=LR)
    g = torch.Generator().manual_seed(11)

    def toks(L):
        return (torch.randint(999, VOCAB, (B, L), generator=g).to(dev), torch.ones(B, L, dtype=torch.int64, device=dev))

    q, p, n = toks(LQ), toks(LD), toks(LD)

    def step():
        opt.zero_grad()
        loss = crit(model.encode_queries(q), model.encode_documents(p), model.encode_documents(n))
        loss.backward()
        opt.step()
        return loss

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        loss = step()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / steps
    tokens = B * (LQ + 2 * LD)
    # dense flops of the encoder per token: 6 layers x 2 x 384 x (3*384 + 384 + 1536 + 1536) + attention 4 x L x 384
    enc_flops = sum(B * L * (6 * (2 * 384 * (4 * 384 + 2 * 1536) + 4 * L * 384)) for L in (LQ, LD, LD))
    out = {"workload": f"training step with the frozen MiniLM-L6 backbone: {B} triplets, query {LQ} / doc {LD} tokens, "
                       f"proj-dim {P_DIM}, Adam", "ms_per_step": ms, "triplets_per_s": B / (ms * 1e-3),
           "tokens_per_s": tokens / (ms * 1e-3), "encoder_tflops": enc_flops / (ms * 1e-3) / 1e12,
           "loss": float(loss.item())}
    if not args.no_cpu:
        try:
            from transformers import BertConfig, BertModel

            hf = BertModel(BertConfig(vocab_size=VOCAB, hidden_size=384, num_hidden_layers=6, num_attention_heads=12,
                                      intermediate_size=1536)).eval()
            bs = 8
            ids = torch.randint(999, VOCAB, (bs, LD), generator=g)
            with torch.no_grad():
                hf(input_ids=ids)
                t0 = time.time()
                hf(input_ids=ids)
                dt = time.time() - t0
            cpu_tok_s = bs * LD / dt
            out["cpu_baseline"] = {"tokens_per_s": cpu_tok_s, "triplets_per_s": cpu_tok_s / (LQ + 2 * LD),
                                   "cores": torch.get_num_threads(), "kind": "port",
                                   "sample": f"transformers BertModel forward, {bs} x {LD} tokens in {dt:.2f} s; a triplet is "
                                             f"{LQ + 2 * LD} tokens (forward only: the backbone is frozen)"}
        except Exception as ex:  # the leg is informative: a missing transformers install must not fail the bench
            out["cpu_baseline"] = {"unavailable": repr(ex)}
    del model, opt
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------------------------------
# in-batch negatives named by index: every positive document is pooled once
# --------------------------------------------------------------------------------------------------
def run_negative_reuse_leg(dev, args, ids_dtype, mask_dtype, steps=40, n_sets=16):
    """configs[1] again, the SAME batches as the headline leg's generator makes (negative i = positive neg_index[i], as
    the reference's batcher draws them, backend/data.py:113-137), but the trainer is told the indices
    (tt_step_args.neg_index): the pooled gather then visits each positive once and copies its row to the negatives
    that name it.  Bit-identical results (tests/test_cuda_parity.py::test_in_batch_negative_reuse_gives_the_same_bits);
    a third of the table rows are not read a second time.  NOT the headline: that leg gathers all three token
    tensors like the reference's three tower calls."""
    from two_towers_overlords_b200 import TwoTowersModel
    from two_towers_overlords_b200.training import FusedTrainer

    torch.manual_seed(0)
    model = TwoTowersModel(projection_dim=P_DIM, precision=args.precision).to(dev)
    tr = FusedTrainer(model, MARGIN, LR, B_PER_GPU, LQ, LD, precision=args.precision, ids_dtype=ids_dtype,
                      mask_dtype=mask_dtype, token_slots=n_sets, in_batch_negatives=True)
    negs = []
    sets = token_sets(n_sets, B_PER_GPU, 777, ids_dtype, mask_dtype, pin=False, neg_index=negs)
    for slot, (ts, ng) in enumerate(zip(sets, negs)):
        tr.load_packed(tr.pack_host_tokens(ts, pin=False), slot)
        tr.load_neg_index(ng, slot)
    tr.prepare()
    for i in range(n_sets):
        tr.step(i % n_sets, (i + 1) % n_sets)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(steps):
        tr.step(i % n_sets, (i + 1) % n_sets)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / steps
    for _ in range(3):
        tr._fwd_bwd(0, 1, 0)
    torch.cuda.synchronize()
    ev0.record()
    for i in range(steps):
        tr._fwd_bwd(i % n_sets, 1, 0)
    ev1.record()
    torch.cuda.synchronize()
    pool_us = ev0.elapsed_time(ev1) / steps * 1e3
    err = int(tr.step_obj.err.item())
    out = {"workload": "configs[1] with the in-batch negatives named by index (tt_step_args.neg_index): every positive "
                       "document is pooled once, its row copied to the negatives that name it",
           "ms_per_step": ms, "triplets_per_s": B_PER_GPU / (ms * 1e-3), "gather_us": pool_us,
           "launches_per_step": int(tr.kernel_launches_per_step or 0), "err_flag": err,
           "loss": float(tr.loss_view[0].item()),
           "note": f"{n_sets} rotating token batches ({n_sets * 3.34:.0f} MB); results bit-identical to gathering the negatives' "
                   "tokens; run_training uses this with the device feeder on one GPU (TT_NEG_REUSE=0 turns it off)"}
    tr.close()
    del tr, model
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------------------------------
# the projection chain, both ways of launching it (tt_step_args.chain)
# --------------------------------------------------------------------------------------------------
def run_chain_variant(dev, args, ids_dtype, mask_dtype, host_packed, steps=40):
    """configs[1] on one GPU: everything after the pooled gather (both layers of both towers, loss, backward, bias
    sums, gradient reduction, Adam) as ONE persistent tcgen05 kernel vs one kernel per contraction — each timed alone
    (gather already done, CUDA events around back-to-back launches) and as a whole training step.  Tensor roofline of
    the chain: useful flops (SURVEY section 8d: 7.08 MFLOP per triplet) / time against the sustained bf16 peak; the
    split-bf16 arithmetic issues 3 (6 in layer 1) bf16 products per useful one."""
    from two_towers_overlords_b200 import TwoTowersModel
    from two_towers_overlords_b200.training import FusedTrainer

    _, tensor_peak, peak_kind = peaks()
    flops = B_PER_GPU * 3 * ((768 * P_DIM + 2 * P_DIM * P_DIM) + (4 * P_DIM * P_DIM + 768 * P_DIM))
    issued = B_PER_GPU * 3 * ((6 * 768 * P_DIM + 3 * 2 * P_DIM * P_DIM) + 3 * (4 * P_DIM * P_DIM + 768 * P_DIM))
    out = {"workload": "configs[1] projection chain per step: 3 x 2048 rows, 384 -> 512 -> 512, cosine triplet loss, "
                       "backward, Adam", "useful_gflop": flops / 1e9, "issued_bf16_gflop": issued / 1e9}
    prev = os.environ.get("TT_CHAIN")
    try:
        for name, flag in (("persistent_kernel", "1"), ("kernel_per_contraction", "0")):
            os.environ["TT_CHAIN"] = flag
            torch.manual_seed(0)
            model = TwoTowersModel(projection_dim=P_DIM, precision=args.precision).to(dev)
            tr = FusedTrainer(model, MARGIN, LR, B_PER_GPU, LQ, LD, precision=args.precision, ids_dtype=ids_dtype,
                              mask_dtype=mask_dtype, token_slots=8)
            for slot in range(8):
                tr.load_packed(host_packed[slot], slot)
            tr.prepare()
            for i in range(8):
                tr.step(i % 8, (i + 1) % 8)
            torch.cuda.synchronize()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for i in range(steps):
                tr.step(i % 8, (i + 1) % 8)
            ev1.record()
            torch.cuda.synchronize()
            step_ms = ev0.elapsed_time(ev1) / steps
            launches = int(tr.kernel_launches_per_step or 0)
            # the chain alone: the gather of slot 0 sits in workspace 0, launch its back half repeatedly (gradients
            # only — eager launches; the per-kernel chain forks its independent branches onto library streams)
            tr._fwd_bwd(0, 1, 0)
            for _ in range(3):
                tr._fwd_bwd(0, 2, 0)
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(steps):
                tr._fwd_bwd(0, 2, 0)
            ev1.record()
            torch.cuda.synchronize()
            alone_us = ev0.elapsed_time(ev1) / steps * 1e3
            out[name] = {"step_ms": step_ms, "triplets_per_s": B_PER_GPU / (step_ms * 1e-3),
                         "launches_per_step": launches, "chain_alone_us": alone_us,
                         "roofline": {"bound": "tensor", "achieved": flops / (alone_us * 1e-6) / 1e12, "peak": tensor_peak,
                                      "peak_kind": peak_kind, "unit": "TFLOP/s",
                                      "frac": flops / (alone_us * 1e-6) / 1e12 / tensor_peak,
                                      "issued_frac": issued / (alone_us * 1e-6) / 1e12 / tensor_peak, "traffic": None}}
            tr.close()
            del tr, model
            torch.cuda.empty_cache()
    finally:
        if prev is None:
            os.environ.pop("TT_CHAIN", None)
        else:
            os.environ["TT_CHAIN"] = prev
    out["note"] = ("the persistent kernel holds every SM (one 320-thread CTA with ~190 KB of shared memory each), so a "
                   "step is gather -> chain (2 launches); the per-kernel chain lets the NEXT step's gather run beside "
                   "its 17 small kernels.  FusedTrainer's default is the persistent kernel (TT_CHAIN=0 selects the other)")
    return out


# --------------------------------------------------------------------------------------------------
# data-parallel parity on real peers
# --------------------------------------------------------------------------------------------------
def run_dp_check(dev, world, rank, args, ids_dtype, mask_dtype, n_steps=2):
    """(a) after `n_steps` exchanged steps every rank holds bit-identical parameters; (b) they equal, to rounding, the
    parameters ONE rank reaches on the same global batches (rank-ordered concatenation of the per-rank batches,
    inv_batch = 1 / global batch).  Fresh models from the same seed; eager steps (no graphs)."""
    import torch.distributed as dist

    from two_towers_overlords_b200 import TwoTowersModel
    from two_towers_overlords_b200.training import FusedTrainer

    def fresh(batch, w, r):
        torch.manual_seed(0)
        m = TwoTowersModel(projection_dim=P_DIM, precision=args.precision).to(dev)
        return m, FusedTrainer(m, MARGIN, LR, batch, LQ, LD, precision=args.precision, world_size=w, rank=r,
                               use_graph=False, ids_dtype=ids_dtype, mask_dtype=mask_dtype)

    m_dp, t_dp = fresh(B_PER_GPU, world, rank)
    p0 = t_dp.flat_p.clone()
    sets = token_sets(n_steps, B_PER_GPU, 4321 + rank, ids_dtype, mask_dtype, pin=False)
    losses = []
    for ts in sets:
        for dst, src in zip(t_dp.tok, ts):
            dst.copy_(src)
        t_dp.step()
        losses.append(float(t_dp.loss_view[0].item()))
    torch.cuda.synchronize()
    t_dp.check()
    mine = t_dp.flat_p.clone()
    bits = mine.view(torch.int32).to(torch.int64)
    digest = torch.stack([bits.sum(), (bits * torch.arange(1, bits.numel() + 1, device=dev)).sum()])
    digests = [torch.zeros_like(digest) for _ in range(world)]
    dist.all_gather(digests, digest)
    identical = all(torch.equal(d, digests[0]) for d in digests)
    dist.barrier()
    t_dp.close()
    out = {"steps": n_steps, "replicas_bit_identical": bool(identical), "loss_dp": losses}
    if rank == 0:  # the same global batches on one rank
        m_1, t_1 = fresh(B_PER_GPU * world, 1, 0)
        all_sets = [token_sets(n_steps, B_PER_GPU, 4321 + r, ids_dtype, mask_dtype, pin=False) for r in range(world)]
        l1 = []
        for s_ in range(n_steps):
            for j, dst in enumerate(t_1.tok):
                dst.copy_(torch.cat([all_sets[r][s_][j] for r in range(world)]))
            t_1.step()
            l1.append(float(t_1.loss_view[0].item()))
        torch.cuda.synchronize()
        upd_dp, upd_1 = (mine - p0).double(), (t_1.flat_p - p0).double()
        out["loss_one_rank"] = l1
        out["loss_rel_err_vs_one_rank"] = max(abs(a - b) / abs(b) for a, b in zip(losses, l1))
        out["update_rel_err_vs_one_rank"] = float((upd_dp - upd_1).norm() / upd_1.norm())
        out["note"] = ("update = parameters after the steps minus the initial ones (norm-wise; Adam's g/(|g|+eps) amplifies "
                       "rounding of near-zero gradient elements, and the summation order differs: per-rank sums added in "
                       "rank order vs one sum over the global batch)")
        del t_1, m_1
    dist.barrier()
    ok = torch.tensor([1 if identical else 0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if int(ok.item()) != 1:
        raise SystemExit("dp_check: data-parallel replicas diverged")
    if rank == 0 and (out["loss_rel_err_vs_one_rank"] > 1e-5 or out["update_rel_err_vs_one_rank"] > 5e-3):
        raise SystemExit(f"dp_check: data-parallel result differs from the one-rank run: {out}")
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------------------------------
# configs[2]: saved-model shape, trainable token tables (sorted-segment scatter-add backward)
# --------------------------------------------------------------------------------------------------
def run_config2(dev, world, rank, args, B=4096, P=384, steps=12, l2_peak=None):
    """Per-GPU batch 4096, P = 384, 32/256-token rows, BOTH 30522x384 tables trainable: the whole step (gather -> MLPs
    -> loss -> projection gradients -> dx -> both scatter-adds) and the document-table scatter-add (tt_pool_bwd) alone
    with its HBM roofline (SURVEY.md §8d formula).  Every rank runs its own replica (no exchange: the table gradient
    all-reduce is not part of this leg)."""
    from two_towers_overlords_b200 import TwoTowersModel, _native
    from two_towers_overlords_b200.training import FusedTrainer

    lib = _native.load()
    hbm_peak, _, peak_kind = peaks()
    torch.manual_seed(1)
    m = TwoTowersModel(projection_dim=P, precision=args.precision, train_table=True).to(dev)
    tr = FusedTrainer(m, MARGIN, LR, B, LQ, LD, precision=args.precision, use_graph=False, ids_dtype=torch.int32,
                      mask_dtype=torch.uint8, token_slots=4)
    sets = token_sets(4, B, 99 + rank, torch.int32, torch.uint8, pin=False)
    for slot, ts in enumerate(sets):
        for dst, src in zip(tr.tok_slots[slot], ts):
            dst.copy_(src)
    for i in range(3):
        tr.step(i % 4)
    torch.cuda.synchronize()
    n0 = lib.tt_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(steps):
        tr.step(i % 4)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / steps
    launches = (lib.tt_launch_count() - n0) // steps
    # the document-table scatter-add alone: rows p | n (2B sequences of 256 tokens), gradient rows g [2B,384]
    ids = torch.cat([tr.tok_slots[0][2], tr.tok_slots[0][4]]).contiguous()
    mask = torch.cat([tr.tok_slots[0][3], tr.tok_slots[0][5]]).contiguous()
    R = ids.shape[0]
    dx = torch.randn(R, HIDDEN, device=dev)
    xh = torch.nn.functional.normalize(torch.randn(R, HIDDEN, device=dev), dim=1)
    cnt = torch.full((R,), float(LD), device=dev)
    nrm = torch.ones(R, device=dev)
    dtab = torch.empty(VOCAB, HIDDEN, device=dev)
    ws_bytes = lib.tt_pool_bwd_ws_bytes(R, LD, VOCAB, HIDDEN)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)

    def bwd():
        _native.check(lib.tt_pool_bwd(dx.data_ptr(), xh.data_ptr(), cnt.data_ptr(), nrm.data_ptr(), ids.data_ptr(),
                                      _native.dtype_code(ids), mask.data_ptr(), _native.dtype_code(mask), R, LD, VOCAB,
                                      HIDDEN, dtab.data_ptr(), 0, ws.data_ptr(), ws_bytes, _native.stream()),
                      "tt_pool_bwd")

    for _ in range(3):
        bwd()
    torch.cuda.synchronize()
    n1 = lib.tt_launch_count()
    ev0.record()
    for _ in range(steps):
        bwd()
    ev1.record()
    torch.cuda.synchronize()
    bwd_ms = ev0.elapsed_time(ev1) / steps
    bwd_launches = (lib.tt_launch_count() - n1) // steps
    n_unique = int(torch.unique(ids[mask.bool()].to(torch.int64)).numel())
    alg = R * LD * (4 + 1) + R * LD * 8 + R * HIDDEN * 4 + n_unique * HIDDEN * 4 + (VOCAB - n_unique) * HIDDEN * 4
    # what the reduction really moves: every unmasked token adds the gradient row of ITS sequence into its table row, so
    # the sorted-segment sum reads one 1536-byte row per TOKEN (g is 12.6 MB and cache-resident: the bytes come from L2)
    n_tok = int(mask.bool().sum().item())
    l2_bytes = n_tok * HIDDEN * 4 + alg
    out = {
        "workload": "configs[2] saved-model shape e15.lr4.d384.m3: batch 4096/GPU, proj-dim 384, query 32 / doc 256 "
                    "tokens, both 30522x384 tables trainable (deterministic sorted-segment scatter-add backward)",
        "metric": METRIC, "value": B * world / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
        "gpu_launches_per_step": int(launches), "n_gpus": world, "scaling": "replicas (no exchange in this leg)",
        "roofline_pool_bwd": {
            "kernel": "tt_pool_bwd (document table: 2B x 256 tokens -> stable radix sort by id -> one warp per touched row, rows named by > 256 tokens cut into 2048-entry chunks summed in a fixed order)",
            "bound": "l2", "achieved": l2_bytes / (bwd_ms * 1e-3) / 1e9, "peak": l2_peak,
            "peak_kind": "measured in this run (tt_ubench_l2_read)", "unit": "GB/s",
            "frac": (l2_bytes / (bwd_ms * 1e-3) / 1e9 / l2_peak) if l2_peak else None,
            "ms_per_call": bwd_ms, "launches_per_call": int(bwd_launches), "l2_bytes_per_call": l2_bytes,
            "unmasked_tokens": n_tok, "unique_rows": n_unique,
            "traffic": ncu_traffic("seg_reduce_kernel_doc_table_cfg2"),
            "note": "whole call (sort + reduction, all launches) against the L2->SM ceiling; its dominant kernel, "
                    "seg_reduce_kernel, alone moves 3.17 GB from L2 in 183 us = 17.3 TB/s under ncu "
                    "(profiles/r02_ncu_summary.json), DRAM traffic 26 MB",
            "hbm_formula": {"bound": "hbm", "achieved": alg / (bwd_ms * 1e-3) / 1e9, "peak": hbm_peak, "peak_kind": peak_kind,
                            "unit": "GB/s", "frac": alg / (bwd_ms * 1e-3) / 1e9 / hbm_peak, "algorithmic_bytes_per_call": alg,
                            "formula": "SURVEY 8d: tokens*(4 B id + 1 B mask) + tokens*8 B sort keys (id, position) + "
                                       "rows*1536 B gradient rows read + 30522*1536 B table gradient written; the per-token "
                                       "row reads that dominate the call are served by L2 and are not in this formula"}},
    }
    del tr, m
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------------------------------
# configs[3]: one full-dataset-sized pass through the public epoch loop + NDCG@10
# --------------------------------------------------------------------------------------------------
def run_epoch_leg(dev, world, rank, args):
    """~800k synthetic MS MARCO-shaped triplets, global batch 2048 x N (16384 on 8 GPUs), batches assembled on the
    device (DeviceTripletFeeder), FusedTrainer.train_epoch_device, then evaluate_model (NDCG@10, sharded over the
    ranks) — the calls run_training makes for one epoch, timed on the device, max over ranks."""
    import contextlib
    import io

    import torch.distributed as dist

    from two_towers_overlords_b200 import TwoTowersModel
    from two_towers_overlords_b200.data import DeviceTripletFeeder, MSMarcoDataset
    from two_towers_overlords_b200.training import FusedTrainer, evaluate_model

    gb = B_PER_GPU * world
    with contextlib.redirect_stdout(io.StringIO()):
        train_ds = MSMarcoDataset("train", max_samples=args.epoch_triplets, synthetic=True)
        val_ds = MSMarcoDataset("validation", max_samples=1000, synthetic=True)
    torch.manual_seed(0)
    m = TwoTowersModel(projection_dim=P_DIM, precision=args.precision).to(dev)
    tok = train_ds.tokenizer()
    tok.add(val_ds.tokenizer())
    m.query_tower.tokenizer = m.document_tower.tokenizer = tok
    reuse = world == 1 and os.environ.get("TT_NEG_REUSE", "1") != "0"  # as run_training wires it (one GPU, device feeder)
    tr = FusedTrainer(m, MARGIN, LR, B_PER_GPU, LQ, LD, precision=args.precision, world_size=world, rank=rank,
                      token_slots=2, in_batch_negatives=reuse)
    feeder = DeviceTripletFeeder(train_ds, gb, LQ, LD, dev, rank=rank, world_size=world, seed=17)
    tr.prepare(2)
    steps = len(feeder)
    for _ in range(1):  # untimed pass: first-use graphs of the epoch tail, allocator warm-up
        tr.train_epoch_device(feeder)
    tr.sync_ranks()
    ev0, ev1, ev2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    ev0.record()
    avg = tr.train_epoch_device(feeder)
    ev1.record()
    import random as _random
    _random.seed(5)
    with contextlib.redirect_stdout(io.StringIO()):
        ndcg = evaluate_model(m, val_ds, batch_size=gb)
    ev2.record()
    torch.cuda.synchronize()
    t = torch.tensor([ev0.elapsed_time(ev1), ev1.elapsed_time(ev2)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    train_ms, eval_ms = float(t[0]), float(t[1])
    tr.sync_ranks()
    tr.close()
    out = {"workload": "configs[3] full-dataset pass: synthetic MS MARCO-shaped pairs, global batch 2048 x N, "
                       "device-assembled batches, NDCG@10 evaluation at the end of the epoch",
           "triplets": steps * gb, "global_batch": gb, "steps": steps, "epoch_ms": train_ms,
           "triplets_per_s": steps * gb / (train_ms * 1e-3), "avg_loss": avg, "eval_ms": eval_ms, "val_ndcg_10": ndcg,
           "in_batch_negative_reuse": bool(reuse),
           "note": "includes per-step batch assembly on the device and the host-side launch loop; evaluate_model = "
                   "sampling + sharded document encode + candidate scoring + NDCG@10 (20 queries, reference defaults)"}
    del tr, m, feeder
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------------------------------
# corpus scan (BASELINE.json configs[4]): sharded exhaustive top-10 + NDCG@10
# --------------------------------------------------------------------------------------------------
def run_scan(dev, world, rank, n_docs, n_queries, P, passes, precision="bf16"):
    """Strong scaling: the corpus is split over the ranks, every rank scores all queries against its shard, one
    all-gather of the [Q,10] lists, merge, NDCG@10.  Returns the `scan` object of the JSON line."""
    import torch.distributed as dist

    from two_towers_overlords_b200 import ops, retrieval

    hbm_peak, tensor_peak, peak_kind = peaks()
    lo, hi = retrieval.shard_bounds(n_docs, world, rank)
    n_local = hi - lo
    g = torch.Generator(device=dev).manual_seed(7)          # same stream on every rank: global corpus, own slice
    gq = torch.Generator(device=dev).manual_seed(8)
    Qe = torch.randn(n_queries, P, generator=gq, device=dev)
    # relevant sets: 1..10 documents per query, planted as query + noise so that NDCG@10 is non-trivial
    gr = torch.Generator(device=dev).manual_seed(9)
    n_rel = torch.randint(1, 11, (n_queries,), generator=gr, device=dev)
    owner = torch.repeat_interleave(torch.arange(n_queries, device=dev), n_rel)
    rel_ids = torch.randperm(n_docs, generator=gr, device=dev)[: owner.numel()]
    noise = 1.0 + 5.0 * torch.rand(owner.numel(), generator=gr, device=dev)
    De = torch.empty(n_local, P, device=dev)
    chunk = 1 << 20
    for s0 in range(0, n_docs, chunk):                       # draw the global corpus chunk by chunk, keep my rows
        blk = torch.randn(min(chunk, n_docs - s0), P, generator=g, device=dev)
        a, b = max(lo, s0), min(hi, s0 + blk.shape[0])
        if a < b:
            De[a - lo: b - lo] = blk[a - s0: b - s0]
    mine = (rel_ids >= lo) & (rel_ids < hi)
    gn = torch.Generator(device=dev).manual_seed(10)
    plant_noise = torch.randn(owner.numel(), P, generator=gn, device=dev)
    De[rel_ids[mine] - lo] = Qe[owner[mine]] + noise[mine, None] * plant_noise[mine]
    del plant_noise
    order = torch.argsort(owner * n_docs + rel_ids)
    rel_csr = (torch.cat([torch.zeros(1, dtype=torch.int64, device=dev), torch.cumsum(n_rel, 0)]), rel_ids[order].contiguous())
    shard = retrieval.CorpusShard(De, id_base=lo, precision=precision)
    del De
    torch.cuda.synchronize()

    def one_pass(q):
        return retrieval.retrieve_and_score(shard, q, rel_csr, k=10, world_size=world)

    def timed(fn, n):
        fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    lib = ops.N.load()
    n0 = lib.tt_launch_count()
    ms_full, (top_s, top_i, ndcg) = timed(lambda: one_pass(Qe), passes)
    launches = (lib.tt_launch_count() - n0) // (passes + 1)
    # end to end: query embeddings start in pinned host memory, top-10 ids + NDCG come back to the host
    Qh = Qe.cpu().pin_memory()
    ids_h = torch.empty(n_queries, 10, dtype=torch.int64).pin_memory()
    ndcg_h = torch.empty(n_queries, dtype=torch.float64).pin_memory()

    def e2e_pass():
        q = Qh.to(dev, non_blocking=True)
        _, ti, nd = one_pass(q)
        ids_h.copy_(ti, non_blocking=True)
        ndcg_h.copy_(nd, non_blocking=True)
        return None

    ms_e2e, _ = timed(e2e_pass, passes)
    # streaming regime of the reference's own eval (few queries per pass, training.py:244): one 128-query tile
    q_small = Qe[:128].contiguous()
    torch.cuda.synchronize()
    time.sleep(0.5)  # the batched passes above run at the power limit; let the clocks settle before a bandwidth test
    for _ in range(3):
        shard.search(q_small, 10)
    ms_small, _ = timed(lambda: shard.search(q_small, 10), 20)
    flops = 2.0 * n_queries * n_local * P
    stream_bytes = n_local * P * 2.0
    return {
        "metric": "top10_queries_per_sec", "value": n_queries / (ms_full * 1e-3), "unit": "queries/s", "scaling": "strong",
        "config": {"workload": "configs[4] corpus scan: synthetic unit-norm passages x 384-d, top-10 + NDCG@10",
                   "n_docs": n_docs, "docs_per_gpu": n_local, "n_queries": n_queries, "dim": P, "k": 10,
                   "precision": f"{precision} tensor-core candidates + exact fp32 re-score", "passes": passes},
        "ms_per_pass": ms_full, "mean_ndcg_10": float(ndcg.mean().item()),
        "e2e": {"value": n_queries / (ms_e2e * 1e-3), "unit": "queries/s", "h2d_bytes_per_pass": Qh.numel() * 4,
                "d2h_bytes_per_pass": ids_h.numel() * 8 + ndcg_h.numel() * 8, "ms_per_pass": ms_e2e},
        "gpu_launches_per_pass": int(launches),
        "roofline_batched": {"bound": "tensor", "achieved": flops / (ms_full * 1e-3) / 1e12, "peak": tensor_peak,
                             "peak_kind": peak_kind, "unit": "TFLOP/s",
                             "frac": flops / (ms_full * 1e-3) / 1e12 / tensor_peak,
                             "traffic": ncu_traffic("scan_candidates_kernel_batched_100kq_8.8M")
                             if (n_local == 8_800_000 and P == 384 and n_queries == 100_000) else None,
                             "note": "whole pass (normalise + scan + refine/re-score + merge + NDCG); 2*Q*N_local*P "
                                     "flops; traffic is DRAM bytes of the scan kernel (cta_group::2 tiles on a shard this "
                                     "long: each document tile is loaded once per CTA pair and multicast; the one-CTA "
                                     "kernel moved 1.31 TB per pass)"},
        "roofline_streaming": {"bound": "hbm", "queries": 128, "achieved": stream_bytes / (ms_small * 1e-3) / 1e9,
                               "peak": hbm_peak, "peak_kind": peak_kind, "unit": "GB/s",
                               "frac": stream_bytes / (ms_small * 1e-3) / 1e9 / hbm_peak, "ms_per_pass": ms_small,
                               "traffic": ncu_traffic("scan_candidates_kernel_streaming_128q_8.8M")
                               if (n_local == 8_800_000 and P == 384) else None,
                               "note": "one 128-query tile against the whole bf16 shard (N_local*P*2 algorithmic "
                                       "bytes); timed over the WHOLE search call (normalise + scan kernel + refine/"
                                       "re-score + flag compaction; one CUDA-graph replay), the scan kernel alone is 1.01 ms "
                                       "under ncu and reads the shard exactly once (profiles/r02_ncu_summary.json); passes/s = the reference's "
                                       "per-query eval regime"},
    }


_REAL_STDOUT = None


def quiet_stdout():
    """Native libraries (NCCL's version banner) write to fd 1; keep stdout to the ONE JSON line by pointing fd 1 at
    stderr for the whole run and printing the result on the saved descriptor."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(obj):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("TT_BENCH_PRECISION", "bf16x3"), choices=["fp32", "bf16x3", "bf16"])
    ap.add_argument("--table-dtype", default="f32", choices=["f32", "bf16"])
    ap.add_argument("--ids-dtype", default="u16", choices=["u16", "i32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-scan", action="store_true")
    ap.add_argument("--no-config2", action="store_true", help="skip the configs[2] leg (trainable tables, B=4096, P=384)")
    ap.add_argument("--no-backbone", action="store_true", help="skip the frozen MiniLM-L6 backbone leg")
    ap.add_argument("--no-chain-variant", action="store_true", help="skip the projection-chain leg (persistent kernel vs one kernel per contraction)")
    ap.add_argument("--no-epoch", action="store_true", help="skip the configs[3] leg (~800k-triplet pass + NDCG@10)")
    ap.add_argument("--epoch-triplets", type=int, default=800_000)
    ap.add_argument("--scan-docs", type=int, default=8_800_000)
    ap.add_argument("--scan-queries", type=int, default=100_000)
    ap.add_argument("--scan-passes", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, gradients and parameters of the last timed training step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the B200 arm's timed steps")
    if args.warmup < 3:
        args.warmup = 3
    quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
