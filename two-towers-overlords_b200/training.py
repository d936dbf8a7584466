"""
Training / evaluation for the two-towers model — B200-native drop-in for the reference's
backend/training.py: `clear_gpu_memory`, `train_epoch`, `train_epoch_optimized`, `evaluate_model`,
`run_training` keep the reference's signatures, return values and printed/logged keys, so backend/main.py
runs on top unchanged.

Additions (the B200 path proper):
  * FusedTrainer      one tt_triplet_step (pooled gather -> both tower MLPs -> loss -> all gradients) + Adam per
                      step, captured as one CUDA graph whose branches run in parallel (the next step's pooled
                      gather beside this step's tensor-core chain); data-parallel with ONE fused kernel per step
                      (reduce-scatter over NVLink peer memory -> Adam -> all-gather; NCCL all-reduce + Adam as the
                      baseline); batches assembled on the device (train_epoch_device); checkpoint / resume.
  * evaluate_model    scores every query against the candidate documents with the corpus-scan / candidate
                      kernels and computes NDCG@k on the device; only tie cases that the closed form cannot
                      express fall back to the exact tie-averaged formula.
"""
from __future__ import annotations

import math
import os
import random
import time
from typing import Optional, Union

import numpy as np
import torch
from torch import GradScaler, autocast

try:
    from . import comm, ops, retrieval
    from .data import (DeviceTripletFeeder, HardNegativeMiner, MSMarcoDataset, PooledBank, TokenTripletLoader,
                       TripletDataLoader)
    from .model import TokenBatch, TripletLoss, TwoTowersModel
except ImportError:
    import comm
    import ops
    import retrieval
    from data import (DeviceTripletFeeder, HardNegativeMiner, MSMarcoDataset, PooledBank, TokenTripletLoader,
                      TripletDataLoader)
    from model import TokenBatch, TripletLoss, TwoTowersModel

try:  # wandb is optional at import time; only touched when logging is requested
    import wandb
except Exception:  # noqa: BLE001
    wandb = None


def clear_gpu_memory():
    """Clear GPU memory cache to reduce fragmentation (training.py:19-23)."""
    if torch.cuda.is_available():
        torch.cuda.empty_cache()
        torch.cuda.synchronize()


# --------------------------------------------------------------------------------------------------
# reference-shaped epoch loops (training.py:26-133)
# --------------------------------------------------------------------------------------------------
def train_epoch(model, dataloader, criterion, optimizer, log_wandb: bool = True) -> float:
    """Train for one epoch (training.py:26-63).  The per-batch loss stays on the device; the host only
    reads it where the reference prints/logs it."""
    total_loss = None
    num_batches = 0
    for queries, positives, negatives in dataloader:
        optimizer.zero_grad()
        query_embeds = model.encode_queries(queries)
        positive_embeds = model.encode_documents(positives)
        negative_embeds = model.encode_documents(negatives)
        loss = criterion(query_embeds, positive_embeds, negative_embeds)
        loss.backward()
        optimizer.step()
        total_loss = loss.detach().double() if total_loss is None else total_loss + loss.detach().double()
        num_batches += 1
        if log_wandb and wandb is not None:
            wandb.log({"batch_loss": loss.item(), "batch": num_batches})
        if num_batches % 10 == 0:
            print(f"Batch {num_batches}, Loss: {loss.item():.4f}")
    if num_batches == 0:
        raise ZeroDivisionError("train_epoch: empty dataloader")
    return float(total_loss.item()) / num_batches


def train_epoch_optimized(model, dataloader, criterion, optimizer, device, scaler, accumulation_steps: int = 2,
                          log_wandb: bool = True) -> float:
    """Mixed-precision + gradient-accumulation epoch (training.py:66-133).  The kernels compute in fp32 /
    split-bf16 regardless of autocast, so the GradScaler only ever sees finite fp32 gradients; its
    scale/unscale protocol is kept so that the optimiser-step cadence matches the reference."""
    model.train()
    total_loss = None
    num_batches = 0
    for batch_idx, (queries, positives, negatives) in enumerate(dataloader):
        with autocast(device.type):
            query_embeds = model.encode_queries(queries)
            positive_embeds = model.encode_documents(positives)
            negative_embeds = model.encode_documents(negatives)
            loss = criterion(query_embeds, positive_embeds, negative_embeds)
            loss = loss / accumulation_steps
        scaler.scale(loss).backward()
        if (batch_idx + 1) % accumulation_steps == 0:
            scaler.step(optimizer)
            scaler.update()
            optimizer.zero_grad()
        unscaled = loss.detach().double() * accumulation_steps
        total_loss = unscaled if total_loss is None else total_loss + unscaled
        num_batches += 1
        if log_wandb and wandb is not None and batch_idx % 10 == 0:
            wandb.log({
                "batch_loss": loss.item() * accumulation_steps,
                "batch": num_batches,
                "gpu_memory_allocated": torch.cuda.memory_allocated() / 1e9 if torch.cuda.is_available() else 0,
                "gpu_memory_reserved": torch.cuda.memory_reserved() / 1e9 if torch.cuda.is_available() else 0,
            })
        if batch_idx % 10 == 0:
            print(f"Batch {batch_idx}, Loss: {loss.item() * accumulation_steps:.4f}")
    if num_batches == 0:
        raise ZeroDivisionError("train_epoch_optimized: empty dataloader")
    return float(total_loss.item()) / num_batches


# --------------------------------------------------------------------------------------------------
# fused B200 trainer
# --------------------------------------------------------------------------------------------------
class AccumulationWindow:
    """Optimiser cadence of the reference's gradient accumulation (backend/training.py:66-133) over micro-steps: the
    optimiser runs after micro-batch `batch_idx` whenever (batch_idx + 1) % a == 0, batch_idx restarts at 0 every epoch,
    and a trailing partial window carries its gradient into the next epoch's first window.  Host only."""

    def __init__(self, accumulation_steps: int):
        if (isinstance(accumulation_steps, bool) or int(accumulation_steps) != accumulation_steps
                or accumulation_steps < 1):
            raise ValueError(f"accumulation_steps must be an integer >= 1, got {accumulation_steps!r}")
        self.a = int(accumulation_steps)
        self.batch_idx = 0  # micro-batch position in the epoch
        self.pending = 0    # micro-batches summed in the gradient buffers since the last optimiser step

    def start_epoch(self):
        self.batch_idx = 0

    def mode(self) -> tuple:
        """(accumulate, close) of the next micro-step: add to the gradient buffers (they carry an unstepped gradient)
        instead of overwriting them; run the optimiser after it."""
        return (self.pending > 0, (self.batch_idx + 1) % self.a == 0)

    def advance(self):
        close = self.mode()[1]
        self.batch_idx += 1
        self.pending = 0 if close else self.pending + 1

    def modes(self) -> list:
        """Every mode the schedule can reach: a = 1 overwrites and steps every time; a > 1 opens a window by
        overwriting, continues it by adding, closes it by adding and stepping — and a first window that continues a
        carried partial one starts by adding."""
        return [(False, True)] if self.a == 1 else [(False, False), (True, False), (True, True)]


class FusedTrainer:
    """Whole training step (training.py:37-51) as: tokens into a static slot (one packed H2D copy or the device
    feeder) -> tt_triplet_step -> tt_adam_step_dev (one GPU) / tt_dp_reduce_adam (data parallel, peer memory) /
    NCCL all-reduce + Adam (baseline), on static buffers so the device part replays as one CUDA graph.

    `step(slot, next_slot)` software-pipelines consecutive steps: the pooled gather of `next_slot` runs beside
    the rest of `slot` (it reads tokens and the frozen tables only, so this is still exact synchronous SGD).
    The 8 projection tensors are re-pointed at views of one flat fp32 buffer, so the model's
    `state_dict()` / `parameters()` always see the trained values; gradients live in a second flat buffer
    whose last element carries the loss (one exchange covers both).

    `accumulation_steps = a` reproduces the reference's gradient accumulation (backend/training.py:66-133): every
    micro-batch (one step() call) adds the gradient of loss / a into the flat gradient, and the optimiser (and, data
    parallel, the one exchange) runs after micro-batch `batch_idx` of the epoch whenever (batch_idx + 1) % a == 0.
    `batch_idx` restarts at 0 with every epoch (train_epoch / train_epoch_device / start_epoch()); a trailing partial
    window is not stepped and its gradient carries into the next epoch's first window, as in the reference.  a = 1 is
    the plain trainer.

    `optimize_tables=True` trains the token tables too (the model's tables must be trainable fp32,
    TwoTowersModel(train_table=True)): torch.optim.Adam's dense step on every row of both tables with the projections'
    step count, as `torch.optim.Adam(model.parameters())` applies it.  On one GPU it runs in the epilogue of the table
    gradient's scatter-add inside the step call; data parallel (exchange="peer") the tables live in a second peer
    segment and their flat gradient goes through the same fused reduce-scatter / Adam / all-gather kernel right after
    the projections'.  Off (the default), a trainable-table model only gets its table gradients (`table_grads`)."""

    def __init__(self, model: TwoTowersModel, margin: float, lr: float, batch_size: int, Lq: int = 32, Ld: int = 256,
                 precision: Optional[str] = None, world_size: int = 1, rank: int = 0, use_graph: bool = True,
                 betas=(0.9, 0.999), eps: float = 1e-8, process_group=None, ids_dtype=torch.int32,
                 mask_dtype=torch.uint8, token_slots: int = 1, exchange: Optional[str] = None,
                 exchange_ctas: int = 0, in_batch_negatives: bool = False, pooled=None, accumulation_steps: int = 1,
                 optimize_tables: bool = False):
        qt, dt = model.query_tower, model.document_tower
        if in_batch_negatives and world_size > 1:  # refused before any buffer or peer segment is allocated
            raise ValueError("in_batch_negatives: the negatives of a data-parallel slice name documents of other ranks")
        self.window = AccumulationWindow(accumulation_steps)
        self.accum = self.window.a
        self.model = model
        self.device = qt.pretrained_model.device
        if self.device.type != "cuda":
            raise RuntimeError("FusedTrainer needs the model on a CUDA device (no CPU fallback)")
        self.B, self.Lq, self.Ld = batch_size, Lq, Ld
        self.H = qt.embedding_dim
        self.P = qt.projection[0].out_features
        self.vocab = qt.pretrained_model.config.vocab_size
        self.margin, self.lr, self.betas, self.eps = float(margin), float(lr), betas, float(eps)
        self.world, self.rank, self.pg = world_size, rank, process_group
        self.precision = precision or qt.precision
        # pooled = (bank_q, bank_d), data.PooledBank: the frozen front end (backbone -> masked mean -> normalise) was
        # computed once per text, so a step copies its 3B pooled rows out of the banks by index instead of pooling
        # tokens.  This is how the MiniLM backbone trains: it has no token table to gather from.
        self.pooled = tuple(pooled) if pooled is not None else None
        if self.pooled is None and not hasattr(qt.pretrained_model, "table"):
            raise ValueError("FusedTrainer: this backbone has no token table to gather from (MiniLM); encode the "
                             "training texts once with data.PooledBank.build(tower, bank, L) for each tower and pass "
                             "pooled=(bank_q, bank_d)")
        if self.pooled is not None:
            if any(p.requires_grad for t in (qt, dt) for p in t.pretrained_model.parameters()):
                raise ValueError("FusedTrainer(pooled=...) needs a frozen backbone: pooled rows of a trainable table "
                                 "would go stale at the first step")
            if in_batch_negatives:
                raise ValueError("FusedTrainer(pooled=...): the negatives are named by their own bank rows; "
                                 "in_batch_negatives does not apply")
            self.pooled[0].check(qt, "the query tower's pooled bank")
            self.pooled[1].check(dt, "the document tower's pooled bank")
            if (self.pooled[0].L, self.pooled[1].L) != (Lq, Ld):
                raise ValueError(f"FusedTrainer(pooled=...): the banks truncate texts to {self.pooled[0].L} / "
                                 f"{self.pooled[1].L} tokens, the trainer to Lq = {Lq} / Ld = {Ld}; build them with the "
                                 "trainer's lengths")
            self.train_table = False
        else:
            self.train_table = bool(qt.pretrained_model.table.requires_grad)
        self.optimize_tables = bool(optimize_tables)
        if self.optimize_tables:
            if not self.train_table:
                raise ValueError("FusedTrainer(optimize_tables=True) needs trainable token tables: build the model with "
                                 "TwoTowersModel(train_table=True)")
            if any(t.pretrained_model.table.dtype != torch.float32 for t in (qt, dt)):
                raise ValueError("FusedTrainer(optimize_tables=True) needs fp32 token tables (bf16 tables do not train)")
            if exchange == "nccl" or (world_size > 1 and not exchange
                                      and os.environ.get("TT_DP_EXCHANGE", "peer") == "nccl"):
                raise ValueError("FusedTrainer(optimize_tables=True) exchanges the tables with the peer exchange only; "
                                 "exchange='nccl' is the projections-only baseline")
        params = model.projection_parameters()
        sizes = [p.numel() for p in params]
        self.n_param = sum(sizes)
        dev = self.device
        # data-parallel exchange: "peer" = ONE kernel (reduce-scatter over NVLink peer stores -> Adam on the local
        # slice -> all-gather of the new parameters), overlapped with the next step's pooled gather, which does not
        # read the projection weights; "nccl" = all-reduce + Adam launch, serialised (the baseline)
        if world_size > 1:
            self.exchange = exchange or os.environ.get("TT_DP_EXCHANGE", "peer")
        else:  # one rank: the fused exchange kernel still works (used by tests), the default is the plain Adam launch
            self.exchange = "peer" if exchange == "peer" else "none"
        if self.exchange not in ("none", "peer", "nccl"):
            raise ValueError(f"exchange must be 'peer' or 'nccl', got {self.exchange!r}")
        self.exchange_ctas = int(exchange_ctas or os.environ.get("TT_DP_CTAS", "0"))
        self.xchg = None
        if self.exchange == "peer":
            self.xchg = comm.DpExchange(self.n_param, world_size, rank, dev, group=process_group)
            self.flat_p = self.xchg.flat_p
        else:
            self.flat_p = torch.empty(self.n_param, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(self.n_param + 1, dtype=torch.float32, device=dev)  # [+1]: loss
        self.exp_avg = torch.zeros(self.n_param, dtype=torch.float32, device=dev)
        self.exp_avg_sq = torch.zeros(self.n_param, dtype=torch.float32, device=dev)
        self.adam_state = torch.zeros(4, dtype=torch.float64, device=dev)
        # the tables' optimiser state: flat [2VH] moments (query table | document table); data parallel, a second
        # exchange whose peer segment holds both tables and a flat [2VH + 1] gradient in the same layout
        self.txchg = None
        self.table_grads = None
        self.table_exp_avg = self.table_exp_avg_sq = None
        if self.optimize_tables:
            tables = (qt.pretrained_model.table, dt.pretrained_model.table)
            nt = tables[0].numel()
            self.n_table = 2 * nt
            if self.exchange == "peer":
                self.txchg = comm.DpExchange(self.n_table, world_size, rank, dev, group=process_group)
                self.table_flat_g = torch.zeros(self.n_table + 1, dtype=torch.float32, device=dev)
                with torch.no_grad():
                    for i, t in enumerate(tables):
                        view = self.txchg.flat_p[i * nt: (i + 1) * nt].view_as(t)
                        view.copy_(t.data)
                        t.data = view  # the table Parameter now aliases the peer segment
                self.table_grads = tuple(self.table_flat_g[i * nt: (i + 1) * nt].view_as(t)
                                         for i, t in enumerate(tables))
            self._table_m = torch.zeros(self.n_table, dtype=torch.float32, device=dev)
            self._table_v = torch.zeros(self.n_table, dtype=torch.float32, device=dev)
            self.table_exp_avg = tuple(self._table_m[i * nt: (i + 1) * nt].view_as(t) for i, t in enumerate(tables))
            self.table_exp_avg_sq = tuple(self._table_v[i * nt: (i + 1) * nt].view_as(t) for i, t in enumerate(tables))
        self.p_views, self.g_views = [], []
        off = 0
        with torch.no_grad():
            for p, n in zip(params, sizes):
                view = self.flat_p[off: off + n].view_as(p)
                view.copy_(p.data)
                p.data = view  # the nn.Parameter now aliases the flat buffer
                self.p_views.append(view)
                self.g_views.append(self.flat_g[off: off + n].view_as(p))
                off += n
        # data-parallel replicas must start from the same weights: only gradients are exchanged afterwards (the peer
        # exchange overwrites parameters slice by slice AFTER the first gradients were taken on the local ones)
        self._sync_initial_state()
        # where the step's GLOBAL loss can be read: slot n of the flat gradient (summed in place by NCCL), or slot n
        # of the peer segment (written by the exchange kernel)
        self.loss_view = self.xchg.loss if self.xchg is not None else self.flat_g[self.n_param:]
        # static token buffers (graph replays read these addresses).  The six tensors of a slot are views of ONE
        # byte buffer so that a step's tokens arrive with a single H2D copy (load_packed)
        self._tok_layout = []
        off = 0
        for L, dt_ in ((Lq, ids_dtype), (Lq, mask_dtype), (Ld, ids_dtype), (Ld, mask_dtype), (Ld, ids_dtype),
                       (Ld, mask_dtype)):
            nbytes = batch_size * L * torch.empty((), dtype=dt_).element_size()
            self._tok_layout.append((off, nbytes, L, dt_))
            off += (nbytes + 255) // 256 * 256
        self.tok_bytes = off

        def new_set():
            buf = torch.zeros(self.tok_bytes, dtype=torch.uint8, device=dev)
            return buf, tuple(buf[o: o + nb].view(dt_).view(batch_size, L) for o, nb, L, dt_ in self._tok_layout)

        # token_slots > 1: rotating input buffers (prefetch step i+1 while step i computes; each slot has
        # its own captured graph because a graph replays fixed addresses)
        n_slots = max(1, token_slots)
        self.row_bufs = None
        if self.pooled is None:
            sets = [new_set() for _ in range(n_slots)]
            self.tok_bufs = [b for b, _ in sets]
            self.tok_slots = [v for _, v in sets]
        else:  # no token buffers: a slot is the int32 [3B] bank rows of its batch (q | p | n), see load_rows()
            self.tok_bufs = []
            self.tok_slots = [None] * n_slots
            self.row_bufs = [torch.zeros(3 * batch_size, dtype=torch.int32, device=dev) for _ in range(n_slots)]
            self._rows_loaded = [False] * n_slots  # step() refuses a slot whose rows were never given
        self.tok = self.tok_slots[0]
        if self.train_table and self.table_grads is None:
            self.table_grads = (torch.zeros_like(qt.pretrained_model.table, dtype=torch.float32),
                                torch.zeros_like(dt.pretrained_model.table, dtype=torch.float32))
        # TWO step workspaces: the pooled gather of step i+1 (tokens + frozen tables only, never the projection
        # weights) runs beside everything else of step i, so consecutive steps alternate between them
        # How the projection chain is launched (tt_step_args.chain).  Default: the persistent chain kernel — everything
        # after the pooled gather in ONE launch (115 us alone at configs[1] against 157-162 us for one kernel per
        # contraction).  It wants every SM, so nothing runs beside it: on one GPU a step is gather -> chain in one stream
        # (2 launches, the second a programmatic dependent of the first; 0.230-0.233 ms), under data parallelism the NEXT
        # step's gather runs beside the exchange kernel, which mostly waits (N = 2: 0.272 ms).  The per-kernel chain
        # (TT_CHAIN=0) lets the look-ahead gather's CTAs slip between its small kernels instead; since the chain kernel
        # lost its transposed copies that schedule is the slower one (0.242-0.248 ms; N = 2: 0.275 ms).  A trainable table
        # has no look-ahead in either mode (the gather reads the table the step updates).
        env_chain = os.environ.get("TT_CHAIN")
        if env_chain is not None:
            self.chain_mode = 1 if env_chain != "0" else 2
        else:
            self.chain_mode = 1
        self.step_objs = []
        for _ in range(2):
            so = ops.TripletStep(batch_size, Lq, Ld, self.H, self.P, self.vocab, self.precision, dev,
                                 train_table=self.train_table)
            so.loss = self.flat_g[self.n_param:]  # this rank's loss term lands in the flat gradient's last slot
            tables = None if self.pooled else (qt.pretrained_model.table.data, dt.pretrained_model.table.data)
            # upstream gradient 1/a: the reference backpropagates loss / accumulation_steps
            so.bind(self.tok, tables, self.p_views, self.g_views, self.margin, 1.0 / (batch_size * world_size),
                    1.0 / self.accum, self.table_grads)
            for toks in self.tok_slots[1:]:
                so.add_tokens(toks)
            if self.pooled:
                so.bind_pooled(self.pooled[0].rows, self.pooled[1].rows)
                for slot, buf in enumerate(self.row_bufs):
                    so.set_pooled_index(slot, buf)
            so.set_chain(self.chain_mode)
            if self.exchange == "none" and self.world == 1:
                # single GPU: torch.optim.Adam rides inside the step call (the tail of the persistent chain kernel
                # with the tensor-core precisions; a launch after the step otherwise)
                so.bind_adam(self.adam_state, self.flat_p, self.flat_g, self.exp_avg, self.exp_avg_sq, self.lr,
                             self.betas, self.eps)
                if self.optimize_tables:  # the tables' Adam step rides in the table gradient's epilogue
                    so.bind_table_adam(tables, self.table_exp_avg, self.table_exp_avg_sq)
            self.step_objs.append(so)
        self.step_obj = self.step_objs[0]
        # In-batch negatives (the reference's batcher, backend/data.py:113-137): negative i IS positive neg_index[i], so
        # its pooled row is copied instead of gathered a second time (tt_step_args.neg_index).  One int32 [B] buffer per
        # token slot (static addresses: the step graphs read them); fill them with load_neg_index() / the device feeder.
        # With trainable tables each negative's table-gradient row is folded into the positive it copies.
        self.in_batch_negatives = bool(in_batch_negatives)
        self.neg_bufs = None
        if self.in_batch_negatives:
            self.neg_bufs = [torch.zeros(batch_size, dtype=torch.int32, device=dev) for _ in self.tok_slots]
            self._neg_loaded = [False] * len(self.tok_slots)  # step() refuses a slot whose indices were never given
            for so in self.step_objs:
                for slot, buf in enumerate(self.neg_bufs):
                    so.set_neg_index(slot, buf)
        self.use_graph = use_graph
        self.graphs = {}       # (slot, next_slot, parity) -> CUDAGraph
        self.graph_opt = None  # NCCL mode: Adam after the all-reduce
        self.graph_captures = 0  # bench.py asserts that none happens inside a timed region
        self.side = torch.cuda.Stream(device=dev)
        # graphs are captured on a high-priority stream: the latency-bound chain then takes SM slots ahead of the
        # bandwidth-bound pooled gather running beside it (measured 291 -> 268 us per step)
        self.cap_stream = torch.cuda.Stream(device=dev, priority=-1)
        self._parity = 0       # workspace of the current step
        self._primed = None    # slot whose pooled gather already sits in step_objs[_parity]
        self._warm = False
        self.steps_done = 0
        self.kernel_launches_per_step = None
        # data parallel with accumulation: the exchange (which publishes the global loss) runs on closing micro-steps
        # only, so the epoch's loss is this rank's share of every micro-batch's global loss, summed over the ranks once
        # per epoch
        self._loss_share = (torch.zeros((), dtype=torch.float64, device=dev)
                            if self.world > 1 and self.accum > 1 else None)

    # -- data-parallel hygiene ---------------------------------------------------------------------
    def _dist_ready(self) -> bool:
        import torch.distributed as dist

        return self.world > 1 and dist.is_available() and dist.is_initialized()

    def _sync_initial_state(self):
        """Rank 0's projection weights (and Adam step count) become everybody's.  Collective when world_size > 1 and a
        process group exists (virtual-rank tests run several ranks in one process without one)."""
        if not self._dist_ready():
            return
        import torch.distributed as dist

        tmp = self.flat_p.clone()  # the peer segment is library-owned memory: broadcast through a torch tensor
        dist.broadcast(tmp, src=0, group=self.pg)
        if not torch.equal(tmp, self.flat_p):
            if self.rank != 0:
                print(f"[rank {self.rank}] FusedTrainer: initial projection weights differed from rank 0's; "
                      "taking rank 0's")
            self.flat_p.copy_(tmp)
        st = self.xchg.state if self.xchg is not None else self.adam_state
        dist.broadcast(st, src=0, group=self.pg)
        if self.txchg is not None:  # trained tables: only their gradients are exchanged afterwards, as above
            tmp = self.txchg.flat_p.clone()
            dist.broadcast(tmp, src=0, group=self.pg)
            if not torch.equal(tmp, self.txchg.flat_p):
                if self.rank != 0:
                    print(f"[rank {self.rank}] FusedTrainer: initial token tables differed from rank 0's; taking rank 0's")
                self.txchg.flat_p.copy_(tmp)
            dist.broadcast(self.txchg.state, src=0, group=self.pg)
        torch.cuda.synchronize()

    def sync_ranks(self):
        """Host barrier: call after rank-local work (evaluation, checkpoint writes, graph capture) and before the next
        exchanged step, so that no rank spins in the exchange kernel past its timeout waiting for a busy peer."""
        torch.cuda.synchronize()
        if self._dist_ready():
            import torch.distributed as dist

            dist.barrier(group=self.pg)

    def check(self):
        """Raises if the peer exchange reported an error (a rank that never answered).  Host sync; called wherever the
        loss is read on the host and at the end of every epoch."""
        if self.xchg is not None:
            self.xchg.check()
        if self.txchg is not None:
            self.txchg.check()

    # -- pieces ------------------------------------------------------------------------------------
    def load_tokens(self, q: TokenBatch, p: TokenBatch, n: TokenBatch, slot: int = 0):
        """Host (pinned) or device token batches -> static device buffers, async on the current stream."""
        for dst, src in zip(self.tok_slots[slot], (q.input_ids, q.attention_mask, p.input_ids, p.attention_mask,
                                                   n.input_ids, n.attention_mask)):
            dst.copy_(src, non_blocking=True)

    def load_rows(self, rows: torch.Tensor, slot: int = 0):
        """Bank rows of the batch in `slot` for a trainer over pooled banks: int [3, B] or [3B] (query rows | positive
        rows | negative rows; host or device), async on the current stream."""
        if self.row_bufs is None:
            raise RuntimeError("FusedTrainer.load_rows needs a trainer built with pooled=(bank_q, bank_d)")
        self.row_bufs[slot].copy_(rows.reshape(-1).to(torch.int32), non_blocking=True)
        self._rows_loaded[slot] = True

    def check_banks(self):
        """Raises if a pooled bank no longer matches its tower's backbone (weights changed after the build): a stale
        bank must never train silently.  Called by prepare() and at the start of every epoch."""
        if self.pooled is not None:
            self.pooled[0].check(self.model.query_tower, "the query tower's pooled bank")
            self.pooled[1].check(self.model.document_tower, "the document tower's pooled bank")

    def _load(self, batch, slot: int):
        if self.pooled is not None:
            self.load_rows(batch, slot)
        else:
            self.load_tokens(*batch, slot=slot)

    def load_neg_index(self, neg_index: torch.Tensor, slot: int = 0):
        """Indices of the in-batch negatives of the batch in `slot` (int [B]; host or device), async on the current stream."""
        self.neg_bufs[slot].copy_(neg_index.to(torch.int32), non_blocking=True)
        self._neg_loaded[slot] = True

    def _fwd_bwd(self, slot: int = 0, phases: int = 0, parity: int = 0, optimise: bool = False,
                 accumulate: bool = False):
        self.step_objs[parity].run(slot, phases, optimise=optimise, accumulate=accumulate)

    def _exchange(self):
        """The fused reduce-scatter / Adam / all-gather kernel (tt_dp_reduce_adam) on the current stream; with trained
        tables a second call on their flat gradient follows (its loss slot stays 0)."""
        self.xchg.reduce_adam(self.flat_g, self.exp_avg, self.exp_avg_sq, self.lr, self.betas, self.eps,
                              self.exchange_ctas)
        if self.txchg is not None:
            self.txchg.reduce_adam(self.table_flat_g, self._table_m, self._table_v, self.lr, self.betas, self.eps,
                                   self.exchange_ctas)

    def _pipelined(self, slot: int, next_slot: Optional[int], parity: int, mode=(False, True)):
        """One training step on the current stream, in the schedule __init__ chose: whole step (gather -> persistent
        chain kernel), per-kernel chain beside the look-ahead gather of `next_slot`, or — data parallel — persistent
        chain, then the exchange beside the look-ahead gather.  mode = (accumulate, close): add the gradients to the
        buffers instead of overwriting them; run the optimiser / the exchange (a closing micro-step)."""
        cur = torch.cuda.current_stream()
        acc, close = mode
        fused_opt = self.xchg is None and self.world == 1 and close
        exchange = self.xchg is not None and close
        if self._whole_step():
            # ONE call = pooled gather -> persistent chain kernel (+ Adam in its tail): two launches, the second a
            # programmatic dependent of the first
            self._fwd_bwd(slot, 0, parity, optimise=fused_opt, accumulate=acc)
            return
        chain_mode = self.step_objs[0].chain_active()
        if not chain_mode:
            # per-kernel chain: many small latency-bound kernels, the look-ahead gather's CTAs slip in between them
            if next_slot is not None:
                self.side.wait_stream(cur)
                with torch.cuda.stream(self.side):
                    self._fwd_bwd(next_slot, 1, parity ^ 1)
            self._fwd_bwd(slot, 2, parity, optimise=fused_opt, accumulate=acc)
            if exchange:
                self._exchange()
            if next_slot is not None:
                cur.wait_stream(self.side)
            return
        # Persistent chain kernel + data parallelism: the chain wants one CTA on EVERY SM (its CTAs wait for each other),
        # so nothing runs beside it; the look-ahead gather runs beside the exchange kernel instead, which spends most
        # of its time waiting for the peers' gradient flags on one small CTA per SM.
        self._fwd_bwd(slot, 2, parity, optimise=fused_opt, accumulate=acc)
        if next_slot is not None:
            self.side.wait_stream(cur)
            with torch.cuda.stream(self.side):
                self._fwd_bwd(next_slot, 1, parity ^ 1)
        if exchange:
            self._exchange()
        if next_slot is not None:
            cur.wait_stream(self.side)

    def _whole_step(self) -> bool:
        """Single GPU with the persistent chain kernel: a step is gather -> chain in one stream, no look-ahead."""
        return self.xchg is None and self.world == 1 and self.step_objs[0].chain_active()

    def wait(self):
        """Kept for API symmetry: every step() leaves parameters and `loss_view` final in stream order."""

    def read_loss_async(self, host_dst: torch.Tensor):
        """Copies the last step's global loss into pinned host memory without a sync."""
        host_dst.copy_(self.loss_view.reshape(host_dst.shape), non_blocking=True)

    def pack_host_tokens(self, tensors, pin: bool = True) -> torch.Tensor:
        """(q_ids,q_mask,p_ids,p_mask,n_ids,n_mask) host tensors -> one (pinned) byte buffer in slot layout."""
        buf = torch.zeros(self.tok_bytes, dtype=torch.uint8)
        if pin:
            buf = buf.pin_memory()
        for (o, nb, L, dt_), t in zip(self._tok_layout, tensors):
            assert t.dtype == dt_ and tuple(t.shape) == (self.B, L), (t.dtype, tuple(t.shape))
            buf[o: o + nb].view(dt_).view(self.B, L).copy_(t)
        return buf

    def load_packed(self, host_buf: torch.Tensor, slot: int = 0):
        """One H2D copy of a pack_host_tokens() buffer into the slot's static device buffers (current stream)."""
        self.tok_bufs[slot].copy_(host_buf, non_blocking=True)

    def _optimizer(self):
        b1, b2 = self.betas
        N = ops.N
        N.check(N.load().tt_adam_step_dev(N.ptr(self.flat_p), N.ptr(self.flat_g), N.ptr(self.exp_avg),
                                          N.ptr(self.exp_avg_sq), self.n_param, self.lr, b1, b2, self.eps,
                                          N.ptr(self.adam_state), 1.0, N.stream()), "tt_adam_step_dev")
        # projections only: optimize_tables is refused with this NCCL baseline

    def _warm_up(self):
        # one eager forward/backward on a side stream (first-use kernel attributes), gradients only: harmless, except
        # that it overwrites the gradient buffers, so an open window (a resumed checkpoint) is put back afterwards
        keep = None
        if self.window.pending:
            keep = [t.clone() for t in (self.flat_g,) + tuple(self.table_grads or ())]
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self._fwd_bwd(0, 0, 0)
            self._fwd_bwd(0, 0, 1)
        torch.cuda.current_stream().wait_stream(s)
        if keep is not None:
            for t, k in zip((self.flat_g,) + tuple(self.table_grads or ()), keep):
                t.copy_(k)
        torch.cuda.synchronize()
        self._warm = True

    def _graph(self, slot: int, next_slot: Optional[int], parity: int, mode=(False, True)):
        key = (slot, next_slot, parity, mode)
        g = self.graphs.get(key)
        if g is None:
            lib = ops.N.load()
            n0 = lib.tt_launch_count()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=self.cap_stream):
                self._pipelined(slot, next_slot, parity, mode)
            self.graphs[key] = g
            self.graph_captures += 1
            self.kernel_launches_per_step = lib.tt_launch_count() - n0
            if self.world > 1 and self.xchg is None:
                if self.graph_opt is None:
                    self.graph_opt = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(self.graph_opt):
                        self._optimizer()
                self.kernel_launches_per_step += 2  # adam_advance + adam
        return g

    def start_epoch(self):
        """The reference's batch_idx restarts at 0 every epoch; a trailing partial window stays in the gradient
        buffers and is continued by the next epoch's first window.  train_epoch / train_epoch_device call this."""
        self.window.start_epoch()
        if self._loss_share is not None:
            self._loss_share.zero_()

    def _epoch_average(self, total: torch.Tensor, n: int) -> float:
        if self._loss_share is not None:
            total = self._loss_share.clone()
            if self._dist_ready():
                torch.distributed.all_reduce(total, group=self.pg)
        return float(total.item()) / n

    def prepare(self, n_slots: Optional[int] = None):
        """Captures the steady-state graphs of a round-robin schedule over the first `n_slots` token slots
        (step(s, (s + 1) % n_slots)), so no capture happens inside a timed region."""
        self.check_banks()
        n = n_slots or len(self.tok_slots)
        if not self.use_graph:
            return
        if not self._warm:
            self._warm_up()
        for mode in self.window.modes():
            for s_ in range(n):
                if self._whole_step():
                    self._graph(s_, None, self._parity, mode)  # whole-step graphs: no look-ahead, one workspace
                    continue
                nxt = (s_ + 1) % n
                for parity in ((s_ & 1,) if n % 2 == 0 else (0, 1)):
                    self._graph(s_, nxt, parity, mode)
        self.sync_ranks()  # capture time differs per rank: line the ranks up before the first exchanged step

    def step(self, slot: int = 0, next_slot: Optional[int] = None) -> torch.Tensor:
        """One micro-step on the tokens in the static buffers of `slot` (an optimiser step when it closes a window of
        accumulation_steps micro-batches; always, with a = 1); returns the loss as a device scalar — no host sync: the
        micro-batch's global loss, except on a data-parallel micro-step that does not close its window, which runs no
        exchange and returns this rank's share of the global loss (its hinge sum over the global batch size; the shares
        of all ranks add up to the global loss).  `next_slot`: slot holding the tokens of the FOLLOWING step (already
        resident); its pooled gather then runs beside this step and the following step(next_slot, ...) skips it."""
        if not self._warm:
            self._warm_up()
        if self.neg_bufs is not None and not self._neg_loaded[slot]:
            raise RuntimeError(f"FusedTrainer(in_batch_negatives=True): no negative indices were loaded for slot {slot} "
                               "(load_neg_index / DeviceTripletFeeder.assemble)")
        if self.row_bufs is not None and not self._rows_loaded[slot]:
            raise RuntimeError(f"FusedTrainer(pooled=...): no bank rows were loaded for slot {slot} "
                               "(load_rows / DeviceTripletFeeder.assemble)")
        if self.train_table:
            next_slot = None  # a trainable table changes between steps: its gather cannot run ahead of the update
        lib = ops.N.load()
        whole = self._whole_step()
        if whole:
            next_slot = None  # the gather of THIS step is part of the step's graph
            self._primed = slot
        if self._primed != slot:  # pipeline start (or a schedule change): this step's gather has not run yet
            # nothing is primed, so the workspace is free to choose: make it a function of the slot, which is what
            # prepare() captured for an even slot count (a restart must never land on an uncaptured graph key)
            self._parity = slot & 1
            self._fwd_bwd(slot, 1, self._parity)
        parity = self._parity
        mode = self.window.mode()
        if self.use_graph:
            self._graph(slot, next_slot, parity, mode).replay()
        else:
            n0 = lib.tt_launch_count()
            self._pipelined(slot, next_slot, parity, mode)
            self.kernel_launches_per_step = lib.tt_launch_count() - n0
        if self._loss_share is not None:  # before the all-reduce below sums the loss slot over the ranks
            self._loss_share += self.flat_g[self.n_param].double()
        close = mode[1]
        if self.world > 1 and self.xchg is None and close:
            torch.distributed.all_reduce(self.flat_g, group=self.pg)
            if self.use_graph:
                self.graph_opt.replay()
            else:
                self._optimizer()
                self.kernel_launches_per_step += 2
        self._primed = next_slot
        if next_slot is not None:
            self._parity ^= 1
        self.steps_done += 1
        self.window.advance()
        if not close:  # no exchange published a loss: this rank's term (the whole loss on one GPU)
            return self.flat_g[self.n_param]
        return self.loss_view[0]

    def train_epoch_device(self, feeder, log_every: int = 0) -> float:
        """One pass with batches assembled on the device (data.DeviceTripletFeeder): per step one assembly kernel for
        the NEXT batch, then the step graph — the host only launches."""
        steps = len(feeder)
        if steps == 0:
            raise ZeroDivisionError("FusedTrainer.train_epoch_device: not enough pairs for one batch")
        self.check_banks()
        feeder.start_epoch()
        self.start_epoch()
        total = torch.zeros((), dtype=torch.float64, device=self.device)
        n_slots = len(self.tok_slots)
        feeder.assemble(self, 0, 0)
        for i in range(steps):
            slot = i % n_slots if n_slots >= 2 else 0
            nslot = None
            if i + 1 < steps and n_slots >= 2:
                nslot = (i + 1) % n_slots
                feeder.assemble(self, nslot, i + 1)
            loss = self.step(slot, nslot)
            total += loss.double()
            if i + 1 < steps and n_slots < 2:
                feeder.assemble(self, 0, i + 1)
            if log_every and (i + 1) % log_every == 0:
                if self.rank == 0:
                    print(f"Batch {i + 1}, Loss: {loss.item():.4f}")
                self.check()
        feeder.check()
        avg = self._epoch_average(total, steps)
        self.check()
        return avg

    # -- checkpoint / resume (main.py:142-152 saves `model.state_dict()`; this adds the optimiser so a run can resume) --
    def _slice_bounds(self, n: Optional[int] = None):
        """This rank's slice [lo, hi) of an exchanged flat buffer of n parameters (tt_dp_segment_bytes' layout)."""
        n = self.n_param if n is None else n
        per = (n + 1 + self.world - 1) // self.world
        S = (per + 63) // 64 * 64
        return min(self.rank * S, n), min((self.rank + 1) * S, n)

    def state_dict(self) -> dict:
        """Model weights (reference key names) + Adam moments and step count.  Collective in peer mode with
        world_size > 1 (the moments are sharded over the ranks there).  Inside an open accumulation window it also holds
        the window: "accumulation_steps", "window_batch_idx", "window_pending" and the gradient buffers ("window_grad",
        and "window_table_grads" when the tables train).  Data parallel, every rank's partial gradient differs, so a
        save inside a window raises there."""
        if self.window.pending and self.world > 1:
            raise RuntimeError(f"FusedTrainer.state_dict: {self.window.pending} micro-batches of an accumulation "
                               "window are pending and every rank's partial gradient differs; save at a window "
                               f"boundary (after a micro-step with (batch_idx + 1) % {self.accum} == 0)")
        m, v = self.exp_avg.clone(), self.exp_avg_sq.clone()
        if self.xchg is not None and self.world > 1:
            torch.distributed.all_reduce(m, group=self.pg)   # every rank holds zeros outside its own slice
            torch.distributed.all_reduce(v, group=self.pg)
        st = self.xchg.state if self.xchg is not None else self.adam_state
        sd = {"model": {k: t.detach().cpu().clone() for k, t in self.model.state_dict().items()},
              "exp_avg": m.cpu(), "exp_avg_sq": v.cpu(), "adam_state": st.detach().cpu().clone(),
              "steps_done": self.steps_done, "lr": self.lr, "betas": tuple(self.betas), "eps": self.eps}
        if self.window.pending:
            sd.update(accumulation_steps=self.accum, window_batch_idx=self.window.batch_idx,
                      window_pending=self.window.pending, window_grad=self.flat_g[: self.n_param].cpu().clone())
            if self.table_grads is not None:
                sd["window_table_grads"] = tuple(t.cpu().clone() for t in self.table_grads)
        if self.optimize_tables:
            tm, tv = self._table_m.clone(), self._table_v.clone()
            if self.txchg is not None and self.world > 1:
                torch.distributed.all_reduce(tm, group=self.pg)   # sharded like exp_avg
                torch.distributed.all_reduce(tv, group=self.pg)
            nt = self.n_table // 2
            shape = self.table_exp_avg[0].shape
            sd["table_exp_avg"] = (tm[:nt].view(shape).cpu(), tm[nt:].view(shape).cpu())
            sd["table_exp_avg_sq"] = (tv[:nt].view(shape).cpu(), tv[nt:].view(shape).cpu())
            if self.txchg is not None:
                sd["table_adam_state"] = self.txchg.state.detach().cpu().clone()
        return sd

    def load_state_dict(self, sd: dict):
        pending = int(sd.get("window_pending", 0))
        if pending:
            if int(sd["accumulation_steps"]) != self.accum:
                raise ValueError(f"FusedTrainer.load_state_dict: the checkpoint was saved inside a window of "
                                 f"accumulation_steps = {sd['accumulation_steps']}, this trainer has {self.accum}")
            if self.world > 1:
                raise ValueError("FusedTrainer.load_state_dict: a checkpoint inside an accumulation window holds one "
                                 "rank's partial gradient; data-parallel training resumes at window boundaries only")
            if ("window_table_grads" in sd) != (self.table_grads is not None):
                raise ValueError("FusedTrainer.load_state_dict: the checkpoint's open window and this trainer disagree "
                                 "on whether the token tables train")
        if self.optimize_tables and "table_exp_avg" not in sd:
            raise ValueError("FusedTrainer.load_state_dict: this trainer optimises the token tables, the checkpoint holds "
                             "no table moments (it was saved without optimize_tables)")
        model_sd = sd["model"]
        if self.pooled is not None:
            # The pooled banks were computed from the frozen backbone and are keyed to its tensors' versions: copying the
            # backbone in place, even with equal values, would make them stale.  A checkpoint of this training run holds
            # the same backbone, so equal tensors are left untouched; a different backbone would need new banks.
            cur = self.model.state_dict()
            frozen = [k for k in model_sd if k.split(".", 2)[1:2] == ["pretrained_model"]]
            differ = [k for k in frozen if k not in cur or not torch.equal(cur[k].cpu(), model_sd[k].cpu())]
            if differ:
                raise RuntimeError(f"FusedTrainer(pooled=...): the checkpoint's backbone differs from the model's "
                                   f"({len(differ)} tensors, e.g. {differ[0]}); the pooled banks would be stale. Load it "
                                   "into the model first, rebuild the banks with PooledBank.build() and a new trainer")
            model_sd = {k: v for k, v in model_sd.items() if k not in set(frozen)}
            missing, unexpected = self.model.load_state_dict(model_sd, strict=False)
            if unexpected or set(missing) - set(frozen):
                raise RuntimeError(f"FusedTrainer.load_state_dict: missing keys {sorted(set(missing) - set(frozen))}, "
                                   f"unexpected keys {sorted(unexpected)}")
        else:
            self.model.load_state_dict(model_sd)  # in-place copies: the parameters keep aliasing the flat buffer
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        if self.xchg is not None:
            lo, hi = self._slice_bounds()
            for t in (self.exp_avg, self.exp_avg_sq):  # keep the "zeros outside my slice" invariant
                t[:lo].zero_()
                t[hi:].zero_()
            self.xchg.state.copy_(sd["adam_state"])
        else:
            self.adam_state.copy_(sd["adam_state"])
        if self.optimize_tables:
            for dst, src in ((self.table_exp_avg, sd["table_exp_avg"]), (self.table_exp_avg_sq, sd["table_exp_avg_sq"])):
                for t, x in zip(dst, src):
                    t.copy_(x)
            if self.txchg is not None:
                lo, hi = self._slice_bounds(self.n_table)
                for t in (self._table_m, self._table_v):
                    t[:lo].zero_()
                    t[hi:].zero_()
                self.txchg.state.copy_(sd.get("table_adam_state", sd["adam_state"]))
        self.steps_done = int(sd.get("steps_done", 0))
        # a checkpoint without an open window resumes at a window start
        self.window.pending = pending
        self.window.batch_idx = int(sd["window_batch_idx"]) if pending else 0
        if pending:
            self.flat_g[: self.n_param].copy_(sd["window_grad"])
            for t, src in zip(self.table_grads or (), sd.get("window_table_grads", ())):
                t.copy_(src)
        self._primed = None
        self._sync_initial_state()

    def save_checkpoint(self, path: str):
        sd = self.state_dict()
        if self.rank == 0:
            torch.save(sd, path)
        self.sync_ranks()  # rank 0 was busy writing: nobody enters the next exchange before it is back

    def load_checkpoint(self, path: str):
        self.load_state_dict(torch.load(path, map_location="cpu", weights_only=False))

    def close(self):
        """Releases the peer segment (collective in peer mode: call on every rank after a barrier)."""
        if self.xchg is not None:
            torch.cuda.synchronize()
            self.xchg.check()
            # parameters move back to ordinary torch memory so the model outlives the segment
            with torch.no_grad():
                keep = self.flat_p.clone()
                off = 0
                for p in self.model.projection_parameters():
                    p.data = keep[off: off + p.numel()].view_as(p)
                    off += p.numel()
            self.flat_p = keep
            self.loss_view = self.loss_view.clone()
            self.xchg.close()
            self.xchg = None
            if self.txchg is not None:  # and the trained tables out of theirs
                self.txchg.check()
                with torch.no_grad():
                    keep = self.txchg.flat_p.clone()
                    nt = self.n_table // 2
                    for i, t in enumerate((self.model.query_tower.pretrained_model.table,
                                           self.model.document_tower.pretrained_model.table)):
                        t.data = keep[i * nt: (i + 1) * nt].view_as(t)
                self.txchg.close()
                self.txchg = None
            self.exchange = "closed"

    def train_epoch(self, loader: TokenTripletLoader, log_every: int = 0) -> float:
        """One pass over the loader.  With >= 2 token slots the next batch is staged one step ahead so that its
        pooled gather overlaps the current step."""
        self.check_banks()
        self.start_epoch()
        total = torch.zeros((), dtype=torch.float64, device=self.device)
        nb = 0
        n_slots = len(self.tok_slots)
        it = iter(loader)
        cur = next(it, None)
        if cur is None:
            raise ZeroDivisionError("FusedTrainer.train_epoch: empty loader")
        slot = 0
        self._load(cur, slot)
        while cur is not None:
            nxt = next(it, None)
            nslot = None
            if nxt is not None and n_slots >= 2 and len(nxt[0]) == self.B:
                nslot = (slot + 1) % n_slots
                self._load(nxt, nslot)
            loss = self.step(slot, nslot)
            total += loss.double()
            nb += 1
            if log_every and nb % log_every == 0:
                if self.rank == 0:
                    print(f"Batch {nb}, Loss: {loss.item():.4f}")
                self.check()
            if nxt is not None and nslot is None:
                self._load(nxt, slot)
            else:
                slot = nslot if nslot is not None else slot
            cur = nxt
        avg = self._epoch_average(total, nb)
        self.check()
        return avg


# --------------------------------------------------------------------------------------------------
# evaluation (training.py:136-380)
# --------------------------------------------------------------------------------------------------
_K_SCAN = 16  # candidates kept per query (>= 10) so ties at the top-10 boundary are visible


def _tie_averaged_ndcg(rel: np.ndarray, score: np.ndarray, k: int) -> float:
    """sklearn.metrics.ndcg_score semantics for one query (default ignore_ties=False), used only when a
    tie reaches past the scanned candidates.  Tie groups share the mean gain of their ranks."""
    n = len(rel)
    disc = 1.0 / np.log2(np.arange(n) + 2.0)
    disc[k:] = 0.0
    order = np.argsort(-score, kind="stable")
    s_sorted, r_sorted = score[order], rel[order].astype(np.float64)
    dcg, i = 0.0, 0
    while i < n and i < k:
        j = i
        while j + 1 < n and s_sorted[j + 1] == s_sorted[i]:
            j += 1
        dcg += r_sorted[i: j + 1].mean() * disc[i: j + 1].sum()
        i = j + 1
    ideal = float((np.sort(rel)[::-1].astype(np.float64) * disc).sum())
    return 0.0 if ideal == 0 else dcg / ideal


def _ndcg_from_lists(top_s: np.ndarray, top_i: np.ndarray, relevant: set, n_rel_in_pool: int, k: int,
                     exact_fallback) -> float:
    """NDCG@k of one query from its best _K_SCAN (score,id) pairs; tie groups inside the list are averaged
    exactly; a tie group that runs off the end of the list triggers `exact_fallback()`."""
    m = int((top_i >= 0).sum())
    if m > k and top_s[m - 1] == top_s[k - 1] and m == len(top_i):
        return exact_fallback()
    gains = np.array([1.0 if int(d) in relevant else 0.0 for d in top_i[:m]])
    disc = np.zeros(m)
    disc[: min(k, m)] = 1.0 / np.log2(np.arange(min(k, m)) + 2.0)
    dcg, i = 0.0, 0
    while i < m and i < k:
        j = i
        while j + 1 < m and top_s[j + 1] == top_s[i]:
            j += 1
        dcg += gains[i: j + 1].mean() * disc[i: j + 1].sum()
        i = j + 1
    idcg = float((1.0 / np.log2(np.arange(min(n_rel_in_pool, k)) + 2.0)).sum())
    return 0.0 if idcg == 0 else dcg / idcg


def _dist_info():
    """(world_size, rank) of the default process group, (1, 0) without one."""
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


def _eval_plan(dataset, sample_size: int, min_query_groups: int, candidate_pool_size: int, say=print) -> dict:
    """Host part of evaluate_model (training.py:184-279): sample + group by query_id until enough unique queries
    (same `random` call sequence as the reference), keep the queries with most relevant documents, and build the
    per-query candidate pools.  Pure Python on strings — under data parallelism rank 0 runs it and broadcasts the
    result, so that every rank scores the same queries against the same pools."""
    query_groups: dict[int, dict] = {}
    sample_multiplier = 1
    say(f"Grouping data by queries (target: {min_query_groups} unique queries)...")
    while len(query_groups) < min_query_groups and sample_multiplier <= 10:
        sample_size_current = min(sample_size * sample_multiplier, len(dataset))
        for i in random.sample(range(len(dataset)), sample_size_current):
            item = dataset[i]
            group = query_groups.setdefault(item["query_id"], {"query": item["query"], "relevant_docs": {}})
            group["relevant_docs"].setdefault(item["positive"], None)  # insertion-ordered set
        sample_multiplier += 1
    query_ids = sorted(query_groups, key=lambda qid: len(query_groups[qid]["relevant_docs"]), reverse=True)
    query_ids = query_ids[:min_query_groups]
    if not query_ids:
        raise ZeroDivisionError("evaluate_model: no queries to evaluate")
    rel_docs = [list(query_groups[q]["relevant_docs"]) for q in query_ids]
    cand_docs = None
    if candidate_pool_size != -1:
        cand_docs = []
        for qi, q in enumerate(query_ids):
            rel = query_groups[q]["relevant_docs"]
            # irrelevant = every other selected query's relevant docs (training.py:255-261); sorted so a
            # seeded run is reproducible (the reference's order depends on PYTHONHASHSEED)
            irrelevant = sorted({d for o in query_ids if o != q for d in query_groups[o]["relevant_docs"] if d not in rel})
            if len(irrelevant) > candidate_pool_size:
                irrelevant = random.sample(irrelevant, candidate_pool_size)
            cand_docs.append(rel_docs[qi] + irrelevant)
            if len(cand_docs[-1]) <= 1:
                raise ValueError("Computing NDCG is only meaningful when there is more than 1 document.")
    return {"queries": [query_groups[q]["query"] for q in query_ids], "rel_docs": rel_docs, "cand_docs": cand_docs}


def _gather_rows(t: torch.Tensor, world: int) -> torch.Tensor:
    """Concatenates per-rank row blocks of different heights ([n_r, ...] -> [sum n_r, ...], rank order) on every
    rank: one all-gather of the heights, one of the blocks padded to the tallest."""
    import torch.distributed as dist

    n = torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device)
    ns = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(ns, n)
    ns = [int(x.item()) for x in ns]
    top = max(ns)
    pad = torch.zeros((top,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    pad[: t.shape[0]] = t
    parts = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(parts, pad)
    return torch.cat([p_[:k] for p_, k in zip(parts, ns)], dim=0)


def evaluate_model(
    model: TwoTowersModel,
    dataset,
    sample_size: int = 200,
    min_query_groups: int = 20,
    candidate_pool_size: int = 100,
    comprehensive: bool = False,
    log_wandb: bool = False,
    wandb_prefix: str = "final_",
    batch_size: int = 1024,
) -> Union[float, dict[str, float]]:
    """NDCG evaluation with all relevant documents per query (training.py:136-380): same sampling, same
    candidate pools, same metrics and return type; scoring is one batched device pass instead of a per-query
    CPU cosine + sklearn call.

    Under torch.distributed (one process per GPU) the document universe is sharded over the ranks
    (retrieval.shard_bounds): each rank encodes ITS documents with `encode_documents_batched` — no collective —
    scans its own shard, and the per-shard top lists meet in one all-gather + tt_topk_merge (SURVEY.md §8e); the
    small validation pools gather the shard embeddings instead.  Every rank returns the same value; rank 0 prints."""
    world, rank = _dist_info()
    say = print if rank == 0 else (lambda *a, **k: None)
    say(f"Sampling documents for evaluation (initial sample size: {sample_size})...")
    model.eval()
    clear_gpu_memory()

    if world > 1:  # one plan for everybody (the sampling uses the process-local `random` state)
        import torch.distributed as dist

        box = [_eval_plan(dataset, sample_size, min_query_groups, candidate_pool_size, say) if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        plan = box[0]
    else:
        plan = _eval_plan(dataset, sample_size, min_query_groups, candidate_pool_size, say)
    queries, rel_docs, cand_docs = plan["queries"], plan["rel_docs"], plan["cand_docs"]
    n_q = len(queries)
    total_relevant_docs = sum(len(r) for r in rel_docs)
    avg_relevant_per_query = total_relevant_docs / n_q
    say(f"Selected {n_q} queries for evaluation")
    say(f"  Total relevant documents across these queries: {total_relevant_docs}")
    say(f"  Average relevant docs per query: {avg_relevant_per_query:.2f}")

    # document universe and per-query candidate lists
    full_pool = candidate_pool_size == -1
    if full_pool:
        say("🚀 Pre-encoding *all* documents for efficiency (this may take a moment)...")
        universe = list(dataset.get_unique_passages())
        if world > 1:
            universe = sorted(universe)  # a set-ordered list differs between processes: ids must mean the same everywhere
    else:
        universe = list(dict.fromkeys(d for r in rel_docs for d in r))
    doc_index = {d: i for i, d in enumerate(universe)}
    if len(universe) <= 1:
        raise ValueError("Computing NDCG is only meaningful when there is more than 1 document.")
    cand_lists = None if full_pool else [[doc_index[d] for d in c] for c in cand_docs]
    lo, hi = retrieval.shard_bounds(len(universe), world, rank)

    with torch.no_grad():
        query_embeds = model.encode_queries(queries)
        dev = query_embeds.device
        if hi > lo:
            doc_embeds = model.encode_documents_batched(universe[lo:hi], batch_size=batch_size)  # this rank's shard
        else:
            doc_embeds = torch.zeros(0, query_embeds.shape[1], dtype=torch.float32, device=dev)
        if full_pool:
            say(f"🔥 Pre-encoded {len(universe)} documents to reuse for all queries")
        Dn = ops.l2_normalize_rows(doc_embeds)  # per-vector clamp of torch.cosine_similarity (training.py:297)
        Qn = ops.l2_normalize_rows(query_embeds)
        if full_pool:
            kk = min(_K_SCAN, len(universe))
            top_s, top_i = ops.scan_topk(Qn, Dn, k=kk, id_base=lo, precision="fp32")
            top_s, top_i = retrieval.gather_and_merge(top_s, top_i, world)
            pool_sizes = [len(universe)] * n_q
        else:
            if world > 1:  # small pools: every rank scores all queries against the gathered shard embeddings
                Dn = _gather_rows(Dn, world)
            C = max(len(c) for c in cand_lists)
            cand = torch.full((len(cand_lists), C), -1, dtype=torch.int64)
            for r, c in enumerate(cand_lists):
                cand[r, : len(c)] = torch.tensor(c, dtype=torch.int64)
            cand = cand.to(dev)
            kk = min(_K_SCAN, C)
            top_s, top_i = ops.score_candidates(Qn, Dn, cand, k=kk)
            pool_sizes = [len(c) for c in cand_lists]
        # NDCG on the device (tie-free closed form) ...
        rel_lists = [sorted(doc_index[d] for d in r if d in doc_index) for r in rel_docs]
        offs = torch.tensor(np.concatenate([[0], np.cumsum([len(r) for r in rel_lists])]), dtype=torch.int64, device=dev)
        rel_flat = torch.tensor([d for r in rel_lists for d in r], dtype=torch.int64, device=dev)
        ks = (10, 5, 1) if comprehensive else (10,)
        dev_ndcg = {k: ops.ndcg_at_k(top_i, offs, rel_flat, kk=min(k, kk)).cpu().numpy() for k in ks}
        top_s_h, top_i_h = top_s.cpu().numpy(), top_i.cpu().numpy()

    # ... and exact tie handling for the (rare) queries whose best scores tie past the scanned list.  The merged lists
    # are identical on every rank, so all ranks take this path for the same queries (it is collective when sharded).
    def exact(qi: int, k: int) -> float:
        if full_pool:
            sc = ops.candidate_scores(Qn[qi: qi + 1], Dn, np.arange(hi - lo)) if hi > lo else np.zeros(0, np.float32)
            if world > 1:
                sc = _gather_rows(torch.from_numpy(sc).to(dev), world).cpu().numpy()
            idx = np.arange(len(universe))
        else:
            idx = np.array(cand_lists[qi])
            sc = ops.candidate_scores(Qn[qi: qi + 1], Dn, idx)
        rel_set_q = set(rel_lists[qi])
        rel = np.array([1 if int(d) in rel_set_q else 0 for d in idx])
        return _tie_averaged_ndcg(rel, sc, k)

    scores = {k: [] for k in ks}
    for qi in range(n_q):
        m = int((top_i_h[qi] >= 0).sum())
        has_tie = bool((np.diff(top_s_h[qi][:m]) == 0).any()) if m > 1 else False
        rel_set = set(rel_lists[qi])
        n_rel = len(rel_set)
        for k in ks:
            if not has_tie:
                scores[k].append(float(dev_ndcg[k][qi]))
            else:
                scores[k].append(_ndcg_from_lists(top_s_h[qi], top_i_h[qi], rel_set, n_rel, k,
                                                  lambda qi=qi, k=k: exact(qi, k)))
        if qi == 0:
            say("\nSample evaluation results:")
            say(f"Query: {queries[0]}")
            say(f"Number of relevant docs: {len(rel_set)}")
            say(f"Number of candidate docs: {pool_sizes[0]}")
            say(f"NDCG@10 score for this query: {scores[10][0]:.4f}")
            say("Top 10 ranked documents:")
            for rank_, d in enumerate(top_i_h[0][:10]):
                if d < 0:
                    break
                tag = "RELEVANT" if int(d) in rel_set else "irrelevant"
                text = str(universe[int(d)])
                say(f"  {rank_ + 1}. [{tag}] {text[:100] + '...' if len(text) > 100 else text}")

    mean_ndcg_10 = float(np.mean(scores[10]))
    if not comprehensive:
        say(f"\nMean NDCG@10 across {n_q} queries: {mean_ndcg_10:.4f}")
        return mean_ndcg_10
    results = {
        f"{wandb_prefix}ndcg_10": mean_ndcg_10,
        f"{wandb_prefix}ndcg_5": float(np.mean(scores[5])),
        f"{wandb_prefix}ndcg_1": float(np.mean(scores[1])),
        f"{wandb_prefix}ndcg_10_std": float(np.std(scores[10])),
        f"{wandb_prefix}queries_evaluated": n_q,
        f"{wandb_prefix}total_relevant_docs": total_relevant_docs,
        f"{wandb_prefix}avg_relevant_per_query": avg_relevant_per_query,
    }
    say("\n" + "=" * 60)
    say("COMPREHENSIVE EVALUATION RESULTS")
    say("=" * 60)
    say("📊 Performance Metrics:")
    say(f"   NDCG@1:  {results[f'{wandb_prefix}ndcg_1']:.4f}")
    say(f"   NDCG@5:  {results[f'{wandb_prefix}ndcg_5']:.4f}")
    say(f"   NDCG@10: {results[f'{wandb_prefix}ndcg_10']:.4f} (±{results[f'{wandb_prefix}ndcg_10_std']:.4f})")
    say("\n📈 Evaluation Set Coverage:")
    say(f"   Queries evaluated: {results[f'{wandb_prefix}queries_evaluated']}")
    say(f"   Total relevant documents: {results[f'{wandb_prefix}total_relevant_docs']}")
    say(f"   Avg relevant docs/query: {results[f'{wandb_prefix}avg_relevant_per_query']:.2f}")
    if log_wandb and wandb is not None and rank == 0:
        wandb.log(results)
        say("\n✅ Comprehensive test results logged to wandb")
    return results


# --------------------------------------------------------------------------------------------------
# run driver (training.py:383-529)
# --------------------------------------------------------------------------------------------------
def hard_negative_config(hard_negatives: Union[None, int, dict]) -> Optional[dict]:
    """run_training(hard_negatives=...) -> None (off) or {"miner": HardNegativeMiner kwargs, "warmup_epochs": n}.
    None reads TT_HARD_NEGATIVES (unset / 0 = off, an integer d = depth d)."""
    if hard_negatives is None:
        env = os.environ.get("TT_HARD_NEGATIVES", "0").strip() or "0"
        try:
            hard_negatives = int(env)
        except ValueError:
            raise ValueError(f"TT_HARD_NEGATIVES must be an integer depth (0 = off), got {env!r}") from None
    if isinstance(hard_negatives, bool) or not isinstance(hard_negatives, (int, dict)):
        raise ValueError(f"hard_negatives must be None, an integer depth or a dict, got {hard_negatives!r}")
    if isinstance(hard_negatives, int):
        if hard_negatives < 0:
            raise ValueError(f"hard_negatives depth must be >= 0, got {hard_negatives}")
        hard_negatives = {"depth": hard_negatives} if hard_negatives else None
    if hard_negatives is None:
        return None
    kw = dict(hard_negatives)
    warmup = int(kw.pop("warmup_epochs", 1))
    if warmup < 0:
        raise ValueError(f"warmup_epochs must be >= 0, got {warmup}")
    allowed = {"depth", "skip", "ratio", "k_scan"}
    if set(kw) - allowed:
        raise ValueError(f"hard_negatives: unknown keys {sorted(set(kw) - allowed)} (allowed: {sorted(allowed)} and "
                         "warmup_epochs)")
    d = dict(depth=8, skip=0, ratio=0.5, k_scan=32)
    d.update(kw)
    HardNegativeMiner.check_config(**d)
    return {"miner": kw, "warmup_epochs": warmup}


def train_table_config(train_table: Optional[bool]) -> bool:
    """run_training(train_table=...) -> bool.  None reads TT_TRAIN_TABLE (unset / 0 = off, 1 = on)."""
    if train_table is None:
        env = os.environ.get("TT_TRAIN_TABLE", "0").strip() or "0"
        if env not in ("0", "1"):
            raise ValueError(f"TT_TRAIN_TABLE must be 0 or 1, got {env!r}")
        return env == "1"
    return bool(train_table)


def run_training(
    num_epochs: int = 3,
    batch_size: int = 1024,
    learning_rate: float = 1e-4,
    max_samples: int = 10000,
    projection_dim: int = 128,
    margin: float = 0.1,
    project_name: str = "two-towers-retrieval",
    use_wandb: bool = True,
    wandb_config: Optional[dict] = None,
    accumulation_steps: int = 2,
    use_mixed_precision: bool = True,
    num_workers: int = 4,
    run_comprehensive_test: bool = True,
    fused: Optional[bool] = None,
    table_dtype: torch.dtype = torch.float32,
    backbone: Optional[str] = None,
    hard_negatives: Union[None, int, dict] = None,
    fused_accumulation: Optional[bool] = None,
    train_table: Optional[bool] = None,
) -> TwoTowersModel:
    """Main training function (training.py:383-529).  `fused` (additive) selects the FusedTrainer; by
    default it is used whenever the dataset is token-bank backed and no gradient accumulation / wandb
    gradient hooks require the reference-shaped loop.

    `backbone` (additive): "table" (the token-table backbone) or "minilm" (the reference's frozen MiniLM encoder);
    None reads the TT_BACKBONE environment variable, default "table", so an unmodified main.py can choose.  On the
    fused path a MiniLM model encodes every text of the training split once into pooled banks (data.PooledBank) and
    trains the projections on rows gathered from them; otherwise it runs the reference-shaped loop.

    `hard_negatives` (additive): mined negatives on the fused path with the device feeder (data.HardNegativeMiner).
    None reads TT_HARD_NEGATIVES (unset or 0 = off, the default; an integer d = on with depth d); an int d is the same;
    a dict holds the miner's arguments plus "warmup_epochs" (default 1).  After warmup_epochs epochs of in-batch
    negatives the table is re-mined from the current towers at the start of every epoch.

    `fused_accumulation` (additive): honour `accumulation_steps` on the fused path (FusedTrainer(accumulation_steps=a):
    micro-batches add into the flat gradient, one optimiser step and, data parallel, one exchange per window).  None
    reads TT_FUSED_ACCUMULATION (unset or 0 = off, the default).  Off, one GPU takes the fused path only at
    accumulation_steps == 1 and data-parallel runs step every global batch.

    `train_table` (additive): train both token tables with the projections (TwoTowersModel(train_table=True), every
    parameter under one torch.optim.Adam step count).  None reads TT_TRAIN_TABLE (unset or 0 = off, the default; 1 =
    on).  The fused path runs FusedTrainer(optimize_tables=True), the reference-shaped loops
    torch.optim.Adam(model.parameters()).  Needs the token-table backbone with fp32 tables and no hard negatives."""
    if isinstance(accumulation_steps, bool) or not isinstance(accumulation_steps, int) or accumulation_steps < 1:
        raise ValueError(f"accumulation_steps must be an integer >= 1, got {accumulation_steps!r}")
    if fused_accumulation is None:
        env = os.environ.get("TT_FUSED_ACCUMULATION", "0").strip() or "0"
        try:
            fused_accumulation = int(env) != 0
        except ValueError:
            raise ValueError(f"TT_FUSED_ACCUMULATION must be 0 or 1, got {env!r}") from None
    hn = hard_negative_config(hard_negatives)
    if backbone is None:
        backbone = os.environ.get("TT_BACKBONE", "table")
    if backbone not in ("table", "minilm"):
        raise ValueError(f"backbone must be 'table' or 'minilm', got {backbone!r}")
    train_table = train_table_config(train_table)
    if train_table:
        if backbone == "minilm":
            raise ValueError("train_table needs the token-table backbone: the MiniLM backbone is frozen (model.py:28-30) "
                             "and has no token table")
        if hn is not None:
            raise ValueError("train_table and hard negatives are exclusive: the miner's pooled banks come from the frozen "
                             "table and would go stale at the first step")
        if table_dtype != torch.float32:
            raise ValueError(f"train_table needs fp32 token tables, got table_dtype={table_dtype} (bf16 tables do not "
                             "train)")
    # one process per GPU under torchrun / torch.distributed.run (SURVEY.md §8e): `batch_size` is the GLOBAL batch,
    # every rank trains on its contiguous slice and evaluates its shard of the documents
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    say = print if rank == 0 else (lambda *a, **k: None)
    say("Initializing model and data...")
    if not torch.cuda.is_available():
        raise RuntimeError("two-towers-overlords_b200 needs a CUDA (sm_100a) device; there is no CPU path")
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        device = torch.device("cuda", local_rank)
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=device)
        if batch_size % world != 0:
            raise ValueError(f"batch_size {batch_size} (the global batch) must be a multiple of WORLD_SIZE {world}")
    else:
        device = torch.device("cuda")
    say(f"Using device: {device}")
    say(f"GPU: {torch.cuda.get_device_name(device)}")
    say(f"Memory: {torch.cuda.get_device_properties(device).total_memory / 1e9:.1f}GB")
    if world > 1:
        say(f"Data parallel over {world} GPUs: global batch {batch_size}, {batch_size // world} triplets per GPU")

    use_wandb = bool(use_wandb and wandb is not None and rank == 0)
    if use_wandb:
        config = {
            "epochs": num_epochs, "batch_size": batch_size, "learning_rate": learning_rate,
            "max_samples": max_samples, "model_name": "sentence-transformers/all-MiniLM-L6-v2",
            "loss_function": "triplet_loss", "distance_metric": "cosine", "margin": margin,
            "dataset_type": "ms_marco_all_passages", "device": str(device),
            "device_name": torch.cuda.get_device_name(device),
        }
        if wandb_config:
            config.update(wandb_config)
        if not wandb.run:
            wandb.init(project=project_name, config=config)

    if backbone == "minilm":
        model = TwoTowersModel(projection_dim=projection_dim, backbone="minilm").to(device)
    else:
        model = TwoTowersModel(projection_dim=projection_dim, table_dtype=table_dtype, train_table=train_table).to(device)
    if world > 1:  # random-init tables and projections are drawn per process: rank 0's become everybody's
        for t in list(model.parameters()) + list(model.buffers()):
            dist.broadcast(t.data, src=0)
    criterion = TripletLoss(margin=margin)
    optimizer = torch.optim.Adam(model.parameters(), lr=learning_rate)
    if train_table:
        say(f"Trainable parameters: {sum(p.numel() for p in model.parameters() if p.requires_grad):,} "
            "(token tables included)")
    if use_wandb:
        if world == 1:
            wandb.watch(model, log="all", log_freq=100)
        wandb.log({"total_parameters": sum(p.numel() for p in model.parameters())})

    train_ds = MSMarcoDataset("train", max_samples=max_samples)
    val_ds = MSMarcoDataset("validation", max_samples=1000)

    def use_bank_tokenizer(ds, *more):
        tok = ds.tokenizer() if hasattr(ds, "tokenizer") else None
        if tok is not None:
            for d in more:
                tok.add(d.tokenizer())
            model.query_tower.tokenizer = model.document_tower.tokenizer = tok
        return tok

    bank_backed = use_bank_tokenizer(train_ds, val_ds) is not None
    train_dl = TripletDataLoader(train_ds, batch_size=batch_size, num_workers=num_workers, device=device)
    if fused is None:
        # one GPU: the reference-shaped loops serve wandb's gradient hooks and, unless fused_accumulation, gradient
        # accumulation; several GPUs: only the fused step exchanges gradients, so it is the path
        fused = bank_backed and (world > 1 or ((accumulation_steps == 1 or fused_accumulation) and not use_wandb))
    if world > 1 and not fused:
        raise ValueError("data-parallel training needs the fused step (a token-bank dataset and fused != False)")
    host_feeder = os.environ.get("TT_HOST_FEEDER") == "1" or len(train_ds) < 2 * batch_size
    if hn is not None and (not fused or host_feeder):
        raise ValueError("hard negatives need the fused step with the device feeder (DeviceTripletFeeder); the "
                         "reference-shaped loops and TokenTripletLoader draw in-batch negatives only (unset "
                         "TT_HOST_FEEDER, use at least two batches of pairs)")
    # micro-batches per optimiser step of the fused trainer
    fused_accum = accumulation_steps if fused_accumulation else 1
    if fused and accumulation_steps != 1 and not fused_accumulation:
        say(f"  note: accumulation_steps={accumulation_steps} is ignored by the fused step (TT_FUSED_ACCUMULATION=1 "
            f"honours it); the batch of {batch_size} triplets is one optimiser step")

    say("Training configuration:")
    say(f"  Physical batch size: {batch_size}")
    say(f"  Gradient accumulation steps: {accumulation_steps}")
    say(f"  Effective batch size: {batch_size * (fused_accum if fused else accumulation_steps)}")
    say(f"  Mixed precision: {use_mixed_precision}")
    say(f"  DataLoader workers: {num_workers}")
    say(f"  Fused B200 step: {fused}")

    scaler = GradScaler(device.type) if use_mixed_precision else None
    trainer = token_dl = feeder = miner = None
    if fused:
        seed_box = [random.randrange(2 ** 31)]
        if world > 1:  # the epoch permutation and the in-batch negatives are functions of this seed: share rank 0's
            dist.broadcast_object_list(seed_box, src=0)
        if backbone == "minilm":
            # the frozen encoder runs once per training text, not three times per triplet and step
            t0 = time.perf_counter()
            Lq, Ld = 32, 256  # FusedTrainer's token lengths
            banks = (PooledBank.build(model.query_tower, train_ds.query_bank, Lq, world_size=world, rank=rank),
                     PooledBank.build(model.document_tower, train_ds.doc_bank, Ld, world_size=world, rank=rank))
            torch.cuda.synchronize()
            say(f"Encoded {len(banks[0]) + len(banks[1])} training texts ({len(banks[0])} queries, "
                f"{len(banks[1])} passages) with the frozen MiniLM backbone in {time.perf_counter() - t0:.1f}s")
            trainer = FusedTrainer(model, margin, learning_rate, batch_size // world, Lq, Ld, token_slots=2,
                                   world_size=world, rank=rank, pooled=banks, accumulation_steps=fused_accum)
        else:
            # the device feeder draws the in-batch negatives itself and hands their indices to the trainer, which then
            # pools every positive document once, and with trainable tables scatter-adds its tokens once (TT_NEG_REUSE=0:
            # gather the negatives' tokens like any document)
            reuse = not host_feeder and world == 1 and os.environ.get("TT_NEG_REUSE", "1") != "0"
            if hn is not None:
                reuse = False
                say("  Hard negatives: neg-index reuse is off (a mined negative is not a positive of the batch)")
            trainer = FusedTrainer(model, margin, learning_rate, batch_size // world, token_slots=2, world_size=world,
                                   rank=rank, in_batch_negatives=reuse, accumulation_steps=fused_accum,
                                   optimize_tables=train_table)
            if hn is not None:  # the frozen table's pooled rows, for mining only (the step still pools tokens)
                banks = (PooledBank.build(model.query_tower, train_ds.query_bank, trainer.Lq, world_size=world,
                                          rank=rank),
                         PooledBank.build(model.document_tower, train_ds.doc_bank, trainer.Ld, world_size=world,
                                          rank=rank))
        if host_feeder:
            # host-assembled batches (negatives drawn over the global batch, this rank's slice)
            token_dl = TokenTripletLoader(train_ds, batch_size, trainer.Lq, trainer.Ld, rank=rank, world_size=world,
                                          seed=seed_box[0], rows=trainer.pooled is not None)
        else:  # token bank resident in HBM, batches (and in-batch negatives) assembled by one kernel per step
            feeder = DeviceTripletFeeder(train_ds, batch_size, trainer.Lq, trainer.Ld, device, rank=rank,
                                         world_size=world, seed=seed_box[0], rows_only=trainer.pooled is not None)
            if hn is not None:
                miner = HardNegativeMiner(train_ds, *banks, world_size=world, rank=rank, **hn["miner"])
                feeder.hard_negatives = miner
        trainer.prepare(2)

    say(f"Starting training for {num_epochs} epochs...")
    for epoch in range(num_epochs):
        say(f"\nEpoch {epoch + 1}/{num_epochs}")
        if miner is not None and epoch >= hn["warmup_epochs"]:
            st = miner.refresh(model)
            say(f"Hard negatives refreshed in {st['total_s'] * 1e3:.1f} ms (project {st['project_s'] * 1e3:.1f}, "
                f"normalize {st['normalize_s'] * 1e3:.1f}, scan {st['scan_s'] * 1e3:.1f}, merge "
                f"{st['merge_s'] * 1e3:.1f}, filter {st['filter_s'] * 1e3:.1f}): mean {st['mean_count']:.2f} of "
                f"{miner.depth} per query, {st['empty_queries']} queries without one")
        if trainer is not None and feeder is not None:
            avg_loss = trainer.train_epoch_device(feeder, log_every=10)
        elif trainer is not None:
            avg_loss = trainer.train_epoch(token_dl, log_every=10)
        elif use_mixed_precision and scaler is not None:
            avg_loss = train_epoch_optimized(model=model, dataloader=train_dl, criterion=criterion,
                                             optimizer=optimizer, device=device, scaler=scaler,
                                             accumulation_steps=accumulation_steps, log_wandb=use_wandb)
        else:
            avg_loss = train_epoch(model, train_dl, criterion, optimizer, log_wandb=use_wandb)
        say(f"Average training loss: {avg_loss:.4f}")
        ndcg = evaluate_model(model, val_ds, batch_size=batch_size)
        say(f"Validation NDCG@10: {ndcg:.4f}")
        if trainer is not None:
            trainer.sync_ranks()  # evaluation time differs per rank: line up before the next exchanged step
        if use_wandb:
            wandb.log({"epoch": epoch + 1, "avg_train_loss": avg_loss, "val_ndcg_10": ndcg})

    say("\n" + "=" * 60)
    if run_comprehensive_test:
        say("TRAINING COMPLETED - Starting comprehensive testing")
        say("=" * 60)
        test_dataset = MSMarcoDataset("test", max_samples=10_000)
        use_bank_tokenizer(train_ds, val_ds, test_dataset)
        _ = evaluate_model(model=model, dataset=test_dataset, min_query_groups=200, candidate_pool_size=-1,
                           comprehensive=True, log_wandb=use_wandb, batch_size=batch_size)
    else:
        say("TRAINING COMPLETED - Skipping comprehensive testing")
        say("=" * 60)
    if trainer is not None and world > 1:
        trainer.sync_ranks()
        trainer.close()  # parameters move out of the peer segment so the returned model outlives it
    if use_wandb:
        wandb.finish()
    return model
