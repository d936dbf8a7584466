"""The tensor-core training step (tt_triplet_step with `bf16x3` and single-pass `bf16`) against a float64 oracle at the
shapes where its tiling has tails, for both ways of launching the projection chain: the persistent chain kernel
(csrc/tt_chain_sm100.cu, `set_chain(1)`) and one kernel per contraction (csrc/tt_gemm_sm100.cu, `set_chain(2)`).

The persistent kernel cuts its work by shape: row tiles of 128 triplets (the last one partial when B % 128 != 0),
column tiles of 128 (the last one half empty when P % 128 == 64) and 64-column loss slots, weight-gradient chunks of
`kcb` k-blocks of 64 batch rows (the last chunk partial; `kcb` grows from 8 to 16 past 48 chunks), k-blocks of the
document tower that hold both positive and negative rows (B % 64 != 0).  A wrong guard on any of these tails gives a
subtly wrong gradient, so every case here checks, against float64:

  * the loss, the per-triplet statistics [B, 8] row by row, y and dY [3B, P] row by row (TT_CHAIN_FP32_OUT=1);
  * all 8 projection gradients over the whole tensor AND per 64 x 64 block (64 elements for a bias), so a wrong tail
    tile cannot hide in the norm of a large tensor;
  * that the diagnostic fp32 outputs leave the gradients bit-identical.

The oracle starts from the device's own pooled rows xhat (first checked against oracle.pooled_normalised; pooling is
tested elsewhere) and differentiates through the device's ReLU gate and hinge activity (see
tests/test_step_parity.py::oracle_grads for why); every disagreement must lie inside the rounding band of the
precision.  Tokens are short (Lq = 8, Ld = 24, shape "Z", some all-masked rows) over a 4096-token vocabulary: these
tests are about the projection chain."""
import os
from dataclasses import dataclass

import pytest
import torch

from oracle import two_towers_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda"
PRECISIONS = [p for p in os.environ.get("TT_TEST_PRECISIONS", "fp32,bf16x3").split(",") if p]
X3 = ["bf16x3"] if "bf16x3" in PRECISIONS else []
H = O.HIDDEN
VOCAB = 4096
CHAINS = {"persistent": 1, "kernels": 2}
COS_EPS = 1e-8    # torch.cosine_similarity eps (per-vector clamp), backend/model.py:134
KINK_BAND = 2e-6  # bf16x3: |pre-activation| below which the ReLU gate is undecided (tests/test_step_parity.py)

# Gates per precision: loss (relative), gradients (relative Frobenius over the whole tensor, and per block), y and dY
# rows (row-relative), statistics (cosines and hinge absolute, norms and dot products relative), hinge band (|pre-hinge|
# within which the device and float64 may disagree on whether a triplet is active).  Single-pass bf16: set from the
# worst values measured over this file on a B200 (see the report line each case prints) with a margin of at most 4x.
GATES = {
    "bf16x3": dict(loss=1e-4, grad=1e-3, block=3e-3, y=1e-4, dy=1e-3, stats=1e-4, hinge_band=1e-5),
    # worst measured (B200, 1000 W): loss 1.0e-5, gradients 2.1e-2 whole / 2.1e-2 per block, y 1.9e-3, dY 8.9e-3,
    # statistics 4.1e-4
    "bf16": dict(loss=4e-5, grad=3e-2, block=3e-2, y=5e-3, dy=3e-2, stats=1e-3, hinge_band=1.5e-3),
}
NAMES = ("Wq1", "bq1", "Wq2", "bq2", "Wd1", "bd1", "Wd2", "bd2")


@pytest.fixture(scope="module")
def tt():
    import two_towers_overlords_b200 as pkg
    from two_towers_overlords_b200 import ops

    pkg.ops = ops
    return pkg


# both launch modes of every case run back to back (the innermost parametrisation), so they share one oracle forward
CHAIN = pytest.mark.parametrize("chain", list(CHAINS.values()), ids=list(CHAINS))


# ---------------------------------------------------------------------------------------------------------------------
# inputs and the float64 oracle
# ---------------------------------------------------------------------------------------------------------------------
@dataclass
class Inputs:
    tokens: tuple   # q_ids, q_mask, p_ids, p_mask, n_ids, n_mask: CPU, padded to (Lq, Ld), ids int32, mask uint8
    tables: tuple   # fp32 [V, H] query / document tables
    params: list    # Wq1, bq1, Wq2, bq2, Wd1, bd1, Wd2, bd2 (fp32, nn.Linear's init distribution)
    xhat_ref: torch.Tensor  # oracle.pooled_normalised of all 3B rows


_INPUTS, _TABLES = {}, {}


def _tables(vocab):
    if vocab not in _TABLES:
        gen = torch.Generator().manual_seed(vocab)
        _TABLES[vocab] = tuple(torch.randn(vocab, H, generator=gen) for _ in range(2))
    return _TABLES[vocab]


def make_inputs(B, P, seed, Lq=8, Ld=24, vocab=VOCAB) -> Inputs:
    """One case's CPU inputs, cached per (B, P, seed, Lq, Ld, vocab): negatives are other rows' positives, as the
    reference's batcher makes them.  Every 37th row of each segment (at different
    offsets) is all-masked, so its pooled row is exactly zero."""
    key = (B, P, seed, Lq, Ld, vocab)
    if key not in _INPUTS:
        batch = O.synth_triplet_batch(B, Lq, Ld, "Z", seed=seed, vocab=vocab)
        if B == 1:  # the in-batch derangement of one row is the row itself: draw a negative of its own
            other = O.synth_triplet_batch(1, Lq, Ld, "Z", seed=seed + 1, vocab=vocab)
            batch.n_ids, batch.n_mask = other.p_ids, other.p_mask
        toks = [torch.nn.functional.pad(t, (0, L - t.shape[1])) for t, L in zip(batch.astuple(), (Lq, Lq, Ld, Ld, Ld, Ld))]
        for k, off in ((1, 3), (3, 11), (5, 19)):
            toks[k][off::37] = 0
        toks = tuple(t.to(torch.int32 if k % 2 == 0 else torch.uint8).contiguous() for k, t in enumerate(toks))
        tables = _tables(vocab)
        gen = torch.Generator().manual_seed(seed + 7)
        params = []
        for _ in range(2):
            for fan_in, shape in ((H, (P, H)), (H, (P,)), (P, (P, P)), (P, (P,))):
                params.append((torch.rand(shape, generator=gen) * 2 - 1) * fan_in ** -0.5)
        xr = torch.cat([O.pooled_normalised(tables[0], toks[0], toks[1]), O.pooled_normalised(tables[1], toks[2], toks[3]),
                        O.pooled_normalised(tables[1], toks[4], toks[5])])
        _INPUTS[key] = Inputs(toks, tables, params, xr)
    return _INPUTS[key]


def cosine64(a, b):
    return (a * b).sum(1) / (a.norm(dim=1).clamp_min(COS_EPS) * b.norm(dim=1).clamp_min(COS_EPS))


_FWD = {}


def forward64(x, params, B):
    """Float64 first-layer pre-activations z [3B, P] and Σ_k |x_k W1_jk| (the single-pass bf16 rounding scale) from the
    device's pooled rows, cached while the device returns the same rows for the same parameters."""
    key = (x.shape, tuple(float(p.double().sum()) for p in params))
    hit = _FWD.get(key)
    if hit is not None and torch.equal(hit[0], x):
        return hit[1], hit[2]
    if len(_FWD) >= 4:
        _FWD.pop(next(iter(_FWD)))
    xd = x.double()
    W1 = (params[0].double(), params[4].double())
    b1 = (params[1].double(), params[5].double())
    z = torch.cat([xd[:B] @ W1[0].T + b1[0], xd[B:] @ W1[1].T + b1[1]])
    scale = torch.cat([xd[:B].abs() @ W1[0].abs().T, xd[B:].abs() @ W1[1].abs().T])
    _FWD[key] = (x.clone(), z, scale)
    return z, scale


def oracle64(x, params, gate, active, B, margin, inv_batch, grad_scale):
    """Projection, loss and backward in float64 autograd: x [3B, H] (a leaf, or a function of the token tables),
    params 8 float64 leaves, differentiated through the device's ReLU gate (bool [3B, P]) and hinge activity
    (bool [B]).  Returns y, dY, the pre-hinge values, the statistics [B, 8] and the loss Σ hinge · inv_batch; the
    gradients land in .grad of the leaves (of grad_scale · loss, as the step computes them)."""
    Wq1, bq1, Wq2, bq2, Wd1, bd1, Wd2, bd2 = params
    z = torch.cat([x[:B] @ Wq1.T + bq1, x[B:] @ Wd1.T + bd1])
    h = z * gate.double()
    y = torch.cat([h[:B] @ Wq2.T + bq2, h[B:] @ Wd2.T + bd2])
    y.retain_grad()
    q, p, n = y[:B], y[B: 2 * B], y[2 * B:]
    cos_p, cos_n = cosine64(q, p), cosine64(q, n)
    pre = (1 - cos_p) - (1 - cos_n) + margin
    (grad_scale * inv_batch * (pre * active.double()).sum()).backward()
    with torch.no_grad():
        stats = torch.stack([cos_p, cos_n, pre.clamp_min(0), q.norm(dim=1), p.norm(dim=1), n.norm(dim=1), (q * p).sum(1),
                             (q * n).sum(1)], 1)
    return dict(y=y.detach(), dy=y.grad, pre=pre.detach(), stats=stats, loss=float(stats[:, 2].sum()) * inv_batch)


# ---------------------------------------------------------------------------------------------------------------------
# error measures
# ---------------------------------------------------------------------------------------------------------------------
def rel_err(got, want) -> float:
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).norm() / want.norm().clamp_min(1e-30))


def row_rel(got, want, floor=1e-6):
    """Largest row-relative error and its row."""
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    e = (got - want).norm(dim=1) / want.norm(dim=1).clamp_min(floor)
    i = int(e.argmax())
    return float(e[i]), i


def block_err(got, want):
    """Largest per-block relative error over 64 x 64 blocks (64-element blocks of a vector) and the block's origin:
    ||Δ_T|| / max(||want_T||, 0.1 · ||want|| · sqrt(|T| / N))."""
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    rb = 1 if want.dim() == 1 else 64
    g2, w2 = (got[None], want[None]) if want.dim() == 1 else (got, want)
    n_all, w_norm = want.numel(), float(want.norm())
    worst, where = 0.0, None
    for i in range(0, w2.shape[0], rb):
        for j in range(0, w2.shape[1], 64):
            wt = w2[i: i + rb, j: j + 64]
            den = max(float(wt.norm()), 0.1 * w_norm * (wt.numel() / n_all) ** 0.5, 1e-30)
            e = float((g2[i: i + rb, j: j + 64] - wt).norm()) / den
            if e > worst:
                worst, where = e, (i, j)
    return worst, where


def stats_err(got, want):
    """Per-triplet statistics (cos_p, cos_n, hinge, |q|, |p|, |n|, q.p, q.n): cosines and hinge absolute, norms relative,
    dot products relative to |q||p| / |q||n|.  Largest error and its row."""
    g = got.detach().double().cpu()
    e_abs = (g[:, :3] - want[:, :3]).abs().amax(1)
    e_nrm = ((g[:, 3:6] - want[:, 3:6]).abs() / want[:, 3:6].clamp_min(1e-6)).amax(1)
    e_dot = torch.maximum((g[:, 6] - want[:, 6]).abs() / (want[:, 3] * want[:, 4]).clamp_min(1e-12),
                          (g[:, 7] - want[:, 7]).abs() / (want[:, 3] * want[:, 5]).clamp_min(1e-12))
    e = torch.maximum(torch.maximum(e_abs, e_nrm), e_dot)
    i = int(e.argmax())
    return float(e[i]), i


def max_rel(got, want, floor):
    got, want = got.detach().double().cpu().reshape(-1), want.detach().double().cpu().reshape(-1)
    return float((got - want).abs().max() / want.abs().max().clamp_min(floor))


# ---------------------------------------------------------------------------------------------------------------------
# one step on the device
# ---------------------------------------------------------------------------------------------------------------------
class Step:
    """A TripletStep bound to device copies of `inp`: the 8 projection tensors and their gradients are slices of flat
    fp32 buffers (the layout the fused Adam wants)."""

    def __init__(self, tt, inp, precision, chain, margin=0.3, inv_batch=None, grad_scale=1.0, params=None,
                 train_table=False):
        B, Lq = inp.tokens[0].shape
        Ld = inp.tokens[2].shape[1]
        V = inp.tables[0].shape[0]
        P = inp.params[0].shape[0]
        self.B, self.P, self.precision = B, P, precision
        self.params_cpu = [p.clone() for p in (params or inp.params)]
        self.inp = inp
        self.so = tt.ops.TripletStep(B, Lq, Ld, H, P, V, precision, DEV, train_table=train_table)
        self.so.set_chain(chain)
        self.tokens = tuple(t.to(DEV) for t in inp.tokens)
        self.tables = tuple(t.to(DEV) for t in inp.tables)
        self.flat_p = torch.cat([p.reshape(-1) for p in self.params_cpu]).to(DEV)
        self.flat_g = torch.zeros_like(self.flat_p)
        self.p_views, self.g_views, off = [], [], 0
        for p in self.params_cpu:
            self.p_views.append(self.flat_p[off: off + p.numel()].view_as(p))
            self.g_views.append(self.flat_g[off: off + p.numel()].view_as(p))
            off += p.numel()
        self.table_grads = tuple(torch.zeros_like(t) for t in self.tables) if train_table else None
        self.bind(margin, 1.0 / B if inv_batch is None else inv_batch, grad_scale)

    def bind(self, margin, inv_batch, grad_scale=1.0):
        self.margin, self.inv_batch, self.grad_scale = margin, inv_batch, grad_scale
        self.so.bind(self.tokens, self.tables, self.p_views, self.g_views, margin, inv_batch, grad_scale,
                     self.table_grads)

    def run(self, monkeypatch, fp32_out=False, **kw):
        if fp32_out:
            monkeypatch.setenv("TT_CHAIN_FP32_OUT", "1")
        else:
            monkeypatch.delenv("TT_CHAIN_FP32_OUT", raising=False)
        self.so.run(**kw)
        torch.cuda.synchronize()
        assert int(self.so.err.item()) == 0
        return float(self.so.loss.item()), [g.detach().cpu().clone() for g in self.g_views]


def run_and_check(tt, monkeypatch, inp, precision, chain, tag, margin=0.3, inv_batch=None, grad_scale=1.0, params=None,
                  skip_grads=(), train_table=False):
    """One step without and one with the fp32 diagnostic outputs (gradients must be bit-identical), then everything
    against float64.  Returns the Step and the float64 results."""
    st = Step(tt, inp, precision, chain, margin, inv_batch, grad_scale, params, train_table)
    loss0, grads0 = st.run(monkeypatch)
    loss1, grads1 = st.run(monkeypatch, fp32_out=True)
    monkeypatch.delenv("TT_CHAIN_FP32_OUT", raising=False)
    assert loss1 == loss0, (tag, loss0, loss1)
    assert all(torch.equal(a, b) for a, b in zip(grads0, grads1)), (tag, "TT_CHAIN_FP32_OUT changed the gradients")
    return st, check_step(st, grads1, loss1, tag, skip_grads)


def check_step(st, grads, loss, tag, skip_grads=()):
    g = GATES[st.precision]
    B = st.B
    v = st.so._views()
    xhat = v["xhat"].detach().cpu().clone()
    e_x, r_x = row_rel(xhat, st.inp.xhat_ref)
    assert e_x < 1e-4, (tag, "pooled row", r_x, e_x)
    gate = st.so.relu_gate().cpu()
    stats = v["stats"].detach().cpu().clone()
    active = stats[:, 2] > 0
    z, scale = forward64(xhat, st.params_cpu, B)
    prm = [p.double().requires_grad_(True) for p in st.params_cpu]
    o = oracle64(xhat.double(), prm, gate, active, B, st.margin, st.inv_batch, st.grad_scale)
    # gates the device and float64 may disagree on: only inside the rounding band
    flips = gate != (z > 0)
    band = KINK_BAND if st.precision == "bf16x3" else 2.0 ** -7 * scale
    n_flips = int(flips.sum())
    outside = flips & (z.abs() > band)
    hinge_flips = active != (o["pre"] > 0)
    e = dict(loss=abs(loss - o["loss"]) / max(abs(o["loss"]), 1e-30), flips=n_flips)
    e["stats"], r_s = stats_err(stats, o["stats"])
    e["y"], r_y = row_rel(v["y"], o["y"])
    e["dy"], r_dy = row_rel(v["dy"], o["dy"])
    worst = {}
    for nm, got, p in zip(NAMES, grads, prm):
        if nm in skip_grads:
            continue
        be, where = block_err(got, p.grad)
        worst[nm] = (rel_err(got, p.grad), be, where)
    e["grad"] = max((w[0] for w in worst.values()), default=0.0)
    e["block"] = max((w[1] for w in worst.values()), default=0.0)
    print(f"step_shapes {tag}: loss {e['loss']:.2e} grad {e['grad']:.2e} block {e['block']:.2e} y {e['y']:.2e} "
          f"dy {e['dy']:.2e} stats {e['stats']:.2e} relu flips {n_flips} hinge flips {int(hinge_flips.sum())}")
    assert not bool(outside.any()), (tag, "ReLU gate flip outside the rounding band", z[outside][:8])
    assert not bool((hinge_flips & (o["pre"].abs() > g["hinge_band"])).any()), (tag, "hinge activity")
    if st.precision == "bf16x3":
        assert n_flips <= 16, (tag, n_flips)
    assert e["loss"] < g["loss"], (tag, "loss", loss, o["loss"])
    assert e["stats"] < g["stats"], (tag, "stats row", r_s, stats[r_s], o["stats"][r_s])
    assert e["y"] < g["y"], (tag, "y row (q | p | n)", divmod(r_y, B), e["y"])
    assert e["dy"] < g["dy"], (tag, "dY row (q | p | n)", divmod(r_dy, B), e["dy"])
    for nm, (whole, blk, where) in worst.items():
        assert whole < g["grad"], (tag, nm, "whole tensor", whole)
        assert blk < g["block"], (tag, nm, "block at", where, blk)
    return o


# ---------------------------------------------------------------------------------------------------------------------
# A. tiling sweep: every column-tile shape against row tiles with partial tails, partial chunks, mixed p / n k-blocks
# ---------------------------------------------------------------------------------------------------------------------
@CHAIN
@pytest.mark.parametrize("B", [1, 129, 192, 300, 1100])
@pytest.mark.parametrize("P", [64, 128, 192, 256, 320, 448, 512, 576])
@pytest.mark.parametrize("precision", X3)
def test_step_tiling_sweep_vs_float64(tt, monkeypatch, precision, chain, P, B):
    """B = 129 / 300 / 1100: partial last row tile, partial last weight-gradient chunk, k-blocks of the document tower
    that hold positives and negatives; B = 192: a row tile of 64 rows on a whole k-block; P % 128 == 64: a half-empty
    last column tile beside full ones; P = 576: NC = 5 with a half tile and nine 64-column loss slots."""
    inp = make_inputs(B, P, seed=1000 + B + P)
    run_and_check(tt, monkeypatch, inp, precision, chain, (precision, chain, P, B))


# ---------------------------------------------------------------------------------------------------------------------
# B. large batch: the weight-gradient chunks grow to 16 k-blocks; the host tuning hook for the chunk size
# ---------------------------------------------------------------------------------------------------------------------
@CHAIN
@pytest.mark.parametrize("P", [64, 192])
@pytest.mark.parametrize("precision", X3)
def test_step_large_batch_vs_float64(tt, monkeypatch, precision, chain, P):
    """B = 8256 on one GPU: k-blocks [129, 258] -> kcb = 16, chunk counts [9, 17], last chunks of 1 and 2 k-blocks."""
    inp = make_inputs(8256, P, seed=2000 + P, Lq=4, Ld=8)
    run_and_check(tt, monkeypatch, inp, precision, chain, (precision, chain, P, 8256))


@pytest.mark.parametrize("precision", X3)
def test_step_chunk_size_hook_vs_float64(tt, monkeypatch, precision):
    """TT_CHAIN_KCB=4 (persistent kernel): B = 1100 in chunks of 4 k-blocks, k-blocks [18, 35] -> chunk counts [5, 9],
    last chunks of 2 and 3 k-blocks."""
    monkeypatch.setenv("TT_CHAIN_KCB", "4")
    inp = make_inputs(1100, 192, seed=2100)
    run_and_check(tt, monkeypatch, inp, precision, CHAINS["persistent"], (precision, "kcb4", 192, 1100))


# ---------------------------------------------------------------------------------------------------------------------
# C. shapes people run: run_training's defaults, the README dev run, per-rank shapes of data-parallel configs
# ---------------------------------------------------------------------------------------------------------------------
@CHAIN
@pytest.mark.parametrize("B,P,inv_batch,grad_scale", [
    (1024, 128, 1 / 1024, 1.0),   # run_training / TwoTowersModel defaults
    (256, 64, 1 / 256, 1.0),      # configs[0], the README dev run
    (256, 512, 1 / 2048, 1.0),    # configs[1] on 8 GPUs: one rank's share, the loss is the mean over all 8 ranks
    (2048, 512, 1 / 16384, 1.0),  # configs[3] on 8 GPUs
    (1100, 192, 1 / 1100, 0.75),  # a scaled loss gradient
], ids=["B1024-P128", "B256-P64", "B256-P512-inv2048", "B2048-P512-inv16384", "B1100-P192-scale0.75"])
@pytest.mark.parametrize("precision", X3)
def test_step_user_shapes_vs_float64(tt, monkeypatch, precision, chain, B, P, inv_batch, grad_scale):
    inp = make_inputs(B, P, seed=3000 + B + P)
    run_and_check(tt, monkeypatch, inp, precision, chain, (precision, chain, P, B, inv_batch, grad_scale),
                  inv_batch=inv_batch, grad_scale=grad_scale)


# ---------------------------------------------------------------------------------------------------------------------
# D. single-pass bf16 (TT_PRECISION=bf16)
# ---------------------------------------------------------------------------------------------------------------------
@CHAIN
@pytest.mark.parametrize("B", [129, 1100])
@pytest.mark.parametrize("P", [64, 192, 512])
def test_step_single_pass_bf16_vs_float64(tt, monkeypatch, chain, P, B):
    """One bf16 product per contraction: gates measured on the B200 (GATES["bf16"]); a wrong tile is still an O(1)
    error at these gates.  A ReLU gate may differ from float64 where |z_j| <= 2^-7 · Σ_k |x_k W1_jk|."""
    inp = make_inputs(B, P, seed=4000 + B + P)
    run_and_check(tt, monkeypatch, inp, "bf16", chain, ("bf16", chain, P, B))


# ---------------------------------------------------------------------------------------------------------------------
# E. loss-epilogue edges
# ---------------------------------------------------------------------------------------------------------------------
@CHAIN
@pytest.mark.parametrize("margin", [0.0, 2.5])
@pytest.mark.parametrize("precision", X3)
def test_step_margin_edges_vs_float64(tt, monkeypatch, precision, chain, margin):
    """margin 0: about half the hinges are inactive at random init; margin 2.5: every hinge is active
    (cos_n - cos_p >= -2)."""
    inp = make_inputs(300, 192, seed=5000)
    o = run_and_check(tt, monkeypatch, inp, precision, chain, (precision, chain, "margin", margin), margin=margin)[1]
    n_active = int((o["pre"] > 0).sum())
    assert (n_active == 300) if margin == 2.5 else (50 < n_active < 250), n_active


@CHAIN
@pytest.mark.parametrize("precision", X3)
def test_step_workspace_reuse_across_margins(tt, monkeypatch, precision, chain):
    """The same TripletStep for margin 0.3, then -3 (every hinge 0: the loss and every gradient exactly zero), then 0.3
    again (bit-identical to the first call): no stale partial sums, column sums or counters from an earlier call."""
    inp = make_inputs(300, 192, seed=5000)
    st, _ = run_and_check(tt, monkeypatch, inp, precision, chain, (precision, chain, "reuse"))
    loss0, grads0 = st.run(monkeypatch)
    st.bind(-3.0, st.inv_batch)
    loss, grads = st.run(monkeypatch)
    assert loss == 0.0
    for nm, g in zip(NAMES, grads):
        assert float(g.abs().max()) == 0.0, nm
    st.bind(0.3, st.inv_batch)
    loss, grads = st.run(monkeypatch)
    assert loss == loss0
    assert all(torch.equal(a, b) for a, b in zip(grads0, grads))


@CHAIN
@pytest.mark.parametrize("precision", X3)
def test_step_zero_norm_queries_vs_float64(tt, monkeypatch, precision, chain):
    """All-masked query rows with bq1 < 0 and bq2 = 0: q is exactly 0, both cosines are 0 through the per-vector clamp
    and the hinge is the margin.  The p and n rows of such a triplet get exactly zero dY; its q row gets the (huge)
    gradient of torch's clamped cosine.  dbq2 is left out of the gradient gates: those rows dominate it."""
    inp = make_inputs(300, 192, seed=5100)
    params = [p.clone() for p in inp.params]
    params[1] = -(params[1].abs() + 1e-3)
    params[3] = torch.zeros_like(params[3])
    st, o = run_and_check(tt, monkeypatch, inp, precision, chain, (precision, chain, "zero q"), params=params,
                          skip_grads=("bq2",))
    B = st.B
    zero = (inp.tokens[1].sum(1) == 0).nonzero().flatten()
    assert zero.numel() == len(range(3, B, 37))
    v = st.so._views()
    stats = v["stats"].cpu()[zero]
    for col in (0, 1, 3, 6, 7):  # cos_p, cos_n, |q|, q.p, q.n
        assert float(stats[:, col].abs().max()) == 0.0, col
    assert torch.allclose(stats[:, 2], torch.full_like(stats[:, 2], 0.3))
    dy = v["dy"].cpu()
    assert float(dy[B + zero].abs().max()) == 0.0 and float(dy[2 * B + zero].abs().max()) == 0.0
    assert row_rel(dy[zero], o["dy"][zero])[0] < GATES[precision]["dy"]


# ---------------------------------------------------------------------------------------------------------------------
# F. fused Adam at a ragged shape
# ---------------------------------------------------------------------------------------------------------------------
@CHAIN
@pytest.mark.parametrize("precision", X3)
def test_step_fused_adam_ragged_matches_torch_adam(tt, monkeypatch, precision, chain):
    """Three run(optimise=True) calls on three batches (B = 300, P = 192): after each, the parameters and both moments
    equal torch.optim.Adam applied, from the parameters before the call, to the gradient that call wrote, and the
    device's step count advanced by one."""
    inps = [make_inputs(300, 192, seed=6000 + k) for k in range(3)]
    st = Step(tt, inps[0], precision, chain)
    for inp in inps[1:]:
        st.so.add_tokens(tuple(t.to(DEV) for t in inp.tokens))
    lr, betas, eps = 1e-3, (0.9, 0.999), 1e-8
    state = torch.zeros(4, dtype=torch.float64, device=DEV)
    m, v = torch.zeros_like(st.flat_p), torch.zeros_like(st.flat_p)
    st.so.bind_adam(state, st.flat_p, st.flat_g, m, v, lr, betas, eps)
    ref = st.flat_p.detach().cpu().clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=lr, betas=betas, eps=eps)
    for k in range(3):
        before = st.flat_p.detach().cpu().clone()
        st.run(monkeypatch, slot=k, optimise=True)
        with torch.no_grad():
            ref.copy_(before)
        ref.grad = st.flat_g.detach().cpu().clone()
        assert float(ref.grad.abs().max()) > 0.0
        opt.step()
        assert max_rel(st.flat_p, ref, 1e-3) < 1e-6, (k, max_rel(st.flat_p, ref, 1e-3))
        assert max_rel(m, opt.state[ref]["exp_avg"], 1e-30) < 1e-6, k
        # the library forms 1 - beta2 in fp32 from the fp32 beta2 (9.99987e-4), torch.optim.Adam in double (1e-3): the
        # second moment differs by 1.3e-5 relative, and the bias correction by the same factor, so the update does not
        assert max_rel(v, opt.state[ref]["exp_avg_sq"], 1e-30) < 3e-5, k
        assert float(state[0].item()) == k + 1


# ---------------------------------------------------------------------------------------------------------------------
# G. trainable token tables at a ragged shape
# ---------------------------------------------------------------------------------------------------------------------
@CHAIN
@pytest.mark.parametrize("precision", X3)
def test_step_trainable_tables_ragged_vs_float64(tt, monkeypatch, precision, chain):
    """B = 300, P = 192, V = 2048, both tables trainable: the dxhat rows, and both table gradients against float64
    autograd through nn.Embedding with the device's gates (the method of test_step_parity's configs[2] case); rows no
    unmasked token names stay exactly zero."""
    inp = make_inputs(300, 192, seed=7000, vocab=2048)
    st, _ = run_and_check(tt, monkeypatch, inp, precision, chain, (precision, chain, "tables"), train_table=True)
    B = st.B
    v = st.so._views()
    gate = st.so.relu_gate().cpu()
    active = v["stats"].cpu()[:, 2] > 0
    xhat = v["xhat"].detach().cpu().double().requires_grad_(True)
    prm = [p.double().requires_grad_(True) for p in st.params_cpu]
    oracle64(xhat, prm, gate, active, B, st.margin, st.inv_batch, st.grad_scale)
    e, r = row_rel(v["dxhat"], xhat.grad)
    assert e < 1e-3, ("dxhat row (q | p | n)", divmod(r, B), e)
    tables = [t.double().requires_grad_(True) for t in inp.tables]
    q_ids, q_mask, p_ids, p_mask, n_ids, n_mask = inp.tokens
    x = torch.cat([torch.nn.functional.normalize(O.mean_pooling(torch.nn.functional.embedding(ids.long(), tab),
                                                                mask.long()), p=2, dim=1)
                   for tab, ids, mask in ((tables[0], q_ids, q_mask), (tables[1], p_ids, p_mask),
                                          (tables[1], n_ids, n_mask))])
    prm = [p.double().requires_grad_(True) for p in st.params_cpu]
    oracle64(x, prm, gate, active, B, st.margin, st.inv_batch, st.grad_scale)
    for got, tab in zip(st.table_grads, tables):
        got = got.cpu()
        assert rel_err(got, tab.grad) < 1e-3
        untouched = tab.grad.abs().sum(1) == 0
        assert int(untouched.sum()) > 0
        assert float(got[untouched].abs().max()) == 0.0
