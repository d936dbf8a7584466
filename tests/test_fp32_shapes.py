"""The fp32 CUDA-core path (TT_PREC_FP32, csrc/tt_mlp_simt.cu) and the kernels of the autograd surface against float64
at the shapes where they go wrong.  ops.default_precision trains every model whose H or P is not a multiple of 64 on
the fp32 path, and ops.mlp / ops.triplet_loss run the same kernel families in evaluation, indexing and the reference's
training loops.

  A. the whole fp32 step (tt_triplet_step): the SGEMM works in 64 x 64 x 16 tiles, so B and P hit the M, N and K tails
     (the weight gradients contract over K = B and K = 2B batch rows); B = 8256 puts ~5e4-conditioned column sums
     (positive and negative rows of the document tower's dY nearly cancel) into the bias and weight gradients.
  B. tt_encode_fwd / tt_encode_bwd in all three precisions, through ops.mlp and the raw ABI: y and the saved h, the
     four weight gradients and dx, `accumulate`, dx = NULL, M = 0 and the refused calls.
  C. tt_triplet_loss_fwd / tt_triplet_loss_bwd: the statistics row by row, the loss (strided reduction above 1024
     rows), and every gradient row, zero-norm and sub-eps rows included.
  D. tt_adam_step / tt_adam_step_dev against a float64 replay of torch.optim.Adam's single-tensor formula, compared on
     the UPDATE p_t - p_{t-1}, not on the parameters.

Every check runs against float64 from the device's own inputs and prints its worst measured errors; the gates were
set from those numbers on a B200 (1000 W) with a margin of at least 4x (see GATES)."""
import numpy as np
import pytest
import torch

from oracle import two_towers_oracle as O
from test_step_shapes import COS_EPS, KINK_BAND, NAMES, block_err, cosine64, oracle64, rel_err, row_rel, stats_err

pytestmark = pytest.mark.gpu

DEV = "cuda"
VOCAB = 4096
HINGE_BAND = 1e-5  # |pre-hinge| within which the device and float64 may disagree on whether a triplet is active

# Gates (relative, as in tests/test_step_shapes.py): loss, gradients whole tensor / per 64 x 64 block, h, y and dY rows,
# statistics.  They started from BASELINE's gates (GATES["bf16x3"] there: loss 1e-4, gradients 1e-3 / 3e-3, y 1e-4, dY
# 1e-3, statistics 1e-4) and are set to about 4x the worst value this file measured on a B200 (1000 W); the report line
# each case prints carries its measured values.  Worst measured for the step: loss 1.7e-7, gradients 1.7e-4 whole and per
# block (bd2 at B = 8256), h 2.4e-5 (row-relative, a row whose units are all near 0), y 1.1e-6, dY 4.8e-6, statistics
# 4.8e-7.  Before the weight gradients were summed in row slices, dWd2 was 1.0e-3 off at B = 8256, P = 64 and 8.3e-4
# (9.3e-4 in one block) at P = 192: both above these gates.
GATES = dict(loss=1e-6, grad=7e-4, block=7e-4, h=1e-4, y=5e-6, dy=2e-5, stats=2e-6)
# tt_encode_fwd / tt_encode_bwd per precision: h and y rows, weight gradients whole / per block, dx rows.  Worst measured
# (B200, 1000 W): fp32 h 9.7e-6, y 3.2e-7, gradients 1.2e-6, dx 7.4e-7; bf16x3 h 7.7e-6, y 5.0e-6, gradients 6.8e-6 /
# 8.7e-6, dx 1.1e-5; bf16 h 3.5e-3, y 2.7e-3, gradients 3.5e-3 / 3.8e-3, dx 5.9e-3
MLP_GATES = {
    "fp32": dict(h=4e-5, y=2e-6, grad=5e-6, block=5e-6, dx=3e-6),
    "bf16x3": dict(h=4e-5, y=2e-5, grad=3e-5, block=4e-5, dx=5e-5),
    "bf16": dict(h=1.5e-2, y=1.1e-2, grad=1.4e-2, block=1.6e-2, dx=2.4e-2),
}
# worst measured: loss 2.4e-7, statistics 2.4e-7, gradient rows 3.7e-7
LOSS_GATES = dict(loss=1e-6, stats=1e-6, grad=1.5e-6)
# update: max error over max(largest |update|, lr / (1 - beta1^t)); m over max(largest |m|, sqrt(largest v)); v over the
# largest v.  Worst measured: update 1.9e-5 (the rounding of p_t to fp32 at |p| ~ 0.2), m 3.6e-7, v 2.0e-6
ADAM_GATES = dict(update=1e-4, moments=1e-5)


@pytest.fixture(scope="module")
def tt():
    import two_towers_overlords_b200 as pkg
    from two_towers_overlords_b200 import ops

    pkg.ops = ops
    return pkg


def _lib(tt):
    return tt.ops.N.load()


def _call(tt, rc, what):
    tt.ops.N.check(rc, what)


# ---------------------------------------------------------------------------------------------------------------------
# A. the whole fp32 step
# ---------------------------------------------------------------------------------------------------------------------
_INPUTS = {}


def make_inputs(B, P, seed, H=O.HIDDEN, Lq=8, Ld=24, vocab=VOCAB):
    """tests/test_step_shapes.py::make_inputs for any hidden size H: negatives are other rows' positives, every 37th row
    of each segment (at different offsets) is all-masked, parameters follow nn.Linear's init distribution."""
    key = (B, P, seed, H, Lq, Ld, vocab)
    if key not in _INPUTS:
        batch = O.synth_triplet_batch(B, Lq, Ld, "Z", seed=seed, vocab=vocab)
        if B == 1:  # the in-batch derangement of one row is the row itself: draw a negative of its own
            other = O.synth_triplet_batch(1, Lq, Ld, "Z", seed=seed + 1, vocab=vocab)
            batch.n_ids, batch.n_mask = other.p_ids, other.p_mask
        toks = [torch.nn.functional.pad(t, (0, L - t.shape[1])) for t, L in zip(batch.astuple(), (Lq, Lq, Ld, Ld, Ld, Ld))]
        for k, off in ((1, 3), (3, 11), (5, 19)):
            toks[k][off::37] = 0
        toks = tuple(t.to(torch.int32 if k % 2 == 0 else torch.uint8).contiguous() for k, t in enumerate(toks))
        gen = torch.Generator().manual_seed(vocab + H)
        tables = tuple(torch.randn(vocab, H, generator=gen) for _ in range(2))
        gen = torch.Generator().manual_seed(seed + 7)
        params = []
        for _ in range(2):
            for fan_in, shape in ((H, (P, H)), (H, (P,)), (P, (P, P)), (P, (P,))):
                params.append((torch.rand(shape, generator=gen) * 2 - 1) * fan_in ** -0.5)
        xr = torch.cat([O.pooled_normalised(tables[0], toks[0], toks[1]), O.pooled_normalised(tables[1], toks[2], toks[3]),
                        O.pooled_normalised(tables[1], toks[4], toks[5])])
        if len(_INPUTS) >= 4:
            _INPUTS.pop(next(iter(_INPUTS)))
        _INPUTS[key] = (toks, tables, params, xr)
    return _INPUTS[key]


class Fp32Step:
    """ops.TripletStep in fp32 bound to device copies of one case: the 8 projection tensors and their gradients are
    slices of flat fp32 buffers, as FusedTrainer binds them."""

    def __init__(self, tt, inp, margin=0.3, inv_batch=None, grad_scale=1.0, params=None, train_table=False):
        toks, tables, params0, self.xhat_ref = inp
        B, Lq = toks[0].shape
        Ld = toks[2].shape[1]
        V, H = tables[0].shape
        self.params_cpu = [p.clone() for p in (params or params0)]
        P = self.params_cpu[0].shape[0]
        self.B, self.H, self.P = B, H, P
        self.tables_cpu, self.tokens_cpu = tables, toks
        self.so = tt.ops.TripletStep(B, Lq, Ld, H, P, V, "fp32", DEV, train_table=train_table)
        self.tokens = tuple(t.to(DEV) for t in toks)
        self.tables = tuple(t.to(DEV) for t in tables)
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

    def run(self):
        self.so.run()
        torch.cuda.synchronize()
        assert int(self.so.err.item()) == 0
        return float(self.so.loss.item()), [g.detach().cpu().clone() for g in self.g_views]


def check_fp32_step(st, loss, grads, tag, skip_grads=()):
    """Everything a step wrote against float64 autograd from the device's pooled rows, differentiated through the
    device's ReLU gate and hinge activity.  Returns the float64 results."""
    B, g = st.B, GATES
    v = st.so._views()
    xhat = v["xhat"].detach().cpu().clone()
    e_x, r_x = row_rel(xhat, st.xhat_ref)
    assert e_x < 1e-4, (tag, "pooled row", r_x, e_x)
    gate = v["h"].detach().cpu() > 0
    stats = v["stats"].detach().cpu().clone()
    active = stats[:, 2] > 0
    xd = xhat.double()
    prm = [p.double().requires_grad_(True) for p in st.params_cpu]
    with torch.no_grad():
        z = torch.cat([xd[:B] @ prm[0].T + prm[1], xd[B:] @ prm[4].T + prm[5]])
    o = oracle64(xd, prm, gate, active, B, st.margin, st.inv_batch, st.grad_scale)
    flips = gate != (z > 0)
    hinge_flips = active != (o["pre"] > 0)
    e = dict(loss=abs(loss - o["loss"]) / max(abs(o["loss"]), 1e-30))
    e["stats"], r_s = stats_err(stats, o["stats"])
    e["h"], r_h = row_rel(v["h"], z.clamp_min(0))
    e["y"], r_y = row_rel(v["y"], o["y"])
    e["dy"], r_dy = row_rel(v["dy"], o["dy"])
    worst = {}
    for nm, got, p in zip(NAMES, grads, prm):
        if nm not in skip_grads:
            be, where = block_err(got, p.grad)
            worst[nm] = (rel_err(got, p.grad), be, where)
    e["grad"] = max(w[0] for w in worst.values())
    e["block"] = max(w[1] for w in worst.values())
    arg = max(worst, key=lambda k: worst[k][1])
    print(f"fp32_shapes step {tag}: loss {e['loss']:.2e} grad {e['grad']:.2e} block {e['block']:.2e} ({arg}) "
          f"h {e['h']:.2e} y {e['y']:.2e} dy {e['dy']:.2e} stats {e['stats']:.2e} relu flips {int(flips.sum())} "
          f"hinge flips {int(hinge_flips.sum())}")
    assert not bool((flips & (z.abs() > KINK_BAND)).any()), (tag, "ReLU gate flip outside the rounding band")
    assert not bool((hinge_flips & (o["pre"].abs() > HINGE_BAND)).any()), (tag, "hinge activity")
    assert e["loss"] < g["loss"], (tag, "loss", loss, o["loss"])
    assert e["stats"] < g["stats"], (tag, "stats row", r_s, stats[r_s], o["stats"][r_s])
    assert e["h"] < g["h"], (tag, "h row (q | p | n)", divmod(r_h, B), e["h"])
    assert e["y"] < g["y"], (tag, "y row (q | p | n)", divmod(r_y, B), e["y"])
    assert e["dy"] < g["dy"], (tag, "dY row (q | p | n)", divmod(r_dy, B), e["dy"])
    for nm, (whole, blk, where) in worst.items():
        assert whole < g["grad"], (tag, nm, "whole tensor", whole)
        assert blk < g["block"], (tag, nm, "block at", where, blk)
    return o


def run_step_case(tt, inp, tag, **kw):
    """One step, a second identical call (bit-identical loss and gradients), then the float64 check."""
    skip = kw.pop("skip_grads", ())
    st = Fp32Step(tt, inp, **kw)
    loss0, grads0 = st.run()
    loss1, grads1 = st.run()
    assert loss1 == loss0 and all(torch.equal(a, b) for a, b in zip(grads0, grads1)), (tag, "second run differs")
    return st, check_fp32_step(st, loss1, grads1, tag, skip)


# every P against the B that give the weight gradients' K tails (K = B and 2B rows, 16-row k-steps, 64-row tiles); P in
# {16, 24, 100, 130} can only run on this path
STEP_SHAPES = [(B, P) for B in (1, 17, 65, 300, 1100) for P in (16, 24, 64, 100, 130, 192, 576)]
STEP_SHAPES += [(B, P) for B in (15, 63, 129) for P in (24, 130)]


@pytest.mark.parametrize("B,P", STEP_SHAPES, ids=[f"B{b}-P{p}" for b, p in STEP_SHAPES])
def test_fp32_step_tiling_sweep_vs_float64(tt, B, P):
    run_step_case(tt, make_inputs(B, P, seed=10000 + B + P), ("sweep", B, P))


@pytest.mark.parametrize("H", [128, 256, 768])
def test_fp32_step_hidden_sizes_vs_float64(tt, H):
    """The first layer's K = H and dW1's N = H: 2, 4 and 12 column tiles of dW1 at a ragged B and P."""
    run_step_case(tt, make_inputs(65, 100, seed=11000 + H, H=H), ("hidden", H))


@pytest.mark.parametrize("P", [64, 192])
def test_fp32_step_large_batch_vs_float64(tt, P):
    """B = 8256: the document tower's bias and weight gradients sum 16512 rows whose positive and negative halves nearly
    cancel column by column.  With one fp32 running sum per weight element over all rows (one SGEMM) dWd2 was 1.0e-3
    off here at P = 64; the weight gradients now sum row slices, the bias gradients colsum2's double slices."""
    run_step_case(tt, make_inputs(8256, P, seed=12000 + P, Lq=4, Ld=8), ("large", 8256, P))


def test_fp32_step_margins_on_one_workspace(tt):
    """One TripletStep for margins 0.3, 0 (about half the hinges active), 2.5 (all active), -3 (none: loss and every
    gradient exactly zero) and 0.3 again (bit-identical to the first call)."""
    st, o = run_step_case(tt, make_inputs(300, 100, seed=13000), ("margin", 0.3))
    loss0, grads0 = st.run()
    for margin in (0.0, 2.5):
        st.bind(margin, st.inv_batch)
        loss, grads = st.run()
        o = check_fp32_step(st, loss, grads, ("margin", margin))
        n_active = int((o["pre"] > 0).sum())
        assert (n_active == 300) if margin == 2.5 else (50 < n_active < 250), n_active
    st.bind(-3.0, st.inv_batch)
    loss, grads = st.run()
    assert loss == 0.0
    for nm, g in zip(NAMES, grads):
        assert float(g.abs().max()) == 0.0, nm
    st.bind(0.3, st.inv_batch)
    loss, grads = st.run()
    assert loss == loss0 and all(torch.equal(a, b) for a, b in zip(grads0, grads))


def test_fp32_step_zero_norm_queries_vs_float64(tt):
    """All-masked query rows with bq1 < 0 and bq2 = 0: q is exactly 0, both cosines are 0 through the per-vector clamp,
    the p and n rows of such a triplet get exactly zero dY and its q row the (huge) gradient of torch's clamped cosine.
    dbq2 is left out of the gradient gates: those rows dominate it."""
    inp = make_inputs(300, 100, seed=14000)
    params = [p.clone() for p in inp[2]]
    params[1] = -(params[1].abs() + 1e-3)
    params[3] = torch.zeros_like(params[3])
    st, o = run_step_case(tt, inp, ("zero q",), params=params, skip_grads=("bq2",))
    B = st.B
    zero = (inp[0][1].sum(1) == 0).nonzero().flatten()
    assert zero.numel() == len(range(3, B, 37))
    v = st.so._views()
    stats = v["stats"].cpu()[zero]
    for col in (0, 1, 3, 6, 7):
        assert float(stats[:, col].abs().max()) == 0.0, col
    dy = v["dy"].cpu()
    assert float(dy[B + zero].abs().max()) == 0.0 and float(dy[2 * B + zero].abs().max()) == 0.0
    assert row_rel(dy[zero], o["dy"][zero])[0] < GATES["dy"]


def test_fp32_step_scaled_loss_vs_float64(tt):
    """One rank's share of a data-parallel mean (inv_batch = 1/2048) with a scaled upstream gradient."""
    run_step_case(tt, make_inputs(300, 130, seed=15000), ("scaled",), inv_batch=1 / 2048, grad_scale=0.75)


def test_fp32_step_trainable_tables_vs_float64(tt):
    """B = 300, P = 100, V = 2048, both tables trainable: the dxhat rows and both table gradients against float64 autograd
    through nn.Embedding with the device's gates; rows no unmasked token names stay exactly zero."""
    inp = make_inputs(300, 100, seed=16000, vocab=2048)
    st, _ = run_step_case(tt, inp, ("tables",), train_table=True)
    B = st.B
    v = st.so._views()
    gate = v["h"].cpu() > 0
    active = v["stats"].cpu()[:, 2] > 0
    xhat = v["xhat"].detach().cpu().double().requires_grad_(True)
    prm = [p.double().requires_grad_(True) for p in st.params_cpu]
    oracle64(xhat, prm, gate, active, B, st.margin, st.inv_batch, st.grad_scale)
    e, r = row_rel(v["dxhat"], xhat.grad)
    assert e < GATES["dy"], ("dxhat row (q | p | n)", divmod(r, B), e)
    tables = [t.double().requires_grad_(True) for t in st.tables_cpu]
    q_ids, q_mask, p_ids, p_mask, n_ids, n_mask = st.tokens_cpu
    x = torch.cat([torch.nn.functional.normalize(O.mean_pooling(torch.nn.functional.embedding(ids.long(), tab),
                                                                mask.long()), p=2, dim=1)
                   for tab, ids, mask in ((tables[0], q_ids, q_mask), (tables[1], p_ids, p_mask),
                                          (tables[1], n_ids, n_mask))])
    prm = [p.double().requires_grad_(True) for p in st.params_cpu]
    oracle64(x, prm, gate, active, B, st.margin, st.inv_batch, st.grad_scale)
    for got, tab in zip(st.table_grads, tables):
        got = got.cpu()
        e = rel_err(got, tab.grad)
        print(f"fp32_shapes tables: dxhat {row_rel(v['dxhat'], xhat.grad)[0]:.2e} table {e:.2e}")
        assert e < GATES["grad"]
        untouched = tab.grad.abs().sum(1) == 0
        assert int(untouched.sum()) > 0
        assert float(got[untouched].abs().max()) == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# B. tt_encode_fwd / tt_encode_bwd
# ---------------------------------------------------------------------------------------------------------------------
def mlp_case(M, H, P, seed):
    gen = torch.Generator().manual_seed(seed)
    x = torch.nn.functional.normalize(torch.randn(M, H, generator=gen), dim=1) if M else torch.zeros(0, H)
    W1 = (torch.rand(P, H, generator=gen) * 2 - 1) * H ** -0.5
    b1 = (torch.rand(P, generator=gen) * 2 - 1) * H ** -0.5
    W2 = (torch.rand(P, P, generator=gen) * 2 - 1) * P ** -0.5
    b2 = (torch.rand(P, generator=gen) * 2 - 1) * P ** -0.5
    dy = torch.randn(M, P, generator=gen) / max(M, 1)
    return x, W1, b1, W2, b2, dy


class RawMlp:
    """tt_encode_fwd / tt_encode_bwd on device buffers, with a workspace of exactly tt_mlp_ws_bytes."""

    def __init__(self, tt, precision, x, W1, b1, W2, b2):
        self.tt, self.lib = tt, _lib(tt)
        self.prec = tt.ops.N.PRECISIONS[precision]
        self.M, self.H = x.shape
        self.P = W1.shape[0]
        self.x, self.W1, self.b1, self.W2, self.b2 = (t.contiguous().to(DEV) for t in (x, W1, b1, W2, b2))
        self.ws_bytes = self.lib.tt_mlp_ws_bytes(self.M, self.H, self.P, self.prec)
        self.ws = tt.ops.N.workspace(self.ws_bytes, DEV)

    def fwd(self, ws_bytes=None):
        N = self.tt.ops.N
        h = torch.full((self.M, self.P), float("nan"), device=DEV)
        y = torch.full((self.M, self.P), float("nan"), device=DEV)
        rc = self.lib.tt_encode_fwd(N.ptr(self.x), self.M, self.H, self.P, N.ptr(self.W1), N.ptr(self.b1),
                                    N.ptr(self.W2), N.ptr(self.b2), N.ptr(h), N.ptr(y), self.prec, N.ptr(self.ws),
                                    self.ws_bytes if ws_bytes is None else ws_bytes, N.stream())
        return rc, h, y

    def bwd(self, dy, h, out=None, accumulate=0, want_dx=True, ws_bytes=None):
        """out: (dW1, db1, dW2, db2) to write into (accumulate reads them); else fresh NaN-filled buffers."""
        N = self.tt.ops.N
        M, H, P = self.M, self.H, self.P
        if out is None:
            out = tuple(torch.full(s, float("nan"), device=DEV) for s in ((P, H), (P,), (P, P), (P,)))
        dx = torch.full((M, H), float("nan"), device=DEV) if want_dx else None
        dyd = dy.contiguous().to(DEV)
        rc = self.lib.tt_encode_bwd(N.ptr(dyd), N.ptr(self.x), N.ptr(h), N.ptr(self.W1), N.ptr(self.W2), M, H, P,
                                    *(N.ptr(t) for t in out), N.ptr(dx), accumulate, self.prec, N.ptr(self.ws),
                                    self.ws_bytes if ws_bytes is None else ws_bytes, N.stream())
        torch.cuda.synchronize()
        return rc, out, dx


def mlp64(x, W1, b1, W2, b2, dy, gate):
    """Float64 forward and backward of one tower through the given ReLU gate: z, y and (dW1, db1, dW2, db2), dx."""
    x, W1, b1, W2, b2, dy = (t.double() for t in (x, W1, b1, W2, b2, dy))
    z = x @ W1.T + b1
    h = z * gate.double()
    y = h @ W2.T + b2
    dz = (dy @ W2) * gate.double()
    return z, y, (dz.T @ x, dz.sum(0), dy.T @ h, dy.sum(0)), dz @ W1


def check_mlp(tag, precision, got, want, z, gate, scale):
    g = MLP_GATES[precision]
    (h, y, grads, dx), (y64, grads64, dx64) = got, want
    flips = gate != (z > 0)
    band = 2.0 ** -7 * scale if precision == "bf16" else torch.full_like(z, KINK_BAND)
    e_h, r_h = row_rel(h, z.clamp_min(0))
    e_y, r_y = row_rel(y, y64)
    worst = []
    for nm, a, b in zip(("W1", "b1", "W2", "b2"), grads, grads64):
        worst.append((nm, rel_err(a, b), *block_err(a, b)))
    e_g = max(w[1] for w in worst)
    e_b = max(w[2] for w in worst)
    e_dx = row_rel(dx, dx64)[0] if dx is not None else 0.0
    print(f"fp32_shapes mlp {tag}: h {e_h:.2e} y {e_y:.2e} grad {e_g:.2e} block {e_b:.2e} dx {e_dx:.2e} "
          f"relu flips {int(flips.sum())}")
    assert not bool((flips & (z.abs() > band)).any()), (tag, "ReLU gate flip outside the rounding band")
    assert e_h < g["h"], (tag, "h row", r_h, e_h)
    assert e_y < g["y"], (tag, "y row", r_y, e_y)
    for nm, whole, blk, where in worst:
        assert whole < g["grad"], (tag, nm, "whole tensor", whole)
        assert blk < g["block"], (tag, nm, "block at", where, blk)
    assert e_dx < g["dx"], (tag, "dx row", e_dx)


def run_mlp_case(tt, precision, M, H, P, seed):
    """Raw ABI forward + backward against float64, then ops.mlp (autograd) must give the same bits."""
    x, W1, b1, W2, b2, dy = mlp_case(M, H, P, seed)
    raw = RawMlp(tt, precision, x, W1, b1, W2, b2)
    rc, h, y = raw.fwd()
    _call(tt, rc, "tt_encode_fwd")
    rc, grads, dx = raw.bwd(dy, h)
    _call(tt, rc, "tt_encode_bwd")
    hd, h, y = h, h.cpu(), y.cpu()
    gate = h > 0
    z, y64, grads64, dx64 = mlp64(x, W1, b1, W2, b2, dy, gate)
    scale = x.double().abs() @ W1.double().abs().T
    check_mlp((precision, M, H, P), precision, (h, y, [g.cpu() for g in grads], dx.cpu()), (y64, grads64, dx64), z,
              gate, scale)
    # the autograd surface: same kernels, same bits
    xd = x.to(DEV).requires_grad_(True)
    prm = [t.to(DEV).requires_grad_(True) for t in (W1, b1, W2, b2)]
    ya = tt.ops.mlp(xd, *prm, precision)
    ya.backward(dy.to(DEV))
    assert torch.equal(ya.detach().cpu(), y)
    for a, b in zip(prm, grads):
        assert torch.equal(a.grad, b)
    assert torch.equal(xd.grad, dx)
    return raw, hd, dy, grads, dx


M_LIST = [1, 63, 64, 65, 127, 129, 1025, 16512]
# M against one ragged P, every H at one ragged M, and the 32-split cap of the tensor-core weight gradients (M = 16512:
# 258 k-blocks of 64 rows cut to 29 non-empty splits)
MLP_SHAPES = [(M, 384, 192) for M in M_LIST] + [(129, H, 128) for H in (128, 256, 768)]
MLP_SHAPES += [(16512, 768, 64), (1025, 128, 576)]
# fp32 only: H and P off the 64-multiples, down to P = 1
MLP_FP32_SHAPES = [(65, 17, P) for P in (1, 16, 24, 100)] + [(1025, 100, P) for P in (1, 16, 24, 100)]
MLP_FP32_SHAPES += [(16512, 100, 24), (1, 17, 1), (129, 768, 100)]


@pytest.mark.parametrize("M,H,P", MLP_SHAPES, ids=[f"M{m}-H{h}-P{p}" for m, h, p in MLP_SHAPES])
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_encode_fwd_bwd_vs_float64(tt, precision, M, H, P):
    run_mlp_case(tt, precision, M, H, P, seed=20000 + M + H + P)


@pytest.mark.parametrize("M,H,P", MLP_FP32_SHAPES, ids=[f"M{m}-H{h}-P{p}" for m, h, p in MLP_FP32_SHAPES])
def test_encode_fwd_bwd_fp32_ragged_vs_float64(tt, M, H, P):
    run_mlp_case(tt, "fp32", M, H, P, seed=21000 + M + H + P)


ACC_CASES = [(p, M, 384, P) for p in ("fp32", "bf16x3", "bf16") for M, P in ((129, 192), (16512, 64))]
ACC_CASES += [("fp32", 65, 100, 24)]


@pytest.mark.parametrize("precision,M,H,P", ACC_CASES, ids=[f"{p}-M{m}-H{h}-P{q}" for p, m, h, q in ACC_CASES])
def test_encode_bwd_accumulate_and_no_dx(tt, precision, M, H, P):
    """accumulate = 1 adds to the outputs (within the gate of old + float64 new); dx = NULL leaves the other four outputs
    bit-identical."""
    raw, h, dy, grads, dx = run_mlp_case(tt, precision, M, H, P, seed=22000 + M + P)
    _, nodx, _ = raw.bwd(dy, h, want_dx=False)
    for a, b in zip(grads, nodx):
        assert torch.equal(a, b)
    gen = torch.Generator().manual_seed(M)
    old = [torch.randn(g.shape, generator=gen).to(DEV) * g.std() for g in grads]
    acc = tuple(o.clone() for o in old)
    rc, acc, _ = raw.bwd(dy, h, out=acc, accumulate=1)
    _call(tt, rc, "tt_encode_bwd(accumulate)")
    _, _, grads64, _ = mlp64(raw.x.cpu(), raw.W1.cpu(), raw.b1.cpu(), raw.W2.cpu(), raw.b2.cpu(), dy, h.cpu() > 0)
    g = MLP_GATES[precision]
    for nm, a, o, want in zip(("W1", "b1", "W2", "b2"), acc, old, grads64):
        e = rel_err(a, o.cpu().double() + want)
        print(f"fp32_shapes mlp accumulate {(precision, M, H, P, nm)}: grad {e:.2e}")
        assert e < g["grad"], (nm, e)


@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_encode_empty_batch_and_refusals(tt, precision):
    """M = 0: tt_encode_bwd writes zero gradients, or leaves them untouched with accumulate; tt_encode_fwd writes nothing.
    A workspace one byte short is refused, and so is H % 64 != 0 with a tensor-core precision."""
    x, W1, b1, W2, b2, dy = mlp_case(0, 128, 64, 1)
    raw = RawMlp(tt, precision, x, W1, b1, W2, b2)
    _call(tt, raw.fwd()[0], "tt_encode_fwd(M=0)")
    rc, out, _ = raw.bwd(dy, torch.zeros(0, 64, device=DEV), want_dx=False)
    _call(tt, rc, "tt_encode_bwd(M=0)")
    assert all(float(t.abs().max()) == 0.0 for t in out)
    old = tuple(torch.randn(t.shape, device=DEV) for t in out)
    keep = tuple(t.clone() for t in old)
    rc, out, _ = raw.bwd(dy, torch.zeros(0, 64, device=DEV), out=old, accumulate=1, want_dx=False)
    _call(tt, rc, "tt_encode_bwd(M=0, accumulate)")
    assert all(torch.equal(a, b) for a, b in zip(out, keep))
    # a workspace one byte short
    x, W1, b1, W2, b2, dy = mlp_case(65, 128, 64, 2)
    raw = RawMlp(tt, precision, x, W1, b1, W2, b2)
    rc, h, _ = raw.fwd(ws_bytes=raw.ws_bytes - 1)
    assert rc != 0 and "workspace" in tt.ops.N.last_error()
    rc, h, _ = raw.fwd()
    _call(tt, rc, "tt_encode_fwd")
    rc, _, _ = raw.bwd(dy, h, ws_bytes=raw.ws_bytes - 1)
    assert rc != 0 and "workspace" in tt.ops.N.last_error()
    if precision != "fp32":
        x, W1, b1, W2, b2, dy = mlp_case(65, 100, 64, 3)
        raw = RawMlp(tt, precision, x, W1, b1, W2, b2)
        rc, h, _ = raw.fwd()
        assert rc != 0 and "multiples of 64" in tt.ops.N.last_error()
        rc, _, _ = raw.bwd(dy, h)
        assert rc != 0 and "multiples of 64" in tt.ops.N.last_error()


# ---------------------------------------------------------------------------------------------------------------------
# C. tt_triplet_loss_fwd / tt_triplet_loss_bwd
# ---------------------------------------------------------------------------------------------------------------------
def loss_case(B, P, seed):
    """q, p, n [B, P]; from 4 rows on, row 0 of q and row 2 of n are zero and row 1 of p and row 3 of q are below the
    cosine's eps (|x| < 1e-8): torch clamps their norms, so their cosines have no norm term in the gradient."""
    gen = torch.Generator().manual_seed(seed)
    q, p, n = (torch.randn(B, P, generator=gen) for _ in range(3))
    if B >= 4:
        q[0] = 0
        n[2] = 0
        p[1] = torch.randn(P, generator=gen) * 1e-11
        q[3] = torch.randn(P, generator=gen) * 1e-11
    return q, p, n


def loss64(q, p, n, margin, inv_batch, dloss, active):
    """Float64 statistics, loss and gradients (of dloss · loss) through torch's clamped cosine, differentiated through
    the device's hinge activity."""
    q, p, n = (t.double().requires_grad_(True) for t in (q, p, n))
    cos_p, cos_n = cosine64(q, p), cosine64(q, n)
    pre = (1 - cos_p) - (1 - cos_n) + margin
    (dloss * inv_batch * (pre * active.double()).sum()).backward()
    with torch.no_grad():
        stats = torch.stack([cos_p, cos_n, pre.clamp_min(0), q.norm(dim=1), p.norm(dim=1), n.norm(dim=1), (q * p).sum(1),
                             (q * n).sum(1)], 1)
    return dict(stats=stats, pre=pre.detach(), loss=float(stats[:, 2].sum()) * inv_batch, grads=(q.grad, p.grad, n.grad))


def run_loss_case(tt, B, P, margin, inv_batch, dloss, seed):
    lib, N = _lib(tt), tt.ops.N
    q, p, n = loss_case(B, P, seed)
    qd, pd, nd = (t.to(DEV) for t in (q, p, n))
    stats = torch.full((B, 8), float("nan"), device=DEV)
    loss = torch.full((), float("nan"), device=DEV)
    _call(tt, lib.tt_triplet_loss_fwd(N.ptr(qd), N.ptr(pd), N.ptr(nd), B, P, margin, inv_batch, N.ptr(stats),
                                      N.ptr(loss), N.stream()), "tt_triplet_loss_fwd")
    grads = tuple(torch.full((B, P), float("nan"), device=DEV) for _ in range(3))
    dl = torch.tensor([dloss], device=DEV)
    _call(tt, lib.tt_triplet_loss_bwd(N.ptr(qd), N.ptr(pd), N.ptr(nd), N.ptr(stats), N.ptr(dl), B, P, inv_batch,
                                      *(N.ptr(g) for g in grads), N.stream()), "tt_triplet_loss_bwd")
    torch.cuda.synchronize()
    stats, loss, grads = stats.cpu(), float(loss.item()), [g.cpu() for g in grads]
    active = stats[:, 2] > 0
    o = loss64(q, p, n, margin, inv_batch, dloss, active)
    tag = (B, P, margin)
    e_loss = abs(loss - o["loss"]) / max(abs(o["loss"]), 1e-30) if o["loss"] else abs(loss)
    e_stats, r_s = stats_err(stats, o["stats"])
    # gradient rows: relative to the row, floored at the scale of the cosine's gradient, |dloss| inv_batch / max(|x|, eps)
    # (at P = 1 the cosine is constant and the float64 gradient is 0); rows of inactive triplets are exactly zero
    gh = abs(dloss) * inv_batch
    e_g = 0.0
    for x, got, want in zip((q, p, n), grads, o["grads"]):
        floor = gh / x.double().norm(dim=1).clamp_min(COS_EPS)
        err = (got.double() - want).norm(dim=1) / torch.maximum(want.norm(dim=1), floor)
        assert int((got[~active] != 0).sum()) == 0, (tag, "inactive triplet with a gradient")
        if bool(active.any()):
            e_g = max(e_g, float(err[active].max()))
    hinge_flips = active != (o["pre"] > 0)
    print(f"fp32_shapes loss B{B} P{P} margin {margin}: loss {e_loss:.2e} stats {e_stats:.2e} grad rows {e_g:.2e} "
          f"active {int(active.sum())}/{B} hinge flips {int(hinge_flips.sum())}")
    assert not bool((hinge_flips & (o["pre"].abs() > HINGE_BAND)).any()), (tag, "hinge activity")
    assert e_loss < LOSS_GATES["loss"], (tag, "loss", loss, o["loss"])
    assert e_stats < LOSS_GATES["stats"], (tag, "stats row", r_s, stats[r_s], o["stats"][r_s])
    assert e_g < LOSS_GATES["grad"], (tag, "gradient row", e_g)
    return o, active


LOSS_B = [1, 3, 4, 5, 1023, 1025, 8256]
LOSS_P = [1, 31, 32, 33, 100, 512]


@pytest.mark.parametrize("P", LOSS_P)
@pytest.mark.parametrize("B", LOSS_B)
def test_triplet_loss_fwd_bwd_vs_float64(tt, B, P):
    """One warp per triplet over P columns (P = 31 / 32 / 33 around the warp width); above 1024 rows the loss reduction
    takes its strided path.  inv_batch is not 1/B and the upstream gradient is not 1."""
    run_loss_case(tt, B, P, 0.3, 0.37 / B, 2.5, seed=30000 + B * 7 + P)


@pytest.mark.parametrize("B,P", [(5, 33), (1025, 100), (8256, 512)])
@pytest.mark.parametrize("margin", [-3.0, 2.5])
def test_triplet_loss_hinge_edges_vs_float64(tt, margin, B, P):
    """margin -3: every hinge exactly inactive (loss 0, every gradient exactly 0); 2.5: every hinge active."""
    o, active = run_loss_case(tt, B, P, margin, 1.0 / B, 1.0, seed=31000 + B + P)
    assert int(active.sum()) == (B if margin > 0 else 0)


# ---------------------------------------------------------------------------------------------------------------------
# D. Adam
# ---------------------------------------------------------------------------------------------------------------------
# The kernels form 1 - beta in fp32 from the fp32 beta (1 - 0.999f = 9.9987e-4, not 1e-3), and their bias corrections
# raise the fp32 beta.  The oracle therefore replays torch.optim.Adam's single-tensor formula in float64 with the
# fp32-rounded betas (and the fp32-rounded grad_scale): any remaining difference is the kernels' fp32 rounding.
HYPER = {"default": (1e-3, 0.9, 0.999, 1e-8), "custom": (2e-2, 0.8, 0.95, 1e-6)}
ADAM_CASES = [(1, "default"), (0.25, "custom"), (1 / 3, "default")]


@pytest.mark.parametrize("scale,hyper", ADAM_CASES, ids=["scale1-default", "scale0.25-custom", "scale1/3-default"])
@pytest.mark.parametrize("variant", ["host_step", "dev_state"])
@pytest.mark.parametrize("n", [1, 3, 255, 256, 257, 4097, 2 ** 20 + 3])
def test_adam_update_vs_float64(tt, n, variant, scale, hyper):
    """Every step: the update p_t - p_{t-1}, m and v (relative errors as ADAM_GATES states).  2000 steps at small n,
    so the double beta powers of tt_adam_step_dev run far; elements whose gradient is always exactly zero must not
    move and keep zero moments."""
    lib, N = _lib(tt), tt.ops.N
    lr, beta1, beta2, eps = HYPER[hyper]
    f32 = lambda v: float(np.float32(v))  # noqa: E731
    b1, b2, gs, lr32, eps32 = f32(beta1), f32(beta2), f32(scale), f32(lr), f32(eps)
    steps = 2000 if n <= 257 else (20 if n < 2 ** 20 else 3)
    gen = torch.Generator().manual_seed(n)
    p0 = torch.randn(n, generator=gen) * 0.05  # the projections' scale (nn.Linear's bound 1/sqrt(384) = 0.051)
    zero = torch.zeros(n, dtype=torch.bool)
    zero[:: 3] = n >= 3  # every third element of a long vector has an always-zero gradient
    p, m, v = p0.to(DEV), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    state = torch.zeros(4, dtype=torch.float64, device=DEV)
    hist = torch.empty(steps, 3, n, device=DEV) if n <= 257 else None
    P64, M64, V64 = p0.double(), torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
    # gradients of varied magnitude, some steps much larger than others (what a bias correction must survive)
    grads = []
    for t in range(steps):
        g = torch.randn(n, generator=gen) * (0.1 if t % 7 else 3.0) * torch.exp(torch.randn(n, generator=gen))
        g[zero] = 0.0
        grads.append(g)
    worst = dict(update=0.0, m=0.0, v=0.0)

    def compare(t, p_prev, p_now, m_now, v_now):
        nonlocal P64, M64, V64
        g64 = grads[t].double() * gs
        M64 = M64 + (g64 - M64) * (1 - b1)
        V64 = V64 * b2 + (1 - b2) * g64 * g64
        bc1, bc2 = 1 - b1 ** (t + 1), 1 - b2 ** (t + 1)
        upd64 = -(lr32 / bc1) * M64 / (V64.sqrt() / bc2 ** 0.5 + eps32)
        upd = p_now.double() - p_prev.double()
        # floors: with one or three elements, m can sit near zero in a step (a relative error of an update much
        # smaller than the step size says nothing); Adam's updates are of the order of lr / bc1, m of sqrt(v)
        den = max(float(upd64.abs().max()), lr32 / bc1)
        worst["update"] = max(worst["update"], float((upd - upd64).abs().max()) / den)
        den = max(float(M64.abs().max()), float(V64.max()) ** 0.5, 1e-30)
        worst["m"] = max(worst["m"], float((m_now.double() - M64).abs().max()) / den)
        worst["v"] = max(worst["v"], float((v_now.double() - V64).abs().max() / V64.abs().max().clamp_min(1e-30)))
        if bool(zero.any()):
            assert float(upd[zero].abs().max()) == 0.0 and float(m_now[zero].abs().max()) == 0.0, t
            assert float(v_now[zero].abs().max()) == 0.0, t

    p_prev = p0
    for t in range(steps):
        gd = grads[t].to(DEV, non_blocking=True)
        if variant == "host_step":
            rc = lib.tt_adam_step(N.ptr(p), N.ptr(gd), N.ptr(m), N.ptr(v), n, lr, beta1, beta2, eps, t + 1, scale,
                                  N.stream())
        else:
            rc = lib.tt_adam_step_dev(N.ptr(p), N.ptr(gd), N.ptr(m), N.ptr(v), n, lr, beta1, beta2, eps, N.ptr(state),
                                      scale, N.stream())
        _call(tt, rc, variant)
        if hist is not None:
            hist[t, 0].copy_(p); hist[t, 1].copy_(m); hist[t, 2].copy_(v)  # noqa: E702
        else:
            pc, mc, vc = p.cpu(), m.cpu(), v.cpu()
            compare(t, p_prev, pc, mc, vc)
            p_prev = pc
    if hist is not None:
        hc = hist.cpu()
        for t in range(steps):
            compare(t, p_prev, hc[t, 0], hc[t, 1], hc[t, 2])
            p_prev = hc[t, 0]
    if variant == "dev_state":
        st = state.cpu()
        assert float(st[0]) == steps
        assert abs(float(st[1]) - b1 ** steps) <= 1e-12 * b1 ** steps + 1e-300
        assert abs(float(st[2]) - b2 ** steps) <= 1e-12 * b2 ** steps + 1e-300
    print(f"fp32_shapes adam n {n} {variant} scale {scale:.3g} {hyper}: update {worst['update']:.2e} "
          f"m {worst['m']:.2e} v {worst['v']:.2e}")
    assert worst["update"] < ADAM_GATES["update"], worst
    assert worst["m"] < ADAM_GATES["moments"] and worst["v"] < ADAM_GATES["moments"], worst
