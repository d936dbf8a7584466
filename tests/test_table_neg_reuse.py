"""In-batch negatives named by index (tt_step_args.neg_index) with trainable token tables: every negative's table-gradient
row g_n[i] is folded into the positive it copies, in ascending i, and the document table sums over the positives' tokens
only.

1. The promised order, bit for bit: against a twin step that gathers the negatives' own tokens, loss, pooled rows, the 8
   projection gradients and dtable_q are bit-identical; dtable_d is bit-identical to a float32 replay (the fold, then the
   sorted-segment sum over the positives' occurrences) and within TAU_B of the float64 sum over all p and n occurrences.
2. grad_accumulate = 1 adds fl(old + new).
3. The fused table Adam with neg_index equals gradients with neg_index, then tt_adam_step_dev, bit for bit.
4. FusedTrainer(in_batch_negatives=True, optimize_tables=True) against the same trainer without reuse; schedules,
   checkpoints and the error flag.
5. The device feeder and run_training's default.
6. The refusals that stay.
"""
import os

import numpy as np
import pytest
import torch

from test_pool_shapes import TAU_B, TINY_ID, ZERO_ID, bits, check_table_grad, grad_table, make_step, occurrences, replay
from test_table_training import LR, _adam_dev, _batch, _model, _tables, _trainer

pytestmark = pytest.mark.gpu

DEV = "cuda"
HEAVY_A, HEAVY_B = 101, 1996  # B and 8B entries among the positives' tokens


@pytest.fixture(scope="module")
def tt():
    import two_towers_overlords_b200 as pkg
    from two_towers_overlords_b200 import _native, data, ops, training

    pkg.ops, pkg.training, pkg.data, pkg._native = ops, training, data, _native
    return pkg


@pytest.fixture
def chain_env():
    old = os.environ.get("TT_CHAIN")
    yield
    if old is None:
        os.environ.pop("TT_CHAIN", None)
    else:
        os.environ["TT_CHAIN"] = old


def neg_pattern(kind, B, gen):
    """int64 [B]: negative i copies positive neg[i]."""
    if kind == "self":
        assert B == 1
        return torch.zeros(1, dtype=torch.int64)
    if kind == "derangement":  # one cycle through a random order: no fixed point
        perm = torch.randperm(B, generator=gen)
        neg = torch.empty(B, dtype=torch.int64)
        neg[perm] = torch.roll(perm, -1)
        return neg
    if kind == "roll3":  # positive 5 named three times, positives 0 and 1 never
        neg = torch.roll(torch.arange(B), 1)
        neg[1] = neg[2] = 5
        return neg
    if kind == "zero":
        return torch.zeros(B, dtype=torch.int64)
    raise ValueError(kind)


def fold_tokens(B, Lq, Ld, V, seed):
    """q and p token sets (int32 ids, uint8 masks): ragged masks, two heavy ids among the positives alone (B and 8B
    entries: more than 256 from B = 300, more than 2048 from B = 257), ids >= 65536 when V allows, a zero-norm and a
    tiny-norm positive, an all-masked positive and an all-masked query."""
    gen = torch.Generator().manual_seed(seed)
    q_ids = torch.randint(0, V, (B, Lq), generator=gen)
    p_ids = torch.randint(0, V, (B, Ld), generator=gen)
    q_ids[:, 0] = 102
    p_ids[:, 1] = HEAVY_A
    p_ids[:, 2:10] = HEAVY_B
    if V > 65536:
        p_ids[:, 10] = 65536 + 17
    masks = []
    for L, full in ((Lq, 1), (Ld, 10)):  # the heavy columns are never masked
        lens = torch.randint(1, L + 1, (B, 1), generator=gen)
        m = (torch.arange(L)[None] < lens) & (torch.rand(B, L, generator=gen) < 0.9)
        m[:, :full] = True
        masks.append(m.to(torch.uint8))
    if B >= 5:
        p_ids[2], masks[1][2] = ZERO_ID, 1  # zero norm: the clamped branch of g
        p_ids[3], masks[1][3] = TINY_ID, 1
        masks[1][4] = 0                     # all masked
        masks[0][3] = 0
    return q_ids.to(torch.int32), masks[0], p_ids.to(torch.int32), masks[1]


def fold64(G, neg, B):
    """The fold in float32 on the CPU: g_p[j] = ((g_p[j] + g_n[i1]) + g_n[i2]) + ... in ascending i."""
    F = G.clone()
    for i, j in enumerate(neg.tolist()):
        if 0 <= j < B:
            F[B + j] = F[B + j] + G[2 * B + i]
    return F


def twin_steps(tt, B, Lq, Ld, H, V, precision, chain, kind, seed):
    """(so_reuse, so_twin, tokens, neg, tables, dtables of both): the same step with neg_index and poisoned negative
    tokens (ids V - 1, all-ones mask), and with the negatives' own tokens gathered."""
    gen = torch.Generator().manual_seed(seed)
    tables = tuple(grad_table(V, H, gen).to(DEV) for _ in range(2))
    q_ids, q_mask, p_ids, p_mask = fold_tokens(B, Lq, Ld, V, seed)
    neg = neg_pattern(kind, B, gen)
    twin_tok = (q_ids, q_mask, p_ids, p_mask, p_ids[neg].clone(), p_mask[neg].clone())
    reuse_tok = (q_ids, q_mask, p_ids, p_mask, torch.full_like(p_ids, V - 1), torch.ones_like(p_mask))
    so_r, tg_r = make_step(tt, B, Lq, Ld, H, V, precision, tables, reuse_tok, train_table=True, chain=chain, seed=seed)
    so_t, tg_t = make_step(tt, B, Lq, Ld, H, V, precision, tables, twin_tok, train_table=True, chain=chain, seed=seed)
    nd = neg.to(torch.int32).to(DEV)
    so_r.set_neg_index(0, nd)
    so_r._test_neg = nd
    return so_r, so_t, twin_tok, neg, tables, tg_r, tg_t


# ---------------------------------------------------------------------------------------------------------------------
# 1. the promised order
# ---------------------------------------------------------------------------------------------------------------------
# (precision, chain, B, H, V, index pattern): every precision and chain mode, B in {1, 129, 300, 2100}, every H, the three
# vocabularies (70000: ids >= 65536), the four index patterns
FOLD_CASES = [("fp32", 0, 300, 384, 30522, "derangement"), ("fp32", 0, 129, 768, 4096, "roll3"),
              ("fp32", 0, 1, 128, 4096, "self"), ("bf16x3", 1, 300, 384, 30522, "roll3"),
              ("bf16x3", 1, 2100, 384, 30522, "derangement"), ("bf16x3", 2, 129, 128, 70000, "zero"),
              ("bf16x3", 2, 300, 768, 30522, "derangement"), ("bf16x3", 1, 1, 384, 4096, "self"),
              ("bf16", 1, 129, 768, 70000, "derangement"), ("bf16", 2, 300, 128, 4096, "roll3"),
              ("bf16", 1, 2100, 128, 4096, "zero"), ("bf16", 2, 1, 768, 30522, "self")]


@pytest.mark.parametrize("precision,chain,B,H,V,kind", FOLD_CASES)
def test_fold_is_the_promised_sum(tt, precision, chain, B, H, V, kind):
    Lq, Ld = 8, 24
    so_r, so_t, tok, neg, tables, (dq_r, dd_r), (dq_t, dd_t) = twin_steps(tt, B, Lq, Ld, H, V, precision, chain, kind,
                                                                          seed=B + H + V)
    so_r.run()
    so_t.run()
    torch.cuda.synchronize()
    assert int(so_r.err.item()) == 0 and int(so_t.err.item()) == 0
    tag = (precision, chain, B, H, V, kind)
    vr, vt = so_r._views(), so_t._views()
    assert torch.equal(bits(so_r.loss), bits(so_t.loss)), tag
    for name in ("xhat", "cnt", "nrm", "dxhat"):
        assert torch.equal(bits(vr[name]), bits(vt[name])), (tag, name)
    for gr, gt in zip(so_r._test_keep[1], so_t._test_keep[1]):
        assert torch.equal(bits(gr), bits(gt)), (tag, "projection gradient")
    assert torch.equal(bits(dq_r), bits(dq_t)), (tag, "dtable_q")
    # the fold itself: positives' g rows as promised, the other rows untouched
    G = vt["g"].detach().cpu().clone()
    F = fold64(G, neg, B)
    assert torch.equal(bits(vr["g"]), bits(F)), (tag, "folded g")
    if B >= 5:
        n, c = vt["nrm"][B:2 * B, 0].cpu(), vt["cnt"][B:2 * B, 0].cpu()
        assert bool(((n < 1e-12) & (c > 0)).any()), (tag, "a clamped positive")
    # dtable_d: bit-identical to the replay over the positives' occurrences of the folded g
    occ = occurrences([(tok[2], tok[3], B)])
    want = replay(F, occ[0], occ[1], V)
    bad = (bits(dd_r) != bits(want)).any(1).nonzero()[:, 0]
    assert len(bad) == 0, (tag, "dtable_d rows not bit-identical to the replay", bad[:8].tolist(), len(bad))
    # and within TAU_B of the float64 sum over all p and n occurrences (untouched rows exactly 0)
    ids = torch.cat([tok[2], tok[4]]).long()
    mask = torch.cat([tok[3], tok[5]]).long()
    worst = check_table_grad(tag, dd_r, tables[1].cpu(), ids, mask, vt["dxhat"][B:].detach().cpu())
    if V - 1 not in set(ids[mask != 0].tolist()):
        assert float(dd_r[V - 1].abs().max()) == 0.0  # the poisoned negative tokens were never read
    print(f"neg reuse fold {tag}: bit-identical replay, float64 {worst:.2e} (gate {TAU_B:.0e})")


# ---------------------------------------------------------------------------------------------------------------------
# 2. accumulation
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision,chain", [("fp32", 0), ("bf16x3", 1), ("bf16", 2)])
def test_accumulate_adds_old_plus_new(tt, precision, chain):
    B, Lq, Ld, H, V = 300, 8, 24, 384, 4096
    so, _, _, _, _, (dq, dd), _ = twin_steps(tt, B, Lq, Ld, H, V, precision, chain, "roll3", seed=4)
    so.run()
    torch.cuda.synchronize()
    new = (dq.clone(), dd.clone())
    gen = torch.Generator().manual_seed(8)
    old = tuple(torch.randn(t.shape, generator=gen).to(DEV) for t in new)
    for t, o in zip((dq, dd), old):
        t.copy_(o)
    so.run(accumulate=True)
    torch.cuda.synchronize()
    for got, o, n in zip((dq, dd), old, new):
        assert torch.equal(bits(got), bits(o + n)), precision


# ---------------------------------------------------------------------------------------------------------------------
# 3. the fused table Adam
# ---------------------------------------------------------------------------------------------------------------------
def _poisoned(b, V):
    """_batch's tokens with the negatives replaced by ids V - 1 / all-ones masks (never read with neg_index)."""
    return b[:4] + (torch.full_like(b[4], V - 1), torch.ones_like(b[5]))


def _twin_batch(b, neg):
    return b[:4] + (b[2][neg].clone(), b[3][neg].clone())


@pytest.mark.parametrize("precision,chain,H,V,B", [("fp32", 0, 384, 4096, 300), ("bf16x3", 1, 768, 30522, 1100),
                                                   ("bf16x3", 2, 128, 4096, 300), ("bf16", 1, 384, 4096, 1100)])
def test_fused_table_adam_with_neg_index(tt, chain_env, precision, chain, H, V, B):
    """optimize_tables=True with neg_index leaves the tables, their moments and the projections bit-identical to a
    gradients-only trainer with neg_index whose steps are followed by tt_adam_step_dev on each table."""
    P, Lq, Ld = 128, 12, 24
    os.environ["TT_CHAIN"] = "1" if chain == 1 else "0"
    ma, mb = _model(tt, P, V, H, precision, 3), _model(tt, P, V, H, precision, 3)
    ta = _trainer(tt, ma, B, Lq, Ld, precision, use_graph=False, optimize_tables=True, in_batch_negatives=True)
    tb = _trainer(tt, mb, B, Lq, Ld, precision, use_graph=False, in_batch_negatives=True)
    mom = [torch.zeros_like(t) for t in _tables(mb) for _ in range(2)]
    gen = torch.Generator().manual_seed(B)
    for i in range(3):
        b = _poisoned(_batch(B, Lq, Ld, V, 100 + i, heavy=True), V)
        neg = neg_pattern("derangement" if i % 2 == 0 else "roll3", B, gen)
        for tr in (ta, tb):
            tr.load_packed(tr.pack_host_tokens(b, pin=False))
            tr.load_neg_index(neg)
        st0 = tb.adam_state.clone()
        la, lb = float(ta.step().item()), float(tb.step().item())
        assert la == lb
        for k, (p, g) in enumerate(zip(_tables(mb), tb.table_grads)):
            _adam_dev(tt, p.data, g, mom[2 * k], mom[2 * k + 1], st0.clone())
        torch.cuda.synchronize()
        for x, y in zip(_tables(ma), _tables(mb)):
            assert torch.equal(x, y), (i, precision, chain)
        for x, y in zip(ta.table_exp_avg + ta.table_exp_avg_sq, mom[0::2] + mom[1::2]):
            assert torch.equal(x, y), i
        assert torch.equal(ta.flat_p, tb.flat_p)
    assert int(ta.step_obj.err.item()) == 0


# ---------------------------------------------------------------------------------------------------------------------
# 4. the trainer end to end
# ---------------------------------------------------------------------------------------------------------------------
def _batches(B, Lq, Ld, V, n, seed):
    gen = torch.Generator().manual_seed(seed)
    out = []
    for i in range(n):
        b = _batch(B, Lq, Ld, V, seed + i)
        out.append((b, neg_pattern("derangement" if i % 2 == 0 else "roll3", B, gen)))
    return out


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_trainer_with_reuse_matches_the_trainer_without(tt, precision):
    """3 steps with and without reuse: step-1 loss bit-identical, losses 1e-4, projections 1e-3; tables under the
    elementwise rule of test_fused_trainer_matches_the_reference_shaped_loop (the reference gradient is the no-reuse
    trainer's own table gradient of each step); never-touched rows bit-identical to their initial values."""
    B, Lq, Ld, V, P, H = 256, 16, 48, 4096, 128, 384
    mf, mr = _model(tt, P, V, H, precision, 11), _model(tt, P, V, H, precision, 11)
    init = [t.detach().clone() for t in _tables(mr)]
    tf = _trainer(tt, mf, B, Lq, Ld, precision, use_graph=True, optimize_tables=True, in_batch_negatives=True)
    tr = _trainer(tt, mr, B, Lq, Ld, precision, use_graph=False, optimize_tables=True)
    ok = [torch.ones_like(t, dtype=torch.bool) for t in init]
    touched = [torch.zeros(V, dtype=torch.bool, device=DEV) for _ in init]
    for i, (b, neg) in enumerate(_batches(B, Lq, Ld, V, 3, 300)):
        tf.load_packed(tf.pack_host_tokens(_poisoned(b, V), pin=False))
        tf.load_neg_index(neg)
        bt = _twin_batch(b, neg)
        tr.load_packed(tr.pack_host_tokens(bt, pin=False))
        tr._fwd_bwd()  # gradients only: the reference table gradient of this step
        for k, g in enumerate(tr.table_grads):
            bound = 1e-3 * g.abs().max()
            ok[k] &= (g == 0) | (g.abs() > 10 * bound)
        lf, lr_ = float(tf.step().item()), float(tr.step().item())
        if i == 0:
            assert lf == lr_, (lf, lr_)
        assert abs(lf - lr_) <= 1e-4 * abs(lr_), (i, lf, lr_)
        touched[0][bt[0][bt[1] != 0].to(DEV)] = True
        touched[1][torch.cat([bt[2], bt[4]])[torch.cat([bt[3], bt[5]]) != 0].to(DEV)] = True
    torch.cuda.synchronize()
    assert int(tf.step_obj.err.item()) == 0
    for x, y in zip(mf.projection_parameters(), mr.projection_parameters()):
        assert float((x - y).detach().norm() / y.detach().norm()) < 1e-3
    for k, (a, b_, t0) in enumerate(zip(_tables(mf), _tables(mr), init)):
        du, ur = (a - t0).detach(), (b_ - t0).detach()
        sel = ok[k] & touched[k][:, None]
        err = (du - ur).abs()
        assert float(err[sel].max()) <= 0.02 * LR, float(err[sel].max())
        rest = touched[k][:, None] & ~ok[k]
        n_touched = int(touched[k].sum()) * du.shape[1]
        assert int((rest & (err > 0.02 * LR)).sum()) <= 1e-3 * n_touched + 16
        assert float(err.max()) <= 6 * LR
        cold = ~touched[k]
        assert torch.equal(a[cold], t0[cold]) and torch.equal(b_[cold], t0[cold])
    tf.close()
    tr.close()


@pytest.mark.parametrize("a", [1, 2])
def test_schedules_with_reuse_are_bit_identical(tt, a):
    """Eager, graph replay and 2 token slots with reuse: tables, table moments, projections, step count and losses."""
    B, Lq, Ld, P, V, H = 256, 16, 48, 128, 4096, 384
    batches = _batches(B, Lq, Ld, V, 5, 400)
    out = []
    for mode in ("eager", "graph", "slots"):
        m = _model(tt, P, V, H, "bf16x3", 21)
        tr = _trainer(tt, m, B, Lq, Ld, "bf16x3", use_graph=mode != "eager", accumulation_steps=a,
                      optimize_tables=True, in_batch_negatives=True, token_slots=2 if mode == "slots" else 1)
        tr.prepare()
        tr.start_epoch()
        losses = []
        for i, (b, neg) in enumerate(batches):
            slot = i % 2 if mode == "slots" else 0
            tr.load_packed(tr.pack_host_tokens(_poisoned(b, V), pin=False), slot)
            tr.load_neg_index(neg, slot)
            losses.append(float(tr.step(slot).item()))
        torch.cuda.synchronize()
        assert int(tr.step_obj.err.item()) == 0
        out.append(([t.detach().clone() for t in _tables(m)] + [tr.flat_p.clone(), tr.adam_state.clone(),
                                                                tr._table_m.clone(), tr._table_v.clone()], losses))
        tr.close()
    for other in out[1:]:
        assert out[0][1] == other[1]
        for x, y in zip(out[0][0], other[0]):
            assert torch.equal(x, y)
    assert int(out[0][0][3][0].item()) == len(batches) // a


@pytest.mark.parametrize("a", [1, 2])
def test_resume_with_reuse_is_bit_exact(tt, tmp_path, a):
    """Save after 3 of 6 micro-steps (inside an open window at a = 2) and resume in a trainer built from another seed:
    the negative indices are per-slot inputs like the tokens, so no new state is needed."""
    B, Lq, Ld, P, V, H = 128, 16, 48, 64, 4096, 128
    batches = _batches(B, Lq, Ld, V, 6, 500)

    def make(seed):
        return _trainer(tt, _model(tt, P, V, H, "bf16x3", seed), B, Lq, Ld, "bf16x3", accumulation_steps=a,
                        optimize_tables=True, in_batch_negatives=True)

    def feed(tr, bs):
        for b, neg in bs:
            tr.load_packed(tr.pack_host_tokens(_poisoned(b, V), pin=False))
            tr.load_neg_index(neg)
            tr.step()

    def state(tr):
        torch.cuda.synchronize()
        return [t.detach().clone() for t in _tables(tr.model)] + [tr._table_m.clone(), tr._table_v.clone(),
                                                                  tr.flat_p.clone(), tr.adam_state.clone()]

    t1 = make(9)
    t1.start_epoch()
    feed(t1, batches)
    want = state(t1)
    t2 = make(9)
    t2.start_epoch()
    feed(t2, batches[:3])
    ck = str(tmp_path / "reuse.ckpt")
    t2.save_checkpoint(ck)
    t3 = make(123)
    t3.load_checkpoint(ck)
    feed(t3, batches[3:])
    for x, y in zip(want, state(t3)):
        assert torch.equal(x, y)
    for t in (t1, t2, t3):
        t.close()


def test_out_of_range_index_raises_the_flag_and_the_next_step_is_unaffected(tt):
    """A negative index outside [0, B) raises the error flag and folds nothing; after it (gradients only), the next valid
    step equals a twin's that never saw it."""
    B, Lq, Ld, P, V, H = 128, 16, 48, 64, 2048, 128
    ma, mb = _model(tt, P, V, H, "bf16x3", 2), _model(tt, P, V, H, "bf16x3", 2)
    ta = _trainer(tt, ma, B, Lq, Ld, "bf16x3", use_graph=False, optimize_tables=True, in_batch_negatives=True)
    tb = _trainer(tt, mb, B, Lq, Ld, "bf16x3", use_graph=False, optimize_tables=True, in_batch_negatives=True)
    (b, neg), = _batches(B, Lq, Ld, V, 1, 600)
    bad = neg.clone()
    bad[5] = B
    for tr in (ta, tb):
        tr.load_packed(tr.pack_host_tokens(_poisoned(b, V), pin=False))
    ta.load_neg_index(bad)
    ta._fwd_bwd()  # gradients only
    torch.cuda.synchronize()
    assert int(ta.step_obj.err.item()) != 0
    ta.step_obj.err.zero_()
    for tr in (ta, tb):
        tr.load_neg_index(neg)
        tr.step()
    torch.cuda.synchronize()
    assert int(ta.step_obj.err.item()) == 0
    for x, y in zip(_tables(ma) + [ta.flat_p, ta._table_m, ta._table_v],
                    _tables(mb) + [tb.flat_p, tb._table_m, tb._table_v]):
        assert torch.equal(x, y)
    ta.close()
    tb.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. the device feeder and run_training
# ---------------------------------------------------------------------------------------------------------------------
def test_device_fed_epoch_with_reuse_trains_the_tables(tt):
    B = 256
    ds = tt.data.MSMarcoDataset("train", max_samples=2000, random_seed=42, synthetic=True)
    first = []
    for reuse in (True, False):
        torch.manual_seed(0)
        m = tt.TwoTowersModel(projection_dim=64, precision="bf16x3", train_table=True).to(DEV)
        tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, 32, 256, token_slots=2, ids_dtype=torch.uint16,
                                      mask_dtype=torch.uint8, in_batch_negatives=reuse, optimize_tables=True)
        feeder = tt.data.DeviceTripletFeeder(ds, B, 32, 256, DEV, seed=5)
        feeder.start_epoch()
        tr.start_epoch()
        feeder.assemble(tr, 0, 0)
        first.append(float(tr.step(0).item()))
        tr.close()
    assert first[0] == first[1], first
    torch.manual_seed(0)
    m = tt.TwoTowersModel(projection_dim=64, precision="bf16x3", train_table=True).to(DEV)
    init = [t.detach().clone() for t in _tables(m)]
    tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, 32, 256, token_slots=2, ids_dtype=torch.uint16,
                                  mask_dtype=torch.uint8, in_batch_negatives=True, optimize_tables=True)
    feeder = tt.data.DeviceTripletFeeder(ds, B, 32, 256, DEV, seed=5)
    avg = tr.train_epoch_device(feeder)
    torch.cuda.synchronize()
    assert np.isfinite(avg)
    assert int(tr.step_obj.err.item()) == 0 and int(feeder.err.item()) == 0
    for t, t0 in zip(_tables(m), init):
        assert not torch.equal(t, t0) and bool(torch.isfinite(t).all())
    tr.close()


@pytest.mark.parametrize("env", [{}, {"TT_NEG_REUSE": "0"}, {"TT_HOST_FEEDER": "1"}], ids=["default", "off", "host"])
def test_run_training_reuses_the_negatives_with_trainable_tables(tt, monkeypatch, env):
    monkeypatch.setenv("TT_SYNTHETIC_DATA", "1")
    for k in ("TT_TRAIN_TABLE", "TT_NEG_REUSE", "TT_HOST_FEEDER"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    seen = []
    real = tt.training.FusedTrainer

    def spy(*args, **kw):
        seen.append(kw.get("in_batch_negatives", False))
        return real(*args, **kw)

    monkeypatch.setattr(tt.training, "FusedTrainer", spy)
    torch.manual_seed(0)
    tt.training.run_training(num_epochs=1, batch_size=256, learning_rate=1e-3, max_samples=2000, projection_dim=64,
                             margin=0.3, use_wandb=False, accumulation_steps=1, use_mixed_precision=False,
                             num_workers=0, run_comprehensive_test=False, train_table=True)
    assert seen == [not env], seen


# ---------------------------------------------------------------------------------------------------------------------
# 6. the refusals that stay
# ---------------------------------------------------------------------------------------------------------------------
def test_refusals_that_stay(tt):
    B, Lq, Ld, P, V, H = 64, 8, 16, 64, 2048, 128
    m = _model(tt, P, V, H, "bf16x3", 1)
    with pytest.raises(ValueError, match="other ranks"):
        _trainer(tt, m, B, Lq, Ld, "bf16x3", optimize_tables=True, in_batch_negatives=True, world_size=2)
    # the ABI: pooled rows together with neg_index stay exclusive
    frozen = tt.TwoTowersModel(projection_dim=P, vocab_size=V, hidden_size=H).to(DEV)
    so = tt.ops.TripletStep(B, Lq, Ld, H, P, V, "bf16x3", DEV)
    params = list(frozen.projection_parameters())
    grads = [torch.zeros_like(p) for p in params]
    rows = torch.zeros(4, H, device=DEV)
    so.bind(None, None, [p.data for p in params], grads, 0.3, 1.0 / B, 1.0)
    so.bind_pooled(rows, rows)
    so.set_pooled_index(0, torch.zeros(3 * B, dtype=torch.int32, device=DEV))
    so.set_neg_index(0, torch.zeros(B, dtype=torch.int32, device=DEV))
    N = tt._native
    import ctypes

    assert so.lib.tt_triplet_step(ctypes.byref(so.slots[0]), N.stream()) != 0
    assert "exclusive" in N.last_error()
