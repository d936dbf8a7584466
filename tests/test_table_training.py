"""Trainable token tables on the fused path (tt_step_args.table_*, TripletStep.bind_table_adam,
FusedTrainer(optimize_tables=True), run_training(train_table=...)): the Adam step in the scatter-add's epilogue against
the unfused form (gradients, then tt_adam_step_dev) bit for bit, against a float64 replay of torch.optim.Adam, and end
to end against the reference-shaped loop; bit-identical schedules, the exchange at table size, checkpoints and the
refusals."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import two_towers_oracle as O

DEV = "cuda"
LR = 1e-3


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


def _batch(B, Lq, Ld, V, seed, heavy=False):
    """Random ids in [1, V / 2) with ragged masks (masked positions hold ids too): row 0 and the upper half of the
    table are never touched.  heavy: a constant id in every query row
    (B entries: a heavy row of one chunk above 256) and another one in every document row (2B entries: more than 2048
    at B >= 1100, several chunks)."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for L in (Lq, Ld, Ld):
        ids = torch.randint(1, V // 2, (B, L), generator=g)
        n = torch.randint(1, L + 1, (B,), generator=g)
        mask = (torch.arange(L)[None, :] < n[:, None]).to(torch.int64)
        out += [ids, mask]
    if heavy:
        out[0][:, 0] = 5
        out[1][:, 0] = 1
        for i in (2, 4):
            out[i][:, 0] = 7
            out[i + 1][:, 0] = 1
    return tuple(out)


def _model(tt, P, V, H, precision, seed):
    torch.manual_seed(seed)
    return tt.TwoTowersModel(projection_dim=P, vocab_size=V, hidden_size=H, precision=precision,
                             train_table=True).to(DEV)


def _trainer(tt, m, B, Lq, Ld, precision, **kw):
    return tt.training.FusedTrainer(m, 0.3, LR, B, Lq, Ld, precision=precision, ids_dtype=torch.int64,
                                    mask_dtype=torch.int64, **kw)


def _tables(m):
    return [m.query_tower.pretrained_model.table, m.document_tower.pretrained_model.table]


def _adam_dev(tt, p, g, mom, sq, state):
    N = tt._native
    N.check(N.load().tt_adam_step_dev(N.ptr(p), N.ptr(g), N.ptr(mom), N.ptr(sq), p.numel(), LR, 0.9, 0.999, 1e-8,
                                      N.ptr(state), 1.0, N.stream()), "tt_adam_step_dev")


# ------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------
def test_tt_train_table_switch_parsing(tt, monkeypatch):
    cfg = tt.training.train_table_config
    monkeypatch.delenv("TT_TRAIN_TABLE", raising=False)
    assert cfg(None) is False and cfg(True) is True and cfg(False) is False
    for env, want in (("0", False), ("", False), ("1", True), (" 1 ", True)):
        monkeypatch.setenv("TT_TRAIN_TABLE", env)
        assert cfg(None) is want
    for bad in ("2", "yes", "-1"):
        monkeypatch.setenv("TT_TRAIN_TABLE", bad)
        with pytest.raises(ValueError):
            cfg(None)


@pytest.mark.parametrize("kw", [dict(backbone="minilm"), dict(hard_negatives=4), dict(table_dtype=torch.bfloat16)])
def test_run_training_refuses_what_trainable_tables_cannot_do(tt, monkeypatch, kw):
    monkeypatch.delenv("TT_TRAIN_TABLE", raising=False)
    with pytest.raises(ValueError, match="train_table"):
        tt.training.run_training(num_epochs=1, use_wandb=False, train_table=True, **kw)
    monkeypatch.setenv("TT_TRAIN_TABLE", "1")
    with pytest.raises(ValueError, match="train_table"):
        tt.training.run_training(num_epochs=1, use_wandb=False, **kw)


# ------------------------------------------------------------------------------------------------------------------
# GPU: the fused update against the unfused form, bit for bit
# ------------------------------------------------------------------------------------------------------------------
# (precision, chain, H, V, accumulation_steps, B): every precision and chain mode, every H, both vocabularies, both
# accumulation modes; B = 1100 adds heavy rows of one chunk (> 256 entries) and of several (> 2048)
CASES = [("fp32", 1, 128, 4096, 1, 300), ("fp32", 1, 768, 30522, 2, 1100), ("bf16x3", 1, 384, 30522, 1, 1100),
         ("bf16x3", 2, 256, 4096, 2, 300), ("bf16x3", 1, 128, 30522, 2, 300), ("bf16", 1, 768, 4096, 1, 1100),
         ("bf16", 2, 384, 30522, 2, 300), ("bf16x3", 2, 768, 4096, 1, 1100), ("bf16", 1, 256, 30522, 1, 300)]


@pytest.mark.gpu
@pytest.mark.parametrize("precision,chain,H,V,a,B", CASES)
def test_fused_table_adam_equals_gradients_then_adam_step_dev(tt, chain_env, precision, chain, H, V, a, B):
    """optimize_tables=True leaves the same tables, table moments and projections bit for bit as a gradients-only
    trainer whose closing micro-steps are followed by tt_adam_step_dev on each table (from a copy of the pre-step
    adam_state).  a = 2 runs the closing step on an accumulated table gradient.  Rows never touched stay bit-identical
    to their initial values; heavy rows and masked tokens are in the batches."""
    P, Lq, Ld = 128, 12, 24
    os.environ["TT_CHAIN"] = "1" if chain == 1 else "0"
    ma, mb = _model(tt, P, V, H, precision, 3), _model(tt, P, V, H, precision, 3)
    init = [t.detach().clone() for t in _tables(ma)]
    ta = _trainer(tt, ma, B, Lq, Ld, precision, use_graph=False, accumulation_steps=a, optimize_tables=True)
    tb = _trainer(tt, mb, B, Lq, Ld, precision, use_graph=False, accumulation_steps=a)
    mom = [torch.zeros_like(t) for t in _tables(mb) for _ in range(2)]
    touched = [torch.zeros(V, dtype=torch.bool) for _ in range(2)]
    ta.start_epoch()
    tb.start_epoch()
    n = 3 * a
    for i in range(n):
        b = _batch(B, Lq, Ld, V, 100 + i, heavy=B >= 1100)
        for k, (ids, mask) in enumerate(((b[0], b[1]), (torch.cat([b[2], b[4]]), torch.cat([b[3], b[5]])))):
            touched[k][ids[mask != 0].unique()] = True
        for tr in (ta, tb):
            tr.load_packed(tr.pack_host_tokens(b, pin=False))
        st0 = tb.adam_state.clone()
        close = tb.window.mode()[1]
        la = float(ta.step().item())
        lb = float(tb.step().item())
        assert la == lb
        if close:
            for k, (p, g) in enumerate(zip(_tables(mb), tb.table_grads)):
                _adam_dev(tt, p.data, g, mom[2 * k], mom[2 * k + 1], st0.clone())
        torch.cuda.synchronize()
        for x, y in zip(_tables(ma), _tables(mb)):
            assert torch.equal(x, y), (i, precision, chain)
        for x, y in zip(ta.table_exp_avg + ta.table_exp_avg_sq, mom[0::2] + mom[1::2]):
            assert torch.equal(x, y), i
        assert torch.equal(ta.flat_p, tb.flat_p) and torch.equal(ta.adam_state, tb.adam_state)
    assert int(ta.adam_state[0].item()) == 3
    for t, t0, hit in zip(_tables(ma), init, touched):
        assert bool(hit.any()) and not bool(hit[V // 2:].any())
        assert torch.equal(t[~hit.to(DEV)], t0[~hit.to(DEV)])  # never touched: g = 0 always, m = 0, no move
        assert not torch.equal(t[hit.to(DEV)], t0[hit.to(DEV)])


# ------------------------------------------------------------------------------------------------------------------
# GPU: the arithmetic against float64
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_table_adam_against_a_float64_replay_of_torch_adam(tt):
    """20 steps: before each, the same step with gradients only records the device's own table gradient g_t; a float64
    replay of torch.optim.Adam (betas rounded to fp32 as the kernel sees them) from those gradients predicts the
    moments and the update of every element."""
    B, Lq, Ld, P, V, H = 256, 12, 24, 128, 4096, 128
    m = _model(tt, P, V, H, "bf16x3", 5)
    tr = _trainer(tt, m, B, Lq, Ld, "bf16x3", use_graph=False, optimize_tables=True)
    b1, b2 = float(np.float32(0.9)), float(np.float32(0.999))
    ref_m = [torch.zeros_like(t, dtype=torch.float64) for t in _tables(m)]
    ref_v = [torch.zeros_like(t, dtype=torch.float64) for t in _tables(m)]
    worst_m = worst_u = 0.0
    for step in range(1, 21):
        tr.load_packed(tr.pack_host_tokens(_batch(B, Lq, Ld, V, 200 + step), pin=False))
        tr._fwd_bwd()  # gradients only: the table gradients this step's update consumes
        g = [t.double().clone() for t in tr.table_grads]
        before = [t.detach().double().clone() for t in _tables(m)]
        tr.step()
        torch.cuda.synchronize()
        for k, t in enumerate(_tables(m)):
            ref_m[k] = b1 * ref_m[k] + (1 - b1) * g[k]
            ref_v[k] = b2 * ref_v[k] + (1 - b2) * g[k] * g[k]
            upd = LR / (1 - b1 ** step) * ref_m[k] / ((ref_v[k] / (1 - b2 ** step)).sqrt() + 1e-8)
            got = before[k] - t.detach().double()
            # the fp32 subtraction p - update rounds at ulp(p): that is the floor of the comparison
            tol = 1e-4 * upd.abs() + 2 * before[k].abs() * 2.0 ** -23 + 1e-12
            worst_u = max(worst_u, float(((got - upd).abs() / tol).max()))
            scale = ref_m[k].abs().max().clamp_min(1e-30)
            worst_m = max(worst_m, float((tr.table_exp_avg[k].double() - ref_m[k]).abs().max() / scale))
    assert worst_u <= 1.0, worst_u
    assert worst_m < 1e-5, worst_m


# ------------------------------------------------------------------------------------------------------------------
# GPU: end to end against the reference-shaped loop
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("P", [64, 384])
def test_fused_trainer_matches_the_reference_shaped_loop(tt, P):
    """FusedTrainer(optimize_tables=True) against train_epoch with torch.optim.Adam(model.parameters()) on a copy of
    the model, 3 steps: loss per step 1e-4, projections 1e-3.  Tables: Adam's first steps are about lr * sign(g), so
    the update is compared elementwise wherever every step's reference gradient is 0 or above 10x its error bound; the
    remaining elements are counted, reported and bounded.  Never-touched rows stay bit-identical in both."""
    B, Lq, Ld, V = 256, 16, 48, 4096
    precision = "bf16x3"
    mf = _model(tt, P, V, 384, precision, 11)
    mr = _model(tt, P, V, 384, precision, 11)
    init = [t.detach().clone() for t in _tables(mr)]
    tr = _trainer(tt, mf, B, Lq, Ld, precision, use_graph=True, optimize_tables=True)
    opt = torch.optim.Adam(mr.parameters(), lr=LR)
    crit = tt.TripletLoss(margin=0.3)
    ok = [torch.ones_like(t, dtype=torch.bool) for t in init]
    touched = [torch.zeros(V, dtype=torch.bool, device=DEV) for _ in init]
    for i in range(3):
        b = _batch(B, Lq, Ld, V, 300 + i)
        tr.load_packed(tr.pack_host_tokens(b, pin=False))
        lf = float(tr.step().item())
        toks = [tt.TokenBatch(b[j].to(DEV), b[j + 1].to(DEV)) for j in (0, 2, 4)]
        lr_ = tt.training.train_epoch(mr, [toks], crit, opt, log_wandb=False)
        assert abs(lf - lr_) <= 1e-4 * abs(lr_), (i, lf, lr_)
        for k, t in enumerate(_tables(mr)):
            g = t.grad.detach()
            bound = 1e-3 * g.abs().max()  # relative accuracy of a tensor-core table gradient
            ok[k] &= (g == 0) | (g.abs() > 10 * bound)
        touched[0][b[0][b[1] != 0].to(DEV)] = True
        touched[1][torch.cat([b[2], b[4]])[torch.cat([b[3], b[5]]) != 0].to(DEV)] = True
    torch.cuda.synchronize()
    for x, y in zip(mf.projection_parameters(), mr.projection_parameters()):
        assert float((x - y).detach().norm() / y.detach().norm()) < 1e-3
    for k, (tf, trf, t0) in enumerate(zip(_tables(mf), _tables(mr), init)):
        du, ur = (tf - t0).detach(), (trf - t0).detach()
        sel = ok[k] & touched[k][:, None]
        err = (du - ur).abs()
        assert float(err[sel].max()) <= 0.02 * LR, float(err[sel].max())
        rest = touched[k][:, None] & ~ok[k]
        n_rest = int(rest.sum())
        n_rest_off = int((rest & (err > 0.02 * LR)).sum())
        n_touched = int(touched[k].sum()) * du.shape[1]
        print(f"P={P} table {k}: {int(sel.sum())} of {n_touched} touched elements compared, {n_rest} with a "
              f"near-zero gradient left out, {n_rest_off} of them differ by more than 0.02 lr "
              f"(max |diff| {float(err[rest].max()) if n_rest else 0.0:.2e})")
        # where |g| is near Adam's eps the relative error of g reaches the update: few elements, bounded by Adam
        assert n_rest_off <= 1e-3 * n_touched + 16
        assert float(err.max()) <= 6 * LR  # Adam moves no element more than ~lr per step
        cold = ~touched[k]
        assert torch.equal(tf[cold], t0[cold]) and torch.equal(trf[cold], t0[cold])
    tr.close()


# ------------------------------------------------------------------------------------------------------------------
# GPU: schedules
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("a", [1, 2, 3])
def test_eager_graph_slots_and_peer_schedules_are_bit_identical(tt, a):
    """Eager, graph replay, 2 token slots and the peer exchange at world 1 (the data-parallel code path: tables in the
    second peer segment, their flat gradient through tt_dp_reduce_adam) leave the same tables, table moments,
    projections, step count and losses bit for bit, over 2.5 windows of a micro-batches."""
    B, Lq, Ld, P, V, H = 256, 16, 48, 128, 4096, 384
    n = max(3, (5 * a) // 2)
    batches = [_batch(B, Lq, Ld, V, 400 + i) for i in range(n)]
    out = []
    for mode in ("eager", "graph", "slots", "peer"):
        m = _model(tt, P, V, H, "bf16x3", 21)
        tr = _trainer(tt, m, B, Lq, Ld, "bf16x3", use_graph=mode != "eager", accumulation_steps=a,
                      optimize_tables=True, token_slots=2 if mode == "slots" else 1,
                      exchange="peer" if mode == "peer" else None)
        tr.prepare()
        tr.start_epoch()
        losses = []
        for i, b in enumerate(batches):
            slot = i % 2 if mode == "slots" else 0
            tr.load_packed(tr.pack_host_tokens(b, pin=False), slot)
            losses.append(float(tr.step(slot).item()))
        torch.cuda.synchronize()
        st = tr.xchg.state if tr.xchg is not None else tr.adam_state
        if tr.txchg is not None:
            assert torch.equal(tr.txchg.state, st)
        sd = tr.state_dict()
        out.append(([t.detach().clone() for t in _tables(m)] + [tr.flat_p.clone(), st.clone()]
                    + list(sd["table_exp_avg"]) + list(sd["table_exp_avg_sq"]), losses))
        tr.close()
        assert all(t.data_ptr() != 0 for t in _tables(m))
    for other in out[1:]:
        assert out[0][1] == other[1]
        for x, y in zip(out[0][0], other[0]):
            assert torch.equal(x.cpu(), y.cpu())
    assert int(out[0][0][3][0].item()) == n // a


# ------------------------------------------------------------------------------------------------------------------
# GPU: the exchange at table size
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3, 8])
def test_exchange_at_table_size(tt, world):
    """tt_dp_reduce_adam over 2 x 30522 x 384 parameters on `world` virtual ranks: replicas bit-identical, equal to Adam
    on the rank-ordered sum (1e-6), and the sharded moments of all ranks add up to the reference moments."""
    from two_towers_overlords_b200 import comm

    n = 2 * 30522 * 384
    torch.manual_seed(world)
    xs = comm.DpExchange.virtual_ranks(n, world, DEV)
    p0 = torch.randn(n, device=DEV)
    for x in xs:
        x.flat_p.copy_(p0)
    ms = [torch.zeros(n, device=DEV) for _ in xs]
    vs = [torch.zeros(n, device=DEV) for _ in xs]
    streams = [torch.cuda.Stream() for _ in xs]
    ref_p, ref_m, ref_v = p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    torch.cuda.synchronize()
    try:
        for step in range(1, 3):
            grads = [torch.zeros(n + 1, device=DEV) for _ in xs]
            for g in grads:  # sparse-looking gradients: most rows of a table gradient are zero
                rows = torch.randint(0, n // 384, (2000,), device=DEV)
                g[:n].view(-1, 384)[rows] = torch.randn(2000, 384, device=DEV) * 0.1
            total = grads[0].clone()
            for g in grads[1:]:
                total += g
            torch.cuda.synchronize()
            for x, g, m, v, st in zip(xs, grads, ms, vs, streams):
                with torch.cuda.stream(st):
                    x.reduce_adam(g, m, v, LR, max_ctas=16)
            torch.cuda.synchronize()
            for x in xs:
                x.check()
            tt.ops.adam_step(ref_p, total[:n].contiguous(), ref_m, ref_v, LR, step)
            for x in xs:
                assert torch.equal(x.flat_p, xs[0].flat_p)
            assert float((xs[0].flat_p - ref_p).abs().max()) <= 1e-6
            assert torch.equal(sum(ms), ref_m) and torch.equal(sum(vs), ref_v)
    finally:
        torch.cuda.synchronize()
        for x in xs:
            x.close()


# ------------------------------------------------------------------------------------------------------------------
# GPU: checkpoints
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("a,exchange", [(1, None), (2, None), (1, "peer")])
def test_resume_is_bit_exact(tt, tmp_path, a, exchange):
    """Save after 3 of 6 micro-steps (inside an open window at a = 2), resume in a new trainer built from another seed:
    tables, table moments, projections and the step count equal the uninterrupted run bit for bit.  A checkpoint
    without table moments is refused."""
    B, Lq, Ld, P, V, H = 128, 16, 48, 64, 4096, 128
    batches = [_batch(B, Lq, Ld, V, 500 + i) for i in range(6)]

    def make(seed):
        return _trainer(tt, _model(tt, P, V, H, "bf16x3", seed), B, Lq, Ld, "bf16x3", accumulation_steps=a,
                        optimize_tables=True, exchange=exchange)

    def feed(tr, bs):
        for b in bs:
            tr.load_packed(tr.pack_host_tokens(b, pin=False))
            tr.step()

    def state(tr):
        torch.cuda.synchronize()
        st = tr.xchg.state if tr.xchg is not None else tr.adam_state
        return [t.detach().clone() for t in _tables(tr.model)] + [tr._table_m.clone(), tr._table_v.clone(),
                                                                  tr.flat_p.clone(), st.clone()]

    t1 = make(9)
    t1.start_epoch()
    feed(t1, batches)
    want = state(t1)
    t2 = make(9)
    t2.start_epoch()
    feed(t2, batches[:3])
    ck = str(tmp_path / "tables.ckpt")
    t2.save_checkpoint(ck)
    t3 = make(123)
    t3.load_checkpoint(ck)
    feed(t3, batches[3:])
    for x, y in zip(want, state(t3)):
        assert torch.equal(x, y)
    sd = torch.load(ck, map_location="cpu", weights_only=False)
    del sd["table_exp_avg"]
    with pytest.raises(ValueError, match="table moments"):
        make(1).load_state_dict(sd)
    for t in (t1, t2, t3):
        t.close()


# ------------------------------------------------------------------------------------------------------------------
# GPU: run_training
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("how", ["arg", "env", "fallback", "default"])
def test_run_training_trains_the_tables_behind_the_switch(tt, monkeypatch, capsys, how):
    """run_training(train_table=True) and TT_TRAIN_TABLE=1 (fused path and the reference-shaped fallback) return
    changed tables; the default returns tables bit-identical to their initial values."""
    monkeypatch.setenv("TT_SYNTHETIC_DATA", "1")
    monkeypatch.delenv("TT_TRAIN_TABLE", raising=False)
    if how in ("env", "fallback"):
        monkeypatch.setenv("TT_TRAIN_TABLE", "1")
    torch.manual_seed(0)
    init = tt.TwoTowersModel(projection_dim=64)
    init_tables = [t.detach().clone() for t in _tables(init)]
    torch.manual_seed(0)
    model = tt.training.run_training(num_epochs=1, batch_size=256, learning_rate=1e-3, max_samples=2000,
                                     projection_dim=64, margin=0.3, use_wandb=False, accumulation_steps=1,
                                     use_mixed_precision=False, num_workers=0, run_comprehensive_test=False,
                                     train_table=True if how == "arg" else None,
                                     fused=False if how == "fallback" else None)
    out = capsys.readouterr().out
    assert f"Fused B200 step: {how != 'fallback'}" in out
    tables = [t.detach().cpu() for t in _tables(model)]
    if how == "default":
        assert "Trainable parameters" not in out
        for t, t0 in zip(tables, init_tables):
            assert torch.equal(t, t0)
    else:
        assert "Trainable parameters" in out
        for t, t0 in zip(tables, init_tables):
            assert not torch.equal(t, t0)
            assert torch.isfinite(t).all()


# ------------------------------------------------------------------------------------------------------------------
# GPU: refusals
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals_leave_the_next_valid_call_unaffected(tt, chain_env):
    """A frozen model, exchange='nccl' and bf16 tables are refused by the trainer; at the ABI, table Adam without
    adam_param, only one table, or a param that is not the gathered table.  After each refusal the next valid step
    equals a step of a twin that never saw one."""
    B, Lq, Ld, P, V, H = 128, 16, 48, 64, 2048, 128
    frozen = tt.TwoTowersModel(projection_dim=P, vocab_size=V, hidden_size=H).to(DEV)
    with pytest.raises(ValueError, match="trainable"):
        _trainer(tt, frozen, B, Lq, Ld, "bf16x3", optimize_tables=True)
    with pytest.raises(ValueError, match="nccl"):
        _trainer(tt, _model(tt, P, V, H, "bf16x3", 1), B, Lq, Ld, "bf16x3", optimize_tables=True, exchange="nccl")
    torch.manual_seed(1)
    bf = tt.TwoTowersModel(projection_dim=P, vocab_size=V, hidden_size=H, table_dtype=torch.bfloat16).to(DEV)
    for t in _tables(bf):
        t.requires_grad_(True)
    with pytest.raises(ValueError, match="fp32"):
        _trainer(tt, bf, B, Lq, Ld, "bf16x3", optimize_tables=True)

    ma, mb = _model(tt, P, V, H, "bf16x3", 2), _model(tt, P, V, H, "bf16x3", 2)
    ta = _trainer(tt, ma, B, Lq, Ld, "bf16x3", use_graph=False, optimize_tables=True)
    tb = _trainer(tt, mb, B, Lq, Ld, "bf16x3", use_graph=False, optimize_tables=True)
    b = _batch(B, Lq, Ld, V, 600)
    for tr in (ta, tb):
        tr.load_packed(tr.pack_host_tokens(b, pin=False))
    so = ta.step_obj
    N = tt._native
    table_q, table_d = so.args.table_q, so.args.table_d
    other = torch.zeros_like(_tables(ma)[0])
    bad = [dict(adam=False),                                            # table Adam without adam_param
           dict(fields=dict(table_param_d=None)),                       # only one table
           dict(fields=dict(table_param_q=N.ptr(other)))]               # not the gathered table
    for case in bad:
        a = so.slots[0]
        if case.get("adam", True):
            (a.adam_state, a.adam_param, a.adam_grad, a.adam_exp_avg, a.adam_exp_avg_sq, a.adam_n, a.adam_lr,
             a.adam_beta1, a.adam_beta2, a.adam_eps) = so._adam
        (a.table_param_q, a.table_param_d, a.table_exp_avg_q, a.table_exp_avg_sq_q, a.table_exp_avg_d,
         a.table_exp_avg_sq_d) = so._table_adam
        for k, v in case.get("fields", {}).items():
            setattr(a, k, v)
        rc = so.lib.tt_triplet_step(ctypes.byref(a), N.stream())
        assert rc != 0, case
        assert "table" in N.last_error()
        a.adam_param = None
        a.table_param_q = a.table_param_d = None
    assert (so.args.table_q, so.args.table_d) == (table_q, table_d)
    for tr in (ta, tb):
        tr.step()
    torch.cuda.synchronize()
    for x, y in zip(_tables(ma) + [ta.flat_p, ta._table_m, ta._table_v],
                    _tables(mb) + [tb.flat_p, tb._table_m, tb._table_v]):
        assert torch.equal(x, y)
