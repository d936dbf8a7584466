"""Gradient accumulation in the fused trainer (tt_step_args.grad_accumulate, FusedTrainer(accumulation_steps=a),
run_training(fused_accumulation=...)): the ABI's exact fl(old + new) contract in every precision and chain mode, the
reference's own accumulation loop (golden), the window cadence and its carry-over into the next epoch against the CPU
oracle, bit-identical schedules, and a resume inside an open window."""
import os

import numpy as np
import pytest
import torch

from oracle import two_towers_oracle as O

DEV = "cuda"
NAMES = ("query_tower.projection.0.weight", "query_tower.projection.0.bias", "query_tower.projection.2.weight",
         "query_tower.projection.2.bias", "document_tower.projection.0.weight", "document_tower.projection.0.bias",
         "document_tower.projection.2.weight", "document_tower.projection.2.bias")


@pytest.fixture(scope="module")
def tt():
    import two_towers_overlords_b200 as pkg
    from two_towers_overlords_b200 import data, ops, training

    pkg.ops, pkg.training, pkg.data = ops, training, data
    return pkg


def rel_err(got, want) -> float:
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).norm() / want.norm().clamp_min(1e-30))


def pad_batch(b, Lq, Ld):
    pad = lambda t, L: torch.nn.functional.pad(t, (0, L - t.shape[1]))  # noqa: E731
    return tuple(pad(t, Lq if i < 2 else Ld) for i, t in enumerate(b.astuple()))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the window schedule
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("a", [1, 2, 3, 4])
def test_window_schedule_follows_the_reference_cadence(tt, a):
    """Over several epochs of different lengths: close iff (batch_idx + 1) % a == 0 with batch_idx restarting every
    epoch; the buffers are added to iff an unstepped gradient is carried (inside a window, or a trailing partial window
    of the previous epoch); every mode met is one prepare() captures."""
    w = tt.training.AccumulationWindow(a)
    pending = 0
    for n in (5, 7, 1, 6, 3, 8):
        w.start_epoch()
        for batch_idx in range(n):
            acc, close = w.mode()
            assert close == ((batch_idx + 1) % a == 0)
            assert acc == (pending > 0)
            assert (acc, close) in w.modes()
            w.advance()
            pending = 0 if close else pending + 1
            assert w.pending == pending
    # a = 3, 5 batches per epoch: one step per epoch (2 after epoch 2); epoch 2's step applies 5 micro-batches
    if a == 3:
        w = tt.training.AccumulationWindow(3)
        closes = []
        for _ in range(2):
            w.start_epoch()
            closes.append([])
            for _ in range(5):
                closes[-1].append(w.mode())
                w.advance()
        assert [sum(c for _, c in e) for e in closes] == [1, 1]
        assert closes[1][:3] == [(True, False), (True, False), (True, True)] and w.pending == 2


@pytest.mark.parametrize("bad", [0, -1, 1.5, True])
def test_accumulation_steps_below_one_is_refused(tt, bad):
    with pytest.raises(ValueError):
        tt.training.AccumulationWindow(bad)
    with pytest.raises(ValueError):
        tt.training.run_training(num_epochs=1, use_wandb=False, accumulation_steps=bad)


# ------------------------------------------------------------------------------------------------------------------
# GPU: the ABI contract
# ------------------------------------------------------------------------------------------------------------------
def _trainer(tt, precision, chain, B, P, V=2048, Lq=16, Ld=40, seed=0, **kw):
    torch.manual_seed(seed)
    m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision=precision,
                          train_table=kw.pop("train_table", False)).to(DEV)
    if chain is not None:
        os.environ["TT_CHAIN"] = "1" if chain == 1 else "0"
    tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, Lq, Ld, precision=precision, use_graph=False,
                                  ids_dtype=torch.int64, mask_dtype=torch.int64, **kw)
    return m, tr


@pytest.fixture
def chain_env():
    old = os.environ.get("TT_CHAIN")
    yield
    if old is None:
        os.environ.pop("TT_CHAIN", None)
    else:
        os.environ["TT_CHAIN"] = old


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 129, 300])
@pytest.mark.parametrize("chain", [1, 2])
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_grad_accumulate_adds_exactly_what_an_overwriting_call_writes(tt, chain_env, precision, chain, B):
    """grad_accumulate = 1 over random G0 leaves exactly G0 + g in every gradient, g = the same call with 0; loss and
    pooled rows unchanged.  P = 576 exercises the tile tails of the 128-wide projection tiles."""
    if precision == "fp32" and chain == 2:
        pytest.skip("the fp32 CUDA-core path has no chain modes")
    P, Lq, Ld = 576, 16, 40
    _, tr = _trainer(tt, precision, chain, B, P, Lq=Lq, Ld=Ld)
    b = O.synth_triplet_batch(B, Lq, Ld, "U", seed=3, vocab=2048)
    tr.load_packed(tr.pack_host_tokens(pad_batch(b, Lq, Ld), pin=False))
    tr._fwd_bwd()
    g = tr.flat_g.clone()
    rows = tr.step_obj.pooled_rows().clone()
    g0 = torch.randn_like(tr.flat_g)
    tr.flat_g.copy_(g0)
    tr._fwd_bwd(accumulate=True)
    torch.cuda.synchronize()
    n = tr.n_param
    assert torch.equal(tr.flat_g[:n], g0[:n] + g[:n])
    assert torch.equal(tr.flat_g[n:], g[n:])  # the loss is overwritten
    assert torch.equal(tr.step_obj.pooled_rows(), rows)


@pytest.mark.gpu
@pytest.mark.parametrize("chain", [1, 2])
@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_grad_accumulate_with_trainable_tables(tt, chain_env, precision, chain):
    """Trainable tables: dtable_q / dtable_d become old + new as well (old rows of untouched ids stay)."""
    if precision == "fp32" and chain == 2:
        pytest.skip("the fp32 CUDA-core path has no chain modes")
    B, P, V, Lq, Ld = 129, 128, 2048, 16, 40
    _, tr = _trainer(tt, precision, chain, B, P, V=V, Lq=Lq, Ld=Ld, train_table=True)
    b = O.synth_triplet_batch(B, Lq, Ld, "Z", seed=4, vocab=V)
    tr.load_packed(tr.pack_host_tokens(pad_batch(b, Lq, Ld), pin=False))
    tr._fwd_bwd()
    g = [t.clone() for t in (tr.flat_g,) + tr.table_grads]
    g0 = [torch.randn_like(t) for t in g]
    for t, s in zip((tr.flat_g,) + tr.table_grads, g0):
        t.copy_(s)
    tr._fwd_bwd(accumulate=True)
    torch.cuda.synchronize()
    n = tr.n_param
    assert torch.equal(tr.flat_g[:n], g0[0][:n] + g[0][:n])
    for t, old, new in zip(tr.table_grads, g0[1:], g[1:]):
        assert torch.equal(t, old + new)


@pytest.mark.gpu
@pytest.mark.parametrize("chain", [1, 2])
def test_grad_accumulate_with_the_pooled_front_end(tt, chain_env, chain):
    """Pooled banks (the MiniLM front end's rows, here random unit rows): the same exact contract."""
    B, P, Lq, Ld = 300, 576, 16, 40
    torch.manual_seed(1)
    m = tt.TwoTowersModel(projection_dim=P, vocab_size=2048, precision="bf16x3").to(DEV)
    H = m.query_tower.embedding_dim
    banks = [tt.data.PooledBank(torch.nn.functional.normalize(torch.randn(n, H, device=DEV), dim=1),
                                tt.data.backbone_identity(tower), L)
             for L, n, tower in ((Lq, 500, m.query_tower), (Ld, 700, m.document_tower))]
    os.environ["TT_CHAIN"] = "1" if chain == 1 else "0"
    tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, Lq, Ld, precision="bf16x3", use_graph=False, pooled=banks)
    idx = torch.cat([torch.randint(0, 500, (B,)), torch.randint(0, 700, (2 * B,))]).to(DEV)
    tr.load_rows(idx)
    tr._fwd_bwd()
    g = tr.flat_g.clone()
    g0 = torch.randn_like(g)
    tr.flat_g.copy_(g0)
    tr._fwd_bwd(accumulate=True)
    torch.cuda.synchronize()
    n = tr.n_param
    assert torch.equal(tr.flat_g[:n], g0[:n] + g[:n]) and torch.equal(tr.flat_g[n:], g[n:])


@pytest.mark.gpu
@pytest.mark.parametrize("chain", [1, 2])
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_fused_adam_consumes_the_accumulated_gradient(tt, chain_env, precision, chain):
    """Accumulate + fused Adam in one call == gradients-only accumulate, then tt_adam_step_dev on the same buffers:
    weights, moments, step count and gradients bit for bit."""
    if precision == "fp32" and chain == 2:
        pytest.skip("the fp32 CUDA-core path has no chain modes")
    B, P, Lq, Ld = 129, 576, 16, 40
    b = O.synth_triplet_batch(B, Lq, Ld, "U", seed=8, vocab=2048)
    out = []
    for fused in (True, False):
        _, tr = _trainer(tt, precision, chain, B, P, Lq=Lq, Ld=Ld, seed=2)
        tr.load_packed(tr.pack_host_tokens(pad_batch(b, Lq, Ld), pin=False))
        torch.manual_seed(5)
        tr.flat_g.copy_(torch.randn_like(tr.flat_g) * 1e-3)
        tr.exp_avg.copy_(torch.randn_like(tr.exp_avg) * 1e-4)
        tr.exp_avg_sq.copy_(torch.rand_like(tr.exp_avg_sq) * 1e-6)
        tr.adam_state.copy_(torch.tensor([3.0, 0.9 ** 3, 0.999 ** 3, 0.0], dtype=torch.float64))
        if fused:
            tr._fwd_bwd(optimise=True, accumulate=True)
        else:
            tr._fwd_bwd(accumulate=True)
            tr._optimizer()
        torch.cuda.synchronize()
        out.append([t.clone() for t in (tr.flat_p, tr.flat_g, tr.exp_avg, tr.exp_avg_sq, tr.adam_state)])
    for x, y in zip(*out):
        assert torch.equal(x, y)


# ------------------------------------------------------------------------------------------------------------------
# GPU: the reference's loop, cadence and carry-over
# ------------------------------------------------------------------------------------------------------------------
def _golden_model(tt, g, P, precision):
    V = g["init__query_tower__pretrained_model__emb__weight"].shape[0]
    m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision=precision)
    with torch.no_grad():
        for name in ("query_tower", "document_tower"):
            t = getattr(m, name)
            t.pretrained_model.table.copy_(torch.from_numpy(g[f"init__{name}__pretrained_model__emb__weight"]))
            for i in (0, 2):
                t.projection[i].weight.copy_(torch.from_numpy(g[f"init__{name}__projection__{i}__weight"]))
                t.projection[i].bias.copy_(torch.from_numpy(g[f"init__{name}__projection__{i}__bias"]))
    return m.to(DEV)


@pytest.mark.gpu
@pytest.mark.parametrize("chain", [1, 2])
@pytest.mark.parametrize("use_graph", [False, True])
@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_fused_accumulation_matches_the_reference_train_epoch_optimized(tt, golden_dir, chain_env, precision,
                                                                        use_graph, chain):
    """The reference's train_epoch_optimized (5 batches, accumulation 2; golden): mean loss 1e-4, the weight update
    after its 2 optimiser steps 2e-3, the gradient the unstepped 5th batch leaves in the gradient views 1e-3."""
    if precision == "fp32" and chain == 2:
        pytest.skip("the fp32 CUDA-core path has no chain modes")
    os.environ["TT_CHAIN"] = "1" if chain == 1 else "0"
    g = np.load(os.path.join(golden_dir, "train_epoch_optimized.npz"))
    m = _golden_model(tt, g, 64, precision)
    margin, lr, accum = float(g["margin"]), float(g["lr"]), int(g["accum"])
    nb = int(g["n_batches"])
    batches = [tuple((torch.from_numpy(g[f"b{b}_{nm}_ids"]), torch.from_numpy(g[f"b{b}_{nm}_mask"]))
                     for nm in ("q", "p", "n")) for b in range(nb)]
    B = batches[0][0][0].shape[0]
    Lq = max(b[0][0].shape[1] for b in batches)
    Ld = max(max(b[1][0].shape[1], b[2][0].shape[1]) for b in batches)
    pad = lambda t, L: torch.nn.functional.pad(t, (0, L - t.shape[1]))  # noqa: E731
    tr = tt.training.FusedTrainer(m, margin, lr, B, Lq, Ld, precision=precision, use_graph=use_graph,
                                  ids_dtype=torch.int64, mask_dtype=torch.int64, accumulation_steps=accum)
    tr.prepare()
    tr.start_epoch()
    losses = []
    for (q, p, n) in batches:
        srcs = (pad(q[0], Lq), pad(q[1], Lq), pad(p[0], Ld), pad(p[1], Ld), pad(n[0], Ld), pad(n[1], Ld))
        for dst, src in zip(tr.tok, srcs):
            dst.copy_(src)
        losses.append(float(tr.step().item()))
    avg = float(np.mean(losses))
    assert abs(avg - float(g["avg_loss"])) <= 1e-4 * float(g["avg_loss"])
    for name in ("query_tower", "document_tower"):
        for i in (0, 2):
            for kind in ("weight", "bias"):
                want = torch.from_numpy(g[f"final__{name}__projection__{i}__{kind}"])
                init = torch.from_numpy(g[f"init__{name}__projection__{i}__{kind}"])
                got = getattr(getattr(m, name).projection[i], kind).detach().cpu()
                assert rel_err(got - init, want - init) < 2e-3, (name, i, kind)
    views = dict(zip(NAMES, tr.g_views))
    for name in ("query_tower", "document_tower"):
        for i in (0, 2):
            for kind in ("weight", "bias"):
                want = torch.from_numpy(g[f"leftover_grad__{name}__projection__{i}__{kind}"])
                assert rel_err(views[f"{name}.projection.{i}.{kind}"], want) < 1e-3, (name, i, kind)
    assert int(tr.adam_state[0].item()) == 2
    assert tr.window.pending == 1


@pytest.mark.gpu
@pytest.mark.parametrize("a", [1, 2, 3, 4])
def test_two_epochs_with_carry_over_match_the_oracle(tt, a):
    """Two epochs of 5 batches against oracle.train_epoch_accum called twice on one model (its trailing partial window
    carries into epoch 2 as in the reference): Adam step count after each epoch and epoch mean losses (1e-4) exactly
    as the cadence dictates, and the weight update of all 8 tensors together within 1e-2.  The update gate is wider
    than the golden loop's per-tensor 2e-3: at a = 3 / 4 it is only 2 Adam steps, whose first steps move every element
    by about ±lr whatever its gradient's size, so one near-zero gradient element whose sign differs between the device
    and the CPU oracle moves a 64-element bias update by 3-5e-3 (measured on a B200, at a = 1 too).  A cadence error —
    a missing or extra step, a lost carry — moves the update by tens of percent."""
    B, Lq, Ld, P, V, margin, lr = 64, 12, 24, 64, 1024, 0.3, 1e-3
    batches = [O.synth_triplet_batch(B, Lq, Ld, "U", seed=60 + i, vocab=V) for i in range(5)]
    torch.manual_seed(7)
    m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision="bf16x3").to(DEV)
    ref = O.OracleTwoTowers(P, vocab=V)
    with torch.no_grad():
        for t_new, t_ref in ((m.query_tower, ref.query_tower), (m.document_tower, ref.document_tower)):
            t_ref.table.copy_(t_new.pretrained_model.table.detach().float().cpu())
            for i in (0, 2):
                t_ref.projection[i].weight.copy_(t_new.projection[i].weight.cpu())
                t_ref.projection[i].bias.copy_(t_new.projection[i].bias.cpu())
    init = [p.detach().cpu().clone() for p in m.projection_parameters()]
    opt = torch.optim.Adam(ref.parameters(), lr=lr)
    tr = tt.training.FusedTrainer(m, margin, lr, B, Lq, Ld, precision="bf16x3", ids_dtype=torch.int64,
                                  mask_dtype=torch.int64, accumulation_steps=a)
    tr.prepare()
    steps = []
    for epoch in range(2):
        want_loss = O.train_epoch_accum(ref, opt, [b.astuple() for b in batches], margin, accumulation_steps=a)
        tr.start_epoch()
        losses = []
        for b in batches:
            tr.load_packed(tr.pack_host_tokens(b.astuple(), pin=False))
            losses.append(float(tr.step().item()))
        assert abs(np.mean(losses) - want_loss) <= 1e-4 * want_loss, (epoch, np.mean(losses), want_loss)
        steps.append(int(tr.adam_state[0].item()))
    n_ref = int(next(iter(opt.state.values()))["step"]) if opt.state else 0
    assert steps == [5 // a, 2 * (5 // a)] and steps[-1] == n_ref  # a = 3: 1 step in epoch 1, 2 after epoch 2
    ref_p = [dict(ref.named_parameters())[nm].detach() for nm in NAMES]
    got = torch.cat([(p.detach().cpu() - p0).reshape(-1) for p, p0 in zip(m.projection_parameters(), init)])
    want = torch.cat([(p - p0).reshape(-1) for p, p0 in zip(ref_p, init)])
    assert rel_err(got, want) < 1e-2, rel_err(got, want)


# ------------------------------------------------------------------------------------------------------------------
# GPU: schedules agree exactly; resume inside a window
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("a", [2, 3])
def test_eager_graph_pipelined_and_peer_schedules_are_bit_identical(tt, a):
    """2.5 windows: eager, graph, pipelined (2 token slots, look-ahead gather) and the peer exchange at world 1 give the
    same weights, moments, gradient buffer and losses bit for bit; no graph is captured after prepare() (up to the last
    micro-step, which has no look-ahead: prepare() captures the round-robin schedule, as at a = 1)."""
    B, Lq, Ld, P, V = 256, 16, 64, 128, 4096
    n = (5 * a) // 2
    batches = [O.synth_triplet_batch(B, Lq, Ld, "U", seed=80 + i, vocab=V) for i in range(n)]
    out = []
    for mode in ("eager", "graph", "pipelined", "pipelined+peer"):
        torch.manual_seed(4)
        m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision="bf16x3").to(DEV)
        tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, Lq, Ld, precision="bf16x3", use_graph=mode != "eager",
                                      ids_dtype=torch.int64, mask_dtype=torch.int64, token_slots=2,
                                      exchange="peer" if mode.endswith("peer") else None, accumulation_steps=a)
        tr.prepare(2)
        cap0 = tr.graph_captures
        tr.start_epoch()
        losses = []
        pipelined = mode.startswith("pipelined")
        tr.load_packed(tr.pack_host_tokens(batches[0].astuple(), pin=False), 0)
        for i in range(n):
            if i == n - 1 and mode != "eager":
                assert tr.graph_captures == cap0, mode
            slot, nslot = i % 2, None
            if pipelined and i + 1 < n:
                nslot = (i + 1) % 2
                tr.load_packed(tr.pack_host_tokens(batches[i + 1].astuple(), pin=False), nslot)
            losses.append(float(tr.step(slot, nslot).item()))
            if not pipelined and i + 1 < n:
                tr.load_packed(tr.pack_host_tokens(batches[i + 1].astuple(), pin=False), (i + 1) % 2)
        torch.cuda.synchronize()
        st = tr.xchg.state if tr.xchg is not None else tr.adam_state
        out.append(([t.clone() for t in (tr.flat_p, tr.flat_g[: tr.n_param], tr.exp_avg, tr.exp_avg_sq, st)], losses))
        tr.close()
    for other in out[1:]:
        assert out[0][1] == other[1]
        for x, y in zip(out[0][0], other[0]):
            assert torch.equal(x, y)
    assert int(out[0][0][4][0].item()) == n // a


@pytest.mark.gpu
def test_resume_inside_an_open_window_is_bit_exact(tt, tmp_path):
    """a = 2: save after micro-step 3 (one micro-batch pending), resume in a new trainer and finish == uninterrupted
    (weights, moments, gradient buffer, Adam step count).  An old-format checkpoint loads at a window start; a window
    saved at a = 2 refuses a trainer at a = 3."""
    B, Lq, Ld, P, V = 128, 16, 48, 64, 2048
    batches = [O.synth_triplet_batch(B, Lq, Ld, "U", seed=40 + i, vocab=V) for i in range(6)]

    def make(seed, a=2):
        torch.manual_seed(seed)
        m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision="bf16x3").to(DEV)
        return tt.training.FusedTrainer(m, 0.3, 1e-3, B, Lq, Ld, precision="bf16x3", ids_dtype=torch.int64,
                                        mask_dtype=torch.int64, accumulation_steps=a)

    def feed(tr, bs):
        for b in bs:
            tr.load_packed(tr.pack_host_tokens(b.astuple(), pin=False))
            tr.step()

    def state(tr):
        torch.cuda.synchronize()
        return [t.clone() for t in (tr.flat_p, tr.flat_g[: tr.n_param], tr.exp_avg, tr.exp_avg_sq, tr.adam_state)]

    t1 = make(9)
    t1.start_epoch()
    feed(t1, batches)
    want = state(t1)
    t2 = make(9)
    t2.start_epoch()
    feed(t2, batches[:3])
    ck = str(tmp_path / "mid_window.ckpt")
    t2.save_checkpoint(ck)
    sd = torch.load(ck, map_location="cpu", weights_only=False)
    assert sd["window_pending"] == 1 and sd["accumulation_steps"] == 2
    t3 = make(123)
    t3.load_checkpoint(ck)
    assert t3.window.pending == 1 and t3.window.batch_idx == 3
    feed(t3, batches[3:])
    got = state(t3)
    for x, y in zip(want, got):
        assert torch.equal(x, y)
    with pytest.raises(ValueError):
        make(1, a=3).load_state_dict(sd)
    old = {k: v for k, v in sd.items() if not k.startswith("window_") and k != "accumulation_steps"}
    t4 = make(1, a=3)
    t4.load_state_dict(old)
    assert t4.window.pending == 0 and t4.window.batch_idx == 0


# ------------------------------------------------------------------------------------------------------------------
# GPU: run_training
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("switch", ["1", "0"])
def test_run_training_honours_accumulation_steps_behind_the_switch(tt, monkeypatch, capsys, switch):
    """TT_FUSED_ACCUMULATION=1: accumulation_steps = 2 trains on the fused path with an effective batch of 2 x 256;
    unset / 0: the same call runs the reference-shaped loop as before."""
    monkeypatch.setenv("TT_SYNTHETIC_DATA", "1")
    monkeypatch.setenv("TT_FUSED_ACCUMULATION", switch)
    torch.manual_seed(0)
    model = tt.training.run_training(num_epochs=2, batch_size=256, learning_rate=1e-3, max_samples=3000,
                                     projection_dim=64, margin=0.3, use_wandb=False, accumulation_steps=2,
                                     use_mixed_precision=True, num_workers=0, run_comprehensive_test=False)
    out = capsys.readouterr().out
    assert isinstance(model, tt.TwoTowersModel)
    assert f"Fused B200 step: {switch == '1'}" in out
    assert "Effective batch size: 512" in out
    losses = [float(l.split(":")[1]) for l in out.splitlines() if l.startswith("Average training loss")]
    assert len(losses) == 2 and all(np.isfinite(losses)) and losses[0] < 0.35
