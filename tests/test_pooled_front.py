"""The pooled-row front end of the fused step: a frozen backbone encoded once per text into pooled banks, and steps that
gather rows of those banks by index instead of pooling tokens (tt_step_args.pooled_*, tt_assemble_triplet_rows,
data.PooledBank, FusedTrainer(pooled=...), run_training(backbone="minilm")).

The token-table backbone has both paths, so there the row path must reproduce the token path bit for bit: pooled rows,
their bf16 terms, loss, gradients and weights.  The MiniLM backbone has only the row path; it is checked against the
reference-shaped autograd step, and its banks against `tower.pooled` of the tokens a step would see.
"""
import copy
import ctypes
import math
import types

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def tt():
    import two_towers_overlords_b200 as pkg
    from two_towers_overlords_b200 import _native, data, ops, retrieval, training  # noqa: F401

    pkg.data, pkg.ops, pkg.training, pkg.retrieval, pkg.N = data, ops, training, retrieval, _native
    return pkg


def synth(tt, n_pairs, seed=42):
    return tt.data.MSMarcoDataset("train", max_samples=n_pairs, random_seed=seed, synthetic=True)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the length-sorted batch plan and the loader's row mode
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cap", [1, 64, 300, 4096])
def test_length_batch_plan_covers_every_row_once_within_the_token_cap(tt, cap):
    rng = np.random.default_rng(cap)
    lens = np.concatenate([rng.integers(1, 257, 997), [0, 400, 1, 256]])
    batches = tt.data.plan_length_batches(lens, cap)
    seen = np.concatenate(batches)
    assert np.array_equal(np.sort(seen), np.arange(len(lens)))
    flat = np.maximum(lens[seen], 1)
    assert np.all(np.diff(flat) >= 0)  # sorted by length
    for b in batches:
        padded = len(b) * int(np.maximum(lens[b], 1).max())
        assert padded <= cap or len(b) == 1


@pytest.mark.parametrize("world", [1, 2, 4])
def test_row_loader_matches_negative_sampler_token_mode_and_rank_slices(tt, world):
    ds = synth(tt, 700)
    gb, seed = 64, 11
    per = gb // world
    loaders = [tt.data.TokenTripletLoader(ds, gb, 8, 24, rank=r, world_size=world, seed=seed, rows=True)
               for r in range(world)]
    tok = tt.data.TokenTripletLoader(ds, gb, 8, 24, rank=0, world_size=world, seed=seed)
    q_idx, d_idx, qid = loaders[0].q_idx, loaders[0].d_idx, loaders[0].qid
    rng = np.random.default_rng(seed)
    order = rng.permutation(len(ds))
    steps = list(zip(*[iter(lo) for lo in loaders], iter(tok)))
    assert len(steps) == len(ds) // gb
    for s, step in enumerate(steps):
        g = order[s * gb: (s + 1) * gb]
        neg = g[tt.data.sample_negative_indices(qid[g], rng)]
        want = np.stack([q_idx[g], d_idx[g], d_idx[neg]]).astype(np.int32)
        rows = [r.numpy() for r in step[:world]]
        assert all(r.dtype == np.int32 and r.shape == (3, per) for r in rows)
        assert np.array_equal(np.concatenate(rows, axis=1), want)
        assert np.all(qid[g] != qid[neg])
        # rank 0's token batch is exactly the rows' texts padded to Lq / Ld
        for t, (bank, L, r) in zip(step[world], ((ds.query_bank, 8, rows[0][0]), (ds.doc_bank, 24, rows[0][1]),
                                                  (ds.doc_bank, 24, rows[0][2]))):
            ref = bank.batch(r.astype(np.int64), L, L)
            assert torch.equal(t.input_ids.long(), ref.input_ids) and torch.equal(t.attention_mask.long(),
                                                                                  ref.attention_mask)


# ---------------------------------------------------------------------------------------------------------------------
# 1. negatives: tt_assemble_triplet_rows against tt_assemble_triplets
# ---------------------------------------------------------------------------------------------------------------------
def _pairs(n_pairs, n_q, n_d, n_qid, seed, dev):
    g = torch.Generator().manual_seed(seed)
    pq = torch.randint(0, n_q, (n_pairs,), generator=g, dtype=torch.int32)
    pd = torch.randint(0, n_d, (n_pairs,), generator=g, dtype=torch.int32)
    qid = torch.randint(0, n_qid, (n_pairs,), generator=g, dtype=torch.int32)
    return pq.to(dev), pd.to(dev), qid.to(dev)


def _id_bank(n, dev, N):
    """Token bank whose text r is the two tokens [r, r]: the first id of an assembled row names its bank row."""
    flat = torch.arange(n, dtype=torch.int32).repeat_interleave(2).to(dev)
    off = (torch.arange(n + 1, dtype=torch.int64) * 2).to(dev)
    return flat, off, N.TokenBankDesc(flat.data_ptr(), off.data_ptr(), N.TT_I32, 0)


@gpu
@pytest.mark.parametrize("Bg", [2, 257, 2048])
@pytest.mark.parametrize("seed", [0, 1, 0xDEADBEEF12345])
def test_row_assembly_draws_the_token_assemblys_negatives(tt, Bg, seed):
    N, dev = tt.N, torch.device("cuda")
    lib = N.load()
    n_pairs, n_q, n_d = 5000, 700, 4000
    pq, pd, qid = _pairs(n_pairs, n_q, n_d, 300, seed & 0xFFFF, dev)
    qb, db = _id_bank(n_q, dev, N), _id_bank(n_d, dev, N)
    order = torch.randperm(n_pairs, generator=torch.Generator().manual_seed(seed & 0xFFF))[:Bg].to(torch.int32).to(dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    full_rows = None
    for G in (1, 2, 8):
        parts = []
        for r in range(G):
            lo, hi = tt.retrieval.shard_bounds(Bg, G, r)
            B = hi - lo
            toks = [torch.full((B, L), -1, dtype=torch.int32, device=dev) for L in (1, 1, 2, 2, 2, 2)]
            neg_t = torch.full((max(B, 1),), -1, dtype=torch.int32, device=dev)
            neg_r = torch.full((max(B, 1),), -2, dtype=torch.int32, device=dev)
            rows = torch.full((max(3 * B, 1),), -3, dtype=torch.int32, device=dev)
            N.check(lib.tt_assemble_triplets(ctypes.byref(qb[2]), ctypes.byref(db[2]), N.ptr(pq), N.ptr(pd),
                                             N.ptr(qid), N.ptr(order), Bg, lo, B, seed, 1, 2,
                                             *[N.ptr(t) for t in toks], N.TT_I32, N.TT_I32, N.ptr(neg_t), N.ptr(err),
                                             N.stream()), "tt_assemble_triplets")
            N.check(lib.tt_assemble_triplet_rows(N.ptr(pq), N.ptr(pd), N.ptr(qid), N.ptr(order), Bg, lo, B, seed,
                                                 N.ptr(rows), N.ptr(neg_r), N.ptr(err), N.stream()),
                    "tt_assemble_triplet_rows")
            if B == 0:
                continue
            assert torch.equal(neg_t[:B], neg_r[:B])
            rows = rows[: 3 * B].view(3, B)
            for role, t in enumerate((toks[0], toks[2], toks[4])):
                assert torch.equal(rows[role], t[:, 0])
            o = order.long()
            assert torch.equal(rows[2], pd[o[neg_r[:B].long()]])
            assert torch.equal(rows[0], pq[o[lo:hi]]) and torch.equal(rows[1], pd[o[lo:hi]])
            parts.append(rows)
        cat = torch.cat(parts, dim=1)
        if full_rows is None:
            full_rows = cat
        assert torch.equal(cat, full_rows)
    assert int(err.item()) == 0


@gpu
def test_row_assembly_raises_the_flag_when_no_item_has_a_partner(tt):
    N, dev = tt.N, torch.device("cuda")
    lib = N.load()
    pq, pd, _ = _pairs(100, 10, 50, 5, 3, dev)
    same = torch.zeros(100, dtype=torch.int32, device=dev)
    order = torch.arange(16, dtype=torch.int32, device=dev)
    rows = torch.zeros(48, dtype=torch.int32, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    N.check(lib.tt_assemble_triplet_rows(N.ptr(pq), N.ptr(pd), N.ptr(same), N.ptr(order), 16, 0, 16, 1, N.ptr(rows),
                                         None, N.ptr(err), N.stream()), "tt_assemble_triplet_rows")
    assert int(err.item()) == 2
    # a bad slice is refused on the host with a message, and the next call is fine
    assert lib.tt_assemble_triplet_rows(N.ptr(pq), N.ptr(pd), N.ptr(same), N.ptr(order), 16, 8, 16, 1, N.ptr(rows),
                                        None, None, N.stream()) != 0
    assert "bad slice" in N.last_error()
    qid = torch.arange(100, dtype=torch.int32, device=dev)
    err.zero_()
    N.check(lib.tt_assemble_triplet_rows(N.ptr(pq), N.ptr(pd), N.ptr(qid), N.ptr(order), 16, 0, 16, 1, N.ptr(rows),
                                         None, N.ptr(err), N.stream()), "tt_assemble_triplet_rows")
    assert int(err.item()) == 0 and torch.equal(rows[:16], pq[:16])


# ---------------------------------------------------------------------------------------------------------------------
# 2. front phase, bit for bit against the token path (table backbone)
# ---------------------------------------------------------------------------------------------------------------------
V, LQ, LD = 3000, 16, 48


def _ragged_banks(tt, n_q=300, n_d=500, seed=0):
    """Ragged token banks; some texts are longer than Lq / Ld and get truncated."""
    rng = np.random.default_rng(seed)

    def bank(prefix, n, L):
        lens = rng.integers(1, L + 20, n)
        off = np.concatenate([[0], np.cumsum(lens)])
        return tt.data.TokenBank(prefix, rng.integers(1, V, int(off[-1])), off)

    return bank("q", n_q, LQ), bank("d", n_d, LD)


def _table_model(tt, precision, P=64, seed=0):
    torch.manual_seed(seed)
    return tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision=precision).cuda()


def _pair_of_trainers(tt, model, banks, B, precision, **kw):
    m_tok, m_row = copy.deepcopy(model), copy.deepcopy(model)
    common = dict(precision=precision, ids_dtype=torch.int32, mask_dtype=torch.uint8, **kw)
    t_tok = tt.training.FusedTrainer(m_tok, 0.3, 1e-2, B, LQ, LD, **common)
    pq = tt.data.PooledBank.build(m_row.query_tower, banks[0], LQ)
    pd = tt.data.PooledBank.build(m_row.document_tower, banks[1], LD)
    t_row = tt.training.FusedTrainer(m_row, 0.3, 1e-2, B, LQ, LD, pooled=(pq, pd), **common)
    return t_tok, t_row


@gpu
@pytest.mark.parametrize("B", [1, 129, 300])
@pytest.mark.parametrize("chain", ["1", "0"])
@pytest.mark.parametrize("precision", ["fp32", "bf16x3", "bf16"])
def test_pooled_rows_reproduce_the_token_step_bit_for_bit(tt, monkeypatch, precision, chain, B):
    monkeypatch.setenv("TT_CHAIN", chain)
    banks = _ragged_banks(tt, seed=B)
    model = _table_model(tt, precision)
    t_tok, t_row = _pair_of_trainers(tt, model, banks, B, precision, use_graph=False)
    rng = np.random.default_rng(B)
    H = t_tok.H
    for _ in range(3):  # three Adam steps
        rq, rp, rn = (rng.integers(0, len(banks[k]), B) for k in (0, 1, 1))
        kw = dict(ids_dtype=torch.int32, mask_dtype=torch.uint8)
        t_tok.load_tokens(banks[0].batch(rq, LQ, LQ, **kw), banks[1].batch(rp, LD, LD, **kw),
                          banks[1].batch(rn, LD, LD, **kw))
        t_row.load_rows(torch.from_numpy(np.stack([rq, rp, rn])))
        l_tok, l_row = t_tok.step(), t_row.step()
        torch.cuda.synchronize()
        s_tok, s_row = t_tok.step_objs[0], t_row.step_objs[0]
        assert torch.equal(s_tok.pooled_rows(), s_row.pooled_rows())
        if precision != "fp32":
            names = ("x_hi", "x_lo", "x_lo2") if precision == "bf16x3" else ("x_hi", "x_lo")
            for nm in names:
                assert torch.equal(s_tok.internal(nm, 3 * B, H), s_row.internal(nm, 3 * B, H)), nm
        assert torch.equal(l_tok, l_row)
        for g_tok, g_row in zip(t_tok.g_views, t_row.g_views):
            assert torch.equal(g_tok, g_row)
        assert int(s_row.err.item()) == 0
    assert torch.equal(t_tok.flat_p, t_row.flat_p)
    assert not torch.equal(t_row.flat_p, torch.cat([p.detach().reshape(-1) for p in model.projection_parameters()]))


@gpu
@pytest.mark.parametrize("chain", ["1", "0"])
def test_device_feeder_epoch_gives_equal_weights_in_both_modes(tt, monkeypatch, chain):
    """One FusedTrainer epoch per mode, batches assembled on the device with the same seed, graphs captured."""
    monkeypatch.setenv("TT_CHAIN", chain)
    ds = synth(tt, 2600)
    B, Lq, Ld = 256, 32, 256
    torch.manual_seed(3)
    model = tt.TwoTowersModel(projection_dim=64).cuda()
    m_tok, m_row = copy.deepcopy(model), copy.deepcopy(model)
    t_tok = tt.training.FusedTrainer(m_tok, 0.3, 1e-3, B, Lq, Ld, token_slots=2)
    banks = (tt.data.PooledBank.build(m_row.query_tower, ds.query_bank, Lq),
             tt.data.PooledBank.build(m_row.document_tower, ds.doc_bank, Ld))
    t_row = tt.training.FusedTrainer(m_row, 0.3, 1e-3, B, Lq, Ld, token_slots=2, pooled=banks)
    losses = []
    for tr in (t_tok, t_row):
        # the row trainer's feeder holds no token banks
        feeder = tt.data.DeviceTripletFeeder(ds, B, Lq, Ld, "cuda", seed=5, rows_only=tr is t_row)
        tr.prepare(2)
        losses.append(tr.train_epoch_device(feeder))
        assert tr.graph_captures >= 1
    assert losses[0] == losses[1] and math.isfinite(losses[0])
    assert torch.equal(t_tok.flat_p, t_row.flat_p)
    assert not hasattr(feeder, "d_flat")
    with pytest.raises(RuntimeError, match="rows_only"):
        feeder.assemble(t_tok, 0, 0)


# ---------------------------------------------------------------------------------------------------------------------
# 3. bank build: a MiniLM row does not depend on its batch or its padded length
# ---------------------------------------------------------------------------------------------------------------------
def _random_minilm_tower(tt, vocab=1000, seed=0):
    tower = tt.AveragePoolingTower(projection_dim=64, vocab_size=vocab, backbone="minilm")
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in tower.pretrained_model.named_parameters():
            if name.endswith("LayerNorm.weight"):
                p.copy_(1.0 + 0.3 * torch.randn(p.shape, generator=g))
            elif name.endswith(".bias"):
                p.copy_(0.2 * torch.randn(p.shape, generator=g))
            elif "query.weight" in name or "key.weight" in name:
                p.copy_(0.1 * torch.randn(p.shape, generator=g))
            elif name.endswith("dense.weight") or "value.weight" in name:
                p.copy_(torch.randn(p.shape, generator=g) / math.sqrt(p.shape[1]))
            else:
                p.copy_(0.02 * torch.randn(p.shape, generator=g))
    return tower.cuda()


@gpu
@pytest.mark.parametrize("max_tokens", [200, 5000])
def test_minilm_bank_rows_equal_the_pooled_rows_of_padded_mixed_batches(tt, max_tokens):
    tower = _random_minilm_tower(tt)
    L = 40
    rng = np.random.default_rng(max_tokens)
    lens = np.concatenate([np.arange(1, L + 1), rng.integers(L + 1, 90, 30), rng.integers(1, L + 1, 150)])
    rng.shuffle(lens)
    off = np.concatenate([[0], np.cumsum(lens)])
    bank = tt.data.TokenBank("t", rng.integers(1, 1000, int(off[-1])), off)
    built = tt.data.PooledBank.build(tower, bank, L, max_tokens_per_call=max_tokens)
    assert built.rows.shape == (len(bank), 384) and built.identity == tt.data.backbone_identity(tower)
    for trial in range(4):
        idx = rng.choice(len(bank), 64, replace=False)
        want = tower.pooled(bank.batch(idx, L, pad_to=L).to("cuda"))
        assert torch.equal(built.rows[torch.from_numpy(idx).cuda()], want), trial
    # the data-parallel build without a process group: slices encoded separately, then concatenated
    parts = [tt.data.PooledBank.encode_rows(tower, bank, L, *tt.retrieval.shard_bounds(len(bank), 3, r), max_tokens)
             for r in range(3)]
    assert torch.equal(torch.cat(parts), built.rows)


# ---------------------------------------------------------------------------------------------------------------------
# 4. MiniLM fused step against the reference-shaped autograd step
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_minilm_fused_step_matches_the_reference_step(tt, precision):
    ds = synth(tt, 1200)
    B, Lq, Ld = 96, 32, 256
    torch.manual_seed(1)
    model = tt.TwoTowersModel(projection_dim=64, backbone="minilm", precision=precision).cuda()
    ref = copy.deepcopy(model)
    banks = (tt.data.PooledBank.build(model.query_tower, ds.query_bank, Lq),
             tt.data.PooledBank.build(model.document_tower, ds.doc_bank, Ld))
    tr = tt.training.FusedTrainer(model, 0.3, 1e-3, B, Lq, Ld, pooled=banks, use_graph=False)
    feeder = tt.data.DeviceTripletFeeder(ds, B, Lq, Ld, "cuda", seed=9)
    feeder.start_epoch()
    toks = tuple(torch.zeros(B, L, dtype=dt_, device="cuda") for L in (Lq, Ld, Ld) for dt_ in (torch.int32, torch.uint8))
    feeder.assemble(types.SimpleNamespace(tok_slots=[toks]), 0, 0)
    feeder.assemble(tr, 0, 0)
    loss = tr.step(0)
    torch.cuda.synchronize()
    batches = [tt.TokenBatch(toks[2 * k], toks[2 * k + 1]) for k in range(3)]
    # the step's pooled rows are the towers' pooled rows of the tokens the token assembly wrote, bit for bit
    rows = tr.step_obj.pooled_rows()
    assert torch.equal(rows[:B], model.query_tower.pooled(batches[0]))
    assert torch.equal(rows[B:2 * B], model.document_tower.pooled(batches[1]))
    assert torch.equal(rows[2 * B:], model.document_tower.pooled(batches[2]))
    crit = tt.TripletLoss(0.3)
    ref_loss = crit(ref.encode_queries(batches[0]), ref.encode_documents(batches[1]), ref.encode_documents(batches[2]))
    ref_loss.backward()
    got, want = float(loss), float(ref_loss.detach())
    assert abs(got - want) <= 1e-4 * abs(want) + 1e-7
    for got, p in zip(tr.g_views, ref.projection_parameters()):
        assert float((got - p.grad).norm() / p.grad.norm()) < 1e-3
    feeder.check()


# ---------------------------------------------------------------------------------------------------------------------
# 5. driver
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("host_feeder,via_env", [("0", False), ("1", False), ("0", True)])
def test_run_training_trains_the_minilm_model(tt, monkeypatch, capsys, host_feeder, via_env):
    monkeypatch.setenv("TT_SYNTHETIC_DATA", "1")
    monkeypatch.setenv("TT_HOST_FEEDER", host_feeder)
    kw = {}
    if via_env:
        monkeypatch.setenv("TT_BACKBONE", "minilm")
    else:
        kw["backbone"] = "minilm"
    torch.manual_seed(0)
    model = tt.training.run_training(num_epochs=2, batch_size=256, learning_rate=1e-3, max_samples=3000,
                                     projection_dim=64, margin=0.3, use_wandb=False, accumulation_steps=1,
                                     use_mixed_precision=False, num_workers=0, run_comprehensive_test=False, **kw)
    out = capsys.readouterr().out
    assert isinstance(model, tt.TwoTowersModel) and "Fused B200 step: True" in out
    assert model.query_tower.backbone == "minilm" and model.document_tower.backbone == "minilm"
    assert any(line.startswith("Encoded ") and "MiniLM" in line for line in out.splitlines())
    losses = [float(l.split(":")[1]) for l in out.splitlines() if l.startswith("Average training loss")]
    ndcgs = [float(l.split(":")[1]) for l in out.splitlines() if l.startswith("Validation NDCG@10")]
    assert len(losses) == 2 and len(ndcgs) == 2 and all(np.isfinite(losses)) and all(0.0 <= n <= 1.0 for n in ndcgs)


# ---------------------------------------------------------------------------------------------------------------------
# 6. refusals
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_out_of_range_row_raises_the_flag_reads_row_zero_and_the_next_step_is_clean(tt, precision):
    banks = _ragged_banks(tt)
    model = _table_model(tt, precision)
    B = 8
    pq = tt.data.PooledBank.build(model.query_tower, banks[0], LQ)
    pd = tt.data.PooledBank.build(model.document_tower, banks[1], LD)
    tr = tt.training.FusedTrainer(model, 0.3, 1e-3, B, LQ, LD, precision=precision, pooled=(pq, pd), use_graph=False)
    rows = torch.arange(3 * B, dtype=torch.int32).view(3, B)
    rows[0, 3] = len(pq)        # one past the query bank
    rows[2, 5] = -1             # negative index into the document bank
    tr.load_rows(rows)
    tr.step()
    torch.cuda.synchronize()
    so = tr.step_obj
    x = so.pooled_rows()
    assert int(so.err.item()) == 1
    assert torch.equal(x[3], pq.rows[0]) and torch.equal(x[2 * B + 5], pd.rows[0])
    so.err.zero_()
    good = torch.arange(3 * B, dtype=torch.int32).view(3, B)
    tr.load_rows(good)
    tr.step()
    torch.cuda.synchronize()
    assert int(so.err.item()) == 0
    want = torch.cat([pq.rows[:B], pd.rows[B: 2 * B], pd.rows[2 * B: 3 * B]])
    assert torch.equal(so.pooled_rows(), want)


@gpu
def test_pooled_trainer_refusals(tt):
    banks = _ragged_banks(tt)
    model = _table_model(tt, "bf16x3")
    pq = tt.data.PooledBank.build(model.query_tower, banks[0], LQ)
    pd = tt.data.PooledBank.build(model.document_tower, banks[1], LD)
    with pytest.raises(ValueError, match="in_batch_negatives"):
        tt.training.FusedTrainer(model, 0.3, 1e-3, 8, LQ, LD, pooled=(pq, pd), in_batch_negatives=True)
    # a copy of the model has its own table: the banks of the original are stale for it
    with pytest.raises(RuntimeError, match="stale"):
        tt.training.FusedTrainer(copy.deepcopy(model), 0.3, 1e-3, 8, LQ, LD, pooled=(pq, pd))
    torch.manual_seed(0)
    trainable = tt.TwoTowersModel(projection_dim=64, vocab_size=V, train_table=True).cuda()
    with pytest.raises(ValueError, match="frozen"):
        tt.training.FusedTrainer(trainable, 0.3, 1e-3, 8, LQ, LD, pooled=(pq, pd))
    # the C ABI refuses pooled rows together with neg_index or table gradients, and stays usable
    tr = tt.training.FusedTrainer(model, 0.3, 1e-3, 8, LQ, LD, pooled=(pq, pd), use_graph=False)
    tr.load_rows(torch.zeros(3, 8, dtype=torch.int32))
    so = tr.step_obj
    neg = torch.zeros(8, dtype=torch.int32, device="cuda")
    so.slots[0].neg_index = neg.data_ptr()
    with pytest.raises(tt.N.NativeError, match="exclusive"):
        so.run(0)
    so.slots[0].neg_index = None
    # a step with table gradients (and the workspace they need) refuses pooled rows
    g = torch.zeros(V, 384, device="cuda")
    so2 = tt.ops.TripletStep(8, LQ, LD, 384, 64, V, "bf16x3", "cuda", train_table=True)
    so2.bind(None, None, tr.p_views, tr.g_views, 0.3, 1 / 8, 1.0, table_grads=(g, g))
    a = so2.slots[0]
    a.pooled_q, a.pooled_q_rows, a.pooled_d, a.pooled_d_rows = pq.rows.data_ptr(), len(pq), pd.rows.data_ptr(), len(pd)
    a.pooled_index = tr.row_bufs[0].data_ptr()
    with pytest.raises(tt.N.NativeError, match="frozen tables"):
        so2.run(0)
    tr.step()
    torch.cuda.synchronize()
    assert math.isfinite(float(tr.loss_view[0])) and int(so.err.item()) == 0


@gpu
def test_minilm_refusals_and_stale_banks(tt):
    tower_kw = dict(projection_dim=64, vocab_size=1000, backbone="minilm")
    torch.manual_seed(0)
    model = tt.TwoTowersModel(**tower_kw).cuda()
    with pytest.raises(ValueError, match="pooled="):
        tt.training.FusedTrainer(model, 0.3, 1e-3, 8, LQ, LD)
    banks = _ragged_banks(tt)
    banks = tuple(tt.data.TokenBank(b.prefix, b.flat % 1000, b.offsets) for b in banks)
    pq = tt.data.PooledBank.build(model.query_tower, banks[0], LQ)
    pd = tt.data.PooledBank.build(model.document_tower, banks[1], LD)
    tr = tt.training.FusedTrainer(model, 0.3, 1e-3, 8, LQ, LD, pooled=(pq, pd))
    tr.prepare()
    # backbone weights change after the build: the bank is stale, at construction, prepare() and every epoch
    with torch.no_grad():
        model.document_tower.pretrained_model.encoder.layer[0].output.dense.bias.add_(0.5)
    with pytest.raises(RuntimeError, match="stale"):
        tr.prepare()
    with pytest.raises(RuntimeError, match="stale"):
        tr.train_epoch([torch.zeros(3, 8, dtype=torch.int32)])
    with pytest.raises(RuntimeError, match="stale"):
        tt.training.FusedTrainer(model, 0.3, 1e-3, 8, LQ, LD, pooled=(pq, pd))
    # a rebuilt bank trains again
    pd2 = tt.data.PooledBank.build(model.document_tower, banks[1], LD)
    tr2 = tt.training.FusedTrainer(model, 0.3, 1e-3, 8, LQ, LD, pooled=(pq, pd2), use_graph=False)
    assert math.isfinite(tr2.train_epoch([torch.zeros(3, 8, dtype=torch.int32)]))


# ---------------------------------------------------------------------------------------------------------------------
# 7. checkpoint / resume over pooled banks, and the banks' shape checks
# ---------------------------------------------------------------------------------------------------------------------
def _model_and_banks(tt, backbone):
    banks = _ragged_banks(tt)
    if backbone == "minilm":
        banks = tuple(tt.data.TokenBank(b.prefix, b.flat % 1000, b.offsets) for b in banks)
        torch.manual_seed(0)
        return tt.TwoTowersModel(projection_dim=64, vocab_size=1000, backbone="minilm").cuda(), banks
    return _table_model(tt, "bf16x3"), banks


def _build(tt, model, banks):
    return (tt.data.PooledBank.build(model.query_tower, banks[0], LQ),
            tt.data.PooledBank.build(model.document_tower, banks[1], LD))


@gpu
@pytest.mark.parametrize("backbone", ["table", "minilm"])
def test_pooled_trainer_resumes_from_a_checkpoint_bit_exactly(tt, tmp_path, backbone):
    """Save after 3 of 6 steps, build a new trainer over the same model and banks, load the checkpoint, train on:
    the weights equal those of an uninterrupted run.  Loading must not make the banks stale."""
    model, banks = _model_and_banks(tt, backbone)
    ref = copy.deepcopy(model)
    B = 16
    rng = np.random.default_rng(0)
    batches = [torch.from_numpy(np.stack([rng.integers(0, len(banks[k]), B) for k in (0, 1, 1)])) for _ in range(6)]

    def trainer(m, pb):
        return tt.training.FusedTrainer(m, 0.3, 1e-2, B, LQ, LD, pooled=pb, use_graph=False)

    t_ref = trainer(ref, _build(tt, ref, banks))
    for b in batches:
        t_ref.load_rows(b)
        t_ref.step()
    pb = _build(tt, model, banks)
    t1 = trainer(model, pb)
    for b in batches[:3]:
        t1.load_rows(b)
        t1.step()
    path = str(tmp_path / "ck.pt")
    t1.save_checkpoint(path)
    t2 = trainer(model, pb)
    with torch.no_grad():
        t2.flat_p.add_(1.0)  # the checkpoint, not the aliased parameters, must restore the weights
    t2.load_checkpoint(path)
    t2.prepare()  # the banks are still current
    for b in batches[3:]:
        t2.load_rows(b)
        t2.step()
    torch.cuda.synchronize()
    assert torch.equal(t2.flat_p, t_ref.flat_p) and torch.equal(t2.exp_avg_sq, t_ref.exp_avg_sq)
    # a checkpoint whose backbone differs is refused before anything is loaded
    sd = torch.load(path, map_location="cpu", weights_only=False)
    key = next(k for k in sd["model"] if k.startswith("document_tower.pretrained_model."))
    sd["model"][key] = sd["model"][key] + 1.0
    before = t2.flat_p.clone()
    with pytest.raises(RuntimeError, match="backbone differs"):
        t2.load_state_dict(sd)
    assert torch.equal(t2.flat_p, before)
    t2.check_banks()


@gpu
def test_banks_of_another_length_or_layout_are_refused(tt):
    model, banks = _model_and_banks(tt, "table")
    pq, pd = _build(tt, model, banks)
    with pytest.raises(ValueError, match="truncate"):
        tt.training.FusedTrainer(model, 0.3, 1e-3, 8, LQ + 1, LD, pooled=(pq, pd))
    short = tt.data.PooledBank.build(model.document_tower, banks[1], LQ)
    with pytest.raises(ValueError, match="truncate"):
        tt.training.FusedTrainer(model, 0.3, 1e-3, 8, LQ, LD, pooled=(pq, short))
    # the query tower's bank is not the document tower's (another table)
    with pytest.raises(RuntimeError, match="stale"):
        tt.training.FusedTrainer(model, 0.3, 1e-3, 8, LQ, LD, pooled=(pq, pq))
    wide = torch.zeros(2 * len(pd), pd.rows.shape[1], device="cuda")
    wide[::2] = pd.rows
    strided = tt.data.PooledBank(wide[::2], pd.identity, pd.L)
    with pytest.raises(AssertionError, match="contiguous"):
        tt.training.FusedTrainer(model, 0.3, 1e-3, 8, LQ, LD, pooled=(pq, strided))
