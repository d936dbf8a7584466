"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the golden vectors that the
reference's own modules produced.  Tolerances are BASELINE.json's: pooled embeddings and loss 1e-4 relative,
gradients 1e-3 relative, top-10 ids bit-exact where score gaps exceed 1e-5."""
import os

import numpy as np
import pytest
import torch

from oracle import two_towers_oracle as O

pytestmark = pytest.mark.gpu

PRECISIONS = [p for p in os.environ.get("TT_TEST_PRECISIONS", "fp32,bf16x3").split(",") if p]


@pytest.fixture(scope="module")
def tt():
    import two_towers_overlords_b200 as pkg
    from two_towers_overlords_b200 import data, ops, retrieval, training

    pkg.ops, pkg.training, pkg.data, pkg.retrieval = ops, training, data, retrieval
    return pkg


DEV = "cuda"


def rel_err(got: torch.Tensor, want: torch.Tensor) -> float:
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).norm() / want.norm().clamp_min(1e-30))


def max_rel(got, want, floor):
    """Largest row-wise relative error: max_rows ||got - want||_inf / max(||want||_inf, floor)."""
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    if got.dim() == 1:
        got, want = got[None], want[None]
    num = (got - want).abs().amax(dim=-1)
    den = want.abs().amax(dim=-1).clamp_min(floor)
    return float((num / den).max())


# ---------------------------------------------------------------------------------------------------
# pooled gather
# ---------------------------------------------------------------------------------------------------
def test_pooling_golden(tt, golden_dir):
    g = np.load(os.path.join(golden_dir, "pooling.npz"))
    h = torch.from_numpy(g["h"])  # [6,13,384] -> a table of 78 rows addressed by position
    table = h.reshape(-1, 384).contiguous().to(DEV)
    ids = torch.arange(78).reshape(6, 13)
    x = tt.ops.pool(table, ids, torch.from_numpy(g["mask"]))
    want = torch.from_numpy(g["normed"])
    assert max_rel(x, want, 1e-6) < 1e-4
    assert float(x[2].abs().max()) == 0.0  # all-masked row -> exactly zero


@pytest.mark.parametrize("shape,B,L", [("U", 33, 32), ("U", 17, 256), ("Z", 64, 256), ("Z", 5, 32), ("U", 3, 1),
                                        ("U", 2, 512), ("Z", 9, 300)])
@pytest.mark.parametrize("table_dtype", [torch.float32, torch.bfloat16])
def test_pool_forward_vs_oracle(tt, shape, B, L, table_dtype):
    gen = torch.Generator().manual_seed(B * 1000 + L)
    V = 4099
    table = torch.randn(V, 384, generator=gen).to(table_dtype)
    ids, mask = O.synth_tokens(B, L, shape, gen, "doc", vocab=V)
    if shape == "Z":
        mask[0] = 0  # an all-masked sequence
        mask[1, ::2] = 0  # a non-prefix mask
    want = O.pooled_normalised(table.float(), ids, mask)
    for ids_dt, mask_dt in ((torch.int64, torch.int64), (torch.int32, torch.uint8), (torch.int16, torch.int32)):
        x = tt.ops.pool(table.to(DEV), ids.to(ids_dt), mask.to(mask_dt))
        assert x.shape == want.shape
        assert max_rel(x, want, 1e-3) < 1e-4, (ids_dt, mask_dt)
    xhat, cnt, nrm, err, _, _ = tt.ops.pool_forward(table.to(DEV), ids, mask)
    assert torch.equal(cnt.cpu(), mask.sum(1).float())
    assert int(err.item()) == 0


def test_pool_flags_out_of_range_ids(tt):
    table = torch.randn(100, 384).to(DEV)
    ids = torch.tensor([[1, 2, 100], [3, 4, 5]])
    _, _, _, err, _, _ = tt.ops.pool_forward(table, ids, torch.ones_like(ids))
    assert int(err.item()) == 1
    with pytest.raises(IndexError):
        tt.ops.pool(table, ids, torch.ones_like(ids), check_ids=True)
    # a masked out-of-range id is ignored, like padding
    _, _, _, err, _, _ = tt.ops.pool_forward(table, ids, torch.tensor([[1, 1, 0], [1, 1, 1]]))
    assert int(err.item()) == 0


@pytest.mark.parametrize("shape", ["U", "Z"])
def test_pool_backward_vs_autograd_and_deterministic(tt, shape):
    gen = torch.Generator().manual_seed(7)
    V, B, L = 1031, 40, 64
    table = torch.randn(V, 384, generator=gen)
    ids, mask = O.synth_tokens(B, L, shape, gen, "doc", vocab=V)
    ids[:, 3] = 17  # a hot token present in every sequence (long segment), duplicates inside rows
    ids[5, :10] = 17
    upstream = torch.randn(B, 384, generator=gen)
    t_ref = table.clone().requires_grad_(True)
    x_ref = torch.nn.functional.normalize(
        O.mean_pooling(torch.nn.functional.embedding(ids, t_ref), mask), p=2, dim=1)
    (x_ref * upstream).sum().backward()
    outs = []
    for _ in range(2):
        t = table.to(DEV).requires_grad_(True)
        x = tt.ops.pool(t, ids, mask)
        (x * upstream.to(DEV)).sum().backward()
        outs.append(t.grad.clone())
    assert torch.equal(outs[0], outs[1]), "scatter-add backward must be bit-reproducible"
    assert rel_err(outs[0], t_ref.grad) < 1e-3
    touched = torch.zeros(V, dtype=torch.bool)
    touched[ids[mask.bool()]] = True
    assert float(outs[0].cpu()[~touched].abs().max()) == 0.0


def test_pool_backward_heavy_segment(tt):
    """More than 256 occurrences of one id exercises the split (heavy) reduction."""
    gen = torch.Generator().manual_seed(8)
    V, B, L = 211, 300, 8
    table = torch.randn(V, 384, generator=gen)
    ids = torch.randint(0, V, (B, L), generator=gen)
    ids[:, 0] = 5
    ids[:, 1] = 5
    mask = torch.ones_like(ids)
    upstream = torch.randn(B, 384, generator=gen)
    t_ref = table.clone().requires_grad_(True)
    x_ref = torch.nn.functional.normalize(O.mean_pooling(torch.nn.functional.embedding(ids, t_ref), mask), p=2, dim=1)
    (x_ref * upstream).sum().backward()
    t = table.to(DEV).requires_grad_(True)
    (tt.ops.pool(t, ids, mask) * upstream.to(DEV)).sum().backward()
    assert rel_err(t.grad, t_ref.grad) < 1e-3
    assert rel_err(t.grad[5], t_ref.grad[5]) < 1e-3


# ---------------------------------------------------------------------------------------------------
# projection MLP and loss
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
# (M, P) with P % 128 == 64 and M off the 128-row tiles: a half-empty last column tile and a partial row tile.  The
# reference gates with its own fp32 ReLU, so no case may hold a pre-activation within rounding of the kink: at
# (300, 384, 320) one sits at 3e-8 and its flip alone moves dW1 by 1.9e-3 (see tests/test_step_parity.py::oracle_grads)
@pytest.mark.parametrize("M,H,P", [(64, 384, 64), (300, 384, 128), (1, 384, 64), (513, 384, 512), (130, 384, 384),
                                   (129, 384, 192), (302, 384, 320), (1100, 384, 448)])
def test_mlp_forward_backward_vs_oracle(tt, precision, M, H, P):
    gen = torch.Generator().manual_seed(M + P)
    torch.manual_seed(M * 1000 + P)  # nn.Linear draws from the global generator: keep the case reproducible
    x = torch.nn.functional.normalize(torch.randn(M, H, generator=gen), dim=1)
    lin1, lin2 = torch.nn.Linear(H, P), torch.nn.Linear(P, P)
    up = torch.randn(M, P, generator=gen) / M
    xr = x.clone().requires_grad_(True)
    y_ref = O.projection(xr, lin1.weight, lin1.bias, lin2.weight, lin2.bias)
    (y_ref * up).sum().backward()
    params = [p.detach().clone().to(DEV).requires_grad_(True) for p in (lin1.weight, lin1.bias, lin2.weight, lin2.bias)]
    xd = x.to(DEV).requires_grad_(True)
    y = tt.ops.mlp(xd, *params, precision)
    (y * up.to(DEV)).sum().backward()
    assert rel_err(y, y_ref) < 1e-4
    for got, want in zip(params, (lin1.weight, lin1.bias, lin2.weight, lin2.bias)):
        assert rel_err(got.grad, want.grad) < 1e-3
    assert rel_err(xd.grad, xr.grad) < 1e-3


@pytest.mark.parametrize("B,P", [(7, 16), (256, 64), (1000, 512)])
def test_triplet_loss_forward_backward_vs_oracle(tt, B, P):
    gen = torch.Generator().manual_seed(B)
    q, p, n = (torch.randn(B, P, generator=gen) for _ in range(3))
    q[0] = 0  # zero vector: cos = 0 through the per-vector clamp
    p[1] = 1e-9
    ref_in = [t.clone().requires_grad_(True) for t in (q, p, n)]
    loss_ref = O.triplet_loss(*ref_in, 0.3)
    (loss_ref * 2.5).backward()
    dev_in = [t.to(DEV).requires_grad_(True) for t in (q, p, n)]
    loss = tt.ops.triplet_loss(*dev_in, 0.3)
    (loss * 2.5).backward()
    assert abs(loss.item() - loss_ref.item()) <= 1e-4 * abs(loss_ref.item())
    for got, want in zip(dev_in[1:], ref_in[1:]):
        assert rel_err(got.grad[2:], want.grad[2:]) < 1e-3
    assert rel_err(dev_in[0].grad[2:], ref_in[0].grad[2:]) < 1e-3


# ---------------------------------------------------------------------------------------------------
# model surface against the reference's golden vectors
# ---------------------------------------------------------------------------------------------------
def _model_from_golden(tt, g, P, precision, prefix=""):
    V = g[prefix + "query_tower__pretrained_model__emb__weight"].shape[0]
    m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision=precision)
    with torch.no_grad():
        for name in ("query_tower", "document_tower"):
            t = getattr(m, name)
            t.pretrained_model.table.copy_(torch.from_numpy(g[f"{prefix}{name}__pretrained_model__emb__weight"]))
            for i in (0, 2):
                t.projection[i].weight.copy_(torch.from_numpy(g[f"{prefix}{name}__projection__{i}__weight"]))
                t.projection[i].bias.copy_(torch.from_numpy(g[f"{prefix}{name}__projection__{i}__bias"]))
    return m.to(DEV)


@pytest.mark.parametrize("tag,P,precision", [("p16", 16, "fp32"), ("p64", 64, "fp32")] +
                         ([("p64", 64, "bf16x3")] if "bf16x3" in PRECISIONS else []))
def test_model_step_matches_reference_golden(tt, golden_dir, tag, P, precision):
    g = np.load(os.path.join(golden_dir, f"step_{tag}.npz"))
    m = _model_from_golden(tt, g, P, precision)
    crit = tt.TripletLoss(margin=float(g["margin"]))
    tok = lambda nm: (torch.from_numpy(g[nm + "_ids"]), torch.from_numpy(g[nm + "_mask"]))  # noqa: E731
    q, p, n = m.encode_queries(tok("q")), m.encode_documents(tok("p")), m.encode_documents(tok("n"))
    for got, nm in ((q, "q"), (p, "p"), (n, "n")):
        assert rel_err(got, torch.from_numpy(g[nm])) < 1e-4
    loss = crit(q, p, n)
    assert abs(loss.item() - float(g["loss"])) <= 1e-4 * float(g["loss"])
    loss.backward()
    for name in ("query_tower", "document_tower"):
        for i in (0, 2):
            for kind in ("weight", "bias"):
                want = torch.from_numpy(g[f"grad__{name}__projection__{i}__{kind}"])
                got = getattr(getattr(m, name).projection[i], kind).grad
                assert rel_err(got, want) < 1e-3, (name, i, kind)
    # state_dict keys the reference's search.py relies on (backend/search.py:104-106)
    sd = m.state_dict()
    assert sd["query_tower.projection.2.weight"].shape == (P, P)
    assert "document_tower.projection.0.bias" in sd


@pytest.mark.parametrize("mode", ["train_epoch", "fused", "fused_graph"])
def test_three_adam_steps_match_reference_train_epoch(tt, golden_dir, mode):
    g = np.load(os.path.join(golden_dir, "train_epoch.npz"))
    m = _model_from_golden(tt, g, 32, "fp32", prefix="init__")
    margin, lr = float(g["margin"]), float(g["lr"])
    batches = []
    for b in range(3):
        batches.append(tuple((torch.from_numpy(g[f"b{b}_{nm}_ids"]), torch.from_numpy(g[f"b{b}_{nm}_mask"]))
                             for nm in ("q", "p", "n")))
    if mode == "train_epoch":
        opt = torch.optim.Adam(m.parameters(), lr=lr)
        avg = tt.training.train_epoch(m, batches, tt.TripletLoss(margin), opt, log_wandb=False)
    else:
        # padding=True pads each batch to its own max; masked padding to a common shape changes nothing
        B = batches[0][0][0].shape[0]
        Lq = max(b[0][0].shape[1] for b in batches)
        Ld = max(max(b[1][0].shape[1], b[2][0].shape[1]) for b in batches)
        pad = lambda t, L: torch.nn.functional.pad(t, (0, L - t.shape[1]))  # noqa: E731
        tr = tt.training.FusedTrainer(m, margin, lr, B, Lq, Ld, precision="fp32", use_graph=(mode == "fused_graph"),
                                      ids_dtype=torch.int64, mask_dtype=torch.int64)
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
                # compare the UPDATE (3 Adam steps of size ~lr), not the weights, so the check has teeth
                assert rel_err(got - init, want - init) < 2e-3, (mode, name, i, kind)


# ---------------------------------------------------------------------------------------------------
# fused step at BASELINE sizes: properties instead of a slow oracle
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
def test_fused_step_full_size_properties(tt, precision):
    torch.manual_seed(0)
    B, Lq, Ld, P = 2048, 32, 256, 512
    m = tt.TwoTowersModel(projection_dim=P, precision=precision).to(DEV)
    batch = O.synth_triplet_batch(B, Lq, Ld, "U", seed=5)
    tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, Lq, Ld, precision=precision, use_graph=False,
                                  ids_dtype=torch.int64, mask_dtype=torch.int64)
    for dst, src in zip(tr.tok, batch.astuple()):
        dst.copy_(src)
    tr._fwd_bwd()
    g1, loss1 = tr.flat_g[:-1].clone(), float(tr.loss_view.item())
    assert 0.2 < loss1 < 0.4  # random init: loss ~ margin (BASELINE.md sanity pin)
    # linearity: doubling the upstream gradient doubles every gradient exactly (power of two)
    tr.step_obj.args.grad_scale = 2.0
    tr._fwd_bwd()
    assert torch.equal(tr.flat_g[:-1], 2 * g1)
    tr.step_obj.args.grad_scale = 1.0
    # determinism
    tr._fwd_bwd()
    assert torch.equal(tr.flat_g[:-1], g1)
    # subset oracle: first 64 triplets through the oracle forward agree with the saved activations' loss
    ref = O.OracleTwoTowers(P)
    with torch.no_grad():
        for t_new, t_ref in ((m.query_tower, ref.query_tower), (m.document_tower, ref.document_tower)):
            t_ref.table.copy_(t_new.pretrained_model.table.cpu())
            for i in (0, 2):
                t_ref.projection[i].weight.copy_(t_new.projection[i].weight.cpu())
                t_ref.projection[i].bias.copy_(t_new.projection[i].bias.cpu())
    sub = tuple(t[:64] for t in batch.astuple())
    q, p, n = ref.encode_queries(sub[0], sub[1]), ref.encode_documents(sub[2], sub[3]), ref.encode_documents(sub[4], sub[5])
    qd = m.encode_queries((sub[0], sub[1]))
    assert rel_err(qd, q) < 1e-4
    ref_loss = O.triplet_loss(q, p, n, 0.3).item()
    got_loss = tt.TripletLoss(0.3)(qd, m.encode_documents((sub[2], sub[3])), m.encode_documents((sub[4], sub[5]))).item()
    assert abs(got_loss - ref_loss) <= 1e-4 * ref_loss


def test_fused_step_trainable_table_vs_oracle(tt):
    torch.manual_seed(1)
    V, B, Lq, Ld, P = 997, 48, 12, 40, 64
    m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision="fp32", train_table=True).to(DEV)
    ref = O.OracleTwoTowers(P, vocab=V, train_table=True)
    with torch.no_grad():
        for t_new, t_ref in ((m.query_tower, ref.query_tower), (m.document_tower, ref.document_tower)):
            t_ref.table.copy_(t_new.pretrained_model.table.cpu())
            for i in (0, 2):
                t_ref.projection[i].weight.copy_(t_new.projection[i].weight.cpu())
                t_ref.projection[i].bias.copy_(t_new.projection[i].bias.cpu())
    batch = O.synth_triplet_batch(B, Lq, Ld, "Z", seed=11, vocab=V)
    Lq_, Ld_ = batch.q_ids.shape[1], batch.p_ids.shape[1]
    tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, Lq_, Ld_, precision="fp32", use_graph=False,
                                  ids_dtype=torch.int64, mask_dtype=torch.int64)
    for dst, src in zip(tr.tok, batch.astuple()):
        dst.copy_(src)
    tr._fwd_bwd()
    q = ref.encode_queries(batch.q_ids, batch.q_mask)
    p = ref.encode_documents(batch.p_ids, batch.p_mask)
    n = ref.encode_documents(batch.n_ids, batch.n_mask)
    O.triplet_loss(q, p, n, 0.3).backward()
    assert rel_err(tr.table_grads[0], ref.query_tower.table.grad) < 1e-3
    assert rel_err(tr.table_grads[1], ref.document_tower.table.grad) < 1e-3
    # and the autograd surface gives the same table gradient
    m.zero_grad()
    loss = tt.TripletLoss(0.3)(m.encode_queries((batch.q_ids, batch.q_mask)),
                               m.encode_documents((batch.p_ids, batch.p_mask)),
                               m.encode_documents((batch.n_ids, batch.n_mask)))
    loss.backward()
    assert rel_err(m.document_tower.pretrained_model.table.grad, ref.document_tower.table.grad) < 1e-3


def test_adam_kernel_matches_torch_adam(tt):
    torch.manual_seed(3)
    p0 = torch.randn(5000)
    ref_p = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref_p], lr=3e-3)
    p, m, v = p0.to(DEV), torch.zeros(5000, device=DEV), torch.zeros(5000, device=DEV)
    p2, m2, v2 = p0.to(DEV), torch.zeros(5000, device=DEV), torch.zeros(5000, device=DEV)
    state = torch.zeros(4, dtype=torch.float64, device=DEV)
    N = tt.ops.N
    for step in range(1, 6):
        grad = torch.randn(5000) * 0.1
        ref_p.grad = grad.clone()
        opt.step()
        gd = grad.to(DEV)
        tt.ops.adam_step(p, gd, m, v, 3e-3, step)
        N.check(N.load().tt_adam_step_dev(N.ptr(p2), N.ptr(gd), N.ptr(m2), N.ptr(v2), 5000, 3e-3, 0.9, 0.999, 1e-8,
                                          N.ptr(state), 1.0, N.stream()), "adam_dev")
    assert max_rel(p, ref_p, 1e-3) < 1e-5
    assert max_rel(p2, ref_p, 1e-3) < 1e-5


# ---------------------------------------------------------------------------------------------------
# data-parallel exchange: fused reduce-scatter -> Adam -> all-gather over peer memory (tt_dp_reduce_adam)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world,n", [(1, 5000), (2, 919552), (4, 57600), (8, 919552), (3, 1001)])
def test_dp_exchange_virtual_ranks_match_summed_adam(tt, world, n):
    """`world` ranks on ONE device (own streams, plain pointers instead of IPC mappings) run the real protocol:
    every rank must end with bit-identical parameters == Adam applied to the rank-ordered sum of the gradients."""
    from two_towers_overlords_b200 import comm

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
        for step in range(1, 4):
            grads = [torch.randn(n + 1, device=DEV) * 0.1 for _ in xs]
            total = grads[0].clone()
            for g in grads[1:]:
                total += g  # rank order, fp32: what the kernel does
            torch.cuda.synchronize()
            for x, g, m, v, st in zip(xs, grads, ms, vs, streams):
                with torch.cuda.stream(st):
                    x.reduce_adam(g, m, v, 3e-3, max_ctas=16)
            torch.cuda.synchronize()
            for x in xs:
                x.check()
            tt.ops.adam_step(ref_p, total[:n].contiguous(), ref_m, ref_v, 3e-3, step)
            for x in xs:
                assert torch.equal(x.flat_p, xs[0].flat_p)       # replicas stay bit-identical
                assert torch.equal(x.loss, total[n:])            # loss slot = sum of the ranks' loss terms
            assert max_rel(xs[0].flat_p, ref_p, 1e-3) < 1e-6
        # Adam moments are sharded: rank r owns slice r, together they cover the reference moments
        S = (((n + 1 + world - 1) // world) + 63) // 64 * 64
        m_all = torch.cat([ms[r][r * S: min((r + 1) * S, n)] for r in range(world) if r * S < n])
        assert max_rel(m_all, ref_m, 1e-6) < 1e-6
    finally:
        for x in xs:
            x.close()


@pytest.mark.parametrize("use_graph", [False, True])
def test_fused_trainer_pipelined_and_peer_exchange_equal_plain_steps(tt, use_graph):
    """Three ways to run the same 5 steps must agree bit for bit: (a) plain sequential steps, (b) software-pipelined
    steps (pooled gather of step i+1 beside the rest of step i, alternating workspaces), (c) pipelined with the
    fused peer-memory exchange kernel as the optimiser (world = 1)."""
    B, Lq, Ld, P, V = 256, 16, 64, 128, 4096
    batches = [O.synth_triplet_batch(B, Lq, Ld, "U", seed=20 + i, vocab=V) for i in range(5)]
    out = []
    for mode in ("plain", "pipelined", "pipelined+peer"):
        torch.manual_seed(4)
        m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision="bf16x3").to(DEV)
        tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, Lq, Ld, precision="bf16x3", use_graph=use_graph,
                                      ids_dtype=torch.int64, mask_dtype=torch.int64, token_slots=2,
                                      exchange="peer" if mode.endswith("peer") else None)
        losses = []
        tr.load_packed(tr.pack_host_tokens(batches[0].astuple(), pin=False), 0)
        for i, b in enumerate(batches):
            slot, nslot = i % 2, None
            if mode != "plain" and i + 1 < len(batches):
                nslot = (i + 1) % 2
                tr.load_packed(tr.pack_host_tokens(batches[i + 1].astuple(), pin=False), nslot)
            tr.step(slot, nslot)
            losses.append(float(tr.loss_view[0].item()))
            if mode == "plain" and i + 1 < len(batches):
                tr.load_packed(tr.pack_host_tokens(batches[i + 1].astuple(), pin=False), (i + 1) % 2)
        torch.cuda.synchronize()
        out.append((tr.flat_p.clone(), losses))
        tr.close()
        assert torch.equal(m.query_tower.projection[0].weight.reshape(-1), out[-1][0][: P * 384])
    for other in out[1:]:
        assert out[0][1] == other[1]
        assert torch.equal(out[0][0], other[0])


@pytest.mark.parametrize("exchange", [None, "peer"])
def test_fused_trainer_checkpoint_resume_is_bit_exact(tt, tmp_path, exchange):
    """3 steps + save + fresh trainer + load + 2 steps == 5 uninterrupted steps (weights, Adam moments, step count)."""
    B, Lq, Ld, P, V = 128, 16, 48, 64, 2048
    batches = [O.synth_triplet_batch(B, Lq, Ld, "Z", seed=40 + i, vocab=V) for i in range(5)]
    Lq_, Ld_ = max(b.q_ids.shape[1] for b in batches), max(b.p_ids.shape[1] for b in batches)

    def pad(t, L):
        return torch.nn.functional.pad(t, (0, L - t.shape[1]))

    def feed(tr, b):
        toks = b.astuple()
        toks = tuple(pad(t, Lq_ if i < 2 else Ld_) for i, t in enumerate(toks))
        tr.load_packed(tr.pack_host_tokens(toks, pin=False))
        tr.step()

    def make():
        torch.manual_seed(9)
        m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision="bf16x3").to(DEV)
        return m, tt.training.FusedTrainer(m, 0.3, 1e-3, B, Lq_, Ld_, precision="bf16x3", ids_dtype=torch.int64,
                                           mask_dtype=torch.int64, exchange=exchange)
    m1, t1 = make()
    for b in batches:
        feed(t1, b)
    torch.cuda.synchronize()
    want = t1.flat_p.clone()
    t1.close()
    m2, t2 = make()
    for b in batches[:3]:
        feed(t2, b)
    ck = str(tmp_path / "e3.lr3.d64.m3.ckpt")
    t2.save_checkpoint(ck)
    t2.close()
    torch.manual_seed(123)  # different init: everything must come from the checkpoint
    m3 = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision="bf16x3").to(DEV)
    t3 = tt.training.FusedTrainer(m3, 0.3, 1e-3, B, Lq_, Ld_, precision="bf16x3", ids_dtype=torch.int64,
                                  mask_dtype=torch.int64, exchange=exchange)
    t3.load_checkpoint(ck)
    assert t3.steps_done == 3
    for b in batches[3:]:
        feed(t3, b)
    torch.cuda.synchronize()
    assert torch.equal(t3.flat_p, want)
    t3.close()
    # the model part alone is what the reference's main.py saves and search.py loads
    sd = torch.load(ck, weights_only=False)["model"]
    assert "query_tower.projection.2.weight" in sd and tuple(sd["query_tower.projection.2.weight"].shape) == (P, P)


# ---------------------------------------------------------------------------------------------------
# retrieval
# ---------------------------------------------------------------------------------------------------
def _check_topk(top_s, top_i, scores64, k):
    """ids bit-exact wherever the oracle's adjacent score gaps exceed 1e-5; scores within 1e-5."""
    Q = scores64.shape[0]
    for qi in range(Q):
        order = np.lexsort((np.arange(scores64.shape[1]), -scores64[qi]))[: k + 1]
        s = scores64[qi][order]
        got_i, got_s = top_i[qi], top_s[qi]
        kk = min(k, scores64.shape[1])
        assert np.allclose(got_s[:kk], s[:kk], atol=1e-5)
        for r in range(kk):
            gap_prev = s[r - 1] - s[r] if r > 0 else np.inf
            gap_next = s[r] - s[r + 1] if r + 1 < len(s) else np.inf
            if gap_prev > 1e-5 and gap_next > 1e-5:
                assert got_i[r] == order[r], (qi, r)
        assert (got_i[kk:] == -1).all()


@pytest.mark.parametrize("Q,N,P,k", [(1, 1000, 64, 10), (70, 4097, 384, 10), (200, 9950, 128, 16), (5, 7, 64, 10),
                                     (64, 65, 512, 1)])
def test_scan_topk_fp32_vs_oracle(tt, Q, N, P, k):
    gen = torch.Generator().manual_seed(Q * N)
    Qe, De = torch.randn(Q, P, generator=gen), torch.randn(N, P, generator=gen)
    Qn, Dn = tt.ops.l2_normalize_rows(Qe.to(DEV)), tt.ops.l2_normalize_rows(De.to(DEV))
    top_s, top_i = tt.ops.scan_topk(Qn, Dn, k=k, precision="fp32")
    qn = Qe.double() / Qe.double().norm(dim=1, keepdim=True)
    dn = De.double() / De.double().norm(dim=1, keepdim=True)
    _check_topk(top_s.cpu().numpy(), top_i.cpu().numpy(), (qn @ dn.T).numpy(), k)
    # the oracle's own per-query loop (reference semantics) agrees on the ids
    ids, _ = O.retrieval_eval(Qe[:3], De, [set()] * min(3, Q), k=min(k, N))
    assert np.array_equal(top_i.cpu().numpy()[:3, : min(k, N)], ids[:, :k])


@pytest.mark.parametrize("pair", ["0", "1"])
@pytest.mark.parametrize("Q,N,P,k", [(1, 1000, 64, 10), (70, 4097, 384, 10), (200, 9950, 128, 16), (5, 7, 64, 10),
                                     (64, 65, 512, 1), (300, 50_000, 384, 10), (129, 20_001, 72, 10)])
def test_scan_topk_tensor_core_vs_oracle(tt, monkeypatch, Q, N, P, k, pair):
    """tcgen05 scan: bf16 candidate generation + exact fp32 re-score must return the fp32 ranking.  pair = 1 forces the
    cta_group::2 kernel (256 queries per CTA pair, document tiles multicast) that long shards select by themselves."""
    monkeypatch.setenv("TT_SCAN_PAIR", pair)
    gen = torch.Generator().manual_seed(Q * N + 1)
    Qe, De = torch.randn(Q, P, generator=gen), torch.randn(N, P, generator=gen)
    Qn, Qb = tt.ops.l2_normalize_rows(Qe.to(DEV), want_bf16=True)
    Dn, Db = tt.ops.l2_normalize_rows(De.to(DEV), want_bf16=True)
    top_s, top_i = tt.ops.scan_topk(Qn, Dn, k=k, precision="bf16", Qb=Qb, Db=Db)
    qn = Qe.double() / Qe.double().norm(dim=1, keepdim=True)
    dn = De.double() / De.double().norm(dim=1, keepdim=True)
    _check_topk(top_s.cpu().numpy(), top_i.cpu().numpy(), (qn @ dn.T).numpy(), k)
    # and it is the same list the strict fp32 scan returns
    ref_s, ref_i = tt.ops.scan_topk(Qn, Dn, k=k, precision="fp32")
    same = (top_i == ref_i)
    gaps_ok = same | ((top_s - ref_s).abs() < 1e-5)
    assert bool(gaps_ok.all())


def test_scan_tensor_core_exact_rescan_of_unproven_queries(tt, monkeypatch):
    """With the error bound forced huge no candidate list can be proven complete: every query goes through the
    listed fp32 re-scan, whose result must equal the strict fp32 scan bit for bit."""
    gen = torch.Generator().manual_seed(77)
    Q, N, P, k = 150, 6000, 128, 10
    Qe, De = torch.randn(Q, P, generator=gen), torch.randn(N, P, generator=gen)
    Qn, Qb = tt.ops.l2_normalize_rows(Qe.to(DEV), want_bf16=True)
    Dn, Db = tt.ops.l2_normalize_rows(De.to(DEV), want_bf16=True)
    ref_s, ref_i = tt.ops.scan_topk(Qn, Dn, k=k, precision="fp32", id_base=1000)
    monkeypatch.setenv("TT_SCAN_EPS", "10")
    top_s, top_i = tt.ops.scan_topk(Qn, Dn, k=k, precision="bf16", Qb=Qb, Db=Db, id_base=1000)
    assert torch.equal(top_i, ref_i)
    assert torch.allclose(top_s, ref_s, atol=1e-6)


@pytest.mark.parametrize("pair", ["0", "1"])
def test_scan_tensor_core_full_shard_properties(tt, monkeypatch, pair):
    """1 M x 384 shard, 512 queries: planted neighbours are found, results are reproducible, and sharding the
    corpus over 4 'GPUs' + merge gives the identical list (both scan kernels)."""
    monkeypatch.setenv("TT_SCAN_PAIR", pair)
    gen = torch.Generator(device=DEV).manual_seed(5)
    N, Q, P, k = 1_000_000, 512, 384, 10
    De = torch.randn(N, P, generator=gen, device=DEV)
    Qe = torch.randn(Q, P, generator=gen, device=DEV)
    planted = torch.randint(0, N, (Q,), generator=gen, device=DEV)
    De[planted] = Qe + 0.3 * torch.randn(Q, P, generator=gen, device=DEV)
    shard = tt.retrieval.CorpusShard(De, precision="bf16")
    s1, i1 = shard.search(Qe, k)
    s2, i2 = shard.search(Qe, k)
    assert torch.equal(i1, i2) and torch.equal(s1, s2)
    assert bool((i1[:, 0] == planted).all())
    assert bool((s1[:, :-1] >= s1[:, 1:]).all())
    parts = []
    for r in range(4):
        lo, hi = tt.retrieval.shard_bounds(N, 4, r)
        parts.append(tt.retrieval.CorpusShard(De[lo:hi], id_base=lo, precision="bf16").search(Qe, k))
    ms, mi = tt.ops.topk_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
    assert torch.equal(mi, i1)
    # exactness of the scores: recompute the winners' cosines in float64
    qn = torch.nn.functional.normalize(Qe.double(), dim=1)
    dn = torch.nn.functional.normalize(De[i1[:, 0]].double(), dim=1)
    assert float(((qn * dn).sum(1) - s1[:, 0].double()).abs().max()) < 1e-5


def test_scan_ties_break_by_ascending_id(tt):
    De = torch.randn(50, 64)
    De[10] = De[3]
    De[40] = De[3]  # three identical documents
    Qe = De[3:4].clone()
    top_s, top_i = tt.ops.scan_topk(tt.ops.l2_normalize_rows(Qe.to(DEV)), tt.ops.l2_normalize_rows(De.to(DEV)), k=5)
    assert top_i[0, :3].tolist() == [3, 10, 40]


def test_sharded_scan_merge_equals_single_scan(tt):
    gen = torch.Generator().manual_seed(2)
    Q, N, P, k = 37, 3001, 64, 10
    Qe, De = torch.randn(Q, P, generator=gen).to(DEV), torch.randn(N, P, generator=gen).to(DEV)
    full = tt.retrieval.CorpusShard(De)
    s_all, i_all = full.search(Qe, k)
    for G in (2, 4, 8):
        parts = []
        for r in range(G):
            lo, hi = tt.retrieval.shard_bounds(N, G, r)
            parts.append(tt.retrieval.CorpusShard(De[lo:hi], id_base=lo).search(Qe, k))
        s, i = tt.ops.topk_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
        assert torch.equal(i, i_all) and torch.equal(s, s_all), G


def test_ndcg_kernel_vs_oracle(tt):
    gen = torch.Generator().manual_seed(4)
    Q, N, P = 40, 500, 64
    Qe, De = torch.randn(Q, P, generator=gen), torch.randn(N, P, generator=gen)
    rng = np.random.default_rng(0)
    relevant = [set(rng.choice(N, size=int(rng.integers(0, 12)), replace=False).tolist()) for _ in range(Q)]
    # plant similarity so that NDCG is non-trivial
    for qi, rel in enumerate(relevant):
        for d in list(rel)[:3]:
            De[d] = Qe[qi] + 0.5 * torch.randn(P, generator=gen)
    shard = tt.retrieval.CorpusShard(De.to(DEV))
    csr = tt.retrieval.relevance_csr(relevant, DEV)
    for k in (10, 5, 1):
        _, top_i, ndcg = tt.retrieval.retrieve_and_score(shard, Qe.to(DEV), csr, k=k)
        _, want = O.retrieval_eval(Qe, De, relevant, k=k)
        assert np.allclose(ndcg.cpu().numpy(), want, atol=1e-9)
    assert ndcg.cpu().numpy().max() > 0.5


def test_score_candidates_vs_oracle(tt):
    gen = torch.Generator().manual_seed(6)
    Q, N, P, C, k = 9, 300, 64, 40, 10
    Qe, De = torch.randn(Q, P, generator=gen), torch.randn(N, P, generator=gen)
    cand = torch.stack([torch.randperm(N, generator=gen)[:C] for _ in range(Q)])
    cand[0, 30:] = -1
    Qn, Dn = tt.ops.l2_normalize_rows(Qe.to(DEV)), tt.ops.l2_normalize_rows(De.to(DEV))
    top_s, top_i = tt.ops.score_candidates(Qn, Dn, cand.to(DEV), k=k)
    for qi in range(Q):
        c = cand[qi][cand[qi] >= 0]
        s = O.cosine_scores(Qe[qi: qi + 1], De[c])
        order = np.lexsort((c.numpy(), -s.astype(np.float64)))[:k]
        assert top_i[qi].cpu().tolist() == c[order].tolist()
        assert np.allclose(top_s[qi].cpu().numpy(), s[order], atol=1e-6)


# ---------------------------------------------------------------------------------------------------
# evaluate_model against the reference's evaluate_model (golden)
# ---------------------------------------------------------------------------------------------------
def test_evaluate_model_matches_reference_golden(tt, golden_dir):
    import random

    g = np.load(os.path.join(golden_dir, "evaluate.npz"))
    m = _model_from_golden(tt, g, 24, "fp32")
    flat_q = [g[f"bank_q_{i}"] for i in range(64)]
    flat_d = [g[f"bank_d_{i}"] for i in range(160)]
    mk = lambda pre, rows: tt.data.TokenBank(pre, np.concatenate(rows), np.concatenate([[0], np.cumsum([len(r) for r in rows])]))  # noqa: E731
    tok = tt.data.TokenBankTokenizer(mk("q", flat_q), mk("d", flat_d))
    m.query_tower.tokenizer = m.document_tower.tokenizer = tok

    class DS:
        def __init__(self):
            self.data = [{"query_id": int(q), "query": f"q:{int(q)}", "positive": f"d:{int(d)}"}
                         for q, d in zip(g["ds_query_id"], g["ds_doc"])]
            self.docs = sorted({d["positive"] for d in self.data})

        def __len__(self):
            return len(self.data)

        def __getitem__(self, i):
            return self.data[i]

        def get_unique_passages(self):
            return self.docs

    ds = DS()
    random.seed(1234)
    val = tt.training.evaluate_model(m, ds, sample_size=60, min_query_groups=10, candidate_pool_size=100)
    assert val == pytest.approx(float(g["val_ndcg10"]), abs=1e-9)
    random.seed(4321)
    full = tt.training.evaluate_model(m, ds, sample_size=120, min_query_groups=12, candidate_pool_size=-1,
                                      comprehensive=True, wandb_prefix="final_")
    for key, v in full.items():
        assert v == pytest.approx(float(g["full__" + key]), abs=1e-9), key


@pytest.mark.parametrize("n_unique", [8, 2])
def test_evaluate_model_handles_tied_scores_like_sklearn(tt, n_unique):
    """Duplicate passages tie exactly; the result must equal sklearn's tie-averaged NDCG (oracle restatement)."""
    import random

    torch.manual_seed(5)
    m = tt.TwoTowersModel(projection_dim=16, vocab_size=300, precision="fp32").to(DEV)
    rng = np.random.default_rng(1)
    rows_q = [rng.integers(1, 300, 6) for _ in range(6)]
    base_d = [rng.integers(1, 300, 12) for _ in range(n_unique)]
    rows_d = [base_d[i % n_unique] for i in range(40)]  # each passage appears 5 / 20 times under different handles
    mk = lambda pre, rows: tt.data.TokenBank(pre, np.concatenate(rows), np.concatenate([[0], np.cumsum([len(r) for r in rows])]))  # noqa: E731
    m.query_tower.tokenizer = m.document_tower.tokenizer = tt.data.TokenBankTokenizer(mk("q", rows_q), mk("d", rows_d))

    class DS:
        data = [{"query_id": i % 6, "query": f"q:{i % 6}", "positive": f"d:{(i * 7) % 40}"} for i in range(60)]
        docs = [f"d:{i}" for i in range(40)]

        def __len__(self):
            return len(self.data)

        def __getitem__(self, i):
            return self.data[i]

        def get_unique_passages(self):
            return self.docs

    ds = DS()
    random.seed(9)
    got = tt.training.evaluate_model(m, ds, sample_size=60, min_query_groups=6, candidate_pool_size=-1)
    # oracle: reference loop with tie-averaged NDCG
    with torch.no_grad():
        De = m.encode_documents(ds.docs).cpu()
        vals = []
        for qid in range(6):
            rel_docs = {d["positive"] for d in ds.data if d["query_id"] == qid}
            rel = np.array([1 if d in rel_docs else 0 for d in ds.docs])
            s = O.cosine_scores(m.encode_queries([f"q:{qid}"]).cpu(), De)
            vals.append(O.ndcg_at_k(rel, s, 10))
    assert got == pytest.approx(float(np.mean(vals)), abs=1e-6)


# ---------------------------------------------------------------------------------------------------
# C-ABI error behaviour
# ---------------------------------------------------------------------------------------------------
def test_c_abi_reports_errors_instead_of_crashing(tt):
    N = tt.ops.N
    lib = N.load()
    x = torch.zeros(4, 384, device=DEV)
    rc = lib.tt_pool_fwd(N.ptr(x), 0, 4, 100, N.ptr(x), 2, N.ptr(x), 2, 1, 1, N.ptr(x), None, None, None, N.stream())
    assert rc != 0 and "hidden size" in N.last_error()
    rc = lib.tt_pool_fwd(N.ptr(x), 0, 4, 384, N.ptr(x), 2, N.ptr(x), 2, 1, 600, N.ptr(x), None, None, None, N.stream())
    assert rc != 0 and "L=600" in N.last_error()
    with pytest.raises(N.NativeError):
        tt.ops.pool(torch.zeros(4, 384), torch.zeros(1, 1, dtype=torch.int64), None)  # CPU tensor: no fallback


# ---------------------------------------------------------------------------------------------------
# document index + search (backend/search.py surface over the scan kernel)
# ---------------------------------------------------------------------------------------------------
def test_document_search_engine_matches_cosine_ranking_and_persists(tt, tmp_path):
    from two_towers_overlords_b200 import search

    torch.manual_seed(0)
    model = tt.TwoTowersModel(projection_dim=64, precision="fp32")
    docs = [f"passage {i} mentions item {i % 17} beside thing {(i * 7) % 23} and note {(i * i) % 31}" for i in range(700)]
    eng = search.DocumentSearchEngine(model=model, index_dir=str(tmp_path))
    assert eng.get_index_info()["num_docs"] == 0
    eng.ingest_documents(docs[:300], batch_size=128, clear_existing=True)
    eng.ingest_documents(docs[300:], batch_size=256, persist=True)
    info = eng.get_index_info()
    assert info["num_docs"] == 700 and info["index_name"] == search.DEFAULT_INDEX_NAME
    query = "which passage mentions item 5 beside thing 7"
    res = eng.search(query, top_k=10)
    assert len(res) == 10 and set(res[0]) == {"id", "content", "score", "distance"}
    with torch.no_grad():
        q = model.encode_queries([query]).double().cpu()
        D = torch.cat([model.encode_documents(docs[i: i + 256]) for i in range(0, 700, 256)]).double().cpu()
    cos = torch.nn.functional.cosine_similarity(q, D).numpy()
    order = np.lexsort((np.arange(700), -cos))
    for r, hit in enumerate(res):
        assert abs(hit["score"] - (1.0 + cos[order[r]]) / 2.0) < 1e-5 and abs(hit["distance"] - (1.0 - hit["score"])) < 1e-12
        gap_prev = cos[order[r - 1]] - cos[order[r]] if r else np.inf
        gap_next = cos[order[r]] - cos[order[r + 1]]
        if gap_prev > 1e-5 and gap_next > 1e-5:
            assert hit["id"] == str(order[r]) and hit["content"] == docs[order[r]]
    # deeper than the tensor-core list limit -> fp32 scan, same head
    deep = eng.search(query, top_k=40)
    assert len(deep) == 40 and [h["id"] for h in deep[:10]] == [h["id"] for h in res]
    # the index survives the process like the reference's Redis index: a new engine finds it on disk
    eng2 = search.DocumentSearchEngine(model=model, index_dir=str(tmp_path))
    assert eng2.get_index_info()["num_docs"] == 700
    assert [h["id"] for h in eng2.search(query, top_k=10)] == [h["id"] for h in res]


# ---------------------------------------------------------------------------------------------------
# batch assembly on the device (data.py:113-152 semantics for a token bank resident in HBM)
# ---------------------------------------------------------------------------------------------------
def _feeder_setup(tt, n_pairs=3000, B=256, world=1, rank=0, seed=3):
    ds = tt.data.MSMarcoDataset("train", max_samples=n_pairs, synthetic=True)
    torch.manual_seed(0)
    m = tt.TwoTowersModel(projection_dim=64, precision="bf16x3").to(DEV)
    tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B // world, 32, 256, precision="bf16x3", token_slots=2,
                                  ids_dtype=torch.uint16, mask_dtype=torch.uint8)
    fd = tt.data.DeviceTripletFeeder(ds, B, 32, 256, DEV, rank=rank, world_size=world, seed=seed)
    return ds, m, tr, fd


def test_device_batch_assembly_matches_host_token_bank_and_negative_rule(tt):
    B = 256
    ds, m, tr, fd = _feeder_setup(tt, B=B)
    fd.start_epoch()
    counts = np.zeros(B, dtype=np.int64)
    for step in range(min(4, len(fd))):
        fd.assemble(tr, step % 2, step, want_neg=True)
        torch.cuda.synchronize()
        fd.check()
        order = fd.order[step * B: (step + 1) * B].cpu().numpy()
        neg = fd.neg.cpu().numpy()
        qidx = np.array([int(ds.data[i]["query"].split(":")[1]) for i in order])
        didx = np.array([int(ds.data[i]["positive"].split(":")[1]) for i in order])
        qid = np.array([int(ds.data[i]["query_id"]) for i in order])
        # the reference's rule: never itself, never a passage of the same query
        assert (neg != np.arange(B)).all() and (qid[neg] != qid).all() and neg.min() >= 0 and neg.max() < B
        counts += np.bincount(neg, minlength=B)
        got = [t.cpu() for t in tr.tok_slots[step % 2]]
        for (ids, mask), want in (((got[0], got[1]), ds.query_bank.batch(qidx, 32, 32)),
                                  ((got[2], got[3]), ds.doc_bank.batch(didx, 256, 256)),
                                  ((got[4], got[5]), ds.doc_bank.batch(didx[neg], 256, 256))):
            assert torch.equal(ids.to(torch.int64), want.input_ids) and torch.equal(mask.to(torch.int64), want.attention_mask)
        # a pure function of (seed, epoch, step): assembling again gives the same batch
        before = [t.clone() for t in tr.tok_slots[step % 2]]
        fd.assemble(tr, step % 2, step)
        assert all(torch.equal(a, b) for a, b in zip(before, tr.tok_slots[step % 2]))
    # roughly uniform choice of the partner (1024 draws over 256 bins: no bin should dominate)
    assert counts.max() <= 16 and (counts > 0).sum() > 200


def test_device_batch_assembly_rank_slices_agree_on_global_negatives(tt):
    B = 256
    ds, m, tr, fd = _feeder_setup(tt, B=B)
    fd.start_epoch()
    fd.assemble(tr, 0, 1, want_neg=True)
    full = [t.clone() for t in tr.tok_slots[0]]
    neg_full = fd.neg.clone()
    for rank in range(4):
        ds_r, m_r, tr_r, fd_r = _feeder_setup(tt, B=B, world=4, rank=rank)
        fd_r.start_epoch()
        assert torch.equal(fd_r.order, fd.order)  # same seed -> same permutation on every rank
        fd_r.assemble(tr_r, 0, 1, want_neg=True)
        lo, hi = rank * 64, (rank + 1) * 64
        assert torch.equal(fd_r.neg, neg_full[lo:hi])
        for a, b in zip(tr_r.tok_slots[0], full):
            assert torch.equal(a, b[lo:hi])


def test_train_epoch_device_equals_host_fed_training(tt):
    """Same batches through the device feeder and through pinned host buffers -> bit-identical weights."""
    B = 256
    ds, m, tr, fd = _feeder_setup(tt, n_pairs=1500, B=B)
    avg = tr.train_epoch_device(fd)
    torch.cuda.synchronize()
    assert 0.0 < avg < 0.5
    # replay: rebuild the very same batches on the host from the feeder's permutation and negatives
    ds2, m2, tr2, fd2 = _feeder_setup(tt, n_pairs=1500, B=B)
    fd2.start_epoch()
    assert torch.equal(fd2.order, fd.order)
    for step in range(len(fd2)):
        fd2.assemble(tr2, 0, step, want_neg=True)
        torch.cuda.synchronize()
        order, neg = fd2.order[step * B: (step + 1) * B].cpu().numpy(), fd2.neg.cpu().numpy()
        qidx = np.array([int(ds.data[i]["query"].split(":")[1]) for i in order])
        didx = np.array([int(ds.data[i]["positive"].split(":")[1]) for i in order])
        kw = dict(ids_dtype=torch.uint16, mask_dtype=torch.uint8)
        tr2.load_tokens(ds.query_bank.batch(qidx, 32, 32, **kw), ds.doc_bank.batch(didx, 256, 256, **kw),
                        ds.doc_bank.batch(didx[neg], 256, 256, **kw), slot=1)
        tr2.step(1)
    torch.cuda.synchronize()
    assert torch.equal(tr.flat_p, tr2.flat_p)


@pytest.mark.parametrize("host_feeder", ["0", "1"])
def test_run_training_end_to_end_readme_dev_shape(tt, monkeypatch, capsys, host_feeder):
    """BASELINE configs[0] in small: run_training with the reference's signature on the synthetic corpus (fused step,
    device- or host-assembled batches, validation NDCG@10 every epoch) returns a trained TwoTowersModel."""
    monkeypatch.setenv("TT_SYNTHETIC_DATA", "1")
    monkeypatch.setenv("TT_HOST_FEEDER", host_feeder)
    torch.manual_seed(0)
    model = tt.training.run_training(num_epochs=2, batch_size=256, learning_rate=1e-3, max_samples=3000,
                                     projection_dim=64, margin=0.3, use_wandb=False, accumulation_steps=1,
                                     use_mixed_precision=False, num_workers=0, run_comprehensive_test=False)
    out = capsys.readouterr().out
    assert isinstance(model, tt.TwoTowersModel) and "Fused B200 step: True" in out
    losses = [float(l.split(":")[1]) for l in out.splitlines() if l.startswith("Average training loss")]
    ndcgs = [float(l.split(":")[1]) for l in out.splitlines() if l.startswith("Validation NDCG@10")]
    assert len(losses) == 2 and len(ndcgs) == 2 and all(np.isfinite(losses)) and all(0.0 <= n <= 1.0 for n in ndcgs)
    assert losses[0] < 0.35  # random init starts at the margin (0.3); training must not blow up
    sd = model.state_dict()
    assert tuple(sd["query_tower.projection.2.weight"].shape) == (64, 64)


@pytest.mark.parametrize("world", [1, 2, 8])
def test_peer_list_merge_virtual_ranks_equals_topk_merge(tt, world):
    """tt_peer_barrier + tt_peer_topk_merge (lists read in place from every rank's segment) == tt_topk_merge of the
    gathered lists, ties by ascending id, -1 ids ignored; `world` ranks on one device, one stream each."""
    from two_towers_overlords_b200 import comm

    torch.manual_seed(world)
    Q, k = 300, 10
    pls = comm.PeerLists.virtual_ranks(Q, k, world, DEV)
    parts_s = torch.randn(world, Q, k, device=DEV).sort(dim=2, descending=True).values
    parts_s[:, ::7, 3:5] = 0.25  # ties across and inside lists
    parts_s = parts_s.sort(dim=2, descending=True).values
    parts_i = torch.stack([torch.arange(Q * k, device=DEV).reshape(Q, k) * world + r for r in range(world)])
    parts_i[-1, ::5, 7:] = -1    # a short shard
    want_s, want_i = tt.ops.topk_merge(parts_s, parts_i)
    streams = [torch.cuda.Stream() for _ in range(world)]
    torch.cuda.synchronize()
    outs = []
    try:
        for rep in range(2):  # twice: the epoch counters of the barriers must advance
            outs = []
            for r, (pl, st) in enumerate(zip(pls, streams)):
                with torch.cuda.stream(st):
                    outs.append(pl.merge(parts_s[r], parts_i[r]))
            torch.cuda.synchronize()
            for pl, (s_, i_) in zip(pls, outs):
                pl.check()
                assert torch.equal(i_, want_i) and torch.equal(s_[want_i >= 0], want_s[want_i >= 0])
    finally:
        for pl in pls:
            pl.close()


def test_scan_streaming_regime_is_repeatable_under_stress(tt):
    """128 queries against a 2.2 M-document shard (147 document splits, an odd number of tiles per CTA, a 9-slot ring
    that is not a multiple of the 6 k-blocks of a tile), 600 back-to-back searches: every one must return the ids of
    the first and the kernel must never trap (a two-issuer variant of the kernel failed exactly here)."""
    g = torch.Generator(device=DEV).manual_seed(5)
    De = torch.randn(2_200_000, 384, generator=g, device=DEV)
    Qe = torch.randn(128, 384, generator=g, device=DEV)
    shard = tt.retrieval.CorpusShard(De, precision="bf16")
    del De
    ref_s, ref_i = shard.search(Qe, 10)
    torch.cuda.synchronize()
    for it in range(600):
        s, i = shard.search(Qe, 10)
        if it % 100 == 99:
            torch.cuda.synchronize()
            assert torch.equal(i, ref_i) and torch.equal(s, ref_s)
    # and the list is the exact one: fp32 scan of the same shard (ids may only differ inside a near-tie, gap <= 1e-5)
    s32, i32 = tt.ops.scan_topk(tt.ops.l2_normalize_rows(Qe), shard.Dn, k=11, precision="fp32")
    s32, i32, got_i, got_s = s32.cpu().numpy(), i32.cpu().numpy(), ref_i.cpu().numpy(), ref_s.cpu().numpy()
    assert np.allclose(got_s, s32[:, :10], atol=1e-5)
    for q, r in zip(*np.nonzero(got_i != i32[:, :10])):
        gaps = [abs(s32[q, r] - s32[q, r + 1])] + ([abs(s32[q, r] - s32[q, r - 1])] if r else [])
        assert min(gaps) <= 1e-5, (q, r, gaps)


@pytest.mark.parametrize("K", [64, 320])
def test_mn_major_tcgen05_operands_are_exact(tt, K):
    """The persistent chain kernel reads row-major activations as MN-major tcgen05 operands (no transposed copies).
    D = A^T B over small integers is exact in bf16 x bf16 -> fp32, so the device product must equal the host's bit for
    bit; a wrong leading / stride offset or K step in the shared-memory descriptor scrambles it."""
    from two_towers_overlords_b200 import _native as N

    g = torch.Generator().manual_seed(K)
    A = (torch.randint(-8, 9, (K, 128), generator=g).float() / 8).to(torch.bfloat16)
    B = (torch.randint(-6, 7, (K, 128), generator=g).float() / 4).to(torch.bfloat16)
    want = A.float().t() @ B.float()
    Ad, Bd = A.to(DEV), B.to(DEV)
    D = torch.empty(128, 128, dtype=torch.float32, device=DEV)
    N.check(N.load().tt_selftest_mn_major(N.ptr(Ad), N.ptr(Bd), K, N.ptr(D), N.stream()), "tt_selftest_mn_major")
    assert torch.equal(D.cpu(), want)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("chain", ["1", "0"])
def test_in_batch_negative_reuse_gives_the_same_bits(tt, monkeypatch, precision, chain):
    """The reference's batcher draws every negative among the other items' positives (backend/data.py:113-137).  Given
    their indices (tt_step_args.neg_index) the pooled gather visits each positive once and copies its row to the
    negatives that name it: pooled rows, loss, every gradient and the weights after three Adam steps must be bit-identical
    to gathering the negatives' own tokens.  One positive is named by three negatives, one by none; ragged masks."""
    monkeypatch.setenv("TT_CHAIN", chain)
    B, Lq, Ld, P, V = 300, 16, 48, 64, 2048
    g = torch.Generator().manual_seed(5)

    def batch(seed):
        b = O.synth_triplet_batch(B, Lq, Ld, "Z", seed=seed, vocab=V)
        q_ids, q_mask, p_ids, p_mask, _, _ = b.astuple()
        Ld_ = p_ids.shape[1]
        neg = torch.roll(torch.arange(B), 7)
        neg[:3] = 11  # positive 11 is the negative of three items (and of a fourth through the roll)
        return (q_ids, q_mask, p_ids, p_mask, p_ids[neg].clone(), p_mask[neg].clone()), neg.to(torch.int32), q_ids.shape[1], Ld_

    batches = [batch(70 + i) for i in range(3)]
    Lq_, Ld_ = max(b[2] for b in batches), max(b[3] for b in batches)

    def pad(t, L):
        return torch.nn.functional.pad(t, (0, L - t.shape[1]))

    def run(reuse):
        torch.manual_seed(3)
        m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision=precision).to(DEV)
        tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, Lq_, Ld_, precision=precision, ids_dtype=torch.int64,
                                      mask_dtype=torch.int64, in_batch_negatives=reuse)
        outs = []
        for toks, neg, _, _ in batches:
            toks = tuple(pad(t, Lq_ if i < 2 else Ld_) for i, t in enumerate(toks))
            if reuse:  # the negatives' own token tensors are never read: poison them
                toks = toks[:4] + (torch.full_like(toks[4], V - 1), torch.ones_like(toks[5]))
                tr.load_neg_index(neg)
            tr.load_packed(tr.pack_host_tokens(toks, pin=False))
            loss = tr.step()
            outs.append((float(loss.item()), tr.step_obj.pooled_rows().clone(), [g_.clone() for g_ in tr.g_views]))
        torch.cuda.synchronize()
        assert int(tr.step_obj.err.item()) == 0
        w = tr.flat_p.clone()
        tr.close()
        return outs, w

    a, wa = run(False)
    b, wb = run(True)
    for (la, xa, ga), (lb, xb, gb) in zip(a, b):
        assert la == lb
        assert torch.equal(xa, xb)
        assert all(torch.equal(u, v) for u, v in zip(ga, gb))
    assert torch.equal(wa, wb)


def test_in_batch_negative_index_out_of_range_raises_the_error_flag(tt):
    B, Lq, Ld, P, V = 64, 8, 16, 64, 512
    torch.manual_seed(0)
    m = tt.TwoTowersModel(projection_dim=P, vocab_size=V, precision="bf16x3").to(DEV)
    tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, Lq, Ld, precision="bf16x3", ids_dtype=torch.int64,
                                  mask_dtype=torch.int64, in_batch_negatives=True)
    tr.load_packed(tr.pack_host_tokens(O.synth_triplet_batch(B, Lq, Ld, "U", seed=1, vocab=V).astuple(), pin=False))
    neg = torch.roll(torch.arange(B), 1)
    neg[5] = B  # not a row of this batch
    tr.load_neg_index(neg)
    tr.step()
    torch.cuda.synchronize()
    assert int(tr.step_obj.err.item()) != 0
    tr.close()


# ---------------------------------------------------------------------------------------------------
# bench.py --dump-outputs
# ---------------------------------------------------------------------------------------------------
def test_bench_dumps_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs: loss, the 8 projection gradients and the updated parameters of the last timed step as
    float32 .npy files, the loss equal to the one the JSON line reports, within the 64 MB budget."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "2", "--warmup", "3", "--no-cpu",
                          "--no-scan", "--no-config2", "--no-backbone", "--no-chain-variant", "--no-epoch",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=root)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == 2
    names = [f"{t}.projection.{i}.{k}" for t in ("query_tower", "document_tower") for i in (0, 2)
             for k in ("weight", "bias")]
    want = {"loss.npy"} | {n + ".npy" for n in names} | {"grad." + n + ".npy" for n in names}
    assert set(os.listdir(tmp_path)) == want
    assert sum(os.path.getsize(tmp_path / f) for f in want) <= 64 << 20
    arrays = {f[:-4]: np.load(tmp_path / f) for f in want}
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
    assert arrays["loss"].shape == (1,) and float(arrays["loss"][0]) == d["loss_after"]
    P, H = d["config"]["projection_dim"], 384
    assert arrays["query_tower.projection.0.weight"].shape == (P, H)
    assert arrays["document_tower.projection.2.weight"].shape == (P, P)
    assert all(np.abs(arrays["grad." + n]).max() > 0 for n in names)
