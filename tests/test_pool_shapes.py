"""The pooled gather (csrc/tt_pool.cu) and its table gradient (csrc/tt_pool_bwd.cu) against float64, and the table
gradient against an exact float32 replay of the summation order DESIGN.md §4 promises.

A. `ops.pool_forward` at every hidden size (128, 256, 384, 768), fp32 and bf16 tables, every tail of "4 warps x 4 / 8 / 16
   rows in flight" and of the 128-token compaction loop (n unmasked tokens from 0 to 512), prefix / scattered / last-only
   masks, all id and mask dtypes (bit-identical wherever the values fit), weighted masks, u16 ids >= 32768, 70,000-row
   tables, all-masked and all-zero rows and a near-cancelling row.  Every element must satisfy
   |x - x64| <= TAU_F * max(1, kappa_row), kappa_row = ||sum |w_t| |E_t| ||_2 / ||sum w_t E_t||_2 in float64, so
   cancellation cannot fail a correct kernel.
B. The gather inside `ops.TripletStep` (3 segments reordered longest-first, row offsets, in-batch negative copies, the
   bf16 terms of the tensor-core projection): bit-identical to `ops.pool_forward` of each token set.
C. The table gradient of `ops.pool` against float64 autograd: 1, 2 and 3 radix passes, the masked-token sentinel at the
   top digit value, runs around the 256-entry heavy threshold and the 2048-entry chunks, token counts around the
   1024-item sort slices.  Each touched row must satisfy ||d - d64||_inf <= TAU_B * ||sum_t |w_t| |g64_seq(t)| ||_inf.
D. `TripletStep(train_table=True)`: dtable_q and dtable_d bit-identical to the promised float32 sums of the step's own
   g, including a 1,075,200-token document batch (W = 1050 sort slices: the carry of digit_scan_kernel), and the
   `accumulate = 1` path of the tt_pool_bwd C ABI.
"""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
# Gates.  Worst values measured over this file on one NVIDIA B200 at a 1000 W power limit: forward 3.3e-7 (xhat) and
# 1.5e-7 (nrm), table gradient 9.4e-7, g 1.7e-7.
TAU_F = 1e-6   # forward, per element, times max(1, kappa_row)
TAU_B = 3e-6   # table gradient, per row, relative to || sum |w| |g64| ||_inf
TAU_G = 1e-6   # g = normalize-backward(dxhat) / cnt, per row, relative to || (|dxhat| + |xhat| |dxhat.xhat|) / (nrm cnt) ||_inf
HEAVY, SLICE, CHUNK = 256, 256, 2048  # tt_pool_bwd.cu: kHeavy, kChunk / 8 warps, kChunk

ID_DTYPES = (torch.int64, torch.int32, torch.int16, torch.uint16)
MASK_DTYPES = (torch.int64, torch.int32, torch.uint8, torch.bool)


@pytest.fixture(scope="module")
def tt():
    import two_towers_overlords_b200 as pkg
    from two_towers_overlords_b200 import _native, ops

    pkg.ops, pkg._native = ops, _native
    return pkg


def bits(t):
    t = t.detach().contiguous().cpu()
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16)


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def as_dtype(x, dtype):
    """CPU int64 tensor -> dtype; int16 takes the low 16 bits (the kernels read int16 ids as u16)."""
    if dtype == torch.uint16:
        return torch.from_numpy(x.numpy().astype(np.uint16))
    if dtype == torch.int16:
        return torch.from_numpy(x.numpy().astype(np.uint16).view(np.int16))
    return x.to(dtype)


# ---------------------------------------------------------------------------------------------------------------------
# A. forward against float64
# ---------------------------------------------------------------------------------------------------------------------
NS = (0, 1, 3, 4, 5, 15, 16, 17, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 511, 512)
LS = (1, 33, 128, 129, 512)
V_A = 4099
ZERO_ID, REP_ID, CANCEL_IDS = 7, 5, (11, 12, 13)  # an all-zero table row; a repeated id; E, -E, 1e-3 * E'

_TABLES = {}


def table_a(V, H, dtype):
    key = (V, H, dtype)
    if key not in _TABLES:
        t = torch.randn(V, H, generator=torch.Generator().manual_seed(V * 7 + H)).to(dtype)
        if V > max(CANCEL_IDS):
            t[ZERO_ID] = 0
            t[CANCEL_IDS[1]] = -t[CANCEL_IDS[0]]
            t[CANCEL_IDS[2]] = (t[CANCEL_IDS[2]].float() * 1e-3).to(dtype)
        _TABLES[key] = (t, t.to(DEV))
    return _TABLES[key]


def pool64(table, ids, mask):
    """float64 xhat [B,H], cnt [B], nrm [B], kappa [B] of masked-mean pooling + L2 normalisation (model.py:48-72)."""
    E = table.double()
    w = mask.double()
    B, H = ids.shape[0], E.shape[1]
    seq, pos = torch.nonzero(w != 0, as_tuple=True)
    wt = w[seq, pos][:, None]
    rows = E[ids[seq, pos]]
    s = torch.zeros(B, H, dtype=torch.float64).index_add_(0, seq, rows * wt)
    a = torch.zeros(B, H, dtype=torch.float64).index_add_(0, seq, rows.abs() * wt.abs())
    cnt = w.sum(1)
    m = s / cnt.clamp_min(1e-9)[:, None]
    nrm = m.norm(dim=1)
    x = m / nrm.clamp_min(1e-12)[:, None]
    sn, an = s.norm(dim=1), a.norm(dim=1)
    kappa = torch.where(sn > 0, an / sn.clamp_min(1e-300), torch.where(an > 0, torch.inf, 1.0))
    return x, cnt, nrm, kappa


def check_forward(tag, got, table, ids, mask):
    """got = (xhat, cnt, nrm) of the device; ids as the kernel reads them (int64, low 16 bits for int16).  Returns the
    worst |x - x64| / max(1, kappa) over elements and the worst relative nrm error over max(1, kappa)."""
    xhat, cnt, nrm = (t.detach().cpu() for t in got[:3])
    x64, c64, n64, kap = pool64(table, ids, mask)
    assert torch.equal(cnt, c64.float()), (tag, "cnt")
    k1 = kap.clamp_min(1.0)
    e_x = (xhat.double() - x64).abs().amax(1) / k1
    zero = n64 == 0
    assert bool((xhat[zero] == 0).all()) and bool((nrm[zero] == 0).all()), (tag, "rows of zero norm must be exactly 0")
    e_n = torch.where(zero, 0.0, (nrm.double() - n64).abs() / n64.clamp_min(1e-300) / k1)
    wx, wn = float(e_x.max()), float(e_n.max())
    assert wx <= TAU_F, (tag, "xhat", int(e_x.argmax()), wx)
    assert wn <= TAU_F, (tag, "nrm", int(e_n.argmax()), wn)
    return wx, wn


def forward_rows(L, V, gen):
    """ids [R, L] int64 and binary mask [R, L] int64 covering every n of NS up to L in prefix and scattered layouts, a
    last-only row, a repeated id, ids 0 and V - 1, an all-zero table row, a near-cancelling row and an all-masked row.
    Masked positions hold random ids, some out of range (they must be ignored)."""
    rows_i, rows_m = [], []

    def add(ids, mask):
        rows_i.append(ids)
        rows_m.append(mask)

    def rnd(n):
        return torch.randint(0, V, (n,), generator=gen)

    for n in NS:
        if n > L:
            continue
        m = torch.zeros(L, dtype=torch.int64)
        m[:n] = 1
        add(rnd(L), m)  # prefix
        if 0 < n < L:
            m = torch.zeros(L, dtype=torch.int64)
            m[torch.randperm(L, generator=gen)[:n]] = 1
            add(rnd(L), m)  # scattered
    m = torch.zeros(L, dtype=torch.int64)
    m[-1] = 1
    add(rnd(L), m)  # last position only
    add(torch.full((L,), REP_ID), torch.ones(L, dtype=torch.int64))
    ends = torch.where(torch.arange(L) % 2 == 0, 0, V - 1)
    add(ends, (torch.rand(L, generator=gen) < 0.7).long() | (torch.arange(L) == 0).long())
    add(torch.full((L,), ZERO_ID), torch.ones(L, dtype=torch.int64))
    if L >= 3:
        ids, m = rnd(L), torch.zeros(L, dtype=torch.int64)
        p = torch.randperm(L, generator=gen)[:3]
        ids[p] = torch.tensor(CANCEL_IDS)
        m[p] = 1
        add(ids, m)
    add(rnd(L), torch.zeros(L, dtype=torch.int64))
    ids, mask = torch.stack(rows_i), torch.stack(rows_m)
    junk = (mask == 0) & (torch.rand(ids.shape, generator=gen) < 0.25)
    ids[junk] = V + 3  # masked out-of-range ids
    return ids, mask


@pytest.mark.parametrize("L", LS)
@pytest.mark.parametrize("table_dtype", [torch.float32, torch.bfloat16], ids=["f32", "bf16"])
@pytest.mark.parametrize("H", [128, 256, 384, 768])
def test_pool_forward_tails_vs_float64(tt, H, table_dtype, L):
    table, table_dev = table_a(V_A, H, table_dtype)
    gen = torch.Generator().manual_seed(H * 1000 + L)
    ids, mask = forward_rows(L, V_A, gen)
    base = tt.ops.pool_forward(table_dev, ids, mask)
    assert int(base[3].item()) == 0
    wx, wn = check_forward((H, L), base, table, ids, mask)
    print(f"pool_shapes forward H={H} {table_dtype} L={L}: xhat {wx:.2e} nrm {wn:.2e}")
    again = tt.ops.pool_forward(table_dev, ids, mask)
    assert all(same_bits(a, b) for a, b in zip(base[:3], again[:3])), "second call differs"
    for idt in ID_DTYPES:
        for mdt in MASK_DTYPES:
            got = tt.ops.pool_forward(table_dev, as_dtype(ids, idt), mask.to(mdt))
            assert all(same_bits(a, b) for a, b in zip(base[:3], got[:3])), (idt, mdt)
            assert int(got[3].item()) == 0


@pytest.mark.parametrize("H", [128, 768])
def test_pool_forward_u16_ids_above_32767(tt, H):
    V = 65535
    gen = torch.Generator().manual_seed(H)
    table = torch.randn(V, H, generator=gen)
    table_dev = table.to(DEV)
    B, L = 24, 129
    ids = torch.randint(32768, V, (B, L), generator=gen)
    ids[0, :4] = torch.tensor([0, V - 1, 32768, 32767])
    mask = (torch.rand(B, L, generator=gen) < 0.8).long()
    mask[0, :4] = 1
    mask[1] = 0
    got = tt.ops.pool_forward(table_dev, as_dtype(ids, torch.int16), mask)
    assert int(got[3].item()) == 0
    wx, wn = check_forward(("u16", H), got, table, as_dtype(ids, torch.int16).long() & 0xFFFF, mask)
    print(f"pool_shapes forward u16 ids H={H}: xhat {wx:.2e} nrm {wn:.2e}")
    for idt in (torch.uint16, torch.int32, torch.int64):
        other = tt.ops.pool_forward(table_dev, as_dtype(ids, idt), mask.to(torch.uint8))
        assert all(same_bits(a, b) for a, b in zip(got[:3], other[:3])), idt


def test_pool_forward_70000_row_table_i32_ids(tt):
    V, H, B, L = 70000, 384, 40, 200
    gen = torch.Generator().manual_seed(70000)
    table = torch.randn(V, H, generator=gen)
    table_dev = table.to(DEV)
    ids = torch.randint(0, V, (B, L), generator=gen)
    ids[:, 0] = V - 1
    ids[:, 1] = 65536
    mask = (torch.rand(B, L, generator=gen) < 0.6).long()
    mask[:, :2] = 1
    got = tt.ops.pool_forward(table_dev, ids.to(torch.int32), mask.to(torch.int32))
    assert int(got[3].item()) == 0
    wx, wn = check_forward("V=70000", got, table, ids, mask)
    print(f"pool_shapes forward V=70000: xhat {wx:.2e} nrm {wn:.2e}")
    other = tt.ops.pool_forward(table_dev, ids, mask)
    assert all(same_bits(a, b) for a, b in zip(got[:3], other[:3]))


@pytest.mark.parametrize("H", [384, 768])
def test_pool_forward_weighted_masks(tt, H):
    """Mask values are weights and the count is their sum (model.py:71)."""
    table, table_dev = table_a(V_A, H, torch.float32)
    gen = torch.Generator().manual_seed(23 + H)
    B, L = 20, 512
    ids = torch.randint(0, V_A, (B, L), generator=gen)
    mask = torch.randint(0, 4, (B, L), generator=gen)
    mask[0] = 0
    mask[1] = 3
    mask[2, :] = 0
    mask[2, -1] = 2
    got = tt.ops.pool_forward(table_dev, ids, mask)
    wx, wn = check_forward(("weighted", H), got, table, ids, mask)
    print(f"pool_shapes forward weighted H={H}: xhat {wx:.2e} nrm {wn:.2e}")
    assert float(got[1][1]) == 3.0 * L and float(got[1][2]) == 2.0
    for mdt in (torch.int32, torch.uint8):
        other = tt.ops.pool_forward(table_dev, ids.to(torch.int32), mask.to(mdt))
        assert all(same_bits(a, b) for a, b in zip(got[:3], other[:3])), mdt


def test_pool_forward_rejects_unsupported_shapes(tt):
    N = tt._native
    table = torch.randn(100, 384, device=DEV)
    ids = torch.zeros(2, 513, dtype=torch.int64)
    with pytest.raises(N.NativeError, match="L=513"):
        tt.ops.pool_forward(table, ids, torch.ones_like(ids))
    with pytest.raises(N.NativeError, match="hidden size 192"):
        tt.ops.pool_forward(torch.randn(100, 192, device=DEV), ids[:, :8], torch.ones(2, 8, dtype=torch.int64))
    x = tt.ops.pool_forward(table, ids[:, :512], torch.ones(2, 512, dtype=torch.int64))[0]  # still usable
    torch.cuda.synchronize()
    assert x.shape == (2, 384)


# ---------------------------------------------------------------------------------------------------------------------
# B. the gather inside the step
# ---------------------------------------------------------------------------------------------------------------------
P_STEP = 64
V_B = 4099


def step_tokens(B, Lq, Ld, V, seed, ids_dtype=torch.int32):
    """q, p, n token sets (ids, uint8 mask): random lengths and scattered holes, some all-masked rows, one full row."""
    gen = torch.Generator().manual_seed(seed)
    out = []
    for L, off in ((Lq, 0), (Ld, 1), (Ld, 2)):
        ids = torch.randint(0, V, (B, L), generator=gen)
        lens = torch.randint(0, L + 1, (B, 1), generator=gen)
        mask = (torch.arange(L)[None] < lens) & (torch.rand(B, L, generator=gen) < 0.85)
        mask[off::7] = False
        mask[min(B - 1, 2 + off)] = True
        out += [ids.to(ids_dtype), mask.to(torch.uint8)]
    return tuple(out)


def make_step(tt, B, Lq, Ld, H, V, precision, tables, tokens, train_table=False, chain=0, seed=0):
    gen = torch.Generator().manual_seed(seed + 5)
    params = []
    for _ in range(2):
        for fan_in, shape in ((H, (P_STEP, H)), (H, (P_STEP,)), (P_STEP, (P_STEP, P_STEP)), (P_STEP, (P_STEP,))):
            params.append(((torch.rand(shape, generator=gen) * 2 - 1) * fan_in ** -0.5).to(DEV))
    grads = [torch.zeros_like(p) for p in params]
    so = tt.ops.TripletStep(B, Lq, Ld, H, P_STEP, V, precision, DEV, train_table=train_table)
    so.set_chain(chain)
    tg = tuple(torch.zeros(t.shape, dtype=torch.float32, device=DEV) for t in tables) if train_table else None
    dev_tokens = tuple(t.to(DEV) for t in tokens)
    so.bind(dev_tokens, tables, params, grads, 0.3, 1.0 / B, 1.0, tg)
    so._test_keep = (params, grads, dev_tokens)
    return so, tg


def host_terms(x):
    """hi = bf16_rn(x), lo = bf16_rn(x - hi), lo2 = bf16_rn((x - hi) - lo), in float32 (both subtractions are exact)."""
    hi = x.to(torch.bfloat16)
    r = x - hi.float()
    lo = r.to(torch.bfloat16)
    lo2 = (r - lo.float()).to(torch.bfloat16)
    return hi, lo, lo2


def check_terms(so, precision, rows, H, tag):
    v = so._views()
    xhat = v["xhat"].detach().cpu()
    hi, lo, lo2 = host_terms(xhat)
    assert same_bits(so.internal("x_hi", rows, H).cpu(), hi), (tag, "x_hi")
    assert same_bits(so.internal("x_lo", rows, H).cpu(), lo), (tag, "x_lo")
    if precision == "bf16x3":
        assert same_bits(so.internal("x_lo2", rows, H).cpu(), lo2), (tag, "x_lo2")


STEP_MODES = [("fp32", 384, 0), ("fp32", 768, 0), ("bf16x3", 384, 1), ("bf16x3", 384, 0), ("bf16", 384, 1),
              ("bf16", 384, 0)]


@pytest.mark.parametrize("B", [1, 3, 300])
@pytest.mark.parametrize("Lq,Ld", [(8, 24), (300, 32), (64, 64)])
@pytest.mark.parametrize("precision,H,phases", STEP_MODES,
                         ids=[f"{p}-H{h}-{'gather' if ph else 'step'}" for p, h, ph in STEP_MODES])
def test_step_gather_equals_pool_forward(tt, precision, H, phases, Lq, Ld, B):
    table_q, tq_dev = table_a(V_B, H, torch.float32)
    table_d, td_dev = table_a(V_B + 2, H, torch.float32)  # (a second table; its last two rows are never named)
    tokens = step_tokens(B, Lq, Ld, V_B, seed=B * 7 + Lq)
    so, _ = make_step(tt, B, Lq, Ld, H, V_B, precision, (tq_dev, td_dev), tokens)
    so.run(phases=phases)
    torch.cuda.synchronize()
    assert int(so.err.item()) == 0
    v = so._views()
    tag = (precision, H, phases, Lq, Ld, B)
    for k, table in enumerate((tq_dev, td_dev, td_dev)):
        want = tt.ops.pool_forward(table, tokens[2 * k], tokens[2 * k + 1])
        rs = slice(k * B, (k + 1) * B)
        assert same_bits(v["xhat"][rs], want[0]), (tag, "xhat", "qpn"[k])
        assert same_bits(v["cnt"][rs, 0], want[1]), (tag, "cnt", "qpn"[k])
        assert same_bits(v["nrm"][rs, 0], want[2]), (tag, "nrm", "qpn"[k])
    if precision != "fp32":
        check_terms(so, precision, 3 * B, H, tag)


def neg_index(kind, B, gen):
    if kind == "one":
        return torch.full((B,), 5, dtype=torch.int32)
    # positive 0 named by no negative, 1 once, 2 32 times and 3 33 times (around kMatchCap = 32), the rest at random
    idx = torch.cat([torch.tensor([1]), torch.full((32,), 2), torch.full((33,), 3),
                     torch.randint(4, B, (B - 66,), generator=gen)])
    return idx[torch.randperm(B, generator=gen)].to(torch.int32)


@pytest.mark.parametrize("kind", ["caps", "one"])
@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
def test_step_in_batch_negative_rows_are_bit_copies(tt, precision, kind):
    B, Lq, Ld, H = 300, 8, 24, 384
    table_q, tq_dev = table_a(V_B, H, torch.float32)
    table_d, td_dev = table_a(V_B + 2, H, torch.float32)
    tokens = step_tokens(B, Lq, Ld, V_B, seed=11)
    so, _ = make_step(tt, B, Lq, Ld, H, V_B, precision, (tq_dev, td_dev), tokens)
    idx = neg_index(kind, B, torch.Generator().manual_seed(3))
    so.set_neg_index(0, idx.to(DEV))
    so.run(phases=1)
    torch.cuda.synchronize()
    assert int(so.err.item()) == 0
    v = so._views()
    src = B + idx.long()
    for name in ("xhat", "cnt", "nrm"):
        t = v[name].detach().cpu()
        assert same_bits(t[2 * B:], t[src]), (kind, name)
    want = tt.ops.pool_forward(td_dev, tokens[2], tokens[3])
    assert same_bits(v["xhat"][B: 2 * B], want[0])
    if precision != "fp32":
        check_terms(so, precision, 3 * B, H, kind)


# ---------------------------------------------------------------------------------------------------------------------
# C. table gradient against float64 autograd
# ---------------------------------------------------------------------------------------------------------------------
def grad64(table, ids, mask, dxhat):
    """float64 autograd through embedding, masked mean and F.normalize, on the touched rows only.  Returns (touched
    ids, d64 [T,H], scale [T]: || sum_t |w_t| |g64_seq(t)| ||_inf)."""
    w = mask.double()
    seq, pos = torch.nonzero(w != 0, as_tuple=True)
    tok = ids[seq, pos]
    uniq, inv = torch.unique(tok, return_inverse=True)
    t = table[uniq].double().requires_grad_(True)
    B, H = ids.shape[0], table.shape[1]
    wt = w[seq, pos][:, None]
    s = torch.zeros(B, H, dtype=torch.float64).index_add(0, seq, t[inv] * wt)
    s.retain_grad()
    m = s / w.sum(1).clamp_min(1e-9)[:, None]
    x = torch.nn.functional.normalize(m, p=2, dim=1, eps=1e-12)
    (x * dxhat.double()).sum().backward()
    g64 = s.grad
    scale = torch.zeros(len(uniq), H, dtype=torch.float64).index_add_(0, inv, wt.abs() * g64[seq].abs())
    return uniq, t.grad, scale.amax(1)


def check_table_grad(tag, dtable_dev, table, ids, mask, dxhat):
    uniq, d64, scale = grad64(table, ids, mask, dxhat)
    V = dtable_dev.shape[0]
    touched = torch.zeros(V, dtype=torch.bool, device=DEV)
    touched[uniq.to(DEV)] = True
    if bool((~touched).any()):
        assert float(dtable_dev[~touched].abs().max()) == 0.0, (tag, "untouched rows")
    d = dtable_dev[uniq.to(DEV)].cpu().double()
    e = (d - d64).abs().amax(1) / scale.clamp_min(1e-300)
    e = torch.where(scale > 0, e, (d - d64).abs().amax(1))
    worst = float(e.max())
    assert worst <= TAU_B, (tag, "row", int(uniq[e.argmax()]), worst)
    return worst


def run_pool_grad(tt, table_dev, ids, mask, dxhat_dev):
    t = table_dev.clone().requires_grad_(True)
    x = tt.ops.pool(t, ids, mask)
    (x * dxhat_dev).sum().backward()
    return t.grad


RUNS = (1, 255, 256, 257, 2047, 2048, 2049, 6145)
TINY_ID = 9  # a table row of norm ~1e-14: its sequences normalise by the clamped 1e-12 (the gradient skips the norm)


def grad_table(V, H, gen):
    t = torch.randn(V, H, generator=gen)
    t[ZERO_ID] = 0
    t[TINY_ID] *= 1e-15
    return t


def run_tokens(V, gen, L=64, n_light=3000, weighted=True):
    """[B, L] ids / i64 mask: ids with exactly RUNS[k] unmasked occurrences (0 and V - 1 among the heavy ones), an id with
    257 occurrences of which one is masked, light ids, masked padding, an all-masked row, and rows of the all-zero and the
    tiny table row (both below the normalisation clamp)."""
    special = [0, V - 1] + [int(i) for i in torch.randperm(V - 20, generator=gen)[:len(RUNS) - 1] + 10]
    heavy = dict(zip(special[2:8] + [V - 1, 0], RUNS))  # ..., V - 1: 2049, 0: 6145
    masked_heavy = special[8]
    toks = [(i, 1) for i, n in heavy.items() for _ in range(n)]
    toks += [(masked_heavy, 1)] * 256 + [(masked_heavy, 0)]
    taken = set(heavy) | {masked_heavy, ZERO_ID, TINY_ID}
    light = torch.tensor([i for i in torch.randint(0, V, (n_light * 2,), generator=gen).tolist() if i not in taken][:n_light])
    wl = torch.randint(1, 4, (len(light),), generator=gen) if weighted else torch.ones(len(light), dtype=torch.int64)
    toks += list(zip(light.tolist(), wl.tolist()))
    n = len(toks)
    B = (n + L - 1) // L + 8
    ids = torch.randint(0, V, (B * L,), generator=gen)
    mask = torch.zeros(B * L, dtype=torch.int64)
    slots = torch.randperm((B - 2) * L, generator=gen)[:n] + 2 * L
    t = torch.tensor(toks)
    ids[slots], mask[slots] = t[:, 0], t[:, 1]
    ids, mask = ids.view(B, L), mask.view(B, L)
    ids[0], mask[0] = ZERO_ID, 1  # zero-norm sequence: clamped normalisation
    mask[1] = 0  # all-masked sequence
    ids[2], mask[2] = TINY_ID, 1  # norm ~1e-14: x / 1e-12
    return ids, mask


C_CASES = [(384, 200), (384, 255), (384, 256), (384, 65535), (384, 65536), (128, 256), (256, 65535), (768, 256),
           (768, 65536)]


@pytest.mark.parametrize("H,V", C_CASES)
def test_table_grad_runs_vs_float64(tt, H, V):
    gen = torch.Generator().manual_seed(V + H)
    table = grad_table(V, H, gen)
    table_dev = table.to(DEV)
    ids, mask = run_tokens(V, gen)
    dxhat = torch.randn(ids.shape[0], H, generator=gen)
    d1 = run_pool_grad(tt, table_dev, ids, mask, dxhat.to(DEV))
    d2 = run_pool_grad(tt, table_dev, ids, mask, dxhat.to(DEV))
    assert same_bits(d1, d2), "two runs differ"
    worst = check_table_grad((H, V), d1, table, ids, mask, dxhat)
    print(f"pool_shapes table grad H={H} V={V} N={ids.numel()}: {worst:.2e}")


@pytest.mark.parametrize("B,L", [(33, 31), (32, 32), (25, 41), (17, 241)], ids=["N1023", "N1024", "N1025", "N4097"])
def test_table_grad_token_counts_vs_float64(tt, B, L):
    V, H = 65535, 128
    gen = torch.Generator().manual_seed(B * L)
    table = torch.randn(V, H, generator=gen)
    table_dev = table.to(DEV)
    ids = torch.randint(0, 300, (B, L), generator=gen)
    ids[:, ::3] = V - 1  # a heavy row at N = 4097
    mask = (torch.rand(B, L, generator=gen) < 0.9).long()
    mask[:, -1] = 1
    dxhat = torch.randn(B, H, generator=gen)
    d1 = run_pool_grad(tt, table_dev, ids, mask, dxhat.to(DEV))
    d2 = run_pool_grad(tt, table_dev, ids, mask, dxhat.to(DEV))
    assert same_bits(d1, d2), "two runs differ"
    worst = check_table_grad((B, L), d1, table, ids, mask, dxhat)
    print(f"pool_shapes table grad N={B * L}: {worst:.2e}")


# ---------------------------------------------------------------------------------------------------------------------
# D. exact replay of the reduction order
# ---------------------------------------------------------------------------------------------------------------------
def replay(G, occ_ids, occ_rows, V):
    """dtable [V, H] float32 as the backward promises to sum it, from G [rows, H] float32 (CPU) and the unmasked
    occurrences (ids, g rows; binary mask) in ascending global position: per id, occurrences in position order; a run of
    <= 256 is one sequential sum from +0; a longer run is cut into 2048-entry chunks of 8 slices of 256, each slice a
    sequential sum from +0, the slice sums of a chunk added in order from +0, the chunk sums added in order from +0.
    Vectorised over "the j-th entry of every run / slice" (at most 256 steps)."""
    H = G.shape[1]
    out = torch.zeros(V, H, dtype=torch.float32)
    if len(occ_ids) == 0:
        return out
    order = np.argsort(occ_ids, kind="stable")
    ids_s, rows_s = occ_ids[order], torch.from_numpy(occ_rows[order].astype(np.int64))
    uniq, start, count = np.unique(ids_s, return_index=True, return_counts=True)
    heavy = count > HEAVY
    # units: light runs, then the 256-entry slices of heavy runs
    u_start, u_len, u_owner = [start[~heavy]], [count[~heavy]], [np.arange(len(uniq))[~heavy]]
    for r in np.nonzero(heavy)[0]:
        k = np.arange(0, count[r], SLICE)
        u_start.append(start[r] + k)
        u_len.append(np.minimum(SLICE, count[r] - k))
        u_owner.append(np.full(len(k), r))
    u_start, u_len, u_owner = np.concatenate(u_start), np.concatenate(u_len), np.concatenate(u_owner)
    by_len = np.argsort(-u_len, kind="stable")  # active units form a prefix at every step
    u_start_s, u_len_s = u_start[by_len], u_len[by_len]
    sums = torch.zeros(len(u_start), H, dtype=torch.float32)
    for j in range(int(u_len_s[0])):
        k = int(np.searchsorted(-u_len_s, -j, side="left"))  # units with length > j
        sums[:k] += G[rows_s[torch.from_numpy(u_start_s[:k] + j)]]
    unit_sum = torch.empty_like(sums)
    unit_sum[torch.from_numpy(by_len)] = sums
    n_light = int((~heavy).sum())
    out[torch.from_numpy(uniq[~heavy].astype(np.int64))] = unit_sum[:n_light]
    pos = n_light
    for r in np.nonzero(heavy)[0]:
        n_sl = (int(count[r]) + SLICE - 1) // SLICE
        sl = unit_sum[pos: pos + n_sl]
        pos += n_sl
        row = torch.zeros(H, dtype=torch.float32)
        for c in range(0, n_sl, CHUNK // SLICE):
            chunk = torch.zeros(H, dtype=torch.float32)
            for w in range(CHUNK // SLICE):
                chunk = chunk + (sl[c + w] if c + w < n_sl else torch.zeros(H, dtype=torch.float32))
            row = row + chunk
        out[int(uniq[r])] = row
    return out


def occurrences(segs):
    """segs = [(ids [B,L], mask [B,L], row0)] in global position order -> unmasked (ids, g rows) as numpy."""
    ids_all, rows_all = [], []
    for ids, mask, row0 in segs:
        B, L = ids.shape
        keep = mask.reshape(-1).numpy() != 0
        ids_all.append(ids.reshape(-1).long().numpy()[keep])
        rows_all.append((np.arange(B * L) // L + row0)[keep])
    return np.concatenate(ids_all), np.concatenate(rows_all)


def check_g(v, tag):
    """g = (dxhat - xhat * k) / (max(nrm, 1e-12) * max(cnt, 1e-9)), k = dxhat . xhat unless nrm < 1e-12 (then 0), from
    the device's own fp32 inputs; both clamp branches must occur."""
    d, x = v["dxhat"].detach().cpu().double(), v["xhat"].detach().cpu().double()
    n, c = v["nrm"].detach().cpu().double()[:, 0], v["cnt"].detach().cpu().double()[:, 0]
    clamped = n < 1e-12
    k = torch.where(clamped, 0.0, (d * x).sum(1))
    inv = 1.0 / (n.clamp_min(1e-12) * c.clamp_min(1e-9))
    g64 = (d - x * k[:, None]) * inv[:, None]
    scale = ((d.abs() + x.abs() * k.abs()[:, None]) * inv[:, None]).amax(1)
    e = (v["g"].detach().cpu().double() - g64).abs().amax(1) / scale.clamp_min(1e-300)
    e = torch.where(scale > 0, e, 0.0)
    live = c > 0
    assert bool((clamped & live).any()) and bool((~clamped & live).any()), (tag, "both clamp branches")
    assert float(e.max()) <= TAU_G, (tag, "g row", int(e.argmax()), float(e.max()))
    return float(e.max())


def replay_tokens(B, Lq, Ld, V, seed):
    gen = torch.Generator().manual_seed(seed)
    q_ids = torch.randint(0, V, (B, Lq), generator=gen)
    p_ids = torch.randint(0, V, (B, Ld), generator=gen)
    n_ids = torch.randint(0, V, (B, Ld), generator=gen)
    q_ids[:, :2] = 102             # 2B occurrences in q: heavy
    p_ids[:, 5] = n_ids[:, 5] = 101  # one per document sequence: 2B entries, one partial chunk across the p | n boundary
    p_ids[:, 8:16] = n_ids[:, 8:16] = 1996  # 16B > 2049 entries: several chunks
    p_ids[:, 20] = V - 1
    n_ids[:, 21] = 0
    if V > 65536:
        q_ids[:, 3] = 65536
        n_ids[:, 22] = 65536
    masks = []
    for ids, L in ((q_ids, Lq), (p_ids, Ld), (n_ids, Ld)):
        lens = torch.randint(1, L + 1, (B, 1), generator=gen)
        m = (torch.arange(L)[None] < lens) & (torch.rand(B, L, generator=gen) < 0.9)
        m[:, 5] = True
        m[3::97] = False  # all-masked sequences
        masks.append(m.to(torch.uint8))
    q_ids[1], masks[0][1] = ZERO_ID, 1  # zero-norm sequences: the clamped branch of g
    p_ids[2], masks[1][2] = ZERO_ID, 1
    n_ids[4], masks[2][4] = TINY_ID, 1
    return tuple(t.to(torch.int32) if k % 2 == 0 else t for k, t in
                 enumerate((q_ids, masks[0], p_ids, masks[1], n_ids, masks[2])))


D_CASES = [(300, 32, 256, 30522), (2100, 32, 256, 30522), (300, 32, 256, 70000)]


@pytest.mark.parametrize("precision", ["fp32", "bf16x3"])
@pytest.mark.parametrize("B,Lq,Ld,V", D_CASES, ids=["B300", "B2100", "V70000"])
def test_step_table_grad_is_the_promised_sum(tt, B, Lq, Ld, V, precision):
    H = 384
    gen = torch.Generator().manual_seed(V + 1)
    tables = []
    for _ in range(2):
        tables.append(grad_table(V, H, gen).to(DEV))
    tokens = replay_tokens(B, Lq, Ld, V, seed=B)
    so, (dq, dd) = make_step(tt, B, Lq, Ld, H, V, precision, tuple(tables), tokens, train_table=True,
                             chain=1 if precision != "fp32" else 0)
    so.run()
    torch.cuda.synchronize()
    assert int(so.err.item()) == 0
    v = so._views()
    tag = (B, V, precision)
    eg = check_g(v, tag)
    G = v["g"].detach().cpu().clone()
    q_occ = occurrences([(tokens[0], tokens[1], 0)])
    d_occ = occurrences([(tokens[2], tokens[3], B), (tokens[4], tokens[5], 2 * B)])
    for name, occ, got in (("dtable_q", q_occ, dq), ("dtable_d", d_occ, dd)):
        want = replay(G, occ[0], occ[1], V)
        same = bits(got) == bits(want)
        bad = (~same).any(1).nonzero()[:, 0]
        assert len(bad) == 0, (tag, name, "rows not bit-identical", bad[:8].tolist(), len(bad))
    print(f"pool_shapes replay B={B} V={V} {precision}: bit-identical, g {eg:.2e}")


@pytest.mark.parametrize("V", [255, 3001])
def test_pool_bwd_accumulate_adds_the_promised_sum(tt, V):
    """accumulate = 1 of the tt_pool_bwd C ABI: dtable = promised sum + previous contents (light rows acc + old, heavy rows
    (sum of chunks) + old, untouched rows old); accumulate = 0: the promised sum.  V = 255 sorts in one radix pass, where
    an unstable pass would only reorder the entries of each id; with L = 8 every 32 consecutive tokens span 4 sequences,
    so such a reordering changes the sums."""
    N = tt._native
    lib = N.load()
    H, B, L = 256, 1280, 8
    gen = torch.Generator().manual_seed(V)
    table = torch.randn(V, H, generator=gen).to(DEV)
    ids = torch.randint(0, V, (B, L), generator=gen)
    ids[:, 0] = 17       # ~1150 unmasked entries: one heavy chunk
    ids[:, 1:3] = 18     # ~2300: two chunks
    ids[:, 7] = V - 1
    mask = (torch.rand(B, L, generator=gen) < 0.9).long()
    mask[0] = 0
    ids_d, mask_d = ids.to(torch.int32).to(DEV), mask.to(DEV)
    xhat, cnt, nrm = tt.ops.pool_forward(table, ids_d, mask_d)[:3]
    dxhat = torch.randn(B, H, generator=gen).to(DEV)
    R = torch.randn(V, H, generator=gen)
    ws_bytes = lib.tt_pool_bwd_ws_bytes(B, L, V, H)
    ws = N.workspace(ws_bytes, DEV)
    assert ws.data_ptr() % 256 == 0
    occ = occurrences([(ids, mask, 0)])
    for acc in (0, 1):
        dtable = R.to(DEV) if acc else torch.full((V, H), float("nan"), device=DEV)
        N.check(lib.tt_pool_bwd(N.ptr(dxhat), N.ptr(xhat), N.ptr(cnt), N.ptr(nrm), N.ptr(ids_d), N.dtype_code(ids_d),
                                N.ptr(mask_d), N.dtype_code(mask_d), B, L, V, H, N.ptr(dtable), acc, N.ptr(ws), ws_bytes,
                                N.stream()), "tt_pool_bwd")
        torch.cuda.synchronize()
        G = ws[: B * H * 4].view(torch.float32).view(B, H).cpu()  # g is the first carve of the workspace
        want = replay(G, occ[0], occ[1], V)
        if acc:
            want = want + R
        assert same_bits(dtable, want), ("accumulate", acc)
