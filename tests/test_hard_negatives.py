"""Hard negatives mined with the exact corpus scan (data.HardNegativeMiner, tt_mine_negatives,
tt_assemble_*_mined, run_training(hard_negatives=...)).

The mining filter and the mined draw are checked exactly against numpy replays; the miner's table against a float64
top-k of the device's own normalised projections, ids compared wherever the neighbouring float64 gaps exceed 2 tau
(tau as in test_scan_shapes.py); the feeder and trainer against the in-batch path they extend.  Whether mined
negatives improve NDCG is not checked: the synthetic corpus is random tokens.
"""
import copy
import ctypes

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu
TAU = 1.5e-6
M64 = (1 << 64) - 1


@pytest.fixture(scope="module")
def tt():
    import two_towers_overlords_b200 as pkg
    from two_towers_overlords_b200 import _native, data, ops, retrieval, training  # noqa: F401

    pkg.data, pkg.ops, pkg.training, pkg.retrieval, pkg.N = data, ops, training, retrieval, _native
    return pkg


# ---------------------------------------------------------------------------------------------------------------------
# numpy references
# ---------------------------------------------------------------------------------------------------------------------
def splitmix64(x):
    x = (x + 0x9E3779B97F4A7C15) & M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & M64
    return x ^ (x >> 31)


def mined_pick(seed, i, count, ratio):
    """The documented draw of tt_assemble_*_mined: the table column item i takes, or -1 for its in-batch draw."""
    h0 = splitmix64((seed ^ 0x6A09E667F3BCC909 ^ (i * 0x9E6C63D0676A9A99)) & M64)
    h1 = splitmix64(h0)
    if count <= 0 or not float(h1 >> 40) < float(np.float32(ratio)) * 2.0 ** 24:
        return -1
    return (splitmix64(h1) >> 32) % count


def np_mine(top_id, off, ids, skip, depth):
    Q = top_id.shape[0]
    table = np.full((Q, depth), -1, dtype=np.int32)
    count = np.zeros(Q, dtype=np.int32)
    for r in range(Q):
        excl = set(ids[off[r]: off[r + 1]].tolist())
        surv = [int(d) for d in top_id[r] if d >= 0 and int(d) not in excl][skip: skip + depth]
        table[r, : len(surv)] = surv
        count[r] = len(surv)
    return table, count


def np_exclusions(pq, pd, qid, n_rows):
    qids_of = [set() for _ in range(n_rows)]
    for r, q in zip(pq, qid):
        qids_of[r].add(q)
    docs_of = {}
    for d, q in zip(pd, qid):
        docs_of.setdefault(q, set()).add(d)
    return [sorted(set().union(*[docs_of[q] for q in qs])) if qs else [] for qs in qids_of]


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_splitmix_and_draw_formula_are_pinned():
    # SplitMix64 seeded with 0: the first output of the published generator
    assert splitmix64(0) == 0xE220A8397B1DCDAF
    # ratio 0 and empty rows never draw; ratio 1 always does, uniformly over the row
    assert all(mined_pick(s, i, 8, 0.0) == -1 for s in (0, 7) for i in range(64))
    assert all(mined_pick(s, i, 0, 1.0) == -1 for s in (0, 7) for i in range(64))
    picks = [mined_pick(12345, i, 5, 1.0) for i in range(5000)]
    assert min(picks) == 0 and max(picks) == 4 and abs(np.bincount(picks).min() - 1000) < 150
    # hand-worked: seed 0, item 0 -> h0 = splitmix64(0x6A09E667F3BCC909); hard iff (h1 >> 40) < ratio * 2^24, so a
    # ratio of exactly (h1 >> 40) / 2^24 (a 24-bit fraction: exact in fp32) is the first one that is NOT hard
    h1 = splitmix64(splitmix64(0x6A09E667F3BCC909))
    u = h1 >> 40
    assert mined_pick(0, 0, 7, 1.0) == (splitmix64(h1) >> 32) % 7
    assert mined_pick(0, 0, 7, u / 2 ** 24) == -1
    assert mined_pick(0, 0, 7, float(np.nextafter(np.float32(u / 2 ** 24), np.float32(2)))) >= 0
    assert [mined_pick(0x5EED, i, 8, 0.5) for i in range(12)] == [4, 4, 7, 5, -1, 1, -1, 2, 0, 1, 1, -1]
    frac = np.mean([mined_pick(99, i, 3, 0.3) >= 0 for i in range(20000)])
    assert abs(frac - 0.3) < 0.015


def test_exclusion_csr_shared_passages_and_two_query_ids(tt):
    # row 0 is named under query ids 10 and 12; passage 5 is a positive of ids 10 and 11; row 3 has no pair
    pq = np.array([0, 0, 1, 2, 2, 0, 1])
    pd = np.array([5, 6, 5, 7, 1, 9, 4])
    qid = np.array([10, 10, 11, 10, 12, 12, 11])
    off, ids = tt.data.exclusion_csr(pq, pd, qid, 4)
    assert off.dtype == np.int64 and ids.dtype == np.int32
    got = [ids[off[r]: off[r + 1]].tolist() for r in range(4)]
    assert got == [[1, 5, 6, 7, 9], [4, 5], [1, 5, 6, 7, 9], []]
    assert got == np_exclusions(pq, pd, qid, 4)
    rng = np.random.default_rng(0)
    pq, pd, qid = rng.integers(0, 50, 400), rng.integers(0, 300, 400), rng.integers(0, 70, 400) * 1000003
    off, ids = tt.data.exclusion_csr(pq, pd, qid, 60)
    want = np_exclusions(pq, pd, qid, 60)
    assert [ids[off[r]: off[r + 1]].tolist() for r in range(60)] == want
    assert all(np.all(np.diff(ids[off[r]: off[r + 1]]) > 0) for r in range(60))


def test_miner_config_validation(tt):
    ok = tt.data.HardNegativeMiner.check_config
    assert ok(8, 0, 0.5, 32) == (8, 0, 0.5, 32) and ok(1, 31, 1.0, 32) == (1, 31, 1.0, 32)
    for bad in [(8, 0, 0.5, 33), (8, 0, 0.5, 0), (0, 0, 0.5, 32), (8, -1, 0.5, 32), (9, 24, 0.5, 32), (8, 0, 1.01, 32),
                (8, 0, -0.1, 32), (4, 0, 0.5, 3)]:
        with pytest.raises(ValueError):
            ok(*bad)
    cfg = tt.training.hard_negative_config
    assert cfg(0) is None and cfg(8) == {"miner": {"depth": 8}, "warmup_epochs": 1}
    assert cfg({"depth": 4, "ratio": 1.0, "warmup_epochs": 0}) == {"miner": {"depth": 4, "ratio": 1.0},
                                                                    "warmup_epochs": 0}
    for bad in (-1, {"depth": 40}, {"k_scan": 64}, {"skip": 30}, {"ratio": 2.0}, {"colour": 1}, "8", True):
        with pytest.raises(ValueError):
            cfg(bad)


def test_hard_negative_env_parsing(tt, monkeypatch):
    cfg = tt.training.hard_negative_config
    monkeypatch.delenv("TT_HARD_NEGATIVES", raising=False)
    assert cfg(None) is None
    monkeypatch.setenv("TT_HARD_NEGATIVES", "0")
    assert cfg(None) is None
    monkeypatch.setenv("TT_HARD_NEGATIVES", "8")
    assert cfg(None) == {"miner": {"depth": 8}, "warmup_epochs": 1}
    monkeypatch.setenv("TT_HARD_NEGATIVES", "yes")
    with pytest.raises(ValueError, match="TT_HARD_NEGATIVES"):
        cfg(None)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the mining filter
# ---------------------------------------------------------------------------------------------------------------------
def _lists(Q, k, n_docs, rng):
    """Random scan lists (-1 tails on some rows) and exclusion lists that hit the first rank,
    the last rank, every rank, no rank, and random ranks."""
    top = np.full((Q, k), -1, dtype=np.int64)
    excl = []
    for r in range(Q):
        m = k if r % 5 else int(rng.integers(0, k + 1))
        row = rng.integers(0, n_docs, m)
        top[r, :m] = row
        kind = r % 6
        if kind == 0 and m:
            e = [row[0]]
        elif kind == 1 and m:
            e = [row[m - 1]]
        elif kind == 2:
            e = list(row)  # every rank excluded: count 0
        elif kind == 3:
            e = []
        else:
            e = list(row[rng.random(m) < 0.3])
        e = e + list(rng.integers(0, n_docs, int(rng.integers(0, 4))))  # positives that were not retrieved
        excl.append(sorted(set(int(x) for x in e)))
    off = np.concatenate([[0], np.cumsum([len(e) for e in excl])]).astype(np.int64)
    ids = np.array([x for e in excl for x in e], dtype=np.int32)
    return top, off, ids


def _dev(*arrs):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrs]


@gpu
@pytest.mark.parametrize("Q", [1, 127, 128, 129, 82463])
def test_mine_negatives_matches_numpy(tt, Q):
    rng = np.random.default_rng(Q)
    for k, skip, depth in ((32, 0, 8), (32, 3, 16), (17, 2, 15), (1, 0, 1)):
        top, off, ids = _lists(Q, k, 700_000, rng)
        t_top, t_off, t_ids = _dev(top, off, ids)
        table, count = tt.ops.mine_negatives(t_top, t_off, t_ids, skip, depth)
        want_t, want_c = np_mine(top, off, ids, skip, depth)
        assert np.array_equal(count.cpu().numpy(), want_c), (k, skip, depth)
        assert np.array_equal(table.cpu().numpy(), want_t), (k, skip, depth)
        if Q >= 6:
            assert (want_c == 0).any() and (want_c == min(depth, k - skip)).any()


@gpu
def test_mine_negatives_every_skip_and_depth_at_k32(tt):
    rng = np.random.default_rng(7)
    top, off, ids = _lists(129, 32, 5000, rng)
    t_top, t_off, t_ids = _dev(top, off, ids)
    for skip in range(32):
        for depth in range(1, 33 - skip):
            t, c = tt.ops.mine_negatives(t_top, t_off, t_ids, skip, depth)
            want_t, want_c = np_mine(top, off, ids, skip, depth)
            assert np.array_equal(c.cpu().numpy(), want_c) and np.array_equal(t.cpu().numpy(), want_t), (skip, depth)


@gpu
def test_mine_negatives_refusals_leave_the_library_usable(tt):
    N = tt.N
    lib = N.load()
    top, off, ids = _lists(64, 32, 1000, np.random.default_rng(1))
    t_top, t_off, t_ids = _dev(top, off, ids)
    table = torch.zeros(64, 32, dtype=torch.int32, device="cuda")
    count = torch.zeros(64, dtype=torch.int32, device="cuda")
    p = [N.ptr(t) for t in (t_top, t_off, t_ids, table, count)]
    for k, skip, depth in ((32, 0, 0), (32, 30, 3), (33, 0, 8), (8, -1, 4), (4, 0, 5)):
        assert lib.tt_mine_negatives(p[0], 64, k, p[1], p[2], skip, depth, p[3], p[4], N.stream()) != 0
        assert "tt_mine_negatives" in N.last_error()
    assert lib.tt_mine_negatives(None, 64, 32, p[1], p[2], 0, 8, p[3], p[4], N.stream()) != 0
    assert "null" in N.last_error()
    assert lib.tt_mine_negatives(p[0], -1, 32, p[1], p[2], 0, 8, p[3], p[4], N.stream()) != 0
    t, c = tt.ops.mine_negatives(t_top, t_off, t_ids, 0, 8)
    want_t, want_c = np_mine(top, off, ids, 0, 8)
    assert np.array_equal(t.cpu().numpy(), want_t) and np.array_equal(c.cpu().numpy(), want_c)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the mined draw inside batch assembly
# ---------------------------------------------------------------------------------------------------------------------
def _pairs(n_pairs, n_q, n_d, n_qid, seed, dev):
    g = torch.Generator().manual_seed(seed)
    pq = torch.randint(0, n_q, (n_pairs,), generator=g, dtype=torch.int32)
    pd = torch.randint(0, n_d, (n_pairs,), generator=g, dtype=torch.int32)
    qid = torch.randint(0, n_qid, (n_pairs,), generator=g, dtype=torch.int32)
    return pq.to(dev), pd.to(dev), qid.to(dev)


def _ragged_bank(n, L, seed, dev, N):
    """Ragged token bank (some texts longer than L): the ids of text r start with r so rows can be read back."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, L + 6, n)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    flat = rng.integers(0, 60000, int(off[-1])).astype(np.int32)
    flat[off[:-1]] = np.arange(n)
    t_flat, t_off = torch.from_numpy(flat).to(dev), torch.from_numpy(off).to(dev)
    return flat, off, t_flat, t_off, N.TokenBankDesc(t_flat.data_ptr(), t_off.data_ptr(), N.TT_I32, 0)


N_Q, N_D, LQ, LD = 700, 4000, 3, 7


def _assemble(tt, banks, pq, pd, qid, order, Bg, lo, B, seed, mined):
    """Both entry points (tokens and rows), with the descriptor or without (mined None) -> dict of host arrays."""
    N, dev = tt.N, torch.device("cuda")
    lib = N.load()
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    toks = [torch.full((max(B, 1), L), -7, dtype=torch.int32, device=dev) for L in (LQ, LQ, LD, LD, LD, LD)]
    neg_t = torch.full((max(B, 1),), -9, dtype=torch.int32, device=dev)
    neg_r = torch.full((max(B, 1),), -9, dtype=torch.int32, device=dev)
    rows = torch.full((max(3 * B, 1),), -9, dtype=torch.int32, device=dev)
    targs = (ctypes.byref(banks[0][4]), ctypes.byref(banks[1][4]), N.ptr(pq), N.ptr(pd), N.ptr(qid), N.ptr(order), Bg,
             lo, B, seed, LQ, LD, *[N.ptr(t) for t in toks], N.TT_I32, N.TT_I32, N.ptr(neg_t), N.ptr(err))
    rargs = (N.ptr(pq), N.ptr(pd), N.ptr(qid), N.ptr(order), Bg, lo, B, seed, N.ptr(rows), N.ptr(neg_r), N.ptr(err))
    if mined is None:
        N.check(lib.tt_assemble_triplets(*targs, N.stream()), "tt_assemble_triplets")
        N.check(lib.tt_assemble_triplet_rows(*rargs, N.stream()), "tt_assemble_triplet_rows")
    else:
        N.check(lib.tt_assemble_triplets_mined(*targs, ctypes.byref(mined), N.stream()), "tt_assemble_triplets_mined")
        N.check(lib.tt_assemble_triplet_rows_mined(*rargs, ctypes.byref(mined), N.stream()),
                "tt_assemble_triplet_rows_mined")
    out = {f"t{j}": t[:B].cpu().numpy() for j, t in enumerate(toks)}
    out.update(neg_t=neg_t[:B].cpu().numpy(), neg_r=neg_r[:B].cpu().numpy(), rows=rows[: 3 * B].cpu().numpy(),
               err=int(err.item()))
    return out


def _table(rng, depth, zero=False):
    count = np.zeros(N_Q, dtype=np.int32) if zero else rng.integers(0, depth + 1, N_Q).astype(np.int32)
    table = np.full((N_Q, depth), -1, dtype=np.int32)
    for r in range(N_Q):
        table[r, : count[r]] = rng.choice(N_D, count[r], replace=False)
    return table, count


def _desc(tt, t_table, t_count, depth, ratio):
    return tt.N.MinedNegatives(t_table.data_ptr(), t_count.data_ptr(), depth, N_Q, N_D, ratio)


def _setup(tt, Bg, seed):
    N, dev = tt.N, torch.device("cuda")
    pq, pd, qid = _pairs(5000, N_Q, N_D, 300, seed & 0xFFFF, dev)
    banks = (_ragged_bank(N_Q, LQ, 1, dev, N), _ragged_bank(N_D, LD, 2, dev, N))
    order = torch.randperm(5000, generator=torch.Generator().manual_seed(seed & 0xFFF))[:Bg].to(torch.int32).to(dev)
    return pq, pd, qid, banks, order


@gpu
@pytest.mark.parametrize("Bg", [2, 257, 2048])
@pytest.mark.parametrize("seed", [0, 1, 0xDEADBEEF12345])
def test_mined_assembly_without_hard_items_is_todays_batch(tt, Bg, seed):
    pq, pd, qid, banks, order = _setup(tt, Bg, seed)
    rng = np.random.default_rng(seed & 0xFF)
    base = _assemble(tt, banks, pq, pd, qid, order, Bg, 0, Bg, seed, None)
    for ratio, zero in ((0.0, False), (1.0, True), (0.5, True)):
        table, count = _table(rng, 8, zero)
        t_table, t_count = _dev(table, count)
        got = _assemble(tt, banks, pq, pd, qid, order, Bg, 0, Bg, seed, _desc(tt, t_table, t_count, 8, ratio))
        for key in base:
            assert np.array_equal(got[key], base[key]), (ratio, zero, key)
    assert base["err"] == 0


@gpu
@pytest.mark.parametrize("Bg", [2, 257, 2048])
@pytest.mark.parametrize("ratio", [0.3, 1.0])
def test_mined_assembly_replays_the_documented_draw(tt, Bg, ratio):
    seed = 0xDEADBEEF12345
    pq, pd, qid, banks, order = _setup(tt, Bg, seed)
    rng = np.random.default_rng(Bg)
    depth = 8
    table, count = _table(rng, depth)
    t_table, t_count = _dev(table, count)
    desc = _desc(tt, t_table, t_count, depth, ratio)
    base = _assemble(tt, banks, pq, pd, qid, order, Bg, 0, Bg, seed, None)
    full = _assemble(tt, banks, pq, pd, qid, order, Bg, 0, Bg, seed, desc)
    assert full["err"] == 0
    o, pq_h, pd_h = order.cpu().numpy(), pq.cpu().numpy(), pd.cpu().numpy()
    d_flat, d_off = banks[1][0], banks[1][1]
    n_hard = 0
    for i in range(Bg):
        qrow = int(pq_h[o[i]])
        col = mined_pick(seed, i, int(count[qrow]), ratio)
        if col < 0:  # today's in-batch draw, unchanged
            assert full["neg_t"][i] == base["neg_t"][i] and full["neg_r"][i] == base["neg_r"][i]
            assert full["rows"][2 * Bg + i] == base["rows"][2 * Bg + i]
            assert np.array_equal(full["t4"][i], base["t4"][i]) and np.array_equal(full["t5"][i], base["t5"][i])
            continue
        n_hard += 1
        d = int(table[qrow, col])
        assert full["neg_t"][i] == -1 and full["neg_r"][i] == -1
        assert full["rows"][2 * Bg + i] == d
        # the hard item's tokens are the bank tokens of the chosen passage, truncated and zero padded
        toks = d_flat[d_off[d]: d_off[d + 1]][:LD]
        want = np.zeros(LD, dtype=np.int32)
        want[: len(toks)] = toks
        assert np.array_equal(full["t4"][i], want) and np.array_equal(full["t5"][i], (np.arange(LD) < len(toks)))
    for key in ("t0", "t1", "t2", "t3"):
        assert np.array_equal(full[key], base[key])
    assert np.array_equal(full["rows"][: 2 * Bg], base["rows"][: 2 * Bg])
    if Bg >= 257:  # counts are uniform in 0..8: 8 of 9 rows can draw
        assert n_hard > 0.7 * ratio * Bg
    # data-parallel slices concatenate to the one-rank batch
    for G in (1, 2, 8):
        parts = []
        for r in range(G):
            lo, hi = tt.retrieval.shard_bounds(Bg, G, r)
            if hi == lo:
                continue
            parts.append(_assemble(tt, banks, pq, pd, qid, order, Bg, lo, hi - lo, seed, desc))
        for key in ("t0", "t1", "t2", "t3", "t4", "t5", "neg_t", "neg_r"):
            assert np.array_equal(np.concatenate([p[key] for p in parts]), full[key]), (G, key)
        rows = np.concatenate([p["rows"].reshape(3, -1) for p in parts], axis=1)
        assert np.array_equal(rows, full["rows"].reshape(3, Bg)), G


@gpu
def test_bad_table_entry_or_row_sets_the_flag_and_falls_back(tt):
    Bg, seed = 257, 3
    pq, pd, qid, banks, order = _setup(tt, Bg, seed)
    base = _assemble(tt, banks, pq, pd, qid, order, Bg, 0, Bg, seed, None)
    for bad in (N_D, -5):
        table = np.full((N_Q, 4), bad, dtype=np.int32)
        count = np.full(N_Q, 4, dtype=np.int32)
        t_table, t_count = _dev(table, count)
        got = _assemble(tt, banks, pq, pd, qid, order, Bg, 0, Bg, seed, _desc(tt, t_table, t_count, 4, 1.0))
        assert got["err"] == 3
        assert np.array_equal(got["rows"], base["rows"]) and np.array_equal(got["neg_t"], base["neg_t"])
    # a table with fewer rows than the query bank: rows past it are out of range
    t_table, t_count = _dev(np.zeros((N_Q, 4), np.int32), np.full(N_Q, 4, np.int32))
    short = tt.N.MinedNegatives(t_table.data_ptr(), t_count.data_ptr(), 4, 5, N_D, 1.0)
    assert _assemble(tt, banks, pq, pd, qid, order, Bg, 0, Bg, seed, short)["err"] == 3
    # a bad descriptor is refused on the host, and the library stays usable
    lib, N = tt.N.load(), tt.N
    rows = torch.zeros(3 * Bg, dtype=torch.int32, device="cuda")
    for d in (tt.N.MinedNegatives(t_table.data_ptr(), t_count.data_ptr(), 4, N_Q, N_D, 1.5),
              tt.N.MinedNegatives(t_table.data_ptr(), t_count.data_ptr(), 0, N_Q, N_D, 0.5),
              tt.N.MinedNegatives(None, None, 4, N_Q, N_D, 0.5)):
        assert lib.tt_assemble_triplet_rows_mined(N.ptr(pq), N.ptr(pd), N.ptr(qid), N.ptr(order), Bg, 0, Bg, seed,
                                                  N.ptr(rows), None, None, ctypes.byref(d), N.stream()) != 0
    assert lib.tt_assemble_triplet_rows_mined(N.ptr(pq), N.ptr(pd), N.ptr(qid), N.ptr(order), Bg, 0, Bg, seed,
                                              N.ptr(rows), None, None, None, N.stream()) != 0
    assert "descriptor" in N.last_error()
    assert np.array_equal(_assemble(tt, banks, pq, pd, qid, order, Bg, 0, Bg, seed, None)["rows"], base["rows"])


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the miner against float64
# ---------------------------------------------------------------------------------------------------------------------
def synth(tt, n_pairs, seed=42):
    return tt.data.MSMarcoDataset("train", max_samples=n_pairs, random_seed=seed, synthetic=True)


def _random_banks(tt, model, ds, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    mk = lambda n, L, tower: tt.data.PooledBank(  # noqa: E731
        torch.nn.functional.normalize(torch.randn(n, 384, generator=g, device="cuda"), dim=1),
        tt.data.backbone_identity(tower), L)
    return mk(len(ds.query_bank), 32, model.query_tower), mk(len(ds.doc_bank), 256, model.document_tower)


def _check_table(tt, miner, model, sample=None):
    """The miner's table against the float64 top-k of its own normalised projections minus the exclusions."""
    Qn = tt.ops.l2_normalize_rows(miner._project(model.query_tower, miner.bank_q.rows))
    Dn = tt.ops.l2_normalize_rows(miner._project(model.document_tower, miner.bank_d.rows))
    rows = np.arange(miner.n_rows) if sample is None else sample
    table, count = miner.table.cpu().numpy(), miner.count.cpu().numpy()
    off, ids = miner.excl_offsets.cpu().numpy(), miner.excl_ids.cpu().numpy()
    k, skip, depth = miner.k_scan, miner.skip, miner.depth
    checked = 0
    for s in range(0, len(rows), 64):
        part = rows[s: s + 64]
        S = (Qn[torch.from_numpy(part).cuda()].double() @ Dn.double().T)
        top_v, top_i = torch.topk(S, k + 1, dim=1)
        top_v, top_i = top_v.cpu().numpy(), top_i.cpu().numpy()
        for j, r in enumerate(part):
            excl = set(ids[off[r]: off[r + 1]].tolist())
            got = table[r, : count[r]]
            assert np.all(table[r, count[r]:] == -1) and 0 <= count[r] <= depth
            assert not (set(got.tolist()) & excl), "an excluded passage in the table"
            assert len(set(got.tolist())) == len(got)
            sc = S[j, torch.from_numpy(got.astype(np.int64)).cuda()].cpu().numpy()
            assert np.all(np.diff(sc) <= 2 * TAU), "table row not in descending float64 score"
            v, i_ = top_v[j], top_i[j]
            keep = [t for t in range(k) if int(i_[t]) not in excl][skip: skip + depth]
            if v[k - 1] - v[k] > 2 * TAU:  # the scan's k-th is unambiguous: the counts agree
                assert count[r] == len(keep), r
            for pos, t in enumerate(keep[: count[r]]):
                gap_prev = v[t - 1] - v[t] if t > 0 else np.inf
                gap_next = v[t] - v[t + 1]
                if gap_prev > 2 * TAU and gap_next > 2 * TAU:
                    assert got[pos] == i_[t], (r, pos)
                    checked += 1
                else:
                    assert abs(sc[pos] - v[t]) <= 2 * TAU
    assert checked >= 0.5 * count[rows].sum()
    return checked


@gpu
@pytest.mark.parametrize("P", [64, 128, 512])
def test_miner_table_is_the_float64_top_k_minus_positives(tt, P):
    ds = synth(tt, 3000)
    torch.manual_seed(P)
    model = tt.TwoTowersModel(projection_dim=P, vocab_size=1000).cuda()
    bq, bd = _random_banks(tt, model, ds, seed=P)
    # one projection for both towers and every third positive on its query's pooled row: positives rank first,
    # so the exclusions land inside the lists
    model.document_tower.projection.load_state_dict(model.query_tower.projection.state_dict())
    pq = np.array([int(d["query"].split(":")[1]) for d in ds.data])
    pdoc = np.array([int(d["positive"].split(":")[1]) for d in ds.data])
    with torch.no_grad():
        bd.rows[torch.from_numpy(pdoc[::3]).cuda()] = bq.rows[torch.from_numpy(pq[::3]).cuda()]
    miner = tt.data.HardNegativeMiner(ds, bq, bd, depth=8, skip=2, ratio=1.0, k_scan=32)
    stats = miner.refresh(model)
    for key in ("project_s", "normalize_s", "scan_s", "merge_s", "filter_s", "total_s"):
        assert stats[key] >= 0
    assert stats["empty_queries"] == int((miner.count == 0).sum()) and 0 < stats["mean_count"] <= 8
    _check_table(tt, miner, model)
    ref_t, ref_c = miner.table.clone(), miner.count.clone()
    # G virtual document shards, scanned separately and merged: the same table
    for G in (2, 3, 8):
        parts = [tt.data.HardNegativeMiner(ds, bq, bd, depth=8, skip=2, ratio=1.0, k_scan=32, world_size=G, rank=r)
                 for r in range(G)]
        lists = [p.local_lists(model) for p in parts]
        s, i = tt.ops.topk_merge(torch.stack([a for a, _ in lists]), torch.stack([b for _, b in lists]))
        parts[0].filter(i)
        _check_table(tt, parts[0], model)
        same = (parts[0].table == ref_t).all(1)
        assert float(same.float().mean()) > 0.99, G
        assert torch.equal(parts[0].count[same], ref_c[same])


@gpu
def test_miner_at_the_full_synthetic_train_split(tt):
    ds = tt.data.MSMarcoDataset("train", max_samples=-1, synthetic=True)
    assert len(ds.doc_bank) == 676_193
    torch.manual_seed(0)
    model = tt.TwoTowersModel(projection_dim=128, vocab_size=1000).cuda()
    bq, bd = _random_banks(tt, model, ds, seed=1)
    miner = tt.data.HardNegativeMiner(ds, bq, bd, depth=8, k_scan=32)
    assert miner.n_rows == len(ds.query_bank)
    st = miner.refresh(model)
    print(f"\n[hard negatives] full split refresh: {st}")
    table, count = miner.table.cpu().numpy(), miner.count.cpu().numpy()
    assert np.all((count >= 0) & (count <= 8))
    cols = np.arange(8)[None, :]
    assert np.all((table >= 0) == (cols < count[:, None])) and table.max() < len(ds.doc_bank)
    off, ids = miner.excl_offsets.cpu().numpy(), miner.excl_ids.cpu().numpy()
    for r in range(0, miner.n_rows, 97):
        assert not set(table[r, : count[r]].tolist()) & set(ids[off[r]: off[r + 1]].tolist())
    sample = np.random.default_rng(0).choice(miner.n_rows, 256, replace=False)
    _check_table(tt, miner, model, sample)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: training with mined negatives
# ---------------------------------------------------------------------------------------------------------------------
def _table_banks(tt, model, ds, Lq=32, Ld=256):
    return (tt.data.PooledBank.build(model.query_tower, ds.query_bank, Lq),
            tt.data.PooledBank.build(model.document_tower, ds.doc_bank, Ld))


@gpu
def test_step_fed_mined_rows_equals_the_step_fed_the_same_rows(tt):
    ds = synth(tt, 2600)
    B = 256
    torch.manual_seed(2)
    model = tt.TwoTowersModel(projection_dim=64).cuda()
    banks = _table_banks(tt, model, ds)
    m2 = copy.deepcopy(model)
    banks2 = _table_banks(tt, m2, ds)
    t1 = tt.training.FusedTrainer(model, 0.3, 1e-3, B, 32, 256, pooled=banks, use_graph=False)
    t2 = tt.training.FusedTrainer(m2, 0.3, 1e-3, B, 32, 256, pooled=banks2, use_graph=False)
    miner = tt.data.HardNegativeMiner(ds, *banks, depth=8, ratio=1.0)
    miner.refresh(model)
    feeder = tt.data.DeviceTripletFeeder(ds, B, 32, 256, "cuda", seed=4, rows_only=True)
    feeder.hard_negatives = miner
    feeder.start_epoch()
    for step in range(3):
        feeder.assemble(t1, 0, step)
        t2.load_rows(t1.row_bufs[0].clone())
        t1.step(), t2.step()
    torch.cuda.synchronize()
    feeder.check()
    assert torch.equal(t1.flat_p, t2.flat_p) and torch.equal(t1.exp_avg_sq, t2.exp_avg_sq)
    assert torch.equal(t1.step_obj.pooled_rows(), t2.step_obj.pooled_rows())


def _batch_stats(tt, model, banks, rows, margin):
    with torch.no_grad():
        q = model.query_tower.projection(banks[0].rows[rows[0].long()])
        p = model.document_tower.projection(banks[1].rows[rows[1].long()])
        n = model.document_tower.projection(banks[1].rows[rows[2].long()])
        cp, cn = (torch.nn.functional.cosine_similarity(q, x, dim=1) for x in (p, n))
        return float(cn.mean()), float(((cn - cp + margin) > 0).float().mean())


@gpu
@pytest.mark.parametrize("backbone", ["table", "minilm"])
def test_mined_negatives_are_harder_than_in_batch_ones(tt, backbone):
    ds = synth(tt, 3000)
    B = 1024
    torch.manual_seed(5)
    model = tt.TwoTowersModel(projection_dim=128, backbone=backbone).cuda()
    banks = _table_banks(tt, model, ds)
    tr = tt.training.FusedTrainer(model, 0.1, 1e-3, B, 32, 256, pooled=banks, use_graph=False)
    miner = tt.data.HardNegativeMiner(ds, *banks, depth=8, ratio=1.0)
    miner.refresh(model)
    feeder = tt.data.DeviceTripletFeeder(ds, B, 32, 256, "cuda", seed=6, rows_only=True)
    feeder.start_epoch()
    feeder.assemble(tr, 0, 0)
    plain = tr.row_bufs[0].view(3, B).clone()
    feeder.hard_negatives = miner
    feeder.assemble(tr, 0, 0)
    mined = tr.row_bufs[0].view(3, B).clone()
    feeder.check()
    assert torch.equal(plain[:2], mined[:2])
    # margin 0: at these random-init weights every cosine lies within a few hundredths of 0, so the trainer's margin
    # would make every hinge active with either kind of negative; with margin 0 a hinge is active iff cos_n > cos_p
    cos_b, act_b = _batch_stats(tt, model, banks, plain, 0.0)
    cos_m, act_m = _batch_stats(tt, model, banks, mined, 0.0)
    print(f"\n[hard negatives] {backbone}: mean cos(q, n) {cos_b:.4f} -> {cos_m:.4f}, active hinges {act_b:.3f} -> "
          f"{act_m:.3f}")
    assert cos_m > cos_b and act_m > act_b


def _run(tt, capsys, backbone, **kw):
    torch.manual_seed(0)
    model = tt.training.run_training(num_epochs=2, batch_size=256, learning_rate=1e-3, max_samples=3000,
                                     projection_dim=64, margin=0.3, use_wandb=False, accumulation_steps=1,
                                     use_mixed_precision=False, num_workers=0, run_comprehensive_test=False,
                                     backbone=backbone, **kw)
    return model, capsys.readouterr().out


@gpu
@pytest.mark.parametrize("backbone", ["table", "minilm"])
@pytest.mark.parametrize("via_env", [False, True])
def test_run_training_with_hard_negatives(tt, monkeypatch, capsys, backbone, via_env):
    monkeypatch.setenv("TT_SYNTHETIC_DATA", "1")
    monkeypatch.delenv("TT_HOST_FEEDER", raising=False)
    if via_env:
        monkeypatch.setenv("TT_HARD_NEGATIVES", "8")
        kw = {}
    else:
        kw = {"hard_negatives": {"depth": 6, "ratio": 0.7, "warmup_epochs": 1}}
    model, out = _run(tt, capsys, backbone, **kw)
    lines = out.splitlines()
    assert isinstance(model, tt.TwoTowersModel) and "Fused B200 step: True" in out
    assert sum(line.startswith("Hard negatives refreshed") for line in lines) == 1
    losses = [float(line.split(":")[1]) for line in lines if line.startswith("Average training loss")]
    assert len(losses) == 2 and all(np.isfinite(losses))
    if backbone == "table":
        assert any("neg-index reuse is off" in line for line in lines)


@gpu
def test_refusals(tt, monkeypatch, capsys):
    monkeypatch.setenv("TT_SYNTHETIC_DATA", "1")
    monkeypatch.setenv("TT_HOST_FEEDER", "1")
    with pytest.raises(ValueError, match="device feeder"):
        _run(tt, capsys, "table", hard_negatives=8)
    monkeypatch.delenv("TT_HOST_FEEDER")
    ds = synth(tt, 2600)
    torch.manual_seed(0)
    model = tt.TwoTowersModel(projection_dim=64).cuda()
    banks = _table_banks(tt, model, ds)
    miner = tt.data.HardNegativeMiner(ds, *banks, depth=4)
    # in-batch negative reuse together with a miner
    tr = tt.training.FusedTrainer(model, 0.3, 1e-3, 256, 32, 256, in_batch_negatives=True, use_graph=False)
    feeder = tt.data.DeviceTripletFeeder(ds, 256, 32, 256, "cuda", seed=1)
    feeder.hard_negatives = miner
    feeder.start_epoch()
    with pytest.raises(ValueError, match="in_batch_negatives"):
        feeder.assemble(tr, 0, 0)
    # stale banks (another model's tables), trainable tables, banks of another dataset, bad arguments
    with pytest.raises(RuntimeError, match="stale"):
        miner.refresh(copy.deepcopy(model))
    torch.manual_seed(0)
    trainable = tt.TwoTowersModel(projection_dim=64, train_table=True).cuda()
    tb = _table_banks(tt, trainable, ds)
    with pytest.raises(ValueError, match="frozen"):
        tt.data.HardNegativeMiner(ds, *tb).refresh(trainable)
    with pytest.raises(ValueError, match="same dataset"):
        tt.data.HardNegativeMiner(synth(tt, 2000), *banks)
    for kw in ({"k_scan": 33}, {"skip": 30, "depth": 8}, {"depth": 0}, {"ratio": 1.5}, {"ratio": -0.5}):
        with pytest.raises(ValueError):
            tt.data.HardNegativeMiner(ds, *banks, **kw)
    # a feeder over another dataset refuses the miner
    other = tt.data.DeviceTripletFeeder(synth(tt, 2000), 256, 32, 256, "cuda", seed=1, rows_only=True)
    other.hard_negatives = miner
    other.start_epoch()
    tp = tt.training.FusedTrainer(model, 0.3, 1e-3, 256, 32, 256, pooled=banks, use_graph=False)
    with pytest.raises(ValueError, match="miner"):
        other.assemble(tp, 0, 0)


@gpu
def test_resume_after_epoch_two_refreshes_the_same_table_and_ends_on_the_same_weights(tt, tmp_path):
    ds = synth(tt, 2600)
    B = 256
    torch.manual_seed(8)
    model = tt.TwoTowersModel(projection_dim=64).cuda()
    ref = copy.deepcopy(model)

    def setup(m):
        banks = _table_banks(tt, m, ds)
        tr = tt.training.FusedTrainer(m, 0.3, 1e-3, B, 32, 256, token_slots=2, pooled=banks)
        feeder = tt.data.DeviceTripletFeeder(ds, B, 32, 256, "cuda", seed=3, rows_only=True)
        miner = tt.data.HardNegativeMiner(ds, *banks, depth=8, ratio=0.6)
        feeder.hard_negatives = miner
        tr.prepare(2)
        return tr, feeder, miner

    def epoch(tr, feeder, miner, e):
        if e >= 1:
            miner.refresh(tr.model)
        return tr.train_epoch_device(feeder)

    t_ref, f_ref, m_ref = setup(ref)
    for e in range(3):
        epoch(t_ref, f_ref, m_ref, e)
    table_3 = (m_ref.table.clone(), m_ref.count.clone())
    t1, f1, m1 = setup(model)
    for e in range(2):
        epoch(t1, f1, m1, e)
    path = str(tmp_path / "ck.pt")
    t1.save_checkpoint(path)
    fresh = copy.deepcopy(model)
    t2, f2, m2 = setup(fresh)
    t2.load_checkpoint(path)
    for _ in range(2):  # the feeder's epoch counter and permutation stream, as after two epochs
        f2.start_epoch()
    epoch(t2, f2, m2, 2)
    torch.cuda.synchronize()
    assert torch.equal(m2.table, table_3[0]) and torch.equal(m2.count, table_3[1])
    assert torch.equal(t2.flat_p, t_ref.flat_p)
    assert torch.equal(t2.exp_avg, t_ref.exp_avg) and torch.equal(t2.exp_avg_sq, t_ref.exp_avg_sq)
