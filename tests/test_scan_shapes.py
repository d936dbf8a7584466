"""The corpus scan (tt_scan_topk: the strict fp32 scan, and the tensor-core scan_candidates_kernel + refine_kernel +
listed fp32 re-scan of csrc/tt_scan_sm100.cu) against a float64 top-k oracle at the shapes and data where its
completeness proof does the work (DESIGN.md §4, "Scan exactness").

The tensor-core scan keeps KC candidates per query and document split (16, 32 or 48 by plan and k) behind a threshold
that compaction raises, shares a per-query floor between splits, selects at most kSelCap = 256 candidates for the
exact re-score and re-scans every query it cannot prove in fp32, in rounds of 8192 listed queries.  I.i.d. Gaussian
corpora never stress any of that, so the cases here are built to: every k up to 32 (KC = 16 / 32 / 48), partial query
tiles and the phantom CTA of the pair kernel, partial document tiles and one-document splits, P from 8 to 512,
64-bit id bases, near-tie corpora (thousands of documents within the bf16 error of the k-th score), exact duplicates
across splits and shards, all-negative scores, zero rows, more than 8192 unproven queries and CUDA-graph replays whose
set of unproven queries changes.

The oracle starts from the device's own normalised rows (Qn, Dn; l2_normalize_rows is checked on its own), so it
judges the scan alone.  Every case runs under the strict fp32 scan and the tensor-core scan with one CTA per query
tile and with CTA pairs (TT_SCAN_PAIR = 0 / 1)."""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"
# Largest |returned score - float64 dot of the returned id| allowed.  Worst measured over this file on a B200 (1000 W
# power limit): fp32 9.6e-7, bf16 one CTA 5.1e-7, bf16 CTA pairs 4.5e-7 (the report printed at the end of the module).
TAU = 1.5e-6
CONFIGS = ["fp32", "bf16-cta", "bf16-pair"]
BIG_BASE = 3 * 2 ** 31 + 5
WORST = {}     # configuration -> worst score error seen
ID_DIFFS = {}  # configuration -> [ranks whose id differs from the strict fp32 scan, rows whose scores differ in bits,
#                                  the cases with differing ids]


@pytest.fixture(scope="module")
def tt():
    import two_towers_overlords_b200 as pkg
    from two_towers_overlords_b200 import ops, retrieval

    pkg.ops, pkg.retrieval = ops, retrieval
    yield pkg
    for cfg in sorted(WORST):
        d = ID_DIFFS.get(cfg, [0, 0, []])
        print(f"\n[scan shapes] {cfg}: worst score error {WORST[cfg]:.3e} (tau {TAU:.1e}); vs the strict fp32 scan: "
              f"{d[0]} ranks with another id {d[2]}, {d[1]} rows with other score bits")


@pytest.fixture(params=CONFIGS)
def cfg(request, monkeypatch):
    if request.param != "fp32":
        monkeypatch.setenv("TT_SCAN_PAIR", "1" if request.param == "bf16-pair" else "0")
    return request.param


# ---------------------------------------------------------------------------------------------------------------------
# the oracle
# ---------------------------------------------------------------------------------------------------------------------
def _oracle_order(S64):
    """(scores, local ids) of every row sorted by (score desc, id asc)."""
    order = torch.sort(S64, dim=1, descending=True, stable=True).indices  # stable: equal scores keep ascending ids
    return S64.gather(1, order), order


def _dup_groups(Dn):
    """Sets of bit-identical document rows (ascending local ids), as tensors on the device."""
    if Dn.shape[0] < 2:
        return []
    _, inv, cnt = torch.unique(Dn, dim=0, return_inverse=True, return_counts=True)
    groups = []
    for g in torch.nonzero(cnt > 1).flatten().tolist():
        groups.append(torch.nonzero(inv == g).flatten())
    return groups


def safe_ranks(S64, k):
    """[Q, min(k, N)] mask of ranks whose oracle neighbours are both more than 2 tau away (ids must be exact there)."""
    s, _ = _oracle_order(S64)
    kk = min(k, S64.shape[1])
    inf = torch.full((s.shape[0], 1), float("inf"), dtype=s.dtype, device=s.device)
    ext = torch.cat([inf, s, -inf], 1)  # the rank past N has no neighbour
    prev_gap = ext[:, :kk] - ext[:, 1: kk + 1]
    next_gap = ext[:, 1: kk + 1] - ext[:, 2: kk + 2]
    return (prev_gap > 2 * TAU) & (next_gap > 2 * TAU)


def check_exact_topk(top_s, top_i, Qn, Dn, k, id_base, cfg="fp32", S64=None):
    """Asserts, for every query row, that (top_s, top_i) [Q, k] is the exact top k of Qn . Dn^T by (score desc, id
    asc): padding, no duplicate ids, order, every score within TAU of float64, the set within 2 TAU of the oracle's,
    the oracle's ids where its gaps exceed 2 TAU, and ascending ids inside every group of bit-identical documents."""
    Q, N = Qn.shape[0], Dn.shape[0]
    assert top_s.shape == (Q, k) and top_i.shape == (Q, k)
    top_s, top_i = top_s.to(DEV), top_i.to(DEV)
    kk = min(k, N)
    # padding
    assert bool((top_i[:, kk:] == -1).all()), "ids past min(k, N) must be -1"
    assert bool((top_s[:, kk:] == float("-inf")).all()), "scores past min(k, N) must be -inf"
    if kk == 0:
        return
    ids = top_i[:, :kk]
    loc = ids - id_base
    assert bool(((loc >= 0) & (loc < N)).all()), f"ids outside [{id_base}, {id_base + N})"
    # no duplicates
    srt = torch.sort(loc, dim=1).values
    assert bool((srt[:, 1:] != srt[:, :-1]).all()), "an id appears twice in a row"
    # order: (score desc, id asc), strictly
    s = top_s[:, :kk]
    ok = (s[:, :-1] > s[:, 1:]) | ((s[:, :-1] == s[:, 1:]) & (ids[:, :-1] < ids[:, 1:]))
    assert bool(ok.all()), "rows are not sorted by (score desc, id asc)"
    # scores against float64 dots of their own ids
    if S64 is None:
        S64 = Qn.double() @ Dn.double().T
    own = S64.gather(1, loc)
    err = float((s.double() - own).abs().max())
    WORST[cfg] = max(WORST.get(cfg, 0.0), err)
    assert err <= TAU, f"score error {err:.3e} > {TAU:.0e}"
    # the top-k set: nothing left out scores more than 2 tau above the returned k-th, nothing returned more than 2 tau
    # below the oracle's (k+1)-th
    kth = own[:, kk - 1]
    left = S64.clone()
    left.scatter_(1, loc, float("-inf"))
    assert bool((left.max(1).values <= kth + 2 * TAU).all()), "a document left out beats the returned k-th"
    os_, oi = _oracle_order(S64)
    if N > kk:
        assert bool((own.min(1).values >= os_[:, kk] - 2 * TAU).all()), "a returned document is below the (k+1)-th"
    # exact ids where the oracle's gaps allow
    safe = safe_ranks(S64, k)
    bad = safe & (loc != oi[:, :kk])
    assert not bool(bad.any()), f"{int(bad.sum())} ranks with a wrong id where the gaps exceed 2 tau"
    # bit-identical documents: a returned member implies every smaller-id member (same score, smaller id) is returned
    for g in _dup_groups(Dn):
        member = (loc[:, :, None] == g[None, None, :]).any(1)  # [Q, |g|]
        assert not bool((member[:, 1:] & ~member[:, :-1]).any()), f"duplicates {g.tolist()[:4]}... out of id order"


def run_scan(tt, Qn, Dn, k, id_base, cfg, Qb=None, Db=None):
    if cfg == "fp32":
        return tt.ops.scan_topk(Qn, Dn, k=k, id_base=id_base, precision="fp32")
    Qb = Qn.to(torch.bfloat16) if Qb is None else Qb
    Db = Dn.to(torch.bfloat16) if Db is None else Db
    return tt.ops.scan_topk(Qn, Dn, k=k, id_base=id_base, precision="bf16", Qb=Qb, Db=Db)


def scan_and_check(tt, Qe, De, k, cfg, id_base=0):
    """Normalise on the device, scan under `cfg`, check against float64; tensor-core runs are also compared with the
    strict fp32 scan.  -> (top_s, top_i, Qn, Dn)"""
    Qn, Qb = tt.ops.l2_normalize_rows(Qe.to(DEV), want_bf16=True)
    Dn, Db = tt.ops.l2_normalize_rows(De.to(DEV), want_bf16=True)
    top_s, top_i = run_scan(tt, Qn, Dn, k, id_base, cfg, Qb, Db)
    S64 = Qn.double() @ Dn.double().T
    check_exact_topk(top_s, top_i, Qn, Dn, k, id_base, cfg, S64)
    if cfg != "fp32":
        ref_s, ref_i = run_scan(tt, Qn, Dn, k, id_base, "fp32")
        kk = min(k, Dn.shape[0])
        safe = safe_ranks(S64, k)
        assert bool((top_i[:, :kk] == ref_i[:, :kk])[safe].all()), "ids differ from the strict fp32 scan"
        # (proven rows carry refine's scores, whose summation order is not the fp32 scan's: DESIGN.md §4)
        d = ID_DIFFS.setdefault(cfg, [0, 0, []])
        n_ids = int((top_i != ref_i).sum())
        d[0] += n_ids
        d[1] += int(((top_s != ref_s) & (top_i == ref_i)).any(1).sum())
        if n_ids:
            d[2].append(os.environ.get("PYTEST_CURRENT_TEST", "?").split("::")[-1].split(" ")[0])
    return top_s, top_i, Qn, Dn


# ---------------------------------------------------------------------------------------------------------------------
# corpora (CPU, seeded)
# ---------------------------------------------------------------------------------------------------------------------
def gaussian(Q, N, P, seed):
    gen = torch.Generator().manual_seed(seed)
    return torch.randn(Q, P, generator=gen), torch.randn(N, P, generator=gen)


def near_tie(Q, N, P, sigma, seed, n_tie=2000):
    """n_tie documents and every query are one base row plus noise of sigma, the ties spread evenly over the corpus
    (and so over every split); the other documents are Gaussian."""
    gen = torch.Generator().manual_seed(seed)
    base = torch.randn(P, generator=gen)
    base /= base.norm()
    De = torch.randn(N, P, generator=gen)
    ids = torch.linspace(0, N - 1, n_tie).round().long()
    De[ids] = base + sigma * torch.randn(n_tie, P, generator=gen)
    Qe = base + sigma * torch.randn(Q, P, generator=gen)
    return Qe, De


def with_duplicates(Q, N, P, seed, where):
    """Gaussian corpus with one row copied to every id of `where`, a second row copied 40 times; queries near both."""
    gen = torch.Generator().manual_seed(seed)
    Qe, De = torch.randn(Q, P, generator=gen), torch.randn(N, P, generator=gen)
    De[torch.tensor(where)] = De[where[0]].clone()
    many = torch.linspace(1, N - 2, 40).round().long()
    De[many] = De[many[0]].clone()
    Qe[: Q // 2] = De[where[0]] + 0.05 * torch.randn(Q // 2, P, generator=gen)
    Qe[Q // 2:] = De[many[0]] + 0.05 * torch.randn(Q - Q // 2, P, generator=gen)
    return Qe, De


def negative(Q, N, P, seed, zero_docs=()):
    """Every query near +b, every document near -b: all scores negative (except documents that are all zero)."""
    gen = torch.Generator().manual_seed(seed)
    base = torch.randn(P, generator=gen)
    Qe = base + 0.1 * base.norm() * torch.randn(Q, P, generator=gen) / P ** 0.5
    De = -base + 0.3 * base.norm() * torch.randn(N, P, generator=gen) / P ** 0.5
    if zero_docs:
        De[torch.tensor(zero_docs)] = 0.0
    return Qe, De


# ---------------------------------------------------------------------------------------------------------------------
# k: KC steps 16 -> 32 at k = 11 and 32 -> 48 at k = 27 (one query tile: 79 splits of two tiles over N = 20,001)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 2, 9, 10, 11, 16, 17, 26, 27, 30, 31, 32])
def test_k_sweep(tt, cfg, k):
    Q = 300 if cfg == "bf16-pair" else 100
    Qe, De = gaussian(Q, 20_001, 64, seed=100 + k)
    scan_and_check(tt, Qe, De, k, cfg)


@pytest.mark.parametrize("k", [10, 27, 32])
def test_k_sweep_near_tie(tt, cfg, k):
    """Exact gaps of ~1e-4 between the leading documents, inside the bf16 error: compaction decides which of them are
    candidates, and only the proof can tell whether the dropped ones matter."""
    Q = 300 if cfg == "bf16-pair" else 100
    Qe, De = near_tie(Q, 20_001, 64, 1e-2, seed=200 + k)
    scan_and_check(tt, Qe, De, k, cfg)


def test_k_above_32_is_refused_by_the_tensor_core_scan(tt):
    Qe, De = gaussian(4, 500, 64, seed=3)
    Qn, Dn = tt.ops.l2_normalize_rows(Qe.to(DEV)), tt.ops.l2_normalize_rows(De.to(DEV))
    with pytest.raises(tt.ops.N.NativeError, match="at most 32 results"):
        run_scan(tt, Qn, Dn, 33, 0, "bf16-cta")
    # the fp32 scan has no such limit
    top_s, top_i = run_scan(tt, Qn, Dn, 33, 0, "fp32")
    check_exact_topk(top_s, top_i, Qn, Dn, 33, 0)


# ---------------------------------------------------------------------------------------------------------------------
# plan edges
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("id_base", [0, 1000, BIG_BASE])
@pytest.mark.parametrize("Q", [1, 127, 128, 129, 255, 256, 257])
def test_query_tiles(tt, cfg, Q, id_base):
    Qe, De = gaussian(Q, 20_001, 64, seed=300 + Q)
    scan_and_check(tt, Qe, De, 10, cfg, id_base)


# 19,969 = 78 splits of 256 documents + one split holding a single document (one query tile)
@pytest.mark.parametrize("N", [1, 5, 127, 128, 129, 19_969])
def test_document_counts(tt, cfg, N):
    Q = 300 if cfg == "bf16-pair" else 100
    Qe, De = gaussian(Q, N, 64, seed=400 + N)
    scan_and_check(tt, Qe, De, 16, cfg, id_base=1000)


@pytest.mark.parametrize("P", [8, 16, 56, 64, 72, 136, 504, 512])
def test_row_widths(tt, cfg, P):
    Q = 300 if cfg == "bf16-pair" else 100
    Qe, De = gaussian(Q, 5000, P, seed=500 + P)
    near = torch.arange(0, 5000, 7)  # planted neighbours, so that the leading scores are not all Gaussian noise
    De[near] = Qe[near % Q] + 0.1 * torch.randn(len(near), P, generator=torch.Generator().manual_seed(P))
    scan_and_check(tt, Qe, De, 10, cfg, id_base=BIG_BASE)


def test_row_width_not_a_multiple_of_8_is_refused(tt):
    Qe, De = gaussian(4, 500, 20, seed=5)
    Qn, Dn = tt.ops.l2_normalize_rows(Qe.to(DEV)), tt.ops.l2_normalize_rows(De.to(DEV))
    with pytest.raises(tt.ops.N.NativeError, match="P % 8 == 0"):
        run_scan(tt, Qn, Dn, 10, 0, "bf16-cta")


def test_empty_shard_pads_with_minus_infinity(tt, cfg):
    Qe = torch.randn(3, 64)
    Qn = tt.ops.l2_normalize_rows(Qe.to(DEV))
    Dn = torch.empty(0, 64, device=DEV)
    top_s, top_i = run_scan(tt, Qn, Dn, 10, 7, cfg)
    check_exact_topk(top_s, top_i, Qn, Dn, 10, 7)


# ---------------------------------------------------------------------------------------------------------------------
# data where the proof does the work
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sigma", [1e-4, 1e-2])
@pytest.mark.parametrize("k", [10, 32])
def test_near_tie_corpus(tt, cfg, sigma, k):
    """2,000 documents within the bf16 error of each other and of every query (sigma = 1e-4: equal to a few fp32 ulps,
    so every split compacts on every tile and refine selects more than kSelCap; 1e-2: exact gaps of ~1e-4)."""
    Qe, De = near_tie(300, 20_001, 64, sigma, seed=600 + k)
    scan_and_check(tt, Qe, De, k, cfg)


@pytest.mark.parametrize("k", [10, 32])
def test_exact_duplicates(tt, cfg, k):
    N = 20_001
    # ids in different splits, at the ends of the corpus and on both sides of the shard boundaries of a 4-way split
    where = [5, 4999, 5000, 9000, 9999, 10_000, 15_000, N - 1]
    Qe, De = with_duplicates(300, N, 64, 700 + k, where)
    scan_and_check(tt, Qe, De, k, cfg, id_base=BIG_BASE)


@pytest.mark.parametrize("zero_docs", [(), (5, 9000, 20_000)], ids=["negative", "negative+zero_docs"])
def test_all_scores_negative(tt, cfg, zero_docs):
    """N = 20,001 is not a multiple of 128: zero-filled columns of the last tile would score 0 and beat every real
    document if they passed the mask; all-zero documents do score 0 and must lead, in ascending id."""
    Qe, De = negative(300, 20_001, 64, 800, zero_docs)
    top_s, top_i, Qn, Dn = scan_and_check(tt, Qe, De, 10, cfg)
    if zero_docs:
        assert bool((top_i[:, :3] == torch.tensor(zero_docs, device=DEV)).all()) and bool((top_s[:, :3] == 0).all())
    else:
        assert bool((top_s < 0).all())


def test_zero_query_returns_the_first_ids(tt, cfg):
    k, base = 12, 1000
    Qe, De = gaussian(130, 20_001, 64, seed=900)
    Qe[0] = 0.0
    Qe[129] = 0.0
    top_s, top_i, _, _ = scan_and_check(tt, Qe, De, k, cfg, id_base=base)
    for q in (0, 129):
        assert top_i[q].tolist() == list(range(base, base + k)) and bool((top_s[q] == 0).all())


def test_mixed_batch(tt, cfg):
    """Near-tie queries (unprovable) interleaved with random ones (proven): the re-scan writes back to a scattered
    list of rows and must leave the others as refine wrote them."""
    Qt, De = near_tie(300, 20_001, 64, 1e-4, seed=1000)
    Qr, _ = gaussian(300, 1, 64, seed=1001)
    Qe = torch.where((torch.arange(300) % 2 == 0)[:, None], Qt, Qr)
    scan_and_check(tt, Qe, De, 10, cfg)


@pytest.mark.parametrize("pair", ["0", "1"])
def test_more_unproven_queries_than_one_rescan_round(tt, monkeypatch, pair):
    """TT_SCAN_EPS = 10 leaves every query unproven: 8,492 listed queries take two rounds of the listed re-scan
    (8,192 + 300).  Every row, the second round's too, must equal the strict fp32 scan bit for bit.  (N stays well
    above KC: a split that has seen fewer than KC documents reports no bound and refine proves its queries.)"""
    Qe, De = gaussian(8492, 6000, 64, seed=1100)
    Qn, Qb = tt.ops.l2_normalize_rows(Qe.to(DEV), want_bf16=True)
    Dn, Db = tt.ops.l2_normalize_rows(De.to(DEV), want_bf16=True)
    ref_s, ref_i = run_scan(tt, Qn, Dn, 10, 1000, "fp32")
    monkeypatch.setenv("TT_SCAN_PAIR", pair)
    monkeypatch.setenv("TT_SCAN_EPS", "10")
    top_s, top_i = run_scan(tt, Qn, Dn, 10, 1000, "bf16", Qb, Db)
    assert torch.equal(top_i, ref_i) and torch.equal(top_s, ref_s)
    assert torch.equal(top_i[8192:], ref_i[8192:])
    check_exact_topk(top_s, top_i, Qn, Dn, 10, 1000, "bf16-pair" if pair == "1" else "bf16-cta")


# ---------------------------------------------------------------------------------------------------------------------
# sharding, graphs, normalisation, the search engine
# ---------------------------------------------------------------------------------------------------------------------
def _shard_precision(cfg):
    return "fp32" if cfg == "fp32" else "bf16"


@pytest.mark.parametrize("corpus", ["near_tie", "duplicates", "five_docs"])
@pytest.mark.parametrize("G", [1, 2, 4, 8])
def test_sharded_scan_and_merge(tt, cfg, corpus, G):
    k = 10
    if corpus == "near_tie":
        Qe, De = near_tie(200, 20_001, 64, 1e-2, seed=1200)
    elif corpus == "duplicates":
        Qe, De = with_duplicates(200, 20_001, 64, 1201, [5, 4999, 5000, 10_000, 15_000, 20_000])
    else:  # 5 documents over 8 shards: seven of them are empty
        Qe, De = gaussian(200, 5, 64, seed=1202)
    Qe, De = Qe.to(DEV), De.to(DEV)
    N = De.shape[0]
    prec = _shard_precision(cfg)
    whole = tt.retrieval.CorpusShard(De, precision=prec)
    s1, i1 = whole.search(Qe, k, graph=False)
    parts = []
    for r in range(G):
        lo, hi = tt.retrieval.shard_bounds(N, G, r)
        parts.append(tt.retrieval.CorpusShard(De[lo:hi], id_base=lo, precision=prec).search(Qe, k, graph=False))
    ms, mi = tt.ops.topk_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
    Qn = tt.ops.l2_normalize_rows(Qe)
    S64 = Qn.double() @ whole.Dn.double().T
    check_exact_topk(ms, mi, Qn, whole.Dn, k, 0, cfg, S64)
    kk = min(k, N)
    assert bool((mi[:, :kk] == i1[:, :kk])[safe_ranks(S64, k)].all())


def test_graph_replays_follow_the_unproven_set(tt, monkeypatch):
    """CorpusShard.search captures a query shape seen twice into a CUDA graph; the re-scan's query list and count live
    on the device inside it.  Replays with random (mostly proven) and near-tie (all unproven) contents must equal an
    eager search bit for bit."""
    monkeypatch.setenv("TT_SCAN_PAIR", "0")
    Qt, De = near_tie(200, 20_001, 64, 1e-4, seed=1300)
    Qr1, _ = gaussian(200, 1, 64, seed=1301)
    Qr2, _ = gaussian(200, 1, 64, seed=1302)
    shard = tt.retrieval.CorpusShard(De.to(DEV), precision="bf16")
    for _ in range(3):
        shard.search(Qr1.to(DEV), 10)
    assert len(shard._graphs) == 1
    for Qe in (Qr1, Qt, Qr2, Qt):
        Qe = Qe.to(DEV)
        gs, gi = shard.search(Qe, 10)
        es, ei = shard.search(Qe, 10, graph=False)
        assert torch.equal(gi, ei) and torch.equal(gs, es)
        check_exact_topk(gs, gi, tt.ops.l2_normalize_rows(Qe), shard.Dn, 10, 0, "bf16-cta")


@pytest.mark.parametrize("P", [8, 64, 72, 384, 512])
def test_l2_normalize_rows_vs_float64(tt, P):
    gen = torch.Generator().manual_seed(P)
    x = torch.randn(1000, P, generator=gen) * torch.logspace(-3, 3, 1000)[:, None]
    x[[0, 17, 999]] = 0.0
    x[5] = 1e-12  # below the eps clamp of torch.cosine_similarity: divided by 1e-8, not by its norm
    y, yb = tt.ops.l2_normalize_rows(x.to(DEV), want_bf16=True)
    xd = x.double()
    want = xd / xd.norm(dim=1, keepdim=True).clamp_min(1e-8)
    assert float((y.double().cpu() - want).abs().max()) < 1e-6
    assert bool((y[[0, 17, 999]] == 0).all())
    # the scan's error bound assumes the bf16 copy is the fp32 row rounded to nearest
    assert torch.equal(yb, y.to(torch.bfloat16))


@pytest.mark.parametrize("top_k", [30, 31, 32, 33])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_search_engine_top_k(tt, tmp_path, monkeypatch, precision, top_k):
    from two_towers_overlords_b200 import search

    monkeypatch.setenv("TT_SCAN_PAIR", "0")
    torch.manual_seed(0)
    model = tt.TwoTowersModel(projection_dim=64, precision="fp32")
    docs = [f"passage {i} mentions item {i % 17} beside thing {(i * 7) % 23} and note {(i * i) % 31}" for i in range(300)]
    eng = search.DocumentSearchEngine(model=model, index_dir=str(tmp_path), precision=precision)
    eng.ingest_documents(docs, batch_size=128, clear_existing=True)
    queries = ["which passage mentions item 5 beside thing 7", "note 4", "item 16 thing 0 note 9"]
    res = eng.search_batch(queries, top_k=top_k)
    with torch.no_grad():
        Qn = tt.ops.l2_normalize_rows(model.encode_queries(queries).float())
    top_s = torch.full((len(queries), top_k), float("-inf"), dtype=torch.float64)
    top_i = torch.full((len(queries), top_k), -1, dtype=torch.int64)
    for q, hits in enumerate(res):
        assert len(hits) == top_k
        for r, h in enumerate(hits):
            top_s[q, r] = 2.0 * h["score"] - 1.0  # score = (1 + cos) / 2, exact in double
            top_i[q, r] = int(h["id"])
            assert h["content"] == docs[int(h["id"])]
    check_exact_topk(top_s.float(), top_i, Qn, eng.shard.Dn, top_k, 0, "engine-" + precision)
