"""
Datasets and triplet batching — drop-in for the reference's backend/data.py surface
(`MSMarcoDataset`, `TripletDataLoader`) plus the token-level feeder the B200 step needs.

  * MSMarcoDataset        same item format as backend/data.py:40-87 ({"query_id","query","positive"},
                          `get_unique_passages()`).  Loads MS MARCO v1.1 through `datasets` when it is
                          reachable; offline (this build: no network) it builds a seeded synthetic corpus of
                          the same shape whose "texts" are handles into a TokenBank.
  * TripletDataLoader     in-batch negative sampling with the reference's semantics (data.py:113-137:
                          negative_i = positive_j, j != i, query_id_j != query_id_i), vectorised.
  * TokenBank / TokenBankTokenizer   pre-tokenised texts; the tokenizer object plugs into
                          `tower.tokenizer` and returns the HF call's dict (model.py:43-45).
  * TokenTripletLoader    yields device-resident (q,p,n) TokenBatches for the fused step; with
                          world_size > 1 each rank receives its contiguous slice of the global batch.
  * HardNegativeMiner     per-query tables of hard negatives mined with the corpus scan from the current towers,
                          drawn by DeviceTripletFeeder beside the in-batch negatives.
"""
from __future__ import annotations

import ctypes
import math
import os
import random
from typing import Iterator, Optional, Tuple, Union

import numpy as np
import torch

try:
    from . import ops
    from .model import TokenBatch, VOCAB_SIZE
except ImportError:
    import ops
    from model import TokenBatch, VOCAB_SIZE

MsMarcoDatasetItem = dict[str, Union[str, int]]
Triplet = Tuple[list[str], list[str], list[str]]


# --------------------------------------------------------------------------------------------------
# token bank
# --------------------------------------------------------------------------------------------------
class TokenBank:
    """Ragged token lists stored as one flat int32 array + offsets; texts are handles '<prefix>:<index>'."""

    def __init__(self, prefix: str, flat: np.ndarray, offsets: np.ndarray):
        self.prefix, self.flat, self.offsets = prefix, flat.astype(np.int32), offsets.astype(np.int64)

    def __len__(self):
        return len(self.offsets) - 1

    def handle(self, i: int) -> str:
        return f"{self.prefix}:{i}"

    def tokens(self, i: int) -> np.ndarray:
        return self.flat[self.offsets[i]: self.offsets[i + 1]]

    def lengths(self, idx: np.ndarray) -> np.ndarray:
        return (self.offsets[idx + 1] - self.offsets[idx]).astype(np.int64)

    def batch(self, idx: np.ndarray, max_length: int = 512, pad_to: Optional[int] = None,
              ids_dtype=torch.int64, mask_dtype=torch.int64, pin: bool = False) -> TokenBatch:
        """Pads to the batch max like `padding=True` (model.py:44) unless pad_to is given."""
        idx = np.asarray(idx, dtype=np.int64)
        lens = np.minimum(self.lengths(idx), max_length)
        L = int(pad_to) if pad_to else int(lens.max(initial=1))
        ids = np.zeros((len(idx), L), dtype=np.int64)
        pos = np.arange(L)[None, :]
        valid = pos < lens[:, None]
        src = (self.offsets[idx][:, None] + pos)[valid]
        ids[valid] = self.flat[src]
        t_ids = torch.from_numpy(ids).to(ids_dtype)
        t_mask = torch.from_numpy(valid).to(mask_dtype)
        if pin and torch.cuda.is_available():
            t_ids, t_mask = t_ids.pin_memory(), t_mask.pin_memory()
        return TokenBatch(t_ids, t_mask)

    @staticmethod
    def synthetic(prefix: str, n: int, kind: str, seed: int, vocab: int = VOCAB_SIZE, shape: str = "Z",
                  full_len: Optional[int] = None) -> "TokenBank":
        """MS MARCO-shaped lengths/ids (SURVEY.md §8d): shape 'Z' = log-normal lengths, [CLS]/[SEP],
        Zipf interior ids; shape 'U' = every text exactly full_len uniform ids."""
        rng = np.random.default_rng(seed)
        lo = min(999, vocab // 2)
        if shape == "U":
            L = full_len or (32 if kind == "query" else 256)
            flat = rng.integers(lo, vocab, size=n * L, dtype=np.int64)
            return TokenBank(prefix, flat, np.arange(n + 1, dtype=np.int64) * L)
        mu, sigma, mn, mx = (math.log(9.0), 0.4, 4, 32) if kind == "query" else (math.log(90.0), 0.45, 16, 256)
        lens = np.clip(np.rint(rng.lognormal(mu, sigma, n)), mn, mx).astype(np.int64)
        offsets = np.concatenate([[0], np.cumsum(lens)])
        ranks = np.arange(1, vocab - lo + 1, dtype=np.float64)
        cdf = np.cumsum(1.0 / ranks)
        cdf /= cdf[-1]
        perm = np.random.default_rng(4242).permutation(vocab - lo)
        draw = np.searchsorted(cdf, rng.random(int(offsets[-1])))
        flat = perm[np.minimum(draw, vocab - lo - 1)] + lo
        flat[offsets[:-1]] = 101
        flat[offsets[1:] - 1] = 102
        return TokenBank(prefix, flat, offsets)


class TokenBankTokenizer:
    """Resolves text handles ("<bank prefix>:<index>") against token banks; same call/return shape as the HF
    tokenizer.  A batch may mix handles of several banks (e.g. passages of the train and the test split)."""

    def __init__(self, *banks: TokenBank):
        self.banks: dict[str, TokenBank] = {}
        for b in banks:
            self.add_bank(b)

    def add_bank(self, bank: TokenBank):
        have = self.banks.get(bank.prefix)
        if have is not None and have is not bank:
            raise ValueError(f"two different token banks share the handle prefix {bank.prefix!r}")
        self.banks[bank.prefix] = bank

    def add(self, other: "TokenBankTokenizer"):
        for b in other.banks.values():
            self.add_bank(b)

    def __call__(self, texts, padding=True, truncation=True, return_tensors="pt", max_length=512):
        prefixes = [t.split(":", 1)[0] for t in texts]
        idx = np.fromiter((int(t.split(":", 1)[1]) for t in texts), dtype=np.int64, count=len(texts))
        if all(p == prefixes[0] for p in prefixes):
            tb = self.banks[prefixes[0]].batch(idx, max_length=max_length)
            ids, mask = tb.input_ids, tb.attention_mask
        else:  # mixed banks: resolve each group, then pad to the batch max like padding=True does
            groups: dict[str, list[int]] = {}
            for pos, p in enumerate(prefixes):
                groups.setdefault(p, []).append(pos)
            parts = {p: self.banks[p].batch(idx[rows], max_length=max_length) for p, rows in groups.items()}
            L = max(tb.input_ids.shape[1] for tb in parts.values())
            ids = torch.zeros(len(texts), L, dtype=torch.int64)
            mask = torch.zeros(len(texts), L, dtype=torch.int64)
            for p, rows in groups.items():
                tb = parts[p]
                ids[rows, : tb.input_ids.shape[1]] = tb.input_ids.to(torch.int64)
                mask[rows, : tb.input_ids.shape[1]] = tb.attention_mask.to(torch.int64)
        return {"input_ids": ids, "token_type_ids": torch.zeros_like(ids), "attention_mask": mask}


# --------------------------------------------------------------------------------------------------
# pooled banks: the frozen front end of a tower, computed once per text
# --------------------------------------------------------------------------------------------------
def backbone_identity(tower) -> tuple:
    """What a pooled row depends on besides the text: the MiniLM weights (`MiniLMBackbone._key()`: device, tensor
    versions and addresses) or the token table's version and address.  A bank built under one identity is stale
    under any other."""
    bb = tower.pretrained_model
    if hasattr(bb, "_key"):
        return ("minilm",) + tuple(bb._key())
    t = bb.table
    return ("table", str(t.device), t._version, t.data_ptr())


def plan_length_batches(lengths: np.ndarray, max_tokens: int) -> list[np.ndarray]:
    """Indices of `lengths` sorted by length (stable) and cut into consecutive batches whose padded size
    (count x longest) stays within max_tokens; a text longer than max_tokens forms a batch of its own."""
    lengths = np.maximum(np.asarray(lengths, dtype=np.int64), 1)
    order = np.argsort(lengths, kind="stable")
    batches, start = [], 0
    n = len(order)
    while start < n:
        end = start + 1
        # sorted ascending: the batch [start, end) is padded to lengths[order[end - 1]]
        while end < n and (end + 1 - start) * int(lengths[order[end]]) <= max_tokens:
            end += 1
        batches.append(order[start:end])
        start = end
    return batches


class PooledBank:
    """Pooled rows of every text of one TokenBank for one tower: rows [n_texts, H] fp32 on the device, row r =
    F.normalize(masked_mean(backbone(text r truncated to L))), and the backbone identity they were computed under.
    Only valid while the backbone is frozen and unchanged (`check`)."""

    def __init__(self, rows: torch.Tensor, identity: tuple, L: int):
        self.rows, self.identity, self.L = rows, identity, int(L)

    def __len__(self):
        return self.rows.shape[0]

    def check(self, tower, what: str = "pooled bank"):
        if backbone_identity(tower) != self.identity:
            raise RuntimeError(f"{what} is stale: the tower's backbone changed after the bank was built; rebuild it "
                               "with PooledBank.build()")

    @staticmethod
    def encode_rows(tower, bank: TokenBank, L: int, lo: int, hi: int,
                    max_tokens_per_call: Optional[int] = None) -> torch.Tensor:
        """Pooled rows [hi - lo, H] of texts lo .. hi-1 of `bank` (truncated to L tokens) by `tower.pooled`, in
        length-sorted batches of at most max_tokens_per_call tokens, each padded only to its own longest text."""
        dev = tower.pretrained_model.device
        if max_tokens_per_call is None:
            max_tokens_per_call = getattr(tower.pretrained_model, "max_tokens_per_call", 1 << 17)
        mine = np.arange(lo, hi, dtype=np.int64)
        out = torch.empty(hi - lo, tower.embedding_dim, dtype=torch.float32, device=dev)
        lens = np.minimum(bank.lengths(mine), L)
        with torch.no_grad():
            for part in plan_length_batches(lens, int(max_tokens_per_call)):
                tb = bank.batch(mine[part], max_length=L)
                out[torch.from_numpy(part).to(dev)] = tower.pooled(tb.to(dev))
        return out

    @classmethod
    def build(cls, tower, bank: TokenBank, L: int, max_tokens_per_call: Optional[int] = None, world_size: int = 1,
              rank: int = 0, process_group=None) -> "PooledBank":
        """Encodes every text of `bank` (encode_rows).  With world_size > 1 rank r encodes its retrieval.shard_bounds
        slice and one all_gather_into_tensor assembles the bank, so every rank holds the same bits (a collective;
        process_group None = the default group)."""
        try:
            from .retrieval import shard_bounds
        except ImportError:
            from retrieval import shard_bounds
        identity = backbone_identity(tower)
        dev = tower.pretrained_model.device
        H = tower.embedding_dim
        n = len(bank)
        lo, hi = shard_bounds(n, world_size, rank)
        local = cls.encode_rows(tower, bank, L, lo, hi, max_tokens_per_call)
        if world_size == 1:
            return cls(local, identity, L)
        import torch.distributed as dist

        sizes = [shard_bounds(n, world_size, r) for r in range(world_size)]
        m = max(h - l_ for l_, h in sizes)
        padded = torch.zeros(m, H, dtype=torch.float32, device=dev)
        padded[: hi - lo] = local
        everything = torch.empty(world_size * m, H, dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(everything, padded, group=process_group)
        rows = torch.cat([everything[r * m: r * m + (h - l_)] for r, (l_, h) in enumerate(sizes)], dim=0)
        return cls(rows, identity, L)


# --------------------------------------------------------------------------------------------------
# dataset
# --------------------------------------------------------------------------------------------------
class MSMarcoDataset(torch.utils.data.Dataset):
    """MS MARCO query-passage pairs (backend/data.py:13-87).  `synthetic=None` tries the real dataset and
    falls back to the synthetic corpus when it cannot be loaded (no network)."""

    def __init__(self, split: str = "train", max_samples: int = 10_000, random_seed: int = 42,
                 synthetic: Optional[bool] = None, passages_per_query: float = 8.2) -> None:
        if max_samples < -1 or max_samples == 0:
            raise ValueError("max_samples must be -1 (use full dataset) or > 0 (limit to that many samples)")
        self.split = split
        self.query_bank = self.doc_bank = None
        self.data: list[MsMarcoDatasetItem] = []
        self.docs: list[str] = []
        if synthetic is None:
            synthetic = os.environ.get("HF_HUB_OFFLINE", "0") == "1" or os.environ.get("TT_SYNTHETIC_DATA") == "1"
        if not synthetic:
            try:
                self._load_real(split, max_samples, random_seed)
                return
            except Exception as e:  # noqa: BLE001
                print(f"MS MARCO not reachable ({type(e).__name__}); using the synthetic corpus instead")
        self._build_synthetic(split, max_samples, random_seed, passages_per_query)

    def _load_real(self, split, max_samples, random_seed):
        from datasets import load_dataset

        ds = load_dataset("microsoft/ms_marco", "v1.1", split=split)
        g = torch.Generator()
        g.manual_seed(random_seed)
        seen, count = set(), 0
        for idx in torch.randperm(len(ds), generator=g).tolist():
            item = ds[idx]
            for doc in item["passages"]["passage_text"]:
                if doc.strip():
                    self.data.append({"query_id": int(item["query_id"]), "query": str(item["query"]),
                                      "positive": str(doc)})
                    seen.add(str(doc))
                    count += 1
                    if 0 < max_samples <= count:
                        break
            if 0 < max_samples <= count:
                break
        self.docs = list(seen)

    def _build_synthetic(self, split, max_samples, random_seed, ppq):
        n_pairs = max_samples if max_samples > 0 else {"train": 676_193, "validation": 82_360, "test": 79_704}.get(split, 100_000)
        seed = random_seed + {"train": 0, "validation": 1, "test": 2}.get(split, 3) * 1000
        rng = np.random.default_rng(seed)
        n_queries = max(2, int(math.ceil(n_pairs / ppq)))
        # passages per query ~ 1 + Poisson, truncated so that the total is n_pairs
        per = 1 + rng.poisson(ppq - 1, n_queries)
        cum = np.cumsum(per)
        n_queries = int(np.searchsorted(cum, n_pairs) + 1)
        per = per[:n_queries]
        per[-1] -= int(per.sum() - n_pairs)
        if per[-1] <= 0:
            per = per[:-1]
            per[-1] += n_pairs - int(per.sum())
        n_docs = int(per.sum())
        self.query_bank = TokenBank.synthetic(f"{split}.q", len(per), "query", seed + 1)
        self.doc_bank = TokenBank.synthetic(f"{split}.d", n_docs, "doc", seed + 2)
        d = 0
        for qi, c in enumerate(per):
            for _ in range(int(c)):
                self.data.append({"query_id": qi, "query": self.query_bank.handle(qi),
                                  "positive": self.doc_bank.handle(d)})
                d += 1
        self.docs = [self.doc_bank.handle(i) for i in range(n_docs)]
        print(f"Built synthetic {split} dataset with {len(self.data)} query-document pairs, "
              f"including {len(self.docs)} unique passages")

    def tokenizer(self) -> Optional[TokenBankTokenizer]:
        return TokenBankTokenizer(self.query_bank, self.doc_bank) if self.query_bank is not None else None

    def __len__(self) -> int:
        return len(self.data)

    def __getitem__(self, idx: int) -> MsMarcoDatasetItem:
        return self.data[idx]

    def get_unique_passages(self) -> list[str]:
        return self.docs


# --------------------------------------------------------------------------------------------------
# triplet batching
# --------------------------------------------------------------------------------------------------
def sample_negative_indices(query_ids: np.ndarray, rng: np.random.Generator) -> np.ndarray:
    """For each i a j != i with query_ids[j] != query_ids[i], uniform over the eligible j — the accepted
    distribution of the rejection loop at backend/data.py:124-137 — vectorised.  Raises on a batch where
    some item has no eligible partner (the reference loops forever there)."""
    n = len(query_ids)
    j = rng.integers(0, n, n)
    for _ in range(64):
        bad = (j == np.arange(n)) | (query_ids[j] == query_ids)
        if not bad.any():
            return j
        j[bad] = rng.integers(0, n, int(bad.sum()))
    raise ValueError("batch has an item with no in-batch negative (all query_ids equal)")


class TripletDataLoader:
    """Creates triplets for training with random in-batch negative sampling (backend/data.py:90-152)."""

    def __init__(self, dataset, batch_size: int = 1024, num_workers: int = 4, device=None, seed: Optional[int] = None):
        self.dataset = dataset
        self.batch_size = batch_size
        self.num_workers = num_workers  # texts are handles/strings: no worker processes needed
        self.device = device
        self.rng = np.random.default_rng(seed if seed is not None else random.randrange(2**31))

    def __len__(self):
        return (len(self.dataset) + self.batch_size - 1) // self.batch_size

    def create_triplets(self, batch: list[MsMarcoDatasetItem]) -> Triplet:
        qids = np.array([int(b["query_id"]) for b in batch])
        neg = sample_negative_indices(qids, self.rng)
        return ([b["query"] for b in batch], [b["positive"] for b in batch], [batch[j]["positive"] for j in neg])

    def __iter__(self) -> Iterator[Triplet]:
        order = self.rng.permutation(len(self.dataset))  # shuffle=True, data.py:105
        for s in range(0, len(order), self.batch_size):
            yield self.create_triplets([self.dataset[int(i)] for i in order[s: s + self.batch_size]])


class TokenTripletLoader:
    """Token-level feeder for the fused step: shuffles pairs, samples in-batch negatives over the GLOBAL
    batch (SURVEY.md §8e), then hands this rank its contiguous slice as pinned, fixed-shape token tensors
    (ids int32, mask uint8, padded to Lq/Ld so CUDA-graph replays see one shape).

    rows=True yields the same batches as bank rows instead: an int32 [3, B] tensor of query-bank rows, document-bank
    rows of the positives and document-bank rows of the negatives (for a FusedTrainer over pooled banks)."""

    def __init__(self, dataset: MSMarcoDataset, global_batch: int, Lq: int = 32, Ld: int = 256, rank: int = 0,
                 world_size: int = 1, seed: int = 0, drop_last: bool = True, ids_dtype=torch.int32,
                 mask_dtype=torch.uint8, rows: bool = False):
        assert dataset.query_bank is not None, "TokenTripletLoader needs a token-bank dataset"
        assert global_batch % world_size == 0
        self.ds, self.gb, self.Lq, self.Ld = dataset, global_batch, Lq, Ld
        self.rank, self.world = rank, world_size
        self.rng = np.random.default_rng(seed)  # same seed on every rank -> same global batches
        self.drop_last = drop_last
        self.rows = bool(rows)
        self.ids_dtype, self.mask_dtype = ids_dtype, mask_dtype
        self.q_idx = np.array([int(d["query"].split(":")[1]) for d in dataset.data], dtype=np.int64)
        self.d_idx = np.array([int(d["positive"].split(":")[1]) for d in dataset.data], dtype=np.int64)
        self.qid = np.array([int(d["query_id"]) for d in dataset.data], dtype=np.int64)

    def __len__(self):
        n = len(self.ds)
        return n // self.gb if self.drop_last else (n + self.gb - 1) // self.gb

    def __iter__(self):
        order = self.rng.permutation(len(self.ds))
        per = self.gb // self.world
        for s in range(0, len(order) - (self.gb - 1 if self.drop_last else 0), self.gb):
            g = order[s: s + self.gb]
            neg = g[sample_negative_indices(self.qid[g], self.rng)]
            mine = slice(self.rank * per, (self.rank + 1) * per)
            if self.rows:
                rows = np.stack([self.q_idx[g[mine]], self.d_idx[g[mine]], self.d_idx[neg[mine]]]).astype(np.int32)
                yield torch.from_numpy(rows)
                continue
            kw = dict(ids_dtype=self.ids_dtype, mask_dtype=self.mask_dtype, pin=True)
            yield (self.ds.query_bank.batch(self.q_idx[g[mine]], self.Lq, self.Lq, **kw),
                   self.ds.doc_bank.batch(self.d_idx[g[mine]], self.Ld, self.Ld, **kw),
                   self.ds.doc_bank.batch(self.d_idx[neg[mine]], self.Ld, self.Ld, **kw))


def exclusion_csr(pair_q: np.ndarray, pair_d: np.ndarray, pair_qid: np.ndarray, n_rows: int):
    """Positives of every query-bank row as CSR (offsets int64 [n_rows + 1], ids int32 sorted and unique per row).
    Row r excludes every pair_d[i] whose pair_qid[i] is the query id of some pair naming row r: the in-batch draw's
    rule ("a different query_id") applied to mined passages."""
    pair_q, pair_d = np.asarray(pair_q, dtype=np.int64), np.asarray(pair_d, dtype=np.int64)
    _, qid = np.unique(np.asarray(pair_qid), return_inverse=True)  # query ids renumbered 0 .. n_qid-1
    qid = qid.reshape(-1).astype(np.int64)
    n_qid, n_d = int(qid.max(initial=-1)) + 1, max(int(pair_d.max(initial=-1)) + 1, 1)
    # the pairs grouped by query id: group g is by_qid[starts[g] : starts[g + 1]]
    by_qid = np.argsort(qid, kind="stable")
    starts = np.searchsorted(qid[by_qid], np.arange(n_qid + 1))
    # every distinct (row, query id), expanded to every passage of that query id
    rq = np.unique(pair_q * max(n_qid, 1) + qid)
    rows, groups = rq // max(n_qid, 1), rq % max(n_qid, 1)
    per = starts[groups + 1] - starts[groups]
    within = np.arange(int(per.sum())) - np.repeat(np.cumsum(per) - per, per)
    passages = pair_d[by_qid[np.repeat(starts[groups], per) + within]]
    keys = np.unique(np.repeat(rows, per) * n_d + passages)  # sorted by row, then passage
    counts = np.bincount(keys // n_d, minlength=n_rows)[:n_rows]
    return np.concatenate([[0], np.cumsum(counts)]).astype(np.int64), (keys % n_d).astype(np.int32)


class HardNegativeMiner:
    """Hard negatives for DeviceTripletFeeder, mined with the exact corpus scan from the current towers (DPR / ANCE):
    for every query-bank row, the passages the towers rank highest that are not its positives.

    refresh(model) projects every pooled row of both banks with the current weights, ranks all passages for all
    queries with the tensor-core scan (this rank's document shard, then the merge every data-parallel rank ends
    identical on), drops each query's positives and the first `skip` survivors and keeps the next `depth` in rank
    order (tt_mine_negatives).  The table lives in static device buffers; a feeder with `hard_negatives = miner` then
    gives each item a mined negative with probability `ratio` (tt_assemble_*_mined).  The table is a function of the
    weights, so a checkpoint needs no extra state.  Needs frozen backbones: the banks hold their pooled rows."""

    def __init__(self, dataset: MSMarcoDataset, bank_q: "PooledBank", bank_d: "PooledBank", depth: int = 8,
                 skip: int = 0, ratio: float = 0.5, k_scan: int = 32, world_size: int = 1, rank: int = 0,
                 process_group=None):
        self.depth, self.skip, self.ratio, self.k_scan = self.check_config(depth, skip, ratio, k_scan)
        if dataset.query_bank is None:
            raise ValueError("HardNegativeMiner needs a token-bank dataset")
        if (len(bank_q), len(bank_d)) != (len(dataset.query_bank), len(dataset.doc_bank)):
            raise ValueError(f"HardNegativeMiner: the pooled banks hold {len(bank_q)} / {len(bank_d)} rows, the "
                             f"dataset's token banks {len(dataset.query_bank)} / {len(dataset.doc_bank)}; build them "
                             "from the same dataset")
        self.bank_q, self.bank_d = bank_q, bank_d
        self.world, self.rank, self.pg = int(world_size), int(rank), process_group
        pq = np.array([int(d["query"].split(":")[1]) for d in dataset.data], dtype=np.int64)
        pd = np.array([int(d["positive"].split(":")[1]) for d in dataset.data], dtype=np.int64)
        qid = np.array([int(d["query_id"]) for d in dataset.data], dtype=np.int64)
        self.n_rows, self.n_docs = len(bank_q), len(bank_d)
        off, ids = exclusion_csr(pq, pd, qid, self.n_rows)
        dev = bank_q.rows.device
        self.excl_offsets = torch.from_numpy(off).to(dev)
        self.excl_ids = torch.from_numpy(ids).to(dev)
        self.table = torch.full((self.n_rows, self.depth), -1, dtype=torch.int32, device=dev)
        self.count = torch.zeros(self.n_rows, dtype=torch.int32, device=dev)
        self.refreshed = False

    @staticmethod
    def check_config(depth, skip, ratio, k_scan):
        depth, skip, k_scan, ratio = int(depth), int(skip), int(k_scan), float(ratio)
        if not 1 <= k_scan <= 32:
            raise ValueError(f"HardNegativeMiner: k_scan = {k_scan}; the corpus scan keeps at most 32 per query")
        if depth < 1 or skip < 0 or skip + depth > k_scan:
            raise ValueError(f"HardNegativeMiner: need depth >= 1, skip >= 0 and skip + depth <= k_scan (depth {depth}, "
                             f"skip {skip}, k_scan {k_scan})")
        if not 0.0 <= ratio <= 1.0:
            raise ValueError(f"HardNegativeMiner: ratio = {ratio} is a probability, outside [0, 1]")
        return depth, skip, ratio, k_scan

    def _check_towers(self, model):
        qt, dt = model.query_tower, model.document_tower
        if any(p.requires_grad for t in (qt, dt) for p in t.pretrained_model.parameters()):
            raise ValueError("HardNegativeMiner needs frozen backbones: the pooled banks of a trainable table go stale "
                             "at the first step")
        self.bank_q.check(qt, "the query tower's pooled bank")
        self.bank_d.check(dt, "the document tower's pooled bank")

    @staticmethod
    def _project(tower, rows: torch.Tensor, chunk: int = 1 << 16) -> torch.Tensor:
        p0, p2 = tower.projection[0], tower.projection[2]
        out = torch.empty(rows.shape[0], p0.out_features, dtype=torch.float32, device=rows.device)
        with torch.no_grad():
            for s in range(0, rows.shape[0], chunk):
                out[s: s + chunk] = ops.mlp(rows[s: s + chunk], p0.weight, p0.bias, p2.weight, p2.bias, tower.precision)
        return out

    def local_lists(self, model, events=None):
        """Top-k_scan (scores, global ids) of every query over this rank's document shard (id_base = lo)."""
        try:
            from .retrieval import shard_bounds
        except ImportError:
            from retrieval import shard_bounds
        self._check_towers(model)
        ev = events if events is not None else {}
        mark = lambda name: ev.setdefault(name, torch.cuda.Event(enable_timing=True)).record()  # noqa: E731
        lo, hi = shard_bounds(self.n_docs, self.world, self.rank)
        mark("start")
        yq = self._project(model.query_tower, self.bank_q.rows)
        yd = self._project(model.document_tower, self.bank_d.rows[lo:hi])
        mark("project")
        Qn, Qb = ops.l2_normalize_rows(yq, want_bf16=True)
        Dn, Db = ops.l2_normalize_rows(yd, want_bf16=True)
        del yq, yd
        mark("normalize")
        if hi > lo:
            top = ops.scan_topk(Qn, Dn, k=self.k_scan, id_base=lo, precision="bf16", Qb=Qb, Db=Db)
        else:  # an empty shard (more ranks than passages)
            top = (torch.full((self.n_rows, self.k_scan), -math.inf, device=Qn.device),
                   torch.full((self.n_rows, self.k_scan), -1, dtype=torch.int64, device=Qn.device))
        mark("scan")
        return top

    def filter(self, top_id: torch.Tensor):
        """Merged lists [n_rows, k_scan] -> the table and counts (tt_mine_negatives), in place."""
        ops.mine_negatives(top_id, self.excl_offsets, self.excl_ids, self.skip, self.depth, self.table, self.count)
        self.refreshed = True

    def refresh(self, model) -> dict:
        """Re-mines the table from the model's current weights (current stream; ends in a host sync).  Returns the
        seconds of each phase (device events) and the table's mean count and number of empty rows."""
        try:
            from .retrieval import gather_and_merge
        except ImportError:
            from retrieval import gather_and_merge
        ev = {}
        top_s, top_i = self.local_lists(model, ev)
        top_s, top_i = gather_and_merge(top_s, top_i, self.world, self.pg)
        ev.setdefault("merge", torch.cuda.Event(enable_timing=True)).record()
        self.filter(top_i)
        ev.setdefault("filter", torch.cuda.Event(enable_timing=True)).record()
        del top_s, top_i
        ev["filter"].synchronize()
        names = ["start", "project", "normalize", "scan", "merge", "filter"]
        stats = {f"{b}_s": ev[a].elapsed_time(ev[b]) / 1e3 for a, b in zip(names, names[1:])}
        stats["total_s"] = ev["start"].elapsed_time(ev["filter"]) / 1e3
        cnt = self.count.double()
        stats["mean_count"] = float(cnt.mean()) if self.n_rows else 0.0
        stats["empty_queries"] = int((self.count == 0).sum())
        return stats

    def descriptor(self):
        """tt_mined_negatives of the current table (ctypes), or None before the first refresh."""
        if not self.refreshed:
            return None
        try:
            from . import _native as N
        except ImportError:
            import _native as N
        return N.MinedNegatives(self.table.data_ptr(), self.count.data_ptr(), self.depth, self.n_rows, self.n_docs,
                                self.ratio)


class DeviceTripletFeeder:
    """Batch assembly on the device (SURVEY.md §8f rank 1): the tokenised dataset lives in HBM as two ragged token
    banks; every step ONE kernel (`tt_assemble_triplets`) turns a slice of the epoch permutation into the six padded
    token tensors of a FusedTrainer slot and draws the in-batch negatives (same rule as backend/data.py:124-137) — no
    host work and no H2D traffic per step.  Under data parallelism every rank holds the banks, uses the same epoch
    permutation (same seed) and assembles only its slice of the global batch; the negatives are a pure function of
    (seed, position in the global batch), so the ranks agree without communicating.

    rows_only=True: the feeder serves only trainers over pooled banks (bank rows, `tt_assemble_triplet_rows`) and does
    not upload the token banks."""

    def __init__(self, dataset: MSMarcoDataset, global_batch: int, Lq: int = 32, Ld: int = 256, device="cuda",
                 rank: int = 0, world_size: int = 1, seed: int = 0, drop_last: bool = True, rows_only: bool = False):
        assert dataset.query_bank is not None, "DeviceTripletFeeder needs a token-bank dataset"
        assert global_batch % world_size == 0 and global_batch >= 2
        try:
            from . import _native as N
        except ImportError:
            import _native as N
        self.N = N
        N.ensure_sm100()
        self.device = torch.device(device)
        self.gb, self.Lq, self.Ld = int(global_batch), int(Lq), int(Ld)
        self.rank, self.world, self.seed = int(rank), int(world_size), int(seed)
        self.per = self.gb // self.world
        if not drop_last:
            raise ValueError("DeviceTripletFeeder assembles fixed-shape batches only (drop_last=True)")

        def upload(bank: TokenBank):
            small = int(bank.flat.max(initial=0)) < 65536
            flat = torch.from_numpy(bank.flat.astype(np.uint16 if small else np.int32)).to(self.device)
            off = torch.from_numpy(bank.offsets.astype(np.int64)).to(self.device)
            desc = N.TokenBankDesc(flat.data_ptr(), off.data_ptr(), N.dtype_code(flat), 0)
            return flat, off, desc

        self.rows_only = bool(rows_only)
        if not self.rows_only:
            self.q_flat, self.q_off, self.q_desc = upload(dataset.query_bank)
            self.d_flat, self.d_off, self.d_desc = upload(dataset.doc_bank)
        as_dev = lambda a: torch.from_numpy(np.asarray(a, dtype=np.int32)).to(self.device)  # noqa: E731
        self.pair_q = as_dev([int(d["query"].split(":")[1]) for d in dataset.data])
        self.pair_d = as_dev([int(d["positive"].split(":")[1]) for d in dataset.data])
        self.pair_qid = as_dev([int(d["query_id"]) for d in dataset.data])
        self.n = len(dataset.data)
        self.gen = torch.Generator(device=self.device).manual_seed(self.seed)
        self.err = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.neg = torch.zeros(self.per, dtype=torch.int32, device=self.device)
        self.order = None
        self.epoch = 0
        self.n_rows, self.n_docs = len(dataset.query_bank), len(dataset.doc_bank)
        # a HardNegativeMiner: once its table is refreshed, items draw mined negatives (tt_assemble_*_mined)
        self.hard_negatives: Optional[HardNegativeMiner] = None

    def __len__(self):
        return self.n // self.gb

    def start_epoch(self):
        """New shuffle (DataLoader(shuffle=True), data.py:105); the same on every rank because the seed is."""
        self.order = torch.randperm(self.n, generator=self.gen, device=self.device).to(torch.int32)
        self.epoch += 1

    def assemble(self, trainer, slot: int, step: int, want_neg: bool = False):
        """Fills trainer.tok_slots[slot] with the batch of `step` (asynchronous, current stream)."""
        N = self.N
        assert self.order is not None, "call start_epoch() first"
        assert 0 <= step < len(self)
        order = self.order[step * self.gb: (step + 1) * self.gb]
        step_seed = (self.seed * 0x9E3779B1 + self.epoch * 0x85EBCA77 + step) & 0xFFFFFFFFFFFFFFFF
        mined = self._mined_descriptor(trainer)
        row_bufs = getattr(trainer, "row_bufs", None)
        if row_bufs is not None:
            # a trainer over pooled banks takes bank rows (same items, same negatives as the token path would give)
            args = (N.ptr(self.pair_q), N.ptr(self.pair_d), N.ptr(self.pair_qid), order.data_ptr(), self.gb,
                    self.rank * self.per, self.per, step_seed, N.ptr(row_bufs[slot]),
                    N.ptr(self.neg) if want_neg else None, N.ptr(self.err))
            if mined is None:
                N.check(N.load().tt_assemble_triplet_rows(*args, N.stream()), "tt_assemble_triplet_rows")
            else:
                N.check(N.load().tt_assemble_triplet_rows_mined(*args, ctypes.byref(mined), N.stream()),
                        "tt_assemble_triplet_rows_mined")
            trainer._rows_loaded[slot] = True
            return
        if self.rows_only:
            raise RuntimeError("DeviceTripletFeeder(rows_only=True) holds no token banks: it feeds trainers over pooled "
                               "banks only")
        q_ids, q_mask, p_ids, p_mask, n_ids, n_mask = trainer.tok_slots[slot]
        assert tuple(q_ids.shape) == (self.per, self.Lq) and tuple(p_ids.shape) == (self.per, self.Ld)
        # a trainer that reuses the positives' pooled rows for the in-batch negatives wants their indices in its slot
        neg_bufs = getattr(trainer, "neg_bufs", None)
        neg_ptr = N.ptr(neg_bufs[slot]) if neg_bufs is not None else (N.ptr(self.neg) if want_neg else None)
        if neg_bufs is not None:
            trainer._neg_loaded[slot] = True
        args = (ctypes.byref(self.q_desc), ctypes.byref(self.d_desc), N.ptr(self.pair_q), N.ptr(self.pair_d),
                N.ptr(self.pair_qid), order.data_ptr(), self.gb, self.rank * self.per, self.per, step_seed, self.Lq,
                self.Ld, N.ptr(q_ids), N.ptr(q_mask), N.ptr(p_ids), N.ptr(p_mask), N.ptr(n_ids), N.ptr(n_mask),
                N.dtype_code(q_ids), N.dtype_code(q_mask), neg_ptr, N.ptr(self.err))
        if mined is None:
            N.check(N.load().tt_assemble_triplets(*args, N.stream()), "tt_assemble_triplets")
        else:
            N.check(N.load().tt_assemble_triplets_mined(*args, ctypes.byref(mined), N.stream()),
                    "tt_assemble_triplets_mined")

    def _mined_descriptor(self, trainer):
        """tt_mined_negatives of the attached miner once it has a table, else None (in-batch negatives only)."""
        miner = self.hard_negatives
        if miner is None:
            return None
        if getattr(trainer, "neg_bufs", None) is not None:
            raise ValueError("a trainer built with in_batch_negatives=True cannot take mined negatives: a mined negative "
                             "is not a positive of the batch")
        if (miner.n_rows, miner.n_docs) != (self.n_rows, self.n_docs):
            raise ValueError(f"the miner's table covers {miner.n_rows} queries / {miner.n_docs} passages, the feeder's "
                             f"dataset {self.n_rows} / {self.n_docs}")
        return miner.descriptor()

    def check(self):
        """Host sync: raises if some item had no eligible in-batch negative (the reference would loop forever), or a
        mined negative was out of range."""
        err = int(self.err.item())
        if err == 3:
            raise ValueError("a mined negative or its query row was outside the banks")
        if err != 0:
            raise ValueError("batch has an item with no in-batch negative (all query_ids equal)")
