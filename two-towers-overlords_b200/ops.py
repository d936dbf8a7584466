"""
Host-side operators over the C ABI: thin wrappers and autograd Functions so that `loss.backward()`,
`optimizer.step()` and `state_dict()` of the reference's training loop (backend/training.py:36-53)
keep working on ordinary nn.Parameters while all arithmetic runs in libtt_b200.so.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

try:
    from . import _native as N
except ImportError:  # imported as a top-level module (drop-in mode: this directory on sys.path)
    import _native as N


def default_precision(H: int, P: int) -> str:
    env = os.environ.get("TT_PRECISION")
    if env:
        return env
    return "bf16x3" if (H % 64 == 0 and P % 64 == 0) else "fp32"


def _prec(p) -> int:
    return N.PRECISIONS[p] if isinstance(p, str) else int(p)


def _tokens(ids: torch.Tensor, mask: Optional[torch.Tensor], device) -> tuple[torch.Tensor, torch.Tensor]:
    """Token tensors as the kernels take them: contiguous [B,L] on `device`, ids i64|i32|u16, mask i64|i32|u8."""
    if mask is None:
        mask = torch.ones_like(ids, dtype=torch.uint8)
    if ids.dtype not in (torch.int64, torch.int32, torch.uint16, torch.int16):
        ids = ids.to(torch.int64)
    if mask.dtype == torch.bool:
        mask = mask.to(torch.uint8)
    elif mask.dtype not in (torch.int64, torch.int32, torch.uint8):
        mask = mask.to(torch.int64)
    if ids.dim() != 2 or ids.shape != mask.shape:
        raise ValueError(f"ids/mask must be [B,L] of equal shape, got {tuple(ids.shape)} / {tuple(mask.shape)}")
    return (ids.to(device, non_blocking=True).contiguous(), mask.to(device, non_blocking=True).contiguous())


# --------------------------------------------------------------------------------------------------
# pooled gather (model.py:48-56,63-72)
# --------------------------------------------------------------------------------------------------
def pool_forward(table: torch.Tensor, ids: torch.Tensor, mask: Optional[torch.Tensor]):
    """-> (xhat [B,H] f32, cnt [B], nrm [B]).  Raises IndexError on an out-of-range unmasked id."""
    N.ensure_sm100()
    N.require_device(table)
    ids, mask = _tokens(ids, mask, table.device)
    B, L = ids.shape
    V, H = table.shape
    xhat = torch.empty(B, H, dtype=torch.float32, device=table.device)
    cnt = torch.empty(B, dtype=torch.float32, device=table.device)
    nrm = torch.empty(B, dtype=torch.float32, device=table.device)
    err = torch.zeros(1, dtype=torch.int32, device=table.device)
    if B > 0:
        if L == 0:
            xhat.zero_(); cnt.zero_(); nrm.zero_()
        else:
            N.check(N.load().tt_pool_fwd(N.ptr(table), N.dtype_code(table), V, H, N.ptr(ids), N.dtype_code(ids),
                                         N.ptr(mask), N.dtype_code(mask), B, L, N.ptr(xhat), N.ptr(cnt), N.ptr(nrm),
                                         N.ptr(err), N.stream()), "tt_pool_fwd")
    return xhat, cnt, nrm, err, ids, mask


class _PoolFn(torch.autograd.Function):
    """Trainable-table variant (SURVEY.md D2): backward is the sorted-segment scatter-add."""

    @staticmethod
    def forward(ctx, table, ids, mask):
        xhat, cnt, nrm, err, ids, mask = pool_forward(table.detach(), ids, mask)
        ctx.save_for_backward(xhat, cnt, nrm, ids, mask)
        ctx.table_shape = tuple(table.shape)
        ctx.err = err
        return xhat

    @staticmethod
    def backward(ctx, dxhat):
        xhat, cnt, nrm, ids, mask = ctx.saved_tensors
        V, H = ctx.table_shape
        B, L = ids.shape
        dxhat = dxhat.contiguous().float()
        dtable = torch.empty(V, H, dtype=torch.float32, device=xhat.device)
        lib = N.load()
        ws_bytes = lib.tt_pool_bwd_ws_bytes(B, L, V, H)
        ws = N.workspace(ws_bytes, xhat.device)
        N.check(lib.tt_pool_bwd(N.ptr(dxhat), N.ptr(xhat), N.ptr(cnt), N.ptr(nrm), N.ptr(ids), N.dtype_code(ids),
                                N.ptr(mask), N.dtype_code(mask), B, L, V, H, N.ptr(dtable), 0, N.ptr(ws), ws_bytes,
                                N.stream()), "tt_pool_bwd")
        return dtable, None, None


def pool(table: torch.Tensor, ids, mask, check_ids: bool = False) -> torch.Tensor:
    if table.requires_grad and torch.is_grad_enabled():
        if table.dtype != torch.float32:
            raise ValueError("a trainable token table must be fp32")
        return _PoolFn.apply(table, ids, mask)
    xhat, _, _, err, _, _ = pool_forward(table.detach(), ids, mask)
    if check_ids and int(err.item()) != 0:
        raise IndexError("token id out of range of the embedding table")
    return xhat


# --------------------------------------------------------------------------------------------------
# projection MLP (model.py:33-38,59)
# --------------------------------------------------------------------------------------------------
class _MlpFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, W1, b1, W2, b2, precision):
        N.ensure_sm100()
        x = x.contiguous().float()
        M, H = x.shape
        P = W1.shape[0]
        W1c, b1c, W2c, b2c = (t.detach().contiguous().float() for t in (W1, b1, W2, b2))
        h = torch.empty(M, P, dtype=torch.float32, device=x.device)
        y = torch.empty(M, P, dtype=torch.float32, device=x.device)
        lib = N.load()
        prec = _prec(precision)
        ws_bytes = lib.tt_mlp_ws_bytes(M, H, P, prec)
        ws = N.workspace(ws_bytes, x.device)
        N.check(lib.tt_encode_fwd(N.ptr(x), M, H, P, N.ptr(W1c), N.ptr(b1c), N.ptr(W2c), N.ptr(b2c), N.ptr(h),
                                  N.ptr(y), prec, N.ptr(ws), ws_bytes, N.stream()), "tt_encode_fwd")
        ctx.save_for_backward(x, h, W1c, W2c)
        ctx.prec = prec
        ctx.need_dx = x.requires_grad
        return y

    @staticmethod
    def backward(ctx, dy):
        x, h, W1, W2 = ctx.saved_tensors
        M, H = x.shape
        P = W1.shape[0]
        dy = dy.contiguous().float()
        dev = x.device
        dW1 = torch.empty(P, H, dtype=torch.float32, device=dev)
        db1 = torch.empty(P, dtype=torch.float32, device=dev)
        dW2 = torch.empty(P, P, dtype=torch.float32, device=dev)
        db2 = torch.empty(P, dtype=torch.float32, device=dev)
        dx = torch.empty(M, H, dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        lib = N.load()
        ws_bytes = lib.tt_mlp_ws_bytes(M, H, P, ctx.prec)
        ws = N.workspace(ws_bytes, dev)
        N.check(lib.tt_encode_bwd(N.ptr(dy), N.ptr(x), N.ptr(h), N.ptr(W1), N.ptr(W2), M, H, P, N.ptr(dW1), N.ptr(db1),
                                  N.ptr(dW2), N.ptr(db2), N.ptr(dx), 0, ctx.prec, N.ptr(ws), ws_bytes, N.stream()),
                "tt_encode_bwd")
        return dx, dW1, db1, dW2, db2, None


def mlp(x, W1, b1, W2, b2, precision="fp32") -> torch.Tensor:
    return _MlpFn.apply(x, W1, b1, W2, b2, precision)


# --------------------------------------------------------------------------------------------------
# triplet loss (model.py:132-145)
# --------------------------------------------------------------------------------------------------
class _TripletLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, p, n, margin, inv_batch):
        N.ensure_sm100()
        N.require_device(q)
        q, p, n = (t.contiguous().float() for t in (q, p, n))
        if not (q.shape == p.shape == n.shape and q.dim() == 2):
            raise ValueError("anchor/positive/negative must be [B,P] of equal shape")
        B, P = q.shape
        stats = torch.empty(B, 8, dtype=torch.float32, device=q.device)
        loss = torch.empty((), dtype=torch.float32, device=q.device)
        inv = (1.0 / B if B > 0 else float("nan")) if inv_batch is None else float(inv_batch)
        N.check(N.load().tt_triplet_loss_fwd(N.ptr(q), N.ptr(p), N.ptr(n), B, P, float(margin), inv, N.ptr(stats),
                                             N.ptr(loss), N.stream()), "tt_triplet_loss_fwd")
        ctx.save_for_backward(q, p, n, stats)
        ctx.inv = inv
        return loss

    @staticmethod
    def backward(ctx, dloss):
        q, p, n, stats = ctx.saved_tensors
        B, P = q.shape
        dq, dp, dn = (torch.empty_like(q) for _ in range(3))
        dl = dloss.contiguous().float().reshape(1)
        N.check(N.load().tt_triplet_loss_bwd(N.ptr(q), N.ptr(p), N.ptr(n), N.ptr(stats), N.ptr(dl), B, P, ctx.inv,
                                             N.ptr(dq), N.ptr(dp), N.ptr(dn), N.stream()), "tt_triplet_loss_bwd")
        return dq, dp, dn, None, None


def triplet_loss(q, p, n, margin: float, inv_batch: Optional[float] = None) -> torch.Tensor:
    return _TripletLossFn.apply(q, p, n, margin, inv_batch)


# --------------------------------------------------------------------------------------------------
# fused triplet step (training.py:37-50 without the optimiser)
# --------------------------------------------------------------------------------------------------
class TripletStep:
    """Pre-allocated workspace + argument block for tt_triplet_step; graph-capturable (no allocation,
    no host sync inside `run`)."""

    def __init__(self, B, Lq, Ld, H, P, vocab, precision, device, train_table=False):
        N.ensure_sm100()
        self.lib = N.load()
        self.shape = (B, Lq, Ld, H, P, vocab)
        self.prec = _prec(precision)
        self.train_table = bool(train_table)
        self.ws_bytes = self.lib.tt_step_ws_bytes(B, Lq, Ld, H, P, vocab, self.prec, int(self.train_table))
        self.ws = N.workspace(self.ws_bytes, device).zero_()  # tt_triplet_step wants a zero-filled workspace once
        self.loss = torch.zeros((), dtype=torch.float32, device=device)
        self.err = torch.zeros(1, dtype=torch.int32, device=device)
        self.args = N.StepArgs()
        self.slots = []
        self._keep = []
        self._adam = None
        self._table_adam = None
        self.chain = 0

    def bind(self, tokens, tables, params, grads, margin, inv_batch, grad_scale=1.0, table_grads=None):
        """tokens = (q_ids,q_mask,p_ids,p_mask,n_ids,n_mask) CUDA tensors; tables = (table_q, table_d);
        params / grads = 8 fp32 tensors in the order Wq1,bq1,Wq2,bq2,Wd1,bd1,Wd2,bd2.
        tokens and tables are None for a step that reads precomputed pooled rows only (bind_pooled)."""
        B, Lq, Ld, H, P, vocab = self.shape
        a = self.args
        a.Lq, a.Ld, a.B = Lq, Ld, B
        if tokens is not None:
            q_ids, q_mask, p_ids, p_mask, n_ids, n_mask = tokens
            assert tuple(q_ids.shape) == (B, Lq) and tuple(p_ids.shape) == (B, Ld) and tuple(n_ids.shape) == (B, Ld)
            assert q_ids.dtype == p_ids.dtype == n_ids.dtype and q_mask.dtype == p_mask.dtype == n_mask.dtype
            a.q_ids, a.q_mask = N.ptr(q_ids), N.ptr(q_mask)
            a.p_ids, a.p_mask = N.ptr(p_ids), N.ptr(p_mask)
            a.n_ids, a.n_mask = N.ptr(n_ids), N.ptr(n_mask)
            a.ids_dtype, a.mask_dtype = N.dtype_code(q_ids), N.dtype_code(q_mask)
        a.table_dtype, a.vocab, a.H, a.P = N.TT_F32, vocab, H, P
        if tables is not None:
            a.table_q, a.table_d = N.ptr(tables[0]), N.ptr(tables[1])
            assert tables[0].dtype == tables[1].dtype
            a.table_dtype = N.dtype_code(tables[0])
        for name, t in zip(("Wq1", "bq1", "Wq2", "bq2", "Wd1", "bd1", "Wd2", "bd2"), params):
            assert t.dtype == torch.float32
            setattr(a, name, N.ptr(t))
        for name, t in zip(("dWq1", "dbq1", "dWq2", "dbq2", "dWd1", "dbd1", "dWd2", "dbd2"), grads):
            assert t.dtype == torch.float32
            setattr(a, name, N.ptr(t))
        a.margin, a.inv_batch, a.grad_scale = float(margin), float(inv_batch), float(grad_scale)
        a.loss, a.err_flag = N.ptr(self.loss), N.ptr(self.err)
        if self.train_table:
            a.dtable_q, a.dtable_d = N.ptr(table_grads[0]), N.ptr(table_grads[1])
        else:
            a.dtable_q, a.dtable_d = None, None
        a.precision, a.ws, a.ws_bytes = self.prec, N.ptr(self.ws), self.ws_bytes
        a.adam_param = None
        a.chain = self.chain
        self.slots = [a]
        self._keep = [(tokens, tables, params, grads, table_grads)]

    def add_tokens(self, tokens) -> int:
        """Another token-buffer set sharing every other argument (rotating / double-buffered inputs);
        returns its slot index for run(slot).  tokens = None adds a slot of a pooled-row step (set_pooled_index)."""
        B, Lq, Ld = self.shape[:3]
        a = N.StepArgs.from_buffer_copy(self.args)
        a.pooled_index = None
        if tokens is not None:
            q_ids, q_mask, p_ids, p_mask, n_ids, n_mask = tokens
            assert tuple(q_ids.shape) == (B, Lq) and tuple(p_ids.shape) == (B, Ld) and tuple(n_ids.shape) == (B, Ld)
            assert N.dtype_code(q_ids) == a.ids_dtype and N.dtype_code(q_mask) == a.mask_dtype
            a.q_ids, a.q_mask = N.ptr(q_ids), N.ptr(q_mask)
            a.p_ids, a.p_mask = N.ptr(p_ids), N.ptr(p_mask)
            a.n_ids, a.n_mask = N.ptr(n_ids), N.ptr(n_mask)
        self.slots.append(a)
        self._keep.append(tokens)
        return len(self.slots) - 1

    def _views(self) -> dict:
        """fp32 activations of the last run inside the step workspace, rows q | p | n (the leading carves of
        carve_step_ws in csrc/tt_api.cu: 256-byte aligned, in this order).  Read-only views for the parity tests."""
        B, _, _, H, P = self.shape[:5]
        R = 3 * B
        assert self.ws.data_ptr() % 256 == 0
        out, off = {}, 0
        names = [("xhat", R, H), ("cnt", R, 1), ("nrm", R, 1), ("h", R, P), ("y", R, P), ("stats", B, 8), ("dy", R, P),
                 ("dz1", R, P)]
        if self.train_table:
            names += [("dxhat", R, H), ("g", R, H)]
        for name, rows, cols in names:
            off = (off + 255) // 256 * 256
            out[name] = self.ws[off: off + rows * cols * 4].view(torch.float32).view(rows, cols)
            off += rows * cols * 4
        return out

    def pooled_rows(self) -> torch.Tensor:
        """xhat [3B,H]: pooled + L2-normalised rows of the last run."""
        return self._views()["xhat"]

    def internal(self, name: str, rows: int, cols: int, dtype=torch.bfloat16) -> torch.Tensor:
        """View of a named internal buffer of a tensor-core step workspace (tt_debug_step_buffer)."""
        B, Lq, Ld, H, P, vocab = self.shape
        ptr = ctypes.c_void_p()
        N.check(self.lib.tt_debug_step_buffer(N.ptr(self.ws), B, Lq, Ld, H, P, vocab, self.prec, int(self.train_table),
                                              name.encode(), ctypes.byref(ptr)), "tt_debug_step_buffer")
        off = ptr.value - self.ws.data_ptr()
        nbytes = rows * cols * torch.empty((), dtype=dtype).element_size()
        return self.ws[off: off + nbytes].view(dtype).view(rows, cols)

    def set_neg_index(self, slot: int, neg_index: Optional[torch.Tensor]):
        """In-batch negatives for `slot` (tt_step_args.neg_index): int32 [B] on the device, negative row i is the same
        document as positive row neg_index[i]; its pooled row is then a copy instead of a second gather, and with table
        gradients its gradient row is folded into that positive's.  None: the negatives are gathered from their own
        token tensors."""
        a = self.slots[slot]
        if neg_index is None:
            a.neg_index = None
            return
        assert neg_index.dtype == torch.int32 and neg_index.is_cuda and tuple(neg_index.shape) == (self.shape[0],)
        a.neg_index = N.ptr(neg_index)
        self._keep.append(neg_index)

    def bind_pooled(self, rows_q: torch.Tensor, rows_d: torch.Tensor):
        """Frozen front end computed once per text (tt_step_args.pooled_*): fp32 [n, H] banks of pooled rows, one per
        tower.  Every slot then copies its 3B rows out of them by its index buffer (set_pooled_index) instead of
        pooling tokens; the static addresses keep captured graphs valid."""
        assert not self.train_table, "pooled rows need frozen tables"
        H = self.shape[3]
        for t in (rows_q, rows_d):
            assert t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 and t.shape[1] == H and t.shape[0] >= 1
            assert t.is_contiguous(), "pooled rows are read with a row stride of H: pass a contiguous bank"
        for a in self.slots:
            a.pooled_q, a.pooled_q_rows = N.ptr(rows_q), rows_q.shape[0]
            a.pooled_d, a.pooled_d_rows = N.ptr(rows_d), rows_d.shape[0]
        self._keep.append((rows_q, rows_d))

    def set_pooled_index(self, slot: int, index: torch.Tensor):
        """Bank rows of `slot` (tt_step_args.pooled_index): int32 [3B] on the device, query rows | positive rows |
        negative rows."""
        assert self.args.pooled_q is not None, "set_pooled_index needs bind_pooled() first"
        assert index.dtype == torch.int32 and index.is_cuda and tuple(index.shape) == (3 * self.shape[0],)
        self.slots[slot].pooled_index = N.ptr(index)
        self._keep.append(index)

    def set_chain(self, mode: int):
        """tt_step_args.chain: 0 = library default (TT_CHAIN env, else the persistent kernel), 1 = persistent chain
        kernel, 2 = one kernel per contraction."""
        self.chain = int(mode)
        for a in self.slots:
            a.chain = self.chain

    def chain_active(self) -> bool:
        """True when tt_triplet_step runs the persistent chain kernel for this step."""
        if self.prec == N.PRECISIONS["fp32"]:
            return False
        if self.chain:
            return self.chain == 1
        return os.environ.get("TT_CHAIN", "1") != "0"

    def hidden(self) -> torch.Tensor:
        """h [3B,P] fp32 of the last run.  The persistent chain kernel keeps h only as its bf16 terms (hi + lo)."""
        if self.chain_active() and os.environ.get("TT_CHAIN_FP32_OUT", "0") == "0":
            B, P = self.shape[0], self.shape[4]
            return self.internal("h_hi", 3 * B, P).float() + self.internal("h_lo", 3 * B, P).float()
        return self._views()["h"]

    def relu_gate(self) -> torch.Tensor:
        """bool [3B,P]: which hidden units the last run treated as active (h > 0) — the ReLU gate of its backward."""
        if self.chain_active():
            B, P = self.shape[0], self.shape[4]
            return self.internal("h_hi", 3 * B, P).float() > 0
        return self._views()["h"] > 0

    def bind_adam(self, state, param, grad, exp_avg, exp_avg_sq, lr, betas, eps):
        """Optional optimiser inside the step call (tt_step_args.adam_*): flat fp32 buffers the 8 projection tensors
        and their gradients are slices of.  Only run(..., optimise=True) applies it."""
        self._adam = (N.ptr(state), N.ptr(param), N.ptr(grad), N.ptr(exp_avg), N.ptr(exp_avg_sq), param.numel(),
                      float(lr), float(betas[0]), float(betas[1]), float(eps))
        self._keep.append((state, param, grad, exp_avg, exp_avg_sq))

    def bind_table_adam(self, params, exp_avgs, exp_avg_sqs):
        """Optional optimiser of the trainable token tables (tt_step_args.table_*): params = (table_q, table_d) as bound
        with bind() (fp32), exp_avgs / exp_avg_sqs = their fp32 moment pairs.  run(..., optimise=True) then takes one
        dense Adam step on both tables in the table gradient's epilogue, with the projections' step count and
        hyper-parameters (bind_adam)."""
        assert self.train_table, "bind_table_adam needs a step built with train_table=True"
        for t in tuple(params) + tuple(exp_avgs) + tuple(exp_avg_sqs):
            assert t.dtype == torch.float32 and t.shape == params[0].shape
        self._table_adam = (N.ptr(params[0]), N.ptr(params[1]), N.ptr(exp_avgs[0]), N.ptr(exp_avg_sqs[0]),
                            N.ptr(exp_avgs[1]), N.ptr(exp_avg_sqs[1]))
        self._keep.append((params, exp_avgs, exp_avg_sqs))

    def run(self, slot: int = 0, phases: int = 0, optimise: bool = False, accumulate: bool = False):
        """phases: 0 = whole step, 1 = pooled gather only (TT_STEP_FRONT), 2 = the rest (TT_STEP_BACK).
        optimise: also apply the optimiser bound with bind_adam() (gradients only otherwise), and the tables' one bound
        with bind_table_adam().
        accumulate: add this micro-batch's gradients to the gradient buffers (tt_step_args.grad_accumulate)."""
        a = self.slots[slot]
        a.phases = int(phases)
        a.grad_accumulate = int(bool(accumulate))
        if optimise and phases != 1:
            assert self._adam is not None, "run(optimise=True) needs bind_adam() first"
            (a.adam_state, a.adam_param, a.adam_grad, a.adam_exp_avg, a.adam_exp_avg_sq, a.adam_n, a.adam_lr,
             a.adam_beta1, a.adam_beta2, a.adam_eps) = self._adam
            if self._table_adam is not None:
                (a.table_param_q, a.table_param_d, a.table_exp_avg_q, a.table_exp_avg_sq_q, a.table_exp_avg_d,
                 a.table_exp_avg_sq_d) = self._table_adam
        else:
            a.adam_param = None
        try:
            N.check(self.lib.tt_triplet_step(ctypes.byref(a), N.stream()), "tt_triplet_step")
        finally:
            a.phases = 0
            a.adam_param = None
            a.table_param_q = a.table_param_d = None
            a.grad_accumulate = 0
        return self.loss


def adam_step(param, grad, exp_avg, exp_avg_sq, lr, step, beta1=0.9, beta2=0.999, eps=1e-8, grad_scale=1.0):
    N.check(N.load().tt_adam_step(N.ptr(param), N.ptr(grad), N.ptr(exp_avg), N.ptr(exp_avg_sq), param.numel(),
                                  float(lr), float(beta1), float(beta2), float(eps), int(step), float(grad_scale),
                                  N.stream()), "tt_adam_step")


# --------------------------------------------------------------------------------------------------
# retrieval (training.py:244-311)
# --------------------------------------------------------------------------------------------------
def l2_normalize_rows(x: torch.Tensor, eps: float = 1e-8, want_bf16: bool = False):
    N.ensure_sm100()
    N.require_device(x)
    x = x.contiguous().float()
    y = torch.empty_like(x)
    yb = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device) if want_bf16 else None
    if x.shape[0] == 0:  # an empty shard (more ranks than documents)
        return (y, yb) if want_bf16 else y
    N.check(N.load().tt_l2_normalize_rows(N.ptr(x), x.shape[0], x.shape[1], eps, N.ptr(y), N.ptr(yb), N.stream()),
            "tt_l2_normalize_rows")
    return (y, yb) if want_bf16 else y


def scan_topk(Qn, Dn, k=10, id_base=0, precision="fp32", Qb=None, Db=None):
    """Exhaustive scan of normalised docs Dn [N,P] for every normalised query Qn [Q,P]."""
    N.ensure_sm100()
    Q, P = Qn.shape
    Nd = Dn.shape[0]
    prec = _prec(precision)
    lib = N.load()
    top_s = torch.empty(Q, k, dtype=torch.float32, device=Qn.device)
    top_i = torch.empty(Q, k, dtype=torch.int64, device=Qn.device)
    ws_bytes = lib.tt_scan_ws_bytes(Q, Nd, P, k, prec)
    ws = N.workspace(ws_bytes, Qn.device)
    N.check(lib.tt_scan_topk(N.ptr(Qn), N.ptr(Dn), N.ptr(Qb), N.ptr(Db), Q, Nd, P, k, id_base, prec, N.ptr(top_s),
                             N.ptr(top_i), N.ptr(ws), ws_bytes, N.stream()), "tt_scan_topk")
    return top_s, top_i


def score_candidates(Qn, Dn, cand, k, id_base=0, all_scores=None):
    N.ensure_sm100()
    Q, P = Qn.shape
    cand = cand.contiguous().to(torch.int64)
    C = cand.shape[1]
    top_s = torch.empty(Q, k, dtype=torch.float32, device=Qn.device)
    top_i = torch.empty(Q, k, dtype=torch.int64, device=Qn.device)
    N.check(N.load().tt_score_candidates(N.ptr(Qn), N.ptr(Dn), N.ptr(cand), Q, C, P, k, id_base, N.ptr(top_s),
                                         N.ptr(top_i), N.ptr(all_scores), N.stream()), "tt_score_candidates")
    return top_s, top_i


def candidate_scores(Qn_row, Dn, idx, chunk: int = 8192):
    """Exact fp32 scores of ONE query against the documents `idx` (numpy int array) -> numpy float32."""
    import numpy as np

    out = np.empty(len(idx), dtype=np.float32)
    for s in range(0, len(idx), chunk):
        part = torch.as_tensor(np.asarray(idx[s: s + chunk])[None, :], dtype=torch.int64, device=Qn_row.device)
        buf = torch.empty(1, part.shape[1], dtype=torch.float32, device=Qn_row.device)
        score_candidates(Qn_row, Dn, part, k=1, all_scores=buf)
        out[s: s + part.shape[1]] = buf[0].cpu().numpy()
    return out


def topk_merge(parts_s, parts_i):
    """parts [G,Q,k] -> [Q,k] by (score desc, id asc)."""
    N.ensure_sm100()
    G, Q, k = parts_s.shape
    parts_s, parts_i = parts_s.contiguous().float(), parts_i.contiguous().to(torch.int64)
    top_s = torch.empty(Q, k, dtype=torch.float32, device=parts_s.device)
    top_i = torch.empty(Q, k, dtype=torch.int64, device=parts_s.device)
    N.check(N.load().tt_topk_merge(N.ptr(parts_s), N.ptr(parts_i), G, Q, k, N.ptr(top_s), N.ptr(top_i), N.stream()),
            "tt_topk_merge")
    return top_s, top_i


def mine_negatives(top_id, excl_offsets, excl_ids, skip: int, depth: int, table=None, count=None):
    """tt_mine_negatives: scan lists top_id [Q,k] i64 minus each query's exclusion list (CSR, offsets i64 [Q+1], ids
    i32 sorted per query), `skip` survivors dropped, the next `depth` kept in rank order -> (table [Q,depth] i32,
    count [Q] i32).  table / count: optional preallocated outputs."""
    N.ensure_sm100()
    Q, k = top_id.shape
    dev = top_id.device
    table = torch.empty(Q, depth, dtype=torch.int32, device=dev) if table is None else table
    count = torch.empty(Q, dtype=torch.int32, device=dev) if count is None else count
    assert table.dtype == count.dtype == torch.int32 and tuple(table.shape) == (Q, depth) and tuple(count.shape) == (Q,)
    excl_ids = excl_ids if excl_ids.numel() > 0 else torch.zeros(1, dtype=torch.int32, device=dev)
    N.check(N.load().tt_mine_negatives(N.ptr(top_id.contiguous()), Q, k, N.ptr(excl_offsets.contiguous()),
                                       N.ptr(excl_ids.contiguous()), int(skip), int(depth), N.ptr(table), N.ptr(count),
                                       N.stream()), "tt_mine_negatives")
    return table, count


def ndcg_at_k(top_id, rel_offsets, rel_ids, kk=None):
    N.ensure_sm100()
    Q, k = top_id.shape
    kk = k if kk is None else kk
    out = torch.empty(Q, dtype=torch.float64, device=top_id.device)
    rel_ids = rel_ids if rel_ids.numel() > 0 else torch.zeros(1, dtype=torch.int64, device=top_id.device)
    N.check(N.load().tt_ndcg_at_k(N.ptr(top_id.contiguous()), Q, k, kk, N.ptr(rel_offsets.contiguous()),
                                  N.ptr(rel_ids.contiguous()), N.ptr(out), N.stream()), "tt_ndcg_at_k")
    return out
