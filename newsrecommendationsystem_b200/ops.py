"""torch.autograd.Function wrappers over the C-ABI (forward AND backward run in libnrms_b200).

PyTorch is plumbing here: it owns device memory, streams and autograd bookkeeping; every
arithmetic step is a hand-written sm_100a kernel behind `include/nrms_b200.h`.
"""
from __future__ import annotations

import ctypes as C

import os

import torch

from . import _lib
from ._lib import check, ptr, stream_ptr

D, H, QD = 300, 15, 200
# Text lengths with compiled news-encoder kernels (nrms_news_encoder_*: the reference's num_words_title = 20 and
# num_words_abstract = 50).  Every other length 1..64 runs through nrms_text_encoder_*.
TEXT_LENGTHS_COMPILED = (20, 50)
# An embedding parameter marked `_nrms_grad_sink` (optim.FusedAdam marks the parameters it owns) has a .grad that is a
# live view of the optimizer's flat gradient: the news encoder's backward accumulates the embedding gradient directly
# into it instead of returning a fresh 85 MB tensor for autograd to add.  Every other embedding gets its gradient
# through autograd, so torch.autograd.grad and backward(inputs=...) see it.


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("newsrecommendationsystem_b200 ops need CUDA tensors (there is no CPU fallback); "
                               "move the model/inputs to a B200 device")


def _f32c(t):
    return t.detach().contiguous().float()


def _bytes(n, device):
    # at least 256 B so that data_ptr() is a real, 256-byte aligned allocation
    return torch.empty(max(int(n), 256), dtype=torch.uint8, device=device)


def pack_qkv(wq, bq, wk, bk, wv, bv):
    """[W_Q; W_K; W_V] -> [900,300], [b_Q; b_K; b_V] -> [900] (autograd-transparent)."""
    return torch.cat([wq, wk, wv], dim=0), torch.cat([bq, bk, bv], dim=0)


class _NewsEncoderFn(torch.autograd.Function):
    """NewsEncoder.forward (reference src/model/NRMS/news_encoder.py:27-48)."""

    @staticmethod
    def forward(ctx, tokens, emb, wqkv, bqkv, wa, ba, qa, dropout_p, seed, offset, mode, track_grad,
                ln_w=None, ln_b=None, news_rows=None):
        lib = _lib.load()
        _require_cuda(tokens, emb, wqkv, bqkv, wa, ba, qa, news_rows)
        ln = ln_w is not None          # config-5 variant: LayerNorm between self-attention and additive attention
        tokens = tokens.contiguous()
        if tokens.dtype != torch.int64:
            tokens = tokens.long()
        # index-only minibatch (SURVEY 8 f2): `tokens` is the resident [n_news, L] table, `news_rows` picks the titles
        rows = None if news_rows is None else news_rows.contiguous().long().view(-1)
        n_news, L = tokens.shape
        n = n_news if rows is None else rows.numel()
        dev = emb.device
        emb_c, wqkv_c, bqkv_c, wa_c, ba_c, qa_c = map(_f32c, (emb, wqkv, bqkv, wa, ba, qa))
        out = torch.empty((n, D), dtype=torch.float32, device=dev)
        needs_grad = track_grad and any(ctx.needs_input_grad)   # grad mode is always off inside forward()
        stash = None
        if needs_grad or rows is not None:
            stash = _bytes((lib.nrms_encoder_ln_stash_bytes if ln else lib.nrms_encoder_stash_bytes)(n, L), dev)
        ctx.rows = rows
        if L not in TEXT_LENGTHS_COMPILED:
            # any other length: one entry point for the dense and index-only, plain and LayerNorm forms
            if ln:
                _require_cuda(ln_w, ln_b)
            lnw_c, lnb_c = (_f32c(ln_w), _f32c(ln_b)) if ln else (None, None)
            ws = _bytes(lib.nrms_encoder_fwd_workspace_bytes(n, L, mode, 1 if stash is not None else 0, emb_c.shape[0]),
                        dev)
            check(lib.nrms_text_encoder_fwd(ptr(tokens), n_news, ptr(rows), n, L, ptr(emb_c), emb_c.shape[0],
                                            ptr(wqkv_c), ptr(bqkv_c), ptr(lnw_c), ptr(lnb_c), ptr(wa_c), ptr(ba_c),
                                            ptr(qa_c), ptr(out), ptr(stash), ptr(ws), ws.numel(), float(dropout_p),
                                            int(seed), int(offset), mode, stream_ptr(dev)), "nrms_text_encoder_fwd")
            if needs_grad:
                ctx.save_for_backward(tokens, wqkv_c, wa_c, qa_c, stash, *([lnw_c] if ln else []))
                ctx.meta = (n, L, emb_c.shape[0], float(dropout_p), int(seed), int(offset), mode, ln)
                ctx.emb_param = emb if (emb.is_leaf and getattr(emb, "_nrms_grad_sink", False)) else None
            return out
        if rows is not None:
            lnw_c, lnb_c = (_f32c(ln_w), _f32c(ln_b)) if ln else (None, None)
            check(lib.nrms_news_encoder_rows_fwd(ptr(tokens), n_news, ptr(rows), n, L, ptr(emb_c), emb_c.shape[0],
                                                 ptr(wqkv_c), ptr(bqkv_c), ptr(lnw_c), ptr(lnb_c), ptr(wa_c), ptr(ba_c),
                                                 ptr(qa_c), ptr(out), ptr(stash), float(dropout_p), int(seed), int(offset),
                                                 mode, stream_ptr(dev)), "nrms_news_encoder_rows_fwd")
            if needs_grad:
                ctx.save_for_backward(tokens, wqkv_c, wa_c, qa_c, stash, *([lnw_c] if ln else []))
                ctx.meta = (n, L, emb_c.shape[0], float(dropout_p), int(seed), int(offset), mode, ln)
                ctx.emb_param = emb if (emb.is_leaf and getattr(emb, "_nrms_grad_sink", False)) else None
            return out
        ws_bytes = lib.nrms_encoder_fwd_workspace_bytes(n, L, mode, 1 if needs_grad else 0, emb_c.shape[0])
        ws = _bytes(ws_bytes, dev)
        if ln:
            _require_cuda(ln_w, ln_b)
            lnw_c, lnb_c = _f32c(ln_w), _f32c(ln_b)
            check(lib.nrms_news_encoder_ln_fwd(ptr(tokens), n, L, ptr(emb_c), emb_c.shape[0], ptr(wqkv_c), ptr(bqkv_c),
                                               ptr(lnw_c), ptr(lnb_c), ptr(wa_c), ptr(ba_c), ptr(qa_c), ptr(out),
                                               ptr(stash), ptr(ws), ws.numel(), float(dropout_p), int(seed),
                                               int(offset), mode, stream_ptr(dev)), "nrms_news_encoder_ln_fwd")
        else:
            lnw_c = None
            check(lib.nrms_news_encoder_fwd(ptr(tokens), n, L, ptr(emb_c), emb_c.shape[0], ptr(wqkv_c), ptr(bqkv_c),
                                            ptr(wa_c), ptr(ba_c), ptr(qa_c), ptr(out), ptr(stash), ptr(ws), ws.numel(),
                                            float(dropout_p), int(seed), int(offset), mode, stream_ptr(dev)),
                  "nrms_news_encoder_fwd")
        if needs_grad:
            ctx.save_for_backward(tokens, wqkv_c, wa_c, qa_c, stash, *([lnw_c] if ln else []))
            ctx.meta = (n, L, emb_c.shape[0], float(dropout_p), int(seed), int(offset), mode, ln)
            ctx.emb_param = emb if (emb.is_leaf and getattr(emb, "_nrms_grad_sink", False)) else None
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        n, L, V, p, seed, offset, mode, ln = ctx.meta
        tokens, wqkv, wa, qa, stash = ctx.saved_tensors[:5]
        dev = d_out.device
        d_out = d_out.contiguous().float()
        # The embedding gradient is 85 MB: when the optimizer owns a gradient buffer for the table (FusedAdam's flat
        # gradient, zeroed by zero_grad) the scatter kernel accumulates straight into it -- no 85 MB zero fill here and no
        # 85 MB add by autograd afterwards; autograd is told "no gradient" for that input.
        sink = getattr(ctx, "emb_param", None)
        g = sink.grad if sink is not None else None
        in_place = (g is not None and g.dtype == torch.float32 and g.is_contiguous() and tuple(g.shape) == (V, D)
                    and g.device == dev)
        d_emb = g if in_place else torch.zeros((V, D), dtype=torch.float32, device=dev)
        d_wqkv = torch.zeros((3 * D, D), dtype=torch.float32, device=dev)
        d_bqkv = torch.zeros((3 * D,), dtype=torch.float32, device=dev)
        d_wa = torch.zeros((QD, D), dtype=torch.float32, device=dev)
        d_ba = torch.zeros((QD,), dtype=torch.float32, device=dev)
        d_qa = torch.zeros((QD,), dtype=torch.float32, device=dev)
        ws = _bytes(lib.nrms_encoder_bwd_workspace_bytes(n, L, mode), dev)
        d_lnw = d_lnb = None
        if ln:
            lnw = ctx.saved_tensors[5]
            d_lnw = torch.zeros((D,), dtype=torch.float32, device=dev)
            d_lnb = torch.zeros((D,), dtype=torch.float32, device=dev)
        rows = getattr(ctx, "rows", None)
        if L not in TEXT_LENGTHS_COMPILED:
            check(lib.nrms_text_encoder_bwd(ptr(d_out), ptr(tokens), tokens.shape[0], ptr(rows), n, L, V, ptr(wqkv),
                                            ptr(lnw) if ln else None, ptr(wa), ptr(qa), ptr(stash), ptr(d_emb),
                                            ptr(d_wqkv), ptr(d_bqkv), ptr(d_lnw), ptr(d_lnb), ptr(d_wa), ptr(d_ba),
                                            ptr(d_qa), ptr(ws), ws.numel(), p, seed, offset, mode, stream_ptr(dev)),
                  "nrms_text_encoder_bwd")
        elif rows is not None:
            check(lib.nrms_news_encoder_rows_bwd(ptr(d_out), ptr(tokens), tokens.shape[0], ptr(rows), n, L, V, ptr(wqkv),
                                                 ptr(lnw) if ln else None, ptr(wa), ptr(qa), ptr(stash), ptr(d_emb),
                                                 ptr(d_wqkv), ptr(d_bqkv), ptr(d_lnw), ptr(d_lnb), ptr(d_wa), ptr(d_ba),
                                                 ptr(d_qa), ptr(ws), ws.numel(), p, seed, offset, mode, stream_ptr(dev)),
                  "nrms_news_encoder_rows_bwd")
        elif ln:
            check(lib.nrms_news_encoder_ln_bwd(ptr(d_out), ptr(tokens), n, L, V, ptr(wqkv), ptr(lnw), ptr(wa), ptr(qa),
                                               ptr(stash), ptr(d_emb), ptr(d_wqkv), ptr(d_bqkv), ptr(d_lnw), ptr(d_lnb),
                                               ptr(d_wa), ptr(d_ba), ptr(d_qa), ptr(ws), ws.numel(), p, seed, offset,
                                               mode, stream_ptr(dev)), "nrms_news_encoder_ln_bwd")
        else:
            check(lib.nrms_news_encoder_bwd(ptr(d_out), ptr(tokens), n, L, V, ptr(wqkv), ptr(wa), ptr(qa), ptr(stash),
                                            ptr(d_emb), ptr(d_wqkv), ptr(d_bqkv), ptr(d_wa), ptr(d_ba), ptr(d_qa),
                                            ptr(ws), ws.numel(), p, seed, offset, mode, stream_ptr(dev)),
                  "nrms_news_encoder_bwd")
        return (None, (None if in_place else d_emb), d_wqkv, d_bqkv, d_wa, d_ba, d_qa, None, None, None, None, None, d_lnw,
                d_lnb, None)


class _UserEncoderFn(torch.autograd.Function):
    """UserEncoder.forward (reference src/model/NRMS/user_encoder.py:15-26), dense input."""

    @staticmethod
    def forward(ctx, x, wqkv, bqkv, wa, ba, qa, mode, track_grad, ln_w=None, ln_b=None):
        lib = _lib.load()
        _require_cuda(x, wqkv, bqkv, wa, ba, qa)
        ln = ln_w is not None
        n, S, d = x.shape
        if d != D:
            raise RuntimeError(f"user encoder compiled for dim {D}, got {d}")
        dev = x.device
        x_c, wqkv_c, bqkv_c, wa_c, ba_c, qa_c = map(_f32c, (x, wqkv, bqkv, wa, ba, qa))
        out = torch.empty((n, D), dtype=torch.float32, device=dev)
        needs_grad = track_grad and any(ctx.needs_input_grad)
        stash = _bytes((lib.nrms_encoder_ln_stash_bytes if ln else lib.nrms_encoder_stash_bytes)(n, S), dev) \
            if needs_grad else None
        ws = _bytes(lib.nrms_encoder_fwd_workspace_bytes(n, S, mode, 1 if needs_grad else 0, 0), dev)
        if ln:
            _require_cuda(ln_w, ln_b)
            lnw_c, lnb_c = _f32c(ln_w), _f32c(ln_b)
            check(lib.nrms_user_encoder_ln_fwd(ptr(x_c), 0, None, n, S, ptr(wqkv_c), ptr(bqkv_c), ptr(lnw_c), ptr(lnb_c),
                                               ptr(wa_c), ptr(ba_c), ptr(qa_c), ptr(out), ptr(stash), ptr(ws),
                                               ws.numel(), mode, stream_ptr(dev)), "nrms_user_encoder_ln_fwd")
        else:
            lnw_c = None
            check(lib.nrms_user_encoder_fwd(ptr(x_c), 0, None, n, S, ptr(wqkv_c), ptr(bqkv_c), ptr(wa_c), ptr(ba_c),
                                            ptr(qa_c), ptr(out), ptr(stash), ptr(ws), ws.numel(), mode,
                                            stream_ptr(dev)), "nrms_user_encoder_fwd")
        if needs_grad:
            ctx.save_for_backward(wqkv_c, wa_c, qa_c, stash, *([lnw_c] if ln else []))
            ctx.meta = (n, S, mode, ln)
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        n, S, mode, ln = ctx.meta
        wqkv, wa, qa, stash = ctx.saved_tensors[:4]
        dev = d_out.device
        d_out = d_out.contiguous().float()
        d_x = torch.empty((n, S, D), dtype=torch.float32, device=dev)
        d_wqkv = torch.zeros((3 * D, D), dtype=torch.float32, device=dev)
        d_bqkv = torch.zeros((3 * D,), dtype=torch.float32, device=dev)
        d_wa = torch.zeros((QD, D), dtype=torch.float32, device=dev)
        d_ba = torch.zeros((QD,), dtype=torch.float32, device=dev)
        d_qa = torch.zeros((QD,), dtype=torch.float32, device=dev)
        ws = _bytes(lib.nrms_encoder_bwd_workspace_bytes(n, S, mode), dev)
        d_lnw = d_lnb = None
        if ln:
            lnw = ctx.saved_tensors[4]
            d_lnw = torch.zeros((D,), dtype=torch.float32, device=dev)
            d_lnb = torch.zeros((D,), dtype=torch.float32, device=dev)
            check(lib.nrms_user_encoder_ln_bwd(ptr(d_out), n, S, ptr(wqkv), ptr(lnw), ptr(wa), ptr(qa), ptr(stash),
                                               ptr(d_x), ptr(d_wqkv), ptr(d_bqkv), ptr(d_lnw), ptr(d_lnb), ptr(d_wa),
                                               ptr(d_ba), ptr(d_qa), ptr(ws), ws.numel(), mode, stream_ptr(dev)),
                  "nrms_user_encoder_ln_bwd")
        else:
            check(lib.nrms_user_encoder_bwd(ptr(d_out), n, S, ptr(wqkv), ptr(wa), ptr(qa), ptr(stash), ptr(d_x),
                                            ptr(d_wqkv), ptr(d_bqkv), ptr(d_wa), ptr(d_ba), ptr(d_qa), ptr(ws),
                                            ws.numel(), mode, stream_ptr(dev)),
                  "nrms_user_encoder_bwd")
        return d_x, d_wqkv, d_bqkv, d_wa, d_ba, d_qa, None, None, d_lnw, d_lnb


class _ScoreFn(torch.autograd.Function):
    """DotProductClickPredictor.forward (reference .../click_predictor/dot_product.py:8-19)."""

    @staticmethod
    def forward(ctx, cand, user):
        lib = _lib.load()
        _require_cuda(cand, user)
        B, Cn, X = cand.shape
        cand_c, user_c = _f32c(cand), _f32c(user)
        scores = torch.empty((B, Cn), dtype=torch.float32, device=cand.device)
        check(lib.nrms_score_fwd(ptr(cand_c), ptr(user_c), B, Cn, X, ptr(scores), stream_ptr(cand.device)),
              "nrms_score_fwd")
        ctx.save_for_backward(cand_c, user_c)
        return scores

    @staticmethod
    def backward(ctx, d_scores):
        lib = _lib.load()
        cand, user = ctx.saved_tensors
        B, Cn, X = cand.shape
        d_scores = d_scores.contiguous().float()
        d_cand = torch.empty_like(cand)
        d_user = torch.empty_like(user)
        check(lib.nrms_score_bwd(ptr(d_scores), ptr(cand), ptr(user), B, Cn, X, ptr(d_cand), ptr(d_user),
                                 stream_ptr(cand.device)), "nrms_score_bwd")
        return d_cand, d_user


class _CrossEntropyLabel0Fn(torch.autograd.Function):
    """CrossEntropyLoss()(y_pred, zeros) (reference src/train.py:126,205-206)."""

    @staticmethod
    def forward(ctx, logits):
        lib = _lib.load()
        _require_cuda(logits)
        lg = _f32c(logits)
        B, Cn = lg.shape
        loss = torch.empty((), dtype=torch.float32, device=lg.device)
        d_logits = torch.empty_like(lg)
        check(lib.nrms_ce_loss_fwd_bwd(ptr(lg), B, Cn, 1.0, ptr(loss), ptr(d_logits), stream_ptr(lg.device)),
              "nrms_ce_loss_fwd_bwd")
        ctx.save_for_backward(d_logits)
        return loss

    @staticmethod
    def backward(ctx, g):
        (d_logits,) = ctx.saved_tensors
        return d_logits * g


# ---- functional API ---------------------------------------------------------------------------
def news_encoder(tokens, emb, wqkv, bqkv, wa, ba, qa, dropout_p=0.0, seed=0, offset=0, mode=_lib.MODE_TF32,
                 ln=None, news_rows=None):
    """ln = (weight, bias) of the optional LayerNorm(300) (config-5 variant), None for the reference NRMS.
    news_rows (int64 [n], device): index-only minibatch -- `tokens` is then the device-resident pre-tokenised news table
    [n_news, L] and title t of the call is its row news_rows[t], gathered inside the embedding kernels (SURVEY 8 f2)."""
    lw, lb = ln if ln is not None else (None, None)
    return _NewsEncoderFn.apply(tokens, emb, wqkv, bqkv, wa, ba, qa, dropout_p, seed, offset, mode,
                                torch.is_grad_enabled(), lw, lb, news_rows)


def user_encoder(x, wqkv, bqkv, wa, ba, qa, mode=_lib.MODE_TF32, ln=None):
    lw, lb = ln if ln is not None else (None, None)
    return _UserEncoderFn.apply(x, wqkv, bqkv, wa, ba, qa, mode, torch.is_grad_enabled(), lw, lb)


@torch.no_grad()
def user_encoder_indexed(table, rows, wqkv, bqkv, wa, ba, qa, mode=_lib.MODE_TF32, ln=None):
    """Inference-only user encoder whose input rows are gathered from `table` [n_rows,300] by
    int32 `rows` [n_users,S] (replaces the dict/stack loops of reference src/evaluate.py:220-224)."""
    lib = _lib.load()
    _require_cuda(table, rows)
    if rows.dtype != torch.int32:
        rows = rows.int()
    rows = rows.contiguous()
    n, S = rows.shape
    dev = table.device
    out = torch.empty((n, D), dtype=torch.float32, device=dev)
    ws = _bytes(lib.nrms_encoder_fwd_workspace_bytes(n, S, mode, 0, table.shape[0]), dev)
    args = [_f32c(t) for t in (table, wqkv, bqkv, wa, ba, qa)]
    if os.environ.get("NRMS_B200_DEBUG_WS"):
        print(f"user_encoder_indexed: ws {ws.data_ptr():#x} ({ws.numel() / 2**20:.1f} MiB), table {args[0].data_ptr():#x}, "
              f"rows {rows.data_ptr():#x}, out {out.data_ptr():#x}; allocated {torch.cuda.memory_allocated() / 2**20:.0f} MiB, "
              f"reserved {torch.cuda.memory_reserved() / 2**20:.0f} MiB")
    if ln is not None:
        lw, lb = _f32c(ln[0]), _f32c(ln[1])
        check(lib.nrms_user_encoder_ln_fwd(ptr(args[0]), args[0].shape[0], ptr(rows), n, S, ptr(args[1]), ptr(args[2]),
                                           ptr(lw), ptr(lb), ptr(args[3]), ptr(args[4]), ptr(args[5]), ptr(out), None,
                                           ptr(ws), ws.numel(), mode, stream_ptr(dev)),
              "nrms_user_encoder_ln_fwd(indexed)")
        return out
    check(lib.nrms_user_encoder_fwd(ptr(args[0]), args[0].shape[0], ptr(rows), n, S, ptr(args[1]), ptr(args[2]), ptr(args[3]),
                                    ptr(args[4]), ptr(args[5]), ptr(out), None, ptr(ws), ws.numel(), mode,
                                    stream_ptr(dev)), "nrms_user_encoder_fwd(indexed)")
    return out


@torch.no_grad()
def news_encoder_i32(tokens, emb, wqkv, bqkv, wa, ba, qa):
    """Tensor-mode, inference-only news encoder over int32 token ids [n, L] (evaluate's pre-tokenised table).  The
    int32 kernels are compiled for L = 20 and 50; any other length widens the ids and runs news_encoder in tensor mode."""
    lib = _lib.load()
    _require_cuda(tokens, emb)
    if tokens.dtype != torch.int32:
        raise RuntimeError("news_encoder_i32 takes int32 token ids")
    tokens = tokens.contiguous()
    n, L = tokens.shape
    if L not in TEXT_LENGTHS_COMPILED:
        return news_encoder(tokens.long(), emb, wqkv, bqkv, wa, ba, qa, mode=_lib.MODE_TF32)
    dev = emb.device
    out = torch.empty((n, D), dtype=torch.float32, device=dev)
    args = [_f32c(t) for t in (emb, wqkv, bqkv, wa, ba, qa)]
    ws = _bytes(lib.nrms_encoder_fwd_workspace_bytes(n, L, _lib.MODE_TF32, 0, args[0].shape[0]), dev)
    check(lib.nrms_news_encoder_i32_fwd(ptr(tokens), n, L, ptr(args[0]), args[0].shape[0], ptr(args[1]), ptr(args[2]),
                                        ptr(args[3]), ptr(args[4]), ptr(args[5]), ptr(out), ptr(ws), ws.numel(),
                                        stream_ptr(dev)), "nrms_news_encoder_i32_fwd")
    return out


@torch.no_grad()
def user_encoder_table16(table16, rows, wqkv, bqkv, wa, ba, qa):
    """Tensor-mode indexed user encoder over the caller's fp16 copy of the table (`pack_rows_f16` layout:
    [n_rows + 1, 320] halfs, last row zero) -- the form evaluate keeps between its stages."""
    lib = _lib.load()
    _require_cuda(table16, rows)
    if table16.dtype != torch.float16 or table16.dim() != 2 or table16.shape[1] != 320 or not table16.is_contiguous():
        raise RuntimeError("table16 must be a contiguous fp16 [n_rows + 1, 320] tensor (ops.pack_rows_f16)")
    if rows.dtype != torch.int32:
        rows = rows.int()
    rows = rows.contiguous()
    n, S = rows.shape
    n_rows = table16.shape[0] - 1
    out = torch.empty((n, D), dtype=torch.float32, device=table16.device)
    ws = _bytes(lib.nrms_user_encoder_table16_workspace_bytes(n, S, n_rows), table16.device)
    args = [_f32c(t) for t in (wqkv, bqkv, wa, ba, qa)]
    check(lib.nrms_user_encoder_table16_fwd(ptr(table16), n_rows, ptr(rows), n, S, ptr(args[0]), ptr(args[1]), ptr(args[2]),
                                            ptr(args[3]), ptr(args[4]), ptr(out), ptr(ws), ws.numel(),
                                            stream_ptr(table16.device)), "nrms_user_encoder_table16_fwd")
    return out


def click_score(cand, user):
    return _ScoreFn.apply(cand, user)


def cross_entropy_label0(logits):
    return _CrossEntropyLabel0Fn.apply(logits)


@torch.no_grad()
def score_csr(table, cand_rows, offsets, user_vec):
    """Dot products of each impression's candidate rows of `table` with its user vector; rows 300 or 900 wide."""
    lib = _lib.load()
    _require_cuda(table, cand_rows, offsets, user_vec)
    n_imp = offsets.numel() - 1
    scores = torch.empty((cand_rows.numel(),), dtype=torch.float32, device=table.device)
    if table.shape[-1] == D:
        check(lib.nrms_score_csr(ptr(table), ptr(cand_rows), ptr(offsets), ptr(user_vec), n_imp, ptr(scores),
                                 stream_ptr(table.device)), "nrms_score_csr")
    else:
        check(lib.nrms_score_csr_width(ptr(table), ptr(cand_rows), ptr(offsets), ptr(user_vec), n_imp,
                                       table.shape[-1], ptr(scores), stream_ptr(table.device)), "nrms_score_csr_width")
    return scores


@torch.no_grad()
def pack_rows_f16(table, out=None):
    """fp16 copy of an fp32 [n,300] table in the layout the tensor-mode kernels read: [n+1, 320] halfs (300 values, 1.0 in
    column 300, zero tail; the extra last row all zero).  `out`: a contiguous fp16 [>= n+1, 320] view to write into (e.g.
    a rank's slot of the all-gather buffer of evaluate)."""
    lib = _lib.load()
    _require_cuda(table)
    t = _f32c(table)
    if out is None:
        out = torch.empty((t.shape[0] + 1, 320), dtype=torch.float16, device=t.device)
    elif out.dtype != torch.float16 or out.shape[0] < t.shape[0] + 1 or out.shape[1] != 320 or not out.is_contiguous():
        raise RuntimeError("pack_rows_f16: `out` must be a contiguous fp16 [>= n+1, 320] tensor")
    check(lib.nrms_pack_rows_f16(ptr(t), t.shape[0], ptr(out), stream_ptr(t.device)), "nrms_pack_rows_f16")
    return out


@torch.no_grad()
def score_csr_f16(table16, cand_rows, offsets, user_vec):
    lib = _lib.load()
    _require_cuda(table16, cand_rows, offsets, user_vec)
    n_imp = offsets.numel() - 1
    scores = torch.empty((cand_rows.numel(),), dtype=torch.float32, device=table16.device)
    check(lib.nrms_score_csr_f16(ptr(table16), ptr(cand_rows), ptr(offsets), ptr(user_vec), n_imp, ptr(scores),
                                 stream_ptr(table16.device)), "nrms_score_csr_f16")
    return scores


@torch.no_grad()
def rank_metrics(scores, labels, offsets):
    """-> (per_impression [n,4] fp64 with NaN rows for single-class impressions, sums_counts [8] fp64)."""
    lib = _lib.load()
    _require_cuda(scores, labels, offsets)
    n_imp = offsets.numel() - 1
    per = torch.empty((n_imp, 4), dtype=torch.float64, device=scores.device)
    sc = torch.empty((8,), dtype=torch.float64, device=scores.device)
    check(lib.nrms_rank_metrics(ptr(scores), ptr(labels), ptr(offsets), n_imp, ptr(per), ptr(sc),
                                stream_ptr(scores.device)), "nrms_rank_metrics")
    return per, sc


@torch.no_grad()
def gather_rows(src, rows):
    lib = _lib.load()
    _require_cuda(src, rows)
    rows = rows.contiguous().long()
    out = torch.empty((rows.numel(), src.shape[1]), dtype=torch.float32, device=src.device)
    check(lib.nrms_gather_rows(ptr(src), ptr(rows), rows.numel(), src.shape[1], ptr(out), stream_ptr(src.device)),
          "nrms_gather_rows")
    return out


@torch.no_grad()
def adam_step_(p, g, m, v, step, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, decoupled=False,
               grad_scale=1.0):
    lib = _lib.load()
    _require_cuda(p, g, m, v)
    check(lib.nrms_adam_step(ptr(p), ptr(g), ptr(m), ptr(v), p.numel(), lr, betas[0], betas[1], eps, weight_decay,
                             1 if decoupled else 0, int(step), grad_scale, stream_ptr(p.device)), "nrms_adam_step")


@torch.no_grad()
def gemm_nt(a, b, bias=None, mode=_lib.MODE_TF32):
    """C = A @ B^T (+bias) through the library's contraction kernels (tests / profiling)."""
    lib = _lib.load()
    _require_cuda(a, b)
    M, K = a.shape
    N = b.shape[0]
    c = torch.empty((M, N), dtype=torch.float32, device=a.device)
    check(lib.nrms_gemm_nt(ptr(a), a.stride(0), ptr(b), b.stride(0), ptr(bias), ptr(c), c.stride(0), M, N, K, mode,
                           stream_ptr(a.device)), "nrms_gemm_nt")
    return c


def _mhsa_fwd(x, wqkv, bqkv, mode, length):
    """nrms_mhsa_fwd / nrms_mhsa_masked_fwd -> (ctx, x_c, w_c, len_c, ws); ws holds q|k|v [n*S, 900] afterwards."""
    lib = _lib.load()
    _require_cuda(x, wqkv, bqkv)
    n, S, d = x.shape
    if d != D:
        raise RuntimeError(f"compiled for d_model {D}, got {d}")
    x_c, w_c, b_c = map(_f32c, (x, wqkv, bqkv))
    ctx = torch.empty_like(x_c)
    ws = _bytes(n * S * 3 * D * 4, x.device)
    if length is not None:
        if length.numel() != n:
            raise RuntimeError(f"length must hold one entry per sequence ({n}), got {tuple(length.shape)}")
        len_c = length.to(device=x.device, dtype=torch.int32).contiguous().view(-1)
        check(lib.nrms_mhsa_masked_fwd(ptr(x_c), ptr(len_c), n, S, ptr(w_c), ptr(b_c), ptr(ctx), ptr(ws), ws.numel(),
                                       mode, stream_ptr(x.device)), "nrms_mhsa_masked_fwd")
        return ctx, x_c, w_c, len_c, ws
    check(lib.nrms_mhsa_fwd(ptr(x_c), n, S, ptr(w_c), ptr(b_c), ptr(ctx), ptr(ws), ws.numel(), mode,
                            stream_ptr(x.device)), "nrms_mhsa_fwd")
    return ctx, x_c, w_c, None, ws


@torch.no_grad()
def mhsa_forward(x, wqkv, bqkv, mode=_lib.MODE_TF32, length=None):
    """Standalone MultiHeadSelfAttention.forward(Q, length=length) (K=V=Q) without autograd."""
    return _mhsa_fwd(x, wqkv, bqkv, mode, length)[0]


class _MHSAFn(torch.autograd.Function):
    """Standalone MultiHeadSelfAttention.forward(Q, length=length) (reference multihead_self.py:15-23,46-76, K=V=Q) with
    its backward.  The forward is nrms_mhsa_(masked_)fwd, so grad and no-grad forwards give the same bits; its
    workspace (q|k|v) is what the backward reads."""

    @staticmethod
    def forward(ctx, x, wqkv, bqkv, mode, length, track_grad):
        out, x_c, w_c, len_c, ws = _mhsa_fwd(x, wqkv, bqkv, mode, length)
        if track_grad and any(ctx.needs_input_grad):
            ctx.save_for_backward(x_c, w_c, len_c, ws)
            ctx.meta = (mode,)
        return out

    @staticmethod
    def backward(ctx, d_ctx):
        lib = _lib.load()
        x, wqkv, lengths, fws = ctx.saved_tensors
        (mode,) = ctx.meta
        n, S, _ = x.shape
        dev = d_ctx.device
        d_ctx = d_ctx.contiguous().float()
        d_x = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        d_w = torch.zeros((3 * D, D), dtype=torch.float32, device=dev)
        d_b = torch.zeros((3 * D,), dtype=torch.float32, device=dev)
        ws = _bytes(lib.nrms_mhsa_bwd_workspace_bytes(n, S, mode), dev)
        check(lib.nrms_mhsa_bwd(ptr(d_ctx), ptr(x), ptr(lengths), n, S, ptr(wqkv), ptr(fws), ptr(d_x), ptr(d_w), ptr(d_b),
                                ptr(ws), ws.numel(), mode, stream_ptr(dev)), "nrms_mhsa_bwd")
        return (d_x, d_w if ctx.needs_input_grad[1] else None, d_b if ctx.needs_input_grad[2] else None,
                None, None, None)


def mhsa(x, wqkv, bqkv, mode=_lib.MODE_TF32, length=None):
    """MultiHeadSelfAttention.forward(Q, length=length), autograd-connected (forward and backward in libnrms_b200)."""
    return _MHSAFn.apply(x, wqkv, bqkv, mode, length, torch.is_grad_enabled())


MHA_MAX_LEN = 64


def mha_check(q, k, v, length):
    """The shapes nrms_mha_* take (reference multihead_self.py:15-23,46-76); NotImplementedError names what is not
    compiled or not defined by the reference."""
    if q.dim() != 3 or k.dim() != 3 or v.dim() != 3 or not (q.shape[2] == k.shape[2] == v.shape[2] == D):
        raise RuntimeError(f"compiled for [B, S, {D}] inputs, got {tuple(q.shape)}, {tuple(k.shape)}, {tuple(v.shape)}")
    if not (q.shape[0] == k.shape[0] == v.shape[0]):
        raise RuntimeError(f"Q, K and V need the same batch, got {q.shape[0]}, {k.shape[0]}, {v.shape[0]}")
    sq, sk = q.shape[1], k.shape[1]
    if v.shape[1] != sk:
        raise NotImplementedError(f"K and V must have the same number of rows (attn @ V), got {sk} and {v.shape[1]}")
    if not (1 <= sq <= MHA_MAX_LEN and 1 <= sk <= MHA_MAX_LEN):
        raise NotImplementedError(f"libnrms_b200 compiles 1..{MHA_MAX_LEN} queries and keys, got {sq} and {sk}")
    if length is not None and sq != sk and sq != 1:
        raise NotImplementedError(f"the reference's length mask [B, {sq}] does not broadcast over {sk} keys")


def _mha_operands(q, k, v):
    """The fp32 contiguous operands of Q, K and V: one converted copy per distinct tensor object, made before any
    .float().contiguous(), and every role of one object gets that copy.  The library treats equal pointers as one
    input (projected once, one summed gradient), so a distinct tensor whose copy shares storage with an earlier one's
    (a view such as Q.detach() or h[:, :5] of a batch of one) gets its own clone; the roles are assigned only after
    that, so no role keeps a pointer another object's copy was replaced from."""
    copies = []                                   # (tensor object, its operand)
    out = []
    for t in (q, k, v):
        for o, c in copies:
            if t is o:
                out.append(c)
                break
        else:
            c = _f32c(t)
            if any(c.data_ptr() == u.data_ptr() for _, u in copies):
                c = c.clone()
            copies.append((t, c))
            out.append(c)
    return out


class _MHAFn(torch.autograd.Function):
    """MultiHeadSelfAttention.forward(Q, K, V, length) at 1..64 queries and keys (reference multihead_self.py:15-23,
    46-76) with its backward: nrms_mha_fwd / nrms_mha_bwd.  An input passed in two roles (`k is q`, `v is k`, ...)
    reaches the library as one pointer, so it is projected once; its gradient (the sum over its roles) comes back
    once, and None for the alias.  Grad and no-grad forwards run the same call, so they give the same bits."""

    @staticmethod
    def forward(ctx, q, k, v, wqkv, bqkv, mode, length, track_grad):
        lib = _lib.load()
        n, sq, _ = q.shape
        sk = k.shape[1]
        q_c, k_c, v_c = _mha_operands(q, k, v)
        w_c, b_c = _f32c(wqkv), _f32c(bqkv)
        len_c = None
        if length is not None:
            if length.numel() != n:
                raise RuntimeError(f"length must hold one entry per sequence ({n}), got {tuple(length.shape)}")
            len_c = length.to(device=q.device, dtype=torch.int32).contiguous().view(-1)
        out = torch.empty((n, sq, D), dtype=torch.float32, device=q.device)
        ws = _bytes(lib.nrms_mha_fwd_workspace_bytes(n, sq, sk), q.device)
        check(lib.nrms_mha_fwd(ptr(q_c), ptr(k_c), ptr(v_c), n, sq, sk, ptr(len_c), ptr(w_c), ptr(b_c), ptr(out), ptr(ws),
                               ws.numel(), mode, stream_ptr(q.device)), "nrms_mha_fwd")
        if track_grad and any(ctx.needs_input_grad):
            ctx.save_for_backward(q_c, k_c, v_c, w_c, len_c, ws)
            ctx.meta = (mode, k is q, v is q, v is k)
        return out

    @staticmethod
    def backward(ctx, d_ctx):
        lib = _lib.load()
        q, k, v, wqkv, lengths, fws = ctx.saved_tensors
        mode, kq, vq, vk = ctx.meta
        need = ctx.needs_input_grad
        n, sq, _ = q.shape
        sk = k.shape[1]
        dev = d_ctx.device
        d_ctx = d_ctx.contiguous().float()
        need_q = need[0] or (kq and need[1]) or (vq and need[2])
        need_k = not kq and (need[1] or (vk and need[2]))
        need_v = not vq and not vk and need[2]
        d_q = torch.empty_like(q) if need_q else None
        d_k = torch.empty_like(k) if need_k else None
        d_v = torch.empty_like(v) if need_v else None
        d_xk = d_q if kq else d_k
        d_xv = d_q if vq else (d_xk if vk else d_v)
        d_w = torch.zeros((3 * D, D), dtype=torch.float32, device=dev)
        d_b = torch.zeros((3 * D,), dtype=torch.float32, device=dev)
        ws = _bytes(lib.nrms_mha_bwd_workspace_bytes(n, sq, sk, mode), dev)
        check(lib.nrms_mha_bwd(ptr(d_ctx), ptr(q), ptr(k), ptr(v), n, sq, sk, ptr(lengths), ptr(wqkv), ptr(fws), ptr(d_q),
                               ptr(d_xk), ptr(d_xv), ptr(d_w), ptr(d_b), ptr(ws), ws.numel(), mode, stream_ptr(dev)),
              "nrms_mha_bwd")
        return (d_q, d_k, d_v, d_w if need[3] else None, d_b if need[4] else None, None, None, None)


def mha(q, k, v, wqkv, bqkv, mode=_lib.MODE_TF32, length=None):
    """MultiHeadSelfAttention.forward(Q, K, V, length) at 1..64 queries and keys, autograd-connected (forward and
    backward in libnrms_b200).  K = None means K = Q and V = None means V = Q, as in the reference; pass the same tensor
    object for an input used in two roles so that it is projected once."""
    k = q if k is None else k
    v = q if v is None else v
    mha_check(q, k, v, length)
    _require_cuda(q, k, v, wqkv, bqkv)
    return _MHAFn.apply(q, k, v, wqkv, bqkv, mode, length, torch.is_grad_enabled())


class _AdditiveFn(torch.autograd.Function):
    """AdditiveAttention.forward (reference src/model/general/attention/additive.py:27-53) with its backward, for
    candidate sizes 1..64 (20 / 50: encoder lengths, 2..4: the final attention of model/Exp1; below 20 the linear map
    runs on the CUDA cores in either mode)."""

    @staticmethod
    def forward(ctx, c, wa, ba, qa, mode, track_grad):
        lib = _lib.load()
        _require_cuda(c, wa, ba, qa)
        n, S, d = c.shape
        if d != D or wa.shape[0] != QD:
            raise RuntimeError(f"compiled for candidate dim {D} / query dim {QD}")
        c_c, wa_c, ba_c, qa_c = map(_f32c, (c, wa, ba, qa))
        out = torch.empty((n, D), dtype=torch.float32, device=c.device)
        ws = _bytes(n * S * (QD + 1) * 4 + 512, c.device)
        check(lib.nrms_additive_fwd(ptr(c_c), n, S, ptr(wa_c), ptr(ba_c), ptr(qa_c), ptr(out), ptr(ws), ws.numel(), mode,
                                    stream_ptr(c.device)), "nrms_additive_fwd")
        if track_grad and any(ctx.needs_input_grad):
            ctx.save_for_backward(c_c, wa_c, qa_c, ws)
            ctx.meta = (n, S, mode)
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        c, wa, qa, fws = ctx.saved_tensors
        n, S, mode = ctx.meta
        dev = d_out.device
        d_out = d_out.contiguous().float()
        d_c = torch.empty_like(c)
        d_wa = torch.zeros((QD, D), dtype=torch.float32, device=dev)
        d_ba = torch.zeros((QD,), dtype=torch.float32, device=dev)
        d_qa = torch.zeros((QD,), dtype=torch.float32, device=dev)
        ws = _bytes(lib.nrms_additive_bwd_workspace_bytes(n, S, mode), dev)
        check(lib.nrms_additive_bwd(ptr(d_out), ptr(c), n, S, ptr(wa), ptr(qa), ptr(fws), ptr(d_c), ptr(d_wa), ptr(d_ba),
                                    ptr(d_qa), ptr(ws), ws.numel(), mode, stream_ptr(dev)), "nrms_additive_bwd")
        return d_c, d_wa, d_ba, d_qa, None, None


def additive_attention(c, wa, ba, qa, mode=_lib.MODE_TF32):
    """AdditiveAttention.forward, autograd-connected (forward and backward in libnrms_b200)."""
    return _AdditiveFn.apply(c, wa, ba, qa, mode, torch.is_grad_enabled())


CNN_TEXT_MAX_LEN = 64


class _CnnTextEncoderFn(torch.autograd.Function):
    """NAML TextEncoder.forward (reference src/model/NAML/news_encoder.py:9-40): embedding, dropout, Conv2d(1, 300,
    (3, 300), padding=(1, 0)), ReLU, dropout, additive pooling -- nrms_cnn_text_fwd / _bwd.  conv_w is CNN.weight viewed
    as [300, 900].  The embedding gradient goes straight into an optimizer-owned gradient buffer when there is one, as
    in _NewsEncoderFn."""

    @staticmethod
    def forward(ctx, tokens, emb, conv_w, conv_b, wa, ba, qa, dropout_p, seed, offset, mode, track_grad, news_rows):
        lib = _lib.load()
        _require_cuda(tokens, emb, conv_w, conv_b, wa, ba, qa, news_rows)
        tokens = tokens.contiguous()
        if tokens.dtype != torch.int64:
            tokens = tokens.long()
        rows = None if news_rows is None else news_rows.contiguous().long().view(-1)
        n_tok_rows, L = tokens.shape
        n = n_tok_rows if rows is None else rows.numel()
        dev = emb.device
        emb_c, w_c, b_c, wa_c, ba_c, qa_c = map(_f32c, (emb, conv_w, conv_b, wa, ba, qa))
        out = torch.empty((n, D), dtype=torch.float32, device=dev)
        needs_grad = track_grad and any(ctx.needs_input_grad)
        stash = _bytes(lib.nrms_cnn_text_stash_bytes(n, L), dev) if needs_grad else None
        ws = _bytes(lib.nrms_cnn_text_fwd_workspace_bytes(n, L, mode, 1 if needs_grad else 0), dev)
        check(lib.nrms_cnn_text_fwd(ptr(tokens), n_tok_rows, ptr(rows), n, L, ptr(emb_c), emb_c.shape[0], ptr(w_c),
                                    ptr(b_c), ptr(wa_c), ptr(ba_c), ptr(qa_c), ptr(out), ptr(stash), ptr(ws), ws.numel(),
                                    float(dropout_p), int(seed), int(offset), mode, stream_ptr(dev)), "nrms_cnn_text_fwd")
        if needs_grad:
            ctx.save_for_backward(tokens, rows, w_c, wa_c, qa_c, stash)
            ctx.meta = (n, L, emb_c.shape[0], float(dropout_p), int(seed), int(offset), mode)
            ctx.emb_param = emb if (emb.is_leaf and getattr(emb, "_nrms_grad_sink", False)) else None
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        n, L, V, p, seed, offset, mode = ctx.meta
        tokens, rows, conv_w, wa, qa, stash = ctx.saved_tensors
        dev = d_out.device
        d_out = d_out.contiguous().float()
        sink = getattr(ctx, "emb_param", None)
        g = sink.grad if sink is not None else None
        in_place = (g is not None and g.dtype == torch.float32 and g.is_contiguous() and tuple(g.shape) == (V, D)
                    and g.device == dev)
        d_emb = g if in_place else torch.zeros((V, D), dtype=torch.float32, device=dev)
        d_w = torch.zeros((D, 3 * D), dtype=torch.float32, device=dev)
        d_b = torch.zeros((D,), dtype=torch.float32, device=dev)
        d_wa = torch.zeros((QD, D), dtype=torch.float32, device=dev)
        d_ba = torch.zeros((QD,), dtype=torch.float32, device=dev)
        d_qa = torch.zeros((QD,), dtype=torch.float32, device=dev)
        ws = _bytes(lib.nrms_cnn_text_bwd_workspace_bytes(n, L, mode), dev)
        check(lib.nrms_cnn_text_bwd(ptr(d_out), ptr(tokens), tokens.shape[0], ptr(rows), n, L, V, ptr(conv_w), ptr(wa),
                                    ptr(qa), ptr(stash), ptr(d_emb), ptr(d_w), ptr(d_b), ptr(d_wa), ptr(d_ba), ptr(d_qa),
                                    ptr(ws), ws.numel(), p, seed, offset, mode, stream_ptr(dev)), "nrms_cnn_text_bwd")
        return (None, (None if in_place else d_emb), d_w, d_b, d_wa, d_ba, d_qa, None, None, None, None, None, None)


def cnn_text_encoder(tokens, emb, conv_w, conv_b, wa, ba, qa, dropout_p=0.0, seed=0, offset=0, mode=_lib.MODE_TF32,
                     news_rows=None):
    """NAML's CNN text encoder, autograd-connected.  tokens: integer [n, L] (L = 1..64), emb [num_words, 300], conv_w
    [300, 900] (CNN.weight [300, 1, 3, 300] viewed flat), conv_b [300], wa [200, 300], ba / qa [200] -> fp32 [n, 300].
    news_rows (int64 [m], device): `tokens` is a device-resident token column and text t of the call is its row
    news_rows[t], read through the index inside the gather / scatter kernels."""
    L = tokens.shape[-1]
    if tokens.dim() != 2 or not 1 <= L <= CNN_TEXT_MAX_LEN:
        raise RuntimeError(f"cnn_text_encoder takes [n, L] tokens with L in 1..{CNN_TEXT_MAX_LEN}, got {tuple(tokens.shape)}")
    if tuple(conv_w.shape) != (D, 3 * D):
        raise RuntimeError(f"conv_w must be CNN.weight viewed as [{D}, {3 * D}], got {tuple(conv_w.shape)}")
    return _CnnTextEncoderFn.apply(tokens, emb, conv_w, conv_b, wa, ba, qa, dropout_p, seed, offset, mode,
                                   torch.is_grad_enabled(), news_rows)


class _ElementEncoderFn(torch.autograd.Function):
    """ElementEncoder.forward = relu(linear(embedding(element)))  (reference src/model/Exp1/news_encoder.py:37-44)."""

    @staticmethod
    def forward(ctx, idx, emb, w, b, track_grad):
        lib = _lib.load()
        _require_cuda(idx, emb, w, b)
        if emb.shape[1] != 100 or tuple(w.shape) != (D, 100):
            raise RuntimeError("libnrms_b200 is compiled for category_embedding_dim 100 -> word_embedding_dim 300")
        shape = idx.shape
        idx_c = idx.contiguous().long().view(-1)
        emb_c, w_c, b_c = map(_f32c, (emb, w, b))
        n, ncat = idx_c.numel(), emb_c.shape[0]
        out = torch.empty((n, D), dtype=torch.float32, device=emb.device)
        table = _bytes(lib.nrms_element_encoder_table_bytes(ncat), emb.device)
        check(lib.nrms_element_encoder_fwd(ptr(idx_c), n, ptr(emb_c), ncat, ptr(w_c), ptr(b_c), ptr(out), ptr(table),
                                           stream_ptr(emb.device)), "nrms_element_encoder_fwd")
        if track_grad and any(ctx.needs_input_grad):
            ctx.save_for_backward(idx_c, emb_c, w_c, table)
        return out.view(*shape, D)

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        idx, emb, w, table = ctx.saved_tensors
        dev = d_out.device
        n, ncat = idx.numel(), emb.shape[0]
        d_out = d_out.contiguous().float().view(n, D)
        d_emb = torch.zeros_like(emb)
        d_w = torch.zeros_like(w)
        d_b = torch.zeros((D,), dtype=torch.float32, device=dev)
        ws = _bytes(lib.nrms_element_encoder_table_bytes(ncat), dev)
        check(lib.nrms_element_encoder_bwd(ptr(d_out), ptr(idx), n, ptr(emb), ncat, ptr(w), ptr(table), ptr(d_emb),
                                           ptr(d_w), ptr(d_b), ptr(ws), ws.numel(), stream_ptr(dev)),
              "nrms_element_encoder_bwd")
        return None, d_emb, d_w, d_b, None


def element_encoder(idx, emb, w, b):
    return _ElementEncoderFn.apply(idx, emb, w, b, torch.is_grad_enabled())


class _AddPositionFn(torch.autograd.Function):
    """user_vector + position_embedding.expand_as(user_vector)  (reference src/model/Exp1/user_encoder.py:25-26)."""

    @staticmethod
    def forward(ctx, x, pos):
        lib = _lib.load()
        _require_cuda(x, pos)
        n, S, d = x.shape
        if d != D or tuple(pos.shape) != (S, D):
            raise RuntimeError(f"expected x [n, S, {D}] and position_embedding [S, {D}]")
        x_c, pos_c = _f32c(x), _f32c(pos)
        out = torch.empty_like(x_c)
        check(lib.nrms_add_position_fwd(ptr(x_c), ptr(pos_c), n, S, ptr(out), stream_ptr(x.device)), "nrms_add_position_fwd")
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        d_out = d_out.contiguous().float()
        n, S, _ = d_out.shape
        d_pos = None
        if ctx.needs_input_grad[1]:
            d_pos = torch.zeros((S, D), dtype=torch.float32, device=d_out.device)
            ws = _bytes(lib.nrms_add_position_bwd_workspace_bytes(S), d_out.device)
            check(lib.nrms_add_position_bwd(ptr(d_out), n, S, ptr(d_pos), ptr(ws), ws.numel(), stream_ptr(d_out.device)),
                  "nrms_add_position_bwd")
        return (d_out if ctx.needs_input_grad[0] else None), d_pos


def add_position(x, pos):
    return _AddPositionFn.apply(x, pos)


class _StackFn(torch.autograd.Function):
    """torch.stack(vectors, dim=1) of 300-wide rows (reference src/model/Exp1/news_encoder.py:109) through
    nrms_copy_rows_strided; the backward hands every vector its slice."""

    @staticmethod
    def forward(ctx, *vectors):
        lib = _lib.load()
        _require_cuda(*vectors)
        k, n = len(vectors), vectors[0].shape[0]
        dev = vectors[0].device
        out = torch.empty((n, k, D), dtype=torch.float32, device=dev)
        for j, v in enumerate(vectors):
            v_c = _f32c(v)
            check(lib.nrms_copy_rows_strided(ptr(v_c), D, C.c_void_p(out.data_ptr() + 4 * D * j), k * D, n, D,
                                             stream_ptr(dev)), "nrms_copy_rows_strided")
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        d_out = d_out.contiguous().float()
        n, k, _ = d_out.shape
        grads = []
        for j in range(k):
            g = torch.empty((n, D), dtype=torch.float32, device=d_out.device)
            check(lib.nrms_copy_rows_strided(C.c_void_p(d_out.data_ptr() + 4 * D * j), k * D, ptr(g), D, n, D,
                                             stream_ptr(d_out.device)), "nrms_copy_rows_strided")
            grads.append(g)
        return tuple(grads)


def stack_vectors(vectors):
    return _StackFn.apply(*vectors)


@torch.no_grad()
def recommend_user(table, hist_rows, cand_rows, wqkv, bqkv, wa, ba, qa, rank=True):
    """Single-user latency path (reference src/recommend.py:245-341): user vector from the 50 history rows of the
    news-vector table, scores of the candidate rows, and (rank=True) the candidate positions by descending score.
    Two kernel launches; returns (user_vec [300], scores [C], order int32 [C] or None) on the device."""
    lib = _lib.load()
    _require_cuda(table, hist_rows, cand_rows)
    if hist_rows.numel() != 50:
        raise RuntimeError("the latency path is compiled for num_clicked_news_a_user = 50")
    dev = table.device
    table_c = _f32c(table)
    hist = hist_rows.to(torch.int32).contiguous().view(-1)
    cand = cand_rows.to(torch.int32).contiguous().view(-1)
    Cn = cand.numel()
    args = [_f32c(t) for t in (wqkv, bqkv, wa, ba, qa)]
    user = torch.empty((D,), dtype=torch.float32, device=dev)
    scores = torch.empty((Cn,), dtype=torch.float32, device=dev)
    order = torch.empty((Cn,), dtype=torch.int32, device=dev) if rank else None
    ws = _bytes(lib.nrms_recommend_workspace_bytes(), dev)
    check(lib.nrms_recommend_user(ptr(table_c), table_c.shape[0], ptr(hist), ptr(cand), Cn, ptr(args[0]), ptr(args[1]),
                                  ptr(args[2]), ptr(args[3]), ptr(args[4]), ptr(user), ptr(scores), ptr(order), ptr(ws),
                                  ws.numel(), stream_ptr(dev)), "nrms_recommend_user")
    return user, scores, order


@torch.no_grad()
def topk_news(table, n_news, user_vec, k, exclude_rows=None, mode=_lib.MODE_TF32):
    """The k rows of table[:n_news] with the highest dot product with each user vector (nrms_topk_news): returns
    (scores fp32 [U, k], rows int32 [U, k]) on the device, ordered by score descending and equal scores by row ascending;
    tail entries (fewer than k rows left) are row -1, score -inf.  No score matrix is materialised and nothing syncs.
    mode MODE_TF32: `table` is the fp16 [>= n_news, 320] copy of `pack_rows_f16` (tensor cores, user vectors rounded to
    fp16); MODE_FP32: `table` is fp32 [>= n_news, 300].  exclude_rows: int [U, <= 64] rows never returned for that user
    (history rows; values outside [0, n_news) such as pads are ignored), on the host or the device."""
    n_news = int(n_news)
    if mode == _lib.MODE_TF32:
        if table.dtype != torch.float16 or table.dim() != 2 or table.shape[1] != 320:
            raise RuntimeError("topk_news in tensor mode takes the fp16 [n, 320] table of pack_rows_f16, got "
                               f"{table.dtype} {tuple(table.shape)}")
    elif mode == _lib.MODE_FP32:
        if table.dtype != torch.float32 or table.dim() != 2 or table.shape[1] != D:
            raise RuntimeError(f"topk_news in FP32 mode takes an fp32 [n, {D}] table, got {table.dtype} {tuple(table.shape)}")
    else:
        raise ValueError(f"unknown mode {mode!r}")
    if not 0 < n_news <= table.shape[0]:
        raise RuntimeError(f"n_news = {n_news} must be in [1, {table.shape[0]}] (rows of the table)")
    _require_cuda(table, user_vec)
    lib = _lib.load()
    dev = table.device
    table = table.contiguous()
    u = _f32c(user_vec)
    if u.dim() != 2 or u.shape[1] != D:
        raise RuntimeError(f"user_vec must be [U, {D}], got {tuple(u.shape)}")
    U = u.shape[0]
    ex, n_ex = None, 0
    if exclude_rows is not None:
        ex = torch.as_tensor(exclude_rows).to(device=dev, dtype=torch.int32).contiguous()
        if ex.dim() != 2 or ex.shape[0] != U:
            raise RuntimeError(f"exclude_rows must be [U = {U}, n_exclude], got {tuple(ex.shape)}")
        n_ex = ex.shape[1]
        if n_ex == 0:
            ex = None
    scores = torch.empty((U, k), dtype=torch.float32, device=dev)
    rows = torch.empty((U, k), dtype=torch.int32, device=dev)
    ws = _bytes(lib.nrms_topk_workspace_bytes(U, n_news, int(k), n_ex, mode), dev)
    check(lib.nrms_topk_news(ptr(table), n_news, ptr(u), U, ptr(ex), n_ex, int(k), ptr(scores), ptr(rows), ptr(ws),
                             ws.numel(), mode, stream_ptr(dev)), "nrms_topk_news")
    return scores, rows


@torch.no_grad()
def additive_forward(c, wa, ba, qa, mode=_lib.MODE_TF32):
    """Standalone AdditiveAttention.forward, inference only."""
    lib = _lib.load()
    _require_cuda(c, wa, ba, qa)
    n, S, d = c.shape
    if d != D or wa.shape[0] != QD:
        raise RuntimeError(f"compiled for candidate dim {D} / query dim {QD}")
    c_c, wa_c, ba_c, qa_c = map(_f32c, (c, wa, ba, qa))
    out = torch.empty((n, D), dtype=torch.float32, device=c.device)
    ws = _bytes(n * S * (QD + 1) * 4 + 512, c.device)
    check(lib.nrms_additive_fwd(ptr(c_c), n, S, ptr(wa_c), ptr(ba_c), ptr(qa_c), ptr(out), ptr(ws), ws.numel(), mode,
                                stream_ptr(c.device)), "nrms_additive_fwd")
    return out


GRU_SHAPES = ((900, 900), (900, 450))


def _host_lengths(lengths, n_seq, T):
    """int32 host copy of the per-sequence lengths (nrms_gru_* take them in host memory), checked against 0..T."""
    if lengths.is_cuda:
        raise RuntimeError("gru lengths must be a host tensor: the steps are scheduled on the host")
    lh = lengths.detach().reshape(-1).to(torch.int32).contiguous()
    if lh.numel() != n_seq:
        raise RuntimeError(f"gru takes one length per sequence: {lh.numel()} for {n_seq}")
    if lh.numel() and (int(lh.min()) < 0 or int(lh.max()) > T):
        raise RuntimeError(f"gru lengths must lie in 0..{T}, got [{int(lh.min())}, {int(lh.max())}]")
    return lh


class _GRUFn(torch.autograd.Function):
    """The last hidden state of nn.GRU over pack_padded_sequence(x, lengths, batch_first=True) from h0 (reference
    src/model/LSTUR/user_encoder.py) -- nrms_gru_fwd / _bwd."""

    @staticmethod
    def forward(ctx, x, lengths, h0, w_ih, w_hh, b_ih, b_hh, mode, track_grad):
        lib = _lib.load()
        _require_cuda(x, h0, w_ih, w_hh, b_ih, b_hh)
        n_seq, T, I = x.shape
        Hd = w_hh.shape[1]
        lh = _host_lengths(lengths, n_seq, T)
        dev = x.device
        x_c, w_ih_c, w_hh_c, b_ih_c, b_hh_c = map(_f32c, (x, w_ih, w_hh, b_ih, b_hh))
        h0_c = None if h0 is None else _f32c(h0)
        out = torch.empty((n_seq, Hd), dtype=torch.float32, device=dev)
        needs_grad = track_grad and any(ctx.needs_input_grad)
        stash = _bytes(lib.nrms_gru_stash_bytes(n_seq, T, I, Hd), dev) if needs_grad else None
        ws = _bytes(lib.nrms_gru_fwd_workspace_bytes(n_seq, T, n_seq * T, I, Hd), dev)
        check(lib.nrms_gru_fwd(ptr(x_c), n_seq * T, None, n_seq, T, I, Hd, C.c_void_p(lh.data_ptr()), ptr(h0_c),
                               ptr(w_ih_c), ptr(w_hh_c), ptr(b_ih_c), ptr(b_hh_c), ptr(out), ptr(stash), ptr(ws),
                               ws.numel(), mode, stream_ptr(dev)), "nrms_gru_fwd")
        if needs_grad:
            ctx.save_for_backward(x_c, w_ih_c, w_hh_c, stash)
            ctx.lengths = lh
            ctx.meta = (n_seq, T, I, Hd, mode, h0 is not None)
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        n_seq, T, I, Hd, mode, has_h0 = ctx.meta
        x, w_ih, w_hh, stash = ctx.saved_tensors
        dev = d_out.device
        d_out = d_out.contiguous().float()
        d_x = torch.empty((n_seq, T, I), dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        d_h0 = torch.empty((n_seq, Hd), dtype=torch.float32, device=dev) if has_h0 and ctx.needs_input_grad[2] else None
        d_w_ih = torch.zeros((3 * Hd, I), dtype=torch.float32, device=dev)
        d_w_hh = torch.zeros((3 * Hd, Hd), dtype=torch.float32, device=dev)
        d_b_ih = torch.zeros((3 * Hd,), dtype=torch.float32, device=dev)
        d_b_hh = torch.zeros((3 * Hd,), dtype=torch.float32, device=dev)
        ws = _bytes(lib.nrms_gru_bwd_workspace_bytes(n_seq, T, I, Hd, mode), dev)
        check(lib.nrms_gru_bwd(ptr(d_out), ptr(x), n_seq, T, I, Hd, C.c_void_p(ctx.lengths.data_ptr()), ptr(w_ih),
                               ptr(w_hh), ptr(stash), ptr(d_x), ptr(d_h0), ptr(d_w_ih), ptr(d_w_hh), ptr(d_b_ih),
                               ptr(d_b_hh), ptr(ws), ws.numel(), mode, stream_ptr(dev)), "nrms_gru_bwd")
        return d_x, None, d_h0, d_w_ih, d_w_hh, d_b_ih, d_b_hh, None, None


def _gru_check(I, w_ih, w_hh):
    Hd = w_hh.shape[-1]
    if (I, Hd) not in GRU_SHAPES or tuple(w_ih.shape) != (3 * Hd, I) or tuple(w_hh.shape) != (3 * Hd, Hd):
        raise RuntimeError(f"gru is compiled for (input, hidden) in {GRU_SHAPES}, got w_ih {tuple(w_ih.shape)}, "
                           f"w_hh {tuple(w_hh.shape)}")


def gru(x, lengths, h0, w_ih, w_hh, b_ih, b_hh, mode=_lib.MODE_TF32):
    """Last hidden state of a one-layer nn.GRU (weight_ih_l0 = w_ih [3H, I], ...) over steps t < lengths[s] of
    x [n_seq, T, I], started from h0 [n_seq, H] (None: zeros), autograd-connected.  lengths: integer [n_seq] on the
    HOST, each in 0..T (0 runs no step).  (I, H) = (900, 900) or (900, 450)."""
    if x.dim() != 3:
        raise RuntimeError(f"gru takes x [n_seq, T, I], got {tuple(x.shape)}")
    _gru_check(x.shape[2], w_ih, w_hh)
    return _GRUFn.apply(x, lengths, h0, w_ih, w_hh, b_ih, b_hh, mode, torch.is_grad_enabled())


@torch.no_grad()
def gru_indexed(table, rows, lengths, h0, w_ih, w_hh, b_ih, b_hh, mode=_lib.MODE_TF32):
    """Inference form of gru: step t of sequence s reads row rows[s, t] of the table [n_rows, I] (device).  The input
    projection runs once over the table rows, not once per history row.  rows on the host are range-checked against
    the table before they go to the device; rows already on the device must lie in [0, n_rows)."""
    if not rows.is_cuda:
        if rows.numel() and (int(rows.min()) < 0 or int(rows.max()) >= table.shape[0]):
            raise IndexError(f"gru_indexed rows must lie in [0, {table.shape[0]}), got [{int(rows.min())}, "
                             f"{int(rows.max())}]")
        rows = rows.to(table.device)
    _require_cuda(table, rows, h0, w_ih, w_hh, b_ih, b_hh)
    lib = _lib.load()
    n_seq, T = rows.shape
    I = table.shape[1]
    _gru_check(I, w_ih, w_hh)
    Hd = w_hh.shape[1]
    if rows.numel() and table.shape[0] == 0:
        raise RuntimeError("gru_indexed: empty table")
    lh = _host_lengths(lengths, n_seq, T)
    dev = table.device
    tab, w_ih_c, w_hh_c, b_ih_c, b_hh_c = map(_f32c, (table, w_ih, w_hh, b_ih, b_hh))
    h0_c = None if h0 is None else _f32c(h0)
    r = rows.contiguous().long().view(-1)
    out = torch.empty((n_seq, Hd), dtype=torch.float32, device=dev)
    ws = _bytes(lib.nrms_gru_fwd_workspace_bytes(n_seq, T, tab.shape[0], I, Hd), dev)
    check(lib.nrms_gru_fwd(ptr(tab), tab.shape[0], ptr(r), n_seq, T, I, Hd, C.c_void_p(lh.data_ptr()), ptr(h0_c),
                           ptr(w_ih_c), ptr(w_hh_c), ptr(b_ih_c), ptr(b_hh_c), ptr(out), None, ptr(ws), ws.numel(),
                           mode, stream_ptr(dev)), "nrms_gru_fwd")
    return out


class _RowsFn(torch.autograd.Function):
    """weight[idx] (nn.Embedding / F.embedding), optionally under a whole-row dropout mask -- F.dropout2d of
    embedding(idx).unsqueeze(0) zeroes whole rows (reference src/model/LSTUR/__init__.py) -- nrms_rows_fwd / _bwd."""

    @staticmethod
    def forward(ctx, idx, weight, padding_idx, p, seed, offset):
        lib = _lib.load()
        _require_cuda(idx, weight)
        i = idx.contiguous().long().view(-1)
        w = _f32c(weight)
        n, width = i.numel(), w.shape[1]
        out = torch.empty((n, width), dtype=torch.float32, device=w.device)
        check(lib.nrms_rows_fwd(ptr(w), w.shape[0], width, ptr(i), n, width, ptr(out), width, float(p), int(seed),
                                int(offset), stream_ptr(w.device)), "nrms_rows_fwd")
        ctx.save_for_backward(i)
        ctx.meta = (tuple(w.shape), padding_idx, float(p), int(seed), int(offset))
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        (i,) = ctx.saved_tensors
        shape, padding_idx, p, seed, offset = ctx.meta
        d_out = d_out.contiguous().float()
        d_w = torch.zeros(shape, dtype=torch.float32, device=d_out.device)
        check(lib.nrms_rows_bwd(ptr(d_out), shape[1], ptr(i), i.numel(), shape[1], ptr(d_w), shape[1],
                                -1 if padding_idx is None else int(padding_idx), p, seed, offset,
                                stream_ptr(d_out.device)), "nrms_rows_bwd")
        return None, d_w, None, None, None, None


def embedding_rows(idx, weight, padding_idx=0, dropout_p=0.0, seed=0, offset=0):
    """weight[idx] -> fp32 [idx.numel(), width], autograd-connected (padding_idx rows get no gradient).  dropout_p > 0:
    each output row is zeroed with probability p and the others scaled by 1 / (1 - p), from the Philox stream of the
    (seed, offset) pair (row i: counter i + offset)."""
    return _RowsFn.apply(idx, weight, padding_idx, dropout_p, seed, offset)


def _copy_rows(src, ld_src, dst, ld_dst, n, width, lib, dev):
    check(lib.nrms_rows_fwd(ptr(src), n, ld_src, None, n, width, ptr(dst), ld_dst, 0.0, 0, 0, stream_ptr(dev)),
          "nrms_rows_fwd")


class _ConcatRowsFn(torch.autograd.Function):
    """torch.cat(parts, dim=1) of 2-D fp32 row blocks through strided row copies (nrms_rows_fwd with no index)."""

    @staticmethod
    def forward(ctx, *parts):
        lib = _lib.load()
        _require_cuda(*parts)
        n = parts[0].shape[0]
        widths = [p.shape[1] for p in parts]
        dev = parts[0].device
        out = torch.empty((n, sum(widths)), dtype=torch.float32, device=dev)
        col = 0
        for p, w in zip(parts, widths):
            pc = _f32c(p)
            _copy_rows(pc, w, out[:, col:], out.shape[1], n, w, lib, dev)
            col += w
        ctx.widths = widths
        return out

    @staticmethod
    def backward(ctx, d_out):
        lib = _lib.load()
        d_out = d_out.contiguous().float()
        n, dev = d_out.shape[0], d_out.device
        grads, col = [], 0
        for w in ctx.widths:
            g = torch.empty((n, w), dtype=torch.float32, device=dev)
            _copy_rows(d_out[:, col:], d_out.shape[1], g, w, n, w, lib, dev)
            grads.append(g)
            col += w
        return tuple(grads)


def concat_rows(*parts):
    """torch.cat(parts, dim=1) of [n, w_k] row blocks, autograd-connected, with the copies in libnrms_b200."""
    if len({p.shape[0] for p in parts}) != 1 or any(p.dim() != 2 for p in parts):
        raise RuntimeError(f"concat_rows takes [n, w] blocks of one n, got {[tuple(p.shape) for p in parts]}")
    return _ConcatRowsFn.apply(*parts)
