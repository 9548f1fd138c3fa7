"""Exp1 training with the abstract encoder: 50-token news-encoder training (the tensor-mode mma.sync attention of
attn_mma.cu and the CUDA-core kernels of the FP32 mode), Exp1.forward_rows and TrainStep driving Exp1.

CPU part: a torch fp64 autograd restatement of Exp1.forward + CE(label 0), pinned against the live-reference fixtures
(title-configuration gradients, abstract-configuration forward) before it serves as the reference of the abstract
configuration; the C-ABI's length checks and sizes at L = 50.  GPU part (`-m gpu`): every check is against fp64 built
from the exact operands each mode used (the stashed q|k|v rows, the kernels' own dropout masks).
"""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2_rows
from oracle import nrms_oracle as O
from compact import pinned
from test_exp1_recommend import ATTRS, ATTRS_A, _exp1_state, g1  # noqa: F401  (g1: fixture)

N_CAND = 3          # 1 + K candidates of the test batches
N_CLICKED = 50      # config.num_clicked_news_a_user


# ---- the fp64 restatement ------------------------------------------------------------------------------------------
def _shared(P, key):
    """The parameter behind a state_dict key: the word / category embeddings are shared modules, so named_parameters()
    lists them once, under the first text / element encoder."""
    if key in P:
        return P[key]
    part = ".word_embedding.weight" if key.endswith(".word_embedding.weight") else ".embedding.weight"
    return next(v for k, v in P.items() if k.endswith(part))


def _mhsa(x, P, pre, mask2=None):
    """multihead_self.py:15-23,46-76 (no max subtraction, + 1e-8)."""
    n, S, _ = x.shape
    h = [F.linear(x, P[f"{pre}.W_{w}.weight"], P[f"{pre}.W_{w}.bias"]).view(n, S, 15, 20).transpose(1, 2) for w in "QKV"]
    e = torch.exp(h[0] @ h[1].transpose(-1, -2) / np.sqrt(20.0))
    ctx = ((e / (e.sum(-1, keepdim=True) + 1e-8)) @ h[2]).transpose(1, 2).reshape(n, S, 300)
    return ctx if mask2 is None else ctx * mask2


def _additive(c, P, pre):
    """additive.py:27-53."""
    w = torch.softmax(torch.tanh(F.linear(c, P[f"{pre}.linear.weight"], P[f"{pre}.linear.bias"])) @
                      P[f"{pre}.attention_query_vector"], dim=1)
    return (w.unsqueeze(-1) * c).sum(1)


def exp1_fp64(params, news, n_cand, attributes, masks=None):
    """Exp1.forward (reference src/model/Exp1/__init__.py:15-46, news_encoder.py:10-111, user_encoder.py:7-31) and
    CrossEntropyLoss against label 0 in torch fp64 autograd.  params: {named_parameters() name: array};
    news: {attribute: [B, 1+K+N, ...]}; masks: {text attribute: (mask1, mask2)} for train-mode dropout.
    Returns (loss, logits, {name: gradient})."""
    P = {k: torch.tensor(np.asarray(v, dtype=np.float64), requires_grad=True) for k, v in params.items()}
    B, T = news[attributes[0]].shape[:2]
    flat = {a: torch.as_tensor(np.asarray(news[a])).reshape(B * T, *np.asarray(news[a]).shape[2:]) for a in attributes}
    vecs = []
    for a in ("abstract", "title"):                        # NewsEncoder: text encoders, then element encoders (sorted)
        if a in attributes:
            pre = f"news_encoder.text_encoders.{a}"
            x = F.embedding(flat[a], _shared(P, f"{pre}.word_embedding.weight"), padding_idx=0)
            m1, m2 = (masks or {}).get(a, (None, None))
            if m1 is not None:
                x = x * torch.as_tensor(m1, dtype=torch.float64)
            ctx = _mhsa(x, P, f"{pre}.multihead_self_attention",
                        None if m2 is None else torch.as_tensor(m2, dtype=torch.float64))
            vecs.append(_additive(ctx, P, f"{pre}.additive_attention"))
    for a in ("category", "subcategory"):
        if a in attributes:
            pre = f"news_encoder.element_encoders.{a}"
            e = F.embedding(flat[a], _shared(P, f"{pre}.embedding.weight"), padding_idx=0)
            vecs.append(torch.relu(F.linear(e, P[f"{pre}.linear.weight"], P[f"{pre}.linear.bias"])))
    nv = vecs[0] if len(vecs) == 1 else _additive(torch.stack(vecs, dim=1), P, "news_encoder.final_attention")
    nv = nv.view(B, T, 300)
    u = nv[:, n_cand:] + P["user_encoder.position_embedding"]
    uv = _additive(_mhsa(u, P, "user_encoder.multihead_self_attention"), P, "user_encoder.additive_attention")
    logits = (nv[:, :n_cand] * uv[:, None]).sum(-1)
    loss = F.cross_entropy(logits, torch.zeros(B, dtype=torch.long))
    loss.backward()
    return float(loss.detach()), logits.detach().numpy(), {k: v.grad.numpy() for k, v in P.items()}


def _named(m, sd):
    """The state dict restricted to named_parameters() (shared embeddings once)."""
    return {k: sd[k] for k, _ in m.named_parameters()}


def _batch(rng, B, num_words=401, num_categories=31, abstract=True):
    """A random Exp1 batch [B, 1+K+N, ...] with pad-only and one-token texts among the rows."""
    T = N_CAND + N_CLICKED
    news = {"title": rng.integers(1, num_words, size=(B, T, 20)),
            "category": rng.integers(0, num_categories, size=(B, T)),
            "subcategory": rng.integers(0, num_categories, size=(B, T))}
    news["title"][:, :, 12:] = 0
    if abstract:
        a = rng.integers(1, num_words, size=(B, T, 50))
        a[:, :, 35:] = 0
        a[:, ::7] = 0                                    # pad-only abstracts
        a[:, 3::11, 1:] = 0                              # one-token abstracts
        news["abstract"] = a
    return {k: v.astype(np.int64) for k, v in news.items()}


def _items(news, attrs):
    T = news[attrs[0]].shape[1]
    return [{a: torch.from_numpy(np.ascontiguousarray(news[a][:, j])) for a in attrs} for j in range(T)]


# ---- CPU -----------------------------------------------------------------------------------------------------------
def test_fp64_restatement_pinned_against_reference(g1):
    """The restatement reproduces the live reference: title-configuration logits, loss and every gradient, and the
    abstract-configuration news vectors."""
    m, sd = _exp1_state(ATTRS, 101)
    news = {a: g1["train/" + a] for a in ATTRS}
    K1 = int(g1["train/n_cand"])
    loss, logits, grads = exp1_fp64(_named(m, sd), news, K1, ATTRS)
    np.testing.assert_allclose(logits, g1["train/logits"], atol=5e-6)
    assert abs(loss - float(g1["train/loss"])) < 1e-6
    assert set(grads) == {k[5:] for k in g1 if k.startswith("grad/")}
    # gradients that vanish in exact arithmetic (the additive attention's bias before a softmax) hold only the
    # reference's fp32 rounding noise: a floor relative to the largest gradient
    floor = 1e-6 * max(float(g1["absmax/grad/" + k]) for k in grads)
    for k, g in grads.items():
        scale = max(float(g1["absmax/grad/" + k]), 1e-12)
        err = float(np.abs(pinned(g, 48) - g1["grad/" + k]).max())
        assert err <= 2e-5 * scale + floor, (k, err, scale)
        norm = float(g1["gradnorm/" + k])
        assert abs(float(np.linalg.norm(g)) - norm) <= 2e-5 * norm + floor * np.sqrt(g.size), k

    # abstract configuration: the news vectors of the fixture, through the restatement's own news-encoder path
    m, sd = _exp1_state(ATTRS_A, 102)
    news = {a: g1["fwda/" + a][:, None] for a in ATTRS_A}           # [17, 1, ...]: one "candidate" per row
    P = {k: torch.tensor(np.asarray(v, dtype=np.float64)) for k, v in _named(m, sd).items()}
    vecs = []
    for a in ("abstract", "title"):
        pre = f"news_encoder.text_encoders.{a}"
        x = F.embedding(torch.as_tensor(news[a][:, 0]), _shared(P, f"{pre}.word_embedding.weight"), padding_idx=0)
        vecs.append(_additive(_mhsa(x, P, f"{pre}.multihead_self_attention"), P, f"{pre}.additive_attention"))
    for a in ("category", "subcategory"):
        pre = f"news_encoder.element_encoders.{a}"
        e = F.embedding(torch.as_tensor(news[a][:, 0]), _shared(P, f"{pre}.embedding.weight"), padding_idx=0)
        vecs.append(torch.relu(F.linear(e, P[f"{pre}.linear.weight"], P[f"{pre}.linear.bias"])))
    nv = _additive(torch.stack(vecs, dim=1), P, "news_encoder.final_attention").numpy()
    assert rel_l2_rows(nv, g1["fwda/news_vectors"]) < 2e-6


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from newsrecommendationsystem_b200 import _lib
    return _lib.load()


def _al(nbytes):
    return (nbytes + 255) // 256 * 256


def test_abi_lengths_and_sizes_at_50(lib):
    """Training forms take L = 20 or 50; any other length is refused before a CUDA call.  Stash and backward workspace
    at L = 50 hold what the kernels carve out of them."""
    for L in (30, 21, 49):
        rc = lib.nrms_news_encoder_fwd(None, 8, L, None, 10, None, None, None, None, None, None, C.c_void_p(256), None, 0,
                                       0.0, 0, 0, 1, None)
        assert rc == 2 and b"unsupported" in lib.nrms_last_error()
        rc = lib.nrms_news_encoder_bwd(None, None, 8, L, 10, None, None, None, None, None, None, None, None, None, None,
                                       None, 0, 0.0, 0, 0, 1, None)
        assert rc == 2
        rc = lib.nrms_news_encoder_rows_bwd(None, None, 4, C.c_void_p(256), 8, L, 10, *[None] * 14, 0, 0.0, 0, 0, 1, None)
        assert rc == 2
    n = 7040
    rows = n * 50
    assert lib.nrms_encoder_stash_bytes(n, 50) == sum(_al(rows * w * 4) for w in (300, 900, 300, 200, 1))
    ldr = (rows + 3) // 4 * 4
    base = sum(_al(x * 4) for x in (rows * 300, rows * 200, rows * 900, rows * 300, 296 * 900))
    assert lib.nrms_encoder_bwd_workspace_bytes(n, 50, 0) == base + 256
    assert lib.nrms_encoder_bwd_workspace_bytes(n, 50, 1) == base + sum(_al(x * 4) for x in (ldr * 900, ldr * 300,
                                                                                             900 * 300)) + 256
    assert lib.nrms_encoder_fwd_workspace_bytes(n, 50, 1, 1, 401) == 256


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _abstracts(rng, n, num_words):
    toks = rng.integers(1, num_words, size=(n, 50)).astype(np.int64)
    toks[:, 30:] = 0
    toks[0] = 0                                           # a pad-only abstract
    if n > 1:
        toks[1, 1:] = 0                                   # a one-token abstract
    if n > 6:
        toks[5] = 0
        toks[6, 1:] = 0
    return toks


def _weights(golden_sd, dev):
    from newsrecommendationsystem_b200.ops import pack_qkv
    pk = O.enc_keys(O.NEWS)
    sd = {k: torch.from_numpy(v).to(dev) for k, v in golden_sd.items()}
    wqkv, bqkv = pack_qkv(sd[pk["Wq"]], sd[pk["bq"]], sd[pk["Wk"]], sd[pk["bk"]], sd[pk["Wv"]], sd[pk["bv"]])
    return (sd[O.EMB_KEY].contiguous(), wqkv.contiguous(), bqkv.contiguous(), sd[pk["Wa"]].contiguous(),
            sd[pk["ba"]].contiguous(), sd[pk["qa"]].contiguous())


def _encoder_fwd(lib, dev, toks, w, mode, p, seed, offset):
    """One training-form news-encoder forward at L = toks.shape[1] -> (out, stash bytes)."""
    from newsrecommendationsystem_b200._lib import check, ptr
    emb, wqkv, bqkv, wa, ba, qa = w
    n, L = toks.shape
    t_toks = torch.from_numpy(toks).to(dev)
    out = torch.empty((n, 300), dtype=torch.float32, device=dev)
    stash = torch.zeros(int(lib.nrms_encoder_stash_bytes(n, L)), dtype=torch.uint8, device=dev)
    ws = torch.empty(int(lib.nrms_encoder_fwd_workspace_bytes(n, L, mode, 1, emb.shape[0])), dtype=torch.uint8, device=dev)
    check(lib.nrms_news_encoder_fwd(ptr(t_toks), n, L, ptr(emb), emb.shape[0], ptr(wqkv), ptr(bqkv), ptr(wa), ptr(ba),
                                    ptr(qa), ptr(out), ptr(stash), ptr(ws), ws.numel(), p, seed, offset, mode,
                                    _stream(dev)), "nrms_news_encoder_fwd")
    return out, stash, t_toks


def _stash_views(stash, rows):
    """X [rows,300], QKV [rows,900], C [rows,300] of a stash (256-byte aligned pieces)."""
    raw = stash.cpu().numpy()
    o, out = 0, []
    for w in (300, 900, 300):
        out.append(raw[o:o + rows * w * 4].view(np.float32).reshape(rows, w))
        o += _al(rows * w * 4)
    return out


def _attn64(qkv, n, S):
    q, k, v = (qkv[:, i * 300:(i + 1) * 300].reshape(n, S, 15, 20).transpose(0, 2, 1, 3).astype(np.float64) for i in range(3))
    e = np.exp(q @ k.transpose(0, 1, 3, 2) / np.sqrt(20.0))
    attn = e / (e.sum(-1, keepdims=True) + 1e-8)
    return q, k, v, attn


def _merge(a, n, S):
    return a.transpose(0, 2, 1, 3).reshape(n * S, 300)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 5, 6, 7, 333, 7040])
def test_attention50_kernels_vs_fp64(lib, dev, golden_sd, n):
    """The tensor-mode 50-token attention, forward and backward, fed the stashed q|k|v rows, against fp64 attention and
    its gradient (dropout p = 0.2 on the context); dQKV^T equals dQKV bitwise; the masks equal the FP32 mode's."""
    from newsrecommendationsystem_b200 import _lib
    from newsrecommendationsystem_b200._lib import check, ptr
    rng = np.random.default_rng(50 + n)
    toks = _abstracts(rng, n, golden_sd[O.EMB_KEY].shape[0])
    w = _weights(golden_sd, dev)
    S, rows, p, seed, offset = 50, n * 50, 0.2, 4321, 99
    out, stash, t_toks = _encoder_fwd(lib, dev, toks, w, _lib.MODE_TF32, p, seed, offset)
    _, stash32, _ = _encoder_fwd(lib, dev, toks, w, _lib.MODE_FP32, p, seed, offset)
    torch.cuda.synchronize()
    _, QKV, Cm = _stash_views(stash, rows)
    Cm32 = _stash_views(stash32, rows)[2]
    scale = np.float32(1.25)
    mask2 = np.where(Cm != 0, scale, np.float32(0))
    assert np.array_equal(Cm != 0, Cm32 != 0)                    # the same Philox stream in both modes
    # sample the reference for the largest batch (fp64 attention of 7,040 x 15 heads would need 2 GB)
    sel = np.arange(n) if n <= 333 else np.unique(np.concatenate([np.arange(16), np.arange(n - 16, n),
                                                                 rng.choice(n, 32, replace=False)]))
    qkv_s = QKV.reshape(n, S, 900)[sel].reshape(-1, 900)
    q, k, v, attn = _attn64(qkv_s, len(sel), S)
    ctx = _merge(attn @ v, len(sel), S)
    m2s = mask2.reshape(n, S, 300)[sel].reshape(-1, 300)
    got = Cm.reshape(n, S, 300)[sel].reshape(-1, 300)
    vmax = float(np.abs(v).max())
    err_f = float(np.abs(got - ctx * m2s).max())
    assert err_f < 2e-3 * vmax, (err_f, vmax)
    assert np.isfinite(Cm).all()

    # backward through the ABI; the workspace keeps d_c (the attention's incoming gradient, before the mask), dQKV and,
    # in tensor mode, dQKV^T
    emb, wqkv, bqkv, wa, ba, qa = w
    d_out = torch.from_numpy(rng.standard_normal((n, 300)).astype(np.float32)).to(dev)
    grads = [torch.zeros_like(x) for x in (emb, wqkv, bqkv, wa, ba, qa)]
    ws = torch.zeros(int(lib.nrms_encoder_bwd_workspace_bytes(n, S, _lib.MODE_TF32)), dtype=torch.uint8, device=dev)
    check(lib.nrms_news_encoder_bwd(ptr(d_out), ptr(t_toks), n, S, emb.shape[0], ptr(wqkv), ptr(wa), ptr(qa), ptr(stash),
                                    *[ptr(g) for g in (grads[0], grads[1], grads[2], grads[3], grads[4], grads[5])],
                                    ptr(ws), ws.numel(), p, seed, offset, _lib.MODE_TF32, _stream(dev)),
          "nrms_news_encoder_bwd")
    torch.cuda.synchronize()
    raw = ws.cpu().numpy()
    o_dc = 0
    o_dqkv = _al(rows * 300 * 4) + _al(rows * 200 * 4)
    o_t1 = o_dqkv + _al(rows * 900 * 4) + _al(rows * 300 * 4) + _al(296 * 900 * 4)
    ldr = (rows + 3) // 4 * 4
    d_c = raw[o_dc:o_dc + rows * 1200].view(np.float32).reshape(rows, 300)
    d_qkv = raw[o_dqkv:o_dqkv + rows * 3600].view(np.float32).reshape(rows, 900)
    t1 = raw[o_t1:o_t1 + ldr * 3600].view(np.float32).reshape(900, ldr)
    assert np.array_equal(t1[:, :rows], d_qkv.T)
    g = (d_c.reshape(n, S, 300)[sel].reshape(-1, 300) * m2s).reshape(len(sel), S, 15, 20).transpose(0, 2, 1, 3)
    g = g.astype(np.float64)
    dv = attn.transpose(0, 1, 3, 2) @ g
    dattn = g @ v.transpose(0, 1, 3, 2)
    ds = attn * (dattn - (attn * dattn).sum(-1, keepdims=True)) / np.sqrt(20.0)
    dq, dk = ds @ k, ds.transpose(0, 1, 3, 2) @ q
    ref = np.concatenate([_merge(x, len(sel), S) for x in (dq, dk, dv)], axis=1)
    got = d_qkv.reshape(n, S, 900)[sel].reshape(-1, 900)
    # a pad-only text has equal keys and values: its dQ and dK vanish in exact arithmetic and hold rounding noise only
    floor = 1e-5 * float(np.abs(ref).max())
    for i, name in enumerate("QKV"):
        r, a = ref[:, i * 300:(i + 1) * 300], got[:, i * 300:(i + 1) * 300]
        sc = float(np.abs(r).max()) + 1e-30
        err = float(np.abs(a - r).max())
        print(f"attention50[n={n}] d{name}: max err / max |ref| = {err / sc:.2e}")
        assert err < 3e-3 * sc + floor, (name, err, sc)
    assert np.isfinite(d_qkv).all()


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 2e-5), ("tf32", 1e-3)])
def test_dropout_at_50_tokens(lib, dev, golden_sd, precision, tol):
    """The two dropout sites of a 50-token text read back through the stash: masks exactly {0, 1.25}, keep rate
    0.8 +- 4 sigma, and the train-mode output equals the oracle's forward fed with those masks."""
    from newsrecommendationsystem_b200 import _lib
    mode = _lib.MODES[precision]
    n, S, p = 96, 50, 0.2
    rng = np.random.default_rng(5)
    toks = _abstracts(rng, n, golden_sd[O.EMB_KEY].shape[0])
    w = _weights(golden_sd, dev)
    out, stash, _ = _encoder_fwd(lib, dev, toks, w, mode, p, 1234, 17)
    torch.cuda.synchronize()
    rows = n * S
    X, QKV, Cm = _stash_views(stash, rows)
    scale = np.float32(1.25)
    E = golden_sd[O.EMB_KEY][toks.reshape(-1)]
    known = np.abs(E) > 1e-20
    kept = X != 0
    assert np.all(X[known & kept] == E[known & kept] * scale)
    assert np.all(X[~known] == 0)
    mask1 = np.where(known, np.where(kept, scale, np.float32(0)), scale).astype(np.float32)
    rate1 = float((known & kept).sum()) / int(known.sum())
    assert abs(rate1 - 0.8) < 4 * np.sqrt(0.16 / int(known.sum())), rate1
    q, k, v, attn = _attn64(QKV, n, S)
    ctx = _merge(attn @ v, n, S)
    big = np.abs(ctx) > (1e-4 if precision == "fp32" else 5e-2)
    kept2 = Cm != 0
    ratio = Cm[big & kept2] / ctx[big & kept2]
    assert big.mean() > 0.3
    assert np.all(np.abs(ratio - scale) < 2e-2), (ratio.min(), ratio.max())
    rate2 = float((big & kept2).sum()) / int(big.sum())
    assert abs(rate2 - 0.8) < 4 * np.sqrt(0.16 / int(big.sum())), rate2
    mask2 = np.where(kept2, scale, np.float32(0)).astype(np.float32)
    ref, _ = O.news_encoder_forward(golden_sd, toks, mask1=mask1.reshape(n, S, 300), mask2=mask2.reshape(n, S, 300))
    err = rel_l2_rows(out.cpu().numpy(), ref)
    print(f"dropout50[{precision}]: keep rates {rate1:.4f} / {rate2:.4f}; train-mode forward vs oracle {err:.2e}")
    assert err < tol


@pytest.mark.gpu
def test_title_and_abstract_encoders_draw_different_masks(lib, dev, golden_sd, monkeypatch):
    """One train-mode Exp1 step with abstracts: the two text encoders start their streams at the same offset, so their
    keys must differ -- and the masks those keys give differ."""
    from newsrecommendationsystem_b200 import _lib, ops
    m, sd = _exp1_state(ATTRS_A, 102)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.to(dev).train().set_precision("tf32")
    calls = []
    real = ops.news_encoder

    def spy(tokens, *a, **kw):
        calls.append((tokens.shape[1], kw["seed"], kw["offset"], kw["dropout_p"]))
        return real(tokens, *a, **kw)
    monkeypatch.setattr(ops, "news_encoder", spy)
    items = _items(_batch(np.random.default_rng(3), 2), ATTRS_A)
    ops.cross_entropy_label0(m(items[:N_CAND], items[N_CAND:])).backward()
    by_len = {L: (s, o, p) for L, s, o, p in calls}
    assert set(by_len) == {20, 50} and by_len[20][1] == by_len[50][1] == 0 and by_len[20][2] == 0.2
    assert by_len[20][0] != by_len[50][0]
    toks = _abstracts(np.random.default_rng(4), 8, golden_sd[O.EMB_KEY].shape[0])
    toks[:] = np.maximum(toks, 1)
    w = _weights(golden_sd, dev)
    masks = []
    for L in (20, 50):
        _, stash, _ = _encoder_fwd(lib, dev, toks, w, _lib.MODE_TF32, 0.2, by_len[L][0], 0)
        masks.append(_stash_views(stash, 8 * 50)[0] != 0)
    assert not np.array_equal(masks[0], masks[1])


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_text_encoder_backward_at_50_tokens(lib, dev, golden_sd, precision):
    """The autograd news encoder at L = 50 with dropout against O.encoder_backward fed the kernels' masks, every
    gradient including the embedding's (row 0 = padding_idx untouched)."""
    from newsrecommendationsystem_b200 import _lib, ops
    mode = _lib.MODES[precision]
    n, S, p, seed, offset = 64, 50, 0.2, 777, 5
    rng = np.random.default_rng(8)
    toks = _abstracts(rng, n, golden_sd[O.EMB_KEY].shape[0])
    w = _weights(golden_sd, dev)
    _, stash, t_toks = _encoder_fwd(lib, dev, toks, w, mode, p, seed, offset)
    X, _, Cm = _stash_views(stash, n * S)
    E = golden_sd[O.EMB_KEY][toks.reshape(-1)]
    known = np.abs(E) > 1e-20
    mask1 = np.where(known, np.where(X != 0, 1.25, 0.0), 1.25).reshape(n, S, 300)
    mask2 = np.where(Cm != 0, 1.25, 0.0).reshape(n, S, 300)
    leaves = [x.detach().clone().requires_grad_(True) for x in w]
    out = ops.news_encoder(t_toks, *leaves, dropout_p=p, seed=seed, offset=offset, mode=mode)
    d_out = rng.standard_normal((n, 300))
    got = torch.autograd.grad(out, leaves, torch.from_numpy(d_out.astype(np.float32)).to(dev))
    P64 = {k: v.astype(np.float64) for k, v in golden_sd.items()}
    ref_out, cache = O.news_encoder_forward(P64, toks, mask1=mask1, mask2=mask2)
    dx, gr = O.encoder_backward(d_out, cache, O.enc_params(P64, O.NEWS), 15)
    dE = np.zeros_like(P64[O.EMB_KEY])
    np.add.at(dE, toks.reshape(-1), (dx * mask1).reshape(-1, 300))
    dE[0] = 0
    ref = [dE, np.concatenate([gr["Wq"], gr["Wk"], gr["Wv"]]), np.concatenate([gr["bq"], gr["bk"], gr["bv"]]),
           gr["Wa"], gr["ba"], gr["qa"]]
    gtol = {"fp32": 2e-4, "tf32": 3e-3}[precision]
    floor = 1e-6 * max(float(np.abs(r).max()) for r in ref)
    assert rel_l2_rows(out.detach().cpu().numpy(), ref_out) < (2e-5 if precision == "fp32" else 1e-3)
    for name, a, r in zip(("emb", "wqkv", "bqkv", "wa", "ba", "qa"), got, ref):
        a = a.cpu().numpy()
        sc = float(np.abs(r).max()) + 1e-12
        err = float(np.abs(a - r).max())
        print(f"text encoder 50 [{precision}] d{name}: err / scale {err / sc:.2e}")
        assert err <= gtol * sc + floor, (name, err, sc)
    assert not got[0][0].any()


# (loss, gradient / scale) bounds of the single-step title tests; the 50-term sums of the abstract encoder need no more
EXP1_TOL = {"fp32": (1e-5, 2e-4), "tf32": (2e-3, 3e-3)}


def _exp1_model(dev, precision, train=False, seed=102):
    m, sd = _exp1_state(ATTRS_A, seed)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.to(dev).set_precision(precision)
    m.train(train)
    return m, sd


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_exp1_with_abstract_gradients_vs_fp64(dev, precision):
    """Exp1(['category', 'subcategory', 'title', 'abstract']).forward + CE(label 0) + backward, eval-mode dropout:
    logits, loss and every parameter gradient against the fp64 restatement."""
    from newsrecommendationsystem_b200 import ops
    m, sd = _exp1_model(dev, precision)
    news = _batch(np.random.default_rng(11), 6)
    items = _items(news, ATTRS_A)
    logits = m(items[:N_CAND], items[N_CAND:])
    loss = ops.cross_entropy_label0(logits)
    m.zero_grad()
    loss.backward()
    loss_ref, logits_ref, grads = exp1_fp64(_named(m, sd), news, N_CAND, ATTRS_A)
    ltol, gtol = EXP1_TOL[precision]
    np.testing.assert_allclose(logits.detach().cpu().numpy(), logits_ref, atol=10 * ltol)
    assert abs(float(loss.detach()) - loss_ref) < ltol
    floor = 1e-6 * max(float(np.abs(v).max()) for v in grads.values())
    worst = 0.0
    for k, p in m.named_parameters():
        ref = grads[k]
        sc = float(np.abs(ref).max()) + 1e-12
        err = float(np.abs(p.grad.detach().cpu().numpy() - ref).max())
        worst = max(worst, err / (gtol * sc + floor))
        assert err <= gtol * sc + floor, (k, err, sc)
    print(f"exp1+abstract [{precision}]: loss err {abs(float(loss.detach()) - loss_ref):.2e}, worst gradient err / bound "
          f"{worst:.2f}")


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_exp1_forward_rows_and_train_step(dev, precision):
    """forward_rows over a dict news table equals the list-of-dict forward (train mode: same dropout stream), refuses
    out-of-range rows, and TrainStep drives Exp1 with abstracts through step and step_rows; the first step's Adam
    transition matches O.adam_step on the step's own gradients."""
    from newsrecommendationsystem_b200 import ops
    from newsrecommendationsystem_b200.train import TrainStep
    rng = np.random.default_rng(13)
    N, B = 300, 4
    table = {"title": rng.integers(1, 401, size=(N + 1, 20)), "abstract": rng.integers(1, 401, size=(N + 1, 50)),
             "category": rng.integers(1, 31, size=N + 1), "subcategory": rng.integers(1, 31, size=N + 1)}
    table["abstract"][::5, 20:] = 0
    table["abstract"][1::9, 1:] = 0
    for v in table.values():
        v[N] = 0                                             # the pad row
    cand = rng.integers(0, N, size=(B, N_CAND))
    hist = rng.integers(0, N + 1, size=(B, N_CLICKED))
    dev_table = {k: torch.from_numpy(v.astype(np.int64)).to(dev) for k, v in table.items()}
    rows = np.concatenate([cand, hist], axis=1)
    news = {k: v[rows].astype(np.int64) for k, v in table.items()}

    m1, _ = _exp1_model(dev, precision, train=True)
    m2, _ = _exp1_model(dev, precision, train=True)
    l1 = ops.cross_entropy_label0(m1.forward_rows(dev_table, torch.from_numpy(cand), torch.from_numpy(hist)))
    l1.backward()
    items = _items(news, ATTRS_A)
    l2 = ops.cross_entropy_label0(m2(items[:N_CAND], items[N_CAND:]))
    l2.backward()
    assert abs(float(l1.detach()) - float(l2.detach())) < 1e-6
    for (k, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
        sc = max(float(b.grad.abs().max()), 1e-12)
        assert float((a.grad - b.grad).abs().max()) <= 2e-5 * sc + 1e-9, k

    m3, _ = _exp1_model(dev, precision, train=True)
    ts = TrainStep(m3)
    with pytest.raises(IndexError):
        ts.step_rows(dev_table, torch.from_numpy(cand + N + 1), torch.from_numpy(hist))
    names = [n for n, _ in m3.named_parameters()]
    params = dict(m3.named_parameters())
    P0 = {n: params[n].detach().cpu().numpy().astype(np.float64) for n in names}
    losses = [float(ts.step(items[:N_CAND], items[N_CAND:]))]
    f32 = lambda x: float(np.float32(x))                     # noqa: E731  (the fp32 arguments of nrms_adam_step)
    for n in names:
        g = params[n].grad.detach().cpu().numpy().astype(np.float64)
        p_ref, _, _ = O.adam_step(P0[n], g, np.zeros_like(g), np.zeros_like(g), 1, lr=f32(1e-4), beta1=f32(0.9),
                                  beta2=f32(0.999), eps=f32(1e-8))
        e = np.abs(params[n].detach().cpu().numpy() - p_ref)
        assert (e <= 2e-8 + 2 * np.spacing(np.abs(p_ref).astype(np.float32))).all(), (n, float(e.max()))
    for _ in range(2):
        losses.append(float(ts.step_rows(dev_table, torch.from_numpy(cand), torch.from_numpy(hist))))
        losses.append(float(ts.step(items[:N_CAND], items[N_CAND:])))
    assert all(np.isfinite(losses)) and ts.steps == 5, losses
