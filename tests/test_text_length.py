"""Titles and abstracts of any length from 1 to 64 (config.num_words_title / num_words_abstract): the text encoder,
NRMS and Exp1 training, evaluate and the single-user path at lengths other than the compiled 20 and 50.

CPU part: the length rule of nrms_text_encoder_fwd / _bwd, a numpy restatement of the Philox4x32-10 dropout stream pinned
against the Random123 known-answer vectors, and the models' width rule.  GPU part (`-m gpu`): the masks every path draws,
bit for bit against the restatement; every result against the fp64 oracle (`oracle/`) or the fp64 Exp1 restatement of
test_exp1_abstract_train.py, with train-mode dropout fed the restated masks; bitwise identities between the forms.
"""
import csv
import json
import os
import shutil

import numpy as np
import pytest
import torch

from conftest import rel_l2_rows
from oracle import nrms_oracle as O

TOL_VEC = {"fp32": 2e-5, "tf32": 1e-3}          # test_gpu_parity.py: news / user vectors, max row-wise relative L2
GTOL = {"fp32": 2e-4, "tf32": 3e-3}             # gradients, relative to the tensor's largest entry
INFER_CHUNK_ROWS = 2048 * 20                    # encoder.cu: rows per inference pass
STREAM_EMB, STREAM_CTX = 1, 2                   # encoder_kernels.cuh: Philox stream of dropout #1 / #2
NEWS_LN = {"ln_g": "news_encoder.layer_norm.weight", "ln_b": "news_encoder.layer_norm.bias"}


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from newsrecommendationsystem_b200 import _lib
    return _lib.load()


# ---- Philox4x32-10 and dropout_mask4 (common.cuh), vectorised ---------------------------------------------------------
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Arrays of 32-bit words held in uint64 (each product of two words fits)."""
    c0, c1, c2, c3, k0, k1 = (np.asarray(x, dtype=np.uint64) for x in (c0, c1, c2, c3, k0, k1))
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _M32
        k0 = (k0 + np.uint64(0x9E3779B9)) & _M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & _M32
    return c0, c1, c2, c3


def dropout_mask(rows, p, seed, offset, stream):
    """The multiplicative mask of a [rows, 300] activation: element e draws lane e % 4 of Philox((e / 4 + offset,
    stream, 0), seed) and keeps with scale 1 / (1 - p) iff word * 2^-32 >= p, all in fp32 as the kernels do."""
    c = np.arange(rows * 75, dtype=np.uint64) + np.uint64(offset)
    r = philox4x32_10(c & _M32, c >> np.uint64(32), np.full_like(c, stream), np.zeros_like(c),
                      np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32))
    u = np.stack(r, axis=1).astype(np.uint32).astype(np.float32) * np.float32(2.0 ** -32)
    scale = np.float32(1) / (np.float32(1) - np.float32(p))
    return np.where(u >= np.float32(p), scale, np.float32(0)).reshape(rows, 300)


def test_philox_known_answers():
    """Random123's kat_vectors for philox4x32_10."""
    got = philox4x32_10(0, 0, 0, 0, 0, 0)
    assert [int(x) for x in got] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    m = 0xFFFFFFFF
    got = philox4x32_10(m, m, m, m, m, m)
    assert [int(x) for x in got] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    got = philox4x32_10(0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344, 0xa4093822, 0x299f31d0)
    assert [int(x) for x in got] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_dropout_mask_layout():
    """Four consecutive elements share one evaluation; the offset shifts the counter by one per four elements; the
    keep rate is 1 - p."""
    m = dropout_mask(400, 0.2, 1234, 0, STREAM_CTX)
    assert set(np.unique(m)) <= {0.0, 1.25}
    assert abs((m != 0).mean() - 0.8) < 0.01
    shifted = dropout_mask(399, 0.2, 1234, 75, STREAM_CTX)
    assert np.array_equal(m[1:], shifted)
    assert not np.array_equal(m, dropout_mask(400, 0.2, 1234, 0, STREAM_EMB))
    c = philox4x32_10(5, 0, STREAM_CTX, 0, 1234, 0)
    u = np.array([int(x) for x in c], dtype=np.uint32).astype(np.float32) * np.float32(2.0 ** -32)
    assert np.array_equal(m.reshape(-1)[20:24] != 0, u >= np.float32(0.2))


# ---- CPU: the C-ABI length rule ---------------------------------------------------------------------------------------
def _text_calls(lib, L):
    """nrms_text_encoder_fwd / _bwd in the dense, index-only and LayerNorm forms, with null pointers (4 texts; the
    index-only forward names a stash, the form it needs, which the call never reaches)."""
    n, rows, g, stash = None, 1, 1, 256
    return {
        "fwd": lambda: lib.nrms_text_encoder_fwd(n, 4, n, 4, L, n, 10, n, n, n, n, n, n, n, n, n, n, 0, 0.0, 0, 0, 0, n),
        "rows_fwd": lambda: lib.nrms_text_encoder_fwd(n, 10, rows, 4, L, n, 10, n, n, n, n, n, n, n, n, stash, n, 0, 0.0,
                                                      0, 0, 0, n),
        "ln_fwd": lambda: lib.nrms_text_encoder_fwd(n, 4, n, 4, L, n, 10, n, n, g, g, n, n, n, n, n, n, 0, 0.0, 0, 0, 0,
                                                    n),
        "bwd": lambda: lib.nrms_text_encoder_bwd(n, n, 4, n, 4, L, 10, n, n, n, n, n, n, n, n, n, n, n, n, n, n, 0, 0.0,
                                                 0, 0, 0, n),
        "rows_bwd": lambda: lib.nrms_text_encoder_bwd(n, n, 10, rows, 4, L, 10, n, n, n, n, n, n, n, n, n, n, n, n, n, n,
                                                      0, 0.0, 0, 0, 0, n),
        "ln_bwd": lambda: lib.nrms_text_encoder_bwd(n, n, 4, n, 4, L, 10, n, g, n, n, n, n, n, n, g, g, n, n, n, n, 0,
                                                    0.0, 0, 0, 0, n),
    }


@pytest.mark.parametrize("L", [0, -1, 65])
def test_text_encoder_refuses_lengths_outside_1_to_64(lib, L):
    for name, call in _text_calls(lib, L).items():
        assert call() == 2 and b"unsupported" in lib.nrms_last_error(), name


@pytest.mark.parametrize("L", [1, 37, 64])
def test_text_encoder_takes_lengths_1_to_64(lib, L):
    """Past the length check, the null pointers are what the call refuses."""
    for name, call in _text_calls(lib, L).items():
        assert call() == 1, (name, lib.nrms_last_error())


def test_news_encoder_entries_keep_20_and_50(lib):
    """nrms_news_encoder_* keep their rule where the new pair takes the length."""
    n = None
    assert lib.nrms_news_encoder_fwd(n, 4, 30, n, 10, n, n, n, n, n, n, n, n, 0, 0.0, 0, 0, 0, n) == 2
    assert lib.nrms_text_encoder_fwd(n, 4, n, 4, 30, n, 10, n, n, n, n, n, n, n, n, n, n, 0, 0.0, 0, 0, 0, n) == 1


# ---- CPU: the models' width rule --------------------------------------------------------------------------------------
class _Cfg:
    num_words = 401
    word_embedding_dim = 300
    num_attention_heads = 15
    query_vector_dim = 200
    dropout_probability = 0.2
    num_words_title = 30
    num_clicked_news_a_user = 50


def test_nrms_width_rule():
    from newsrecommendationsystem_b200 import NRMS
    m = NRMS(_Cfg)
    with pytest.raises(RuntimeError, match="num_words_title = 30"):
        m.get_news_vector({"title": torch.ones((3, 21), dtype=torch.int64)})
    with pytest.raises(RuntimeError, match="num_words_title = 30"):
        m.news_encoder.encode_tokens(torch.ones((3, 31), dtype=torch.int64))


def test_exp1_width_rule():
    from newsrecommendationsystem_b200 import Exp1
    from test_exp1_recommend import ATTRS_A, _cfg

    class Cfg(_cfg(ATTRS_A)):
        num_words_abstract = 64
    m = Exp1(Cfg)
    enc = m.news_encoder.text_encoders
    assert enc["abstract"].num_words == ("num_words_abstract", 64)
    assert enc["title"].num_words == ("num_words_title", 20)
    with pytest.raises(RuntimeError, match="num_words_abstract = 64"):
        enc["abstract"](torch.ones((2, 63), dtype=torch.int64))
    with pytest.raises(RuntimeError, match="num_words_title = 20"):
        enc["title"](torch.ones((2, 63), dtype=torch.int64))


# ---- GPU helpers ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _params(golden_sd, ln, seed=3):
    """fp64 state dict of the oracle (the golden weights; the LayerNorm weight and bias drawn)."""
    P = {k: v.astype(np.float64) for k, v in golden_sd.items()}
    if ln:
        rng = np.random.default_rng(seed)
        P[NEWS_LN["ln_g"]] = (1 + 0.2 * rng.standard_normal(300)).astype(np.float32).astype(np.float64)
        P[NEWS_LN["ln_b"]] = (0.1 * rng.standard_normal(300)).astype(np.float32).astype(np.float64)
    return P


def _weights(P, dev):
    """Device fp32 (emb, wqkv, bqkv, wa, ba, qa) and the LayerNorm pair (or None)."""
    p = O.enc_params(P, O.NEWS)
    w = [P[O.EMB_KEY], np.concatenate([p["Wq"], p["Wk"], p["Wv"]]), np.concatenate([p["bq"], p["bk"], p["bv"]]),
         p["Wa"], p["ba"], p["qa"]]
    w = [_t(x.astype(np.float32), dev) for x in w]
    ln = (_t(p["ln_g"].astype(np.float32), dev), _t(p["ln_b"].astype(np.float32), dev)) if "ln_g" in p else None
    return w, ln


def _texts(rng, n, L, V):
    """Right-padded texts, with pad-only and one-token texts among them."""
    t = rng.integers(1, V, size=(n, L))
    t[1::3, max(1, L // 2):] = 0
    t[::7] = 0
    t[3::11, 1:] = 0
    return t.astype(np.int64)


def _masks(n_rows, p, seed, offset):
    return dropout_mask(n_rows, p, seed, offset, STREAM_EMB), dropout_mask(n_rows, p, seed, offset, STREAM_CTX)


def _stash_xc(stash, rows):
    al = lambda nfl: (nfl * 4 + 255) // 256 * 256               # the stash carves 256-byte aligned pieces
    raw = stash.cpu().numpy()
    X = raw[:rows * 1200].view(np.float32).reshape(rows, 300)
    o = al(rows * 300) + al(rows * 900)
    C = raw[o:o + rows * 1200].view(np.float32).reshape(rows, 300)
    return X, C


def _ptr(t):
    import ctypes as C
    return None if t is None else C.c_void_p(t.data_ptr())


def _abi_fwd(lib, dev, entry, table, rows, w, ln, L, mode, p, seed, offset):
    """One training forward through the raw ABI: entry "text" (nrms_text_encoder_fwd) or "news" (the
    nrms_news_encoder_* form of the call).  table int64 [*, L] on the device, rows int64 [n] or None.
    -> (out, stash)."""
    from newsrecommendationsystem_b200._lib import check, stream_ptr
    emb, wqkv, bqkv, wa, ba, qa = w
    n = table.shape[0] if rows is None else rows.numel()
    stash = torch.zeros(int((lib.nrms_encoder_ln_stash_bytes if ln else lib.nrms_encoder_stash_bytes)(n, L)),
                        dtype=torch.uint8, device=dev)
    ws = torch.empty(max(256, int(lib.nrms_encoder_fwd_workspace_bytes(n, L, mode, 1, emb.shape[0]))), dtype=torch.uint8,
                     device=dev)
    out = torch.empty((n, 300), dtype=torch.float32, device=dev)
    g, b = ln if ln else (None, None)
    st = stream_ptr(dev)
    P = _ptr
    if entry == "text":
        check(lib.nrms_text_encoder_fwd(P(table), table.shape[0], P(rows), n, L, P(emb), emb.shape[0], P(wqkv), P(bqkv),
                                        P(g), P(b), P(wa), P(ba), P(qa), P(out), P(stash), P(ws), ws.numel(), p, seed,
                                        offset, mode, st), "nrms_text_encoder_fwd")
    elif rows is not None:
        check(lib.nrms_news_encoder_rows_fwd(P(table), table.shape[0], P(rows), n, L, P(emb), emb.shape[0], P(wqkv),
                                             P(bqkv), P(g), P(b), P(wa), P(ba), P(qa), P(out), P(stash), p, seed, offset,
                                             mode, st), "nrms_news_encoder_rows_fwd")
    elif ln:
        check(lib.nrms_news_encoder_ln_fwd(P(table), n, L, P(emb), emb.shape[0], P(wqkv), P(bqkv), P(g), P(b), P(wa),
                                           P(ba), P(qa), P(out), P(stash), P(ws), ws.numel(), p, seed, offset, mode, st),
              "nrms_news_encoder_ln_fwd")
    else:
        check(lib.nrms_news_encoder_fwd(P(table), n, L, P(emb), emb.shape[0], P(wqkv), P(bqkv), P(wa), P(ba), P(qa),
                                        P(out), P(stash), P(ws), ws.numel(), p, seed, offset, mode, st),
              "nrms_news_encoder_fwd")
    return out, stash


def _abi_bwd(lib, dev, entry, table, rows, w, ln, L, mode, p, seed, offset, stash, d_out):
    from newsrecommendationsystem_b200._lib import check, stream_ptr
    emb, wqkv, bqkv, wa, ba, qa = w
    n = table.shape[0] if rows is None else rows.numel()
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
    g = {"emb": z(*emb.shape), "wqkv": z(900, 300), "bqkv": z(900), "wa": z(200, 300), "ba": z(200), "qa": z(200)}
    if ln:
        g["ln_g"], g["ln_b"] = z(300), z(300)
    ws = torch.empty(int(lib.nrms_encoder_bwd_workspace_bytes(n, L, mode)), dtype=torch.uint8, device=dev)
    st = stream_ptr(dev)
    P = _ptr
    lg = ln[0] if ln else None
    dg, db = (g["ln_g"], g["ln_b"]) if ln else (None, None)
    if entry == "text":
        check(lib.nrms_text_encoder_bwd(P(d_out), P(table), table.shape[0], P(rows), n, L, emb.shape[0], P(wqkv), P(lg),
                                        P(wa), P(qa), P(stash), P(g["emb"]), P(g["wqkv"]), P(g["bqkv"]), P(dg), P(db),
                                        P(g["wa"]), P(g["ba"]), P(g["qa"]), P(ws), ws.numel(), p, seed, offset, mode, st),
              "nrms_text_encoder_bwd")
    elif rows is not None:
        check(lib.nrms_news_encoder_rows_bwd(P(d_out), P(table), table.shape[0], P(rows), n, L, emb.shape[0], P(wqkv),
                                             P(lg), P(wa), P(qa), P(stash), P(g["emb"]), P(g["wqkv"]), P(g["bqkv"]),
                                             P(dg), P(db), P(g["wa"]), P(g["ba"]), P(g["qa"]), P(ws), ws.numel(), p, seed,
                                             offset, mode, st), "nrms_news_encoder_rows_bwd")
    elif ln:
        check(lib.nrms_news_encoder_ln_bwd(P(d_out), P(table), n, L, emb.shape[0], P(wqkv), P(lg), P(wa), P(qa),
                                           P(stash), P(g["emb"]), P(g["wqkv"]), P(g["bqkv"]), P(dg), P(db), P(g["wa"]),
                                           P(g["ba"]), P(g["qa"]), P(ws), ws.numel(), p, seed, offset, mode, st),
              "nrms_news_encoder_ln_bwd")
    else:
        check(lib.nrms_news_encoder_bwd(P(d_out), P(table), n, L, emb.shape[0], P(wqkv), P(wa), P(qa), P(stash),
                                        P(g["emb"]), P(g["wqkv"]), P(g["bqkv"]), P(g["wa"]), P(g["ba"]), P(g["qa"]),
                                        P(ws), ws.numel(), p, seed, offset, mode, st), "nrms_news_encoder_bwd")
    return g


# ---- GPU: the masks ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("form", ["dense", "rows"])
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("L", [1, 7, 20, 30, 50, 64])
def test_masks_bit_for_bit(lib, dev, golden_sd, L, precision, form):
    """Both dropout sites read back from the stash equal the numpy restatement: X = E[token] x mask #1 exactly, and C is
    zero exactly where mask #2 is (on entries whose fp64 context is not tiny).  At 20 and 50 the existing
    nrms_news_encoder_* training kernels are checked the same way, so every path draws the same stream."""
    from newsrecommendationsystem_b200 import _lib
    mode = _lib.MODES[precision]
    P = _params(golden_sd, False)
    w, _ = _weights(P, dev)
    rng = np.random.default_rng(L)
    n, p, seed, offset = 97, 0.2, 0xC0FFEE, 12345
    table = _texts(rng, 131, L, golden_sd[O.EMB_KEY].shape[0])
    sel = rng.integers(0, 131, size=n)
    toks = table[sel]
    entries = ["text"] + (["news"] if L in (20, 50) else [])
    for entry in entries:
        if form == "dense":
            _, stash = _abi_fwd(lib, dev, entry, _t(toks, dev), None, w, None, L, mode, p, seed, offset)
        else:
            _, stash = _abi_fwd(lib, dev, entry, _t(table, dev), _t(sel, dev), w, None, L, mode, p, seed, offset)
        torch.cuda.synchronize()
        X, C = _stash_xc(stash, n * L)
        m1, m2 = _masks(n * L, p, seed, offset)
        E = golden_sd[O.EMB_KEY][toks.reshape(-1)]
        assert np.array_equal(X, E * m1), entry
        ctx, _ = O.mhsa_forward(X.astype(np.float64).reshape(n, L, 300), O.enc_params(P, O.NEWS), 15)
        ctx = ctx.reshape(-1, 300)
        big = np.abs(ctx) > 1e-4 * np.abs(ctx).max()
        assert big.mean() > 0.5
        assert np.array_equal((C != 0)[big], (m2 != 0)[big]), (entry, int(((C != 0) != (m2 != 0))[big].sum()))
        assert not C[m2 == 0].any(), entry


# ---- GPU: forward -----------------------------------------------------------------------------------------------------
FWD_LENGTHS = [1, 2, 7, 19, 21, 30, 49, 64]
_worst = {}


@pytest.mark.gpu
@pytest.mark.parametrize("ln", [False, True], ids=["nrms", "ln"])
@pytest.mark.parametrize("L", FWD_LENGTHS)
def test_forward_vs_oracle(dev, golden_sd, L, ln):
    """ops.news_encoder in both modes: eval mode from 1 text to a count that crosses an inference chunk, and train mode
    (p = 0.2, the oracle fed the restated masks) in the dense and index-only forms, which agree bitwise."""
    from newsrecommendationsystem_b200 import ops, _lib
    P = _params(golden_sd, ln)
    w, lnw = _weights(P, dev)
    rng = np.random.default_rng(200 + L)
    V = golden_sd[O.EMB_KEY].shape[0]
    big = _texts(rng, INFER_CHUNK_ROWS // L + 3, L, V)
    ref_big, _ = O.news_encoder_forward(P, big)
    table = _texts(rng, 300, L, V)
    sel = rng.integers(0, 300, size=157)
    seed, offset, p = 99, 4321, 0.2
    m1, m2 = _masks(157 * L, p, seed, offset)
    ref_train, _ = O.news_encoder_forward(P, table[sel], mask1=m1.reshape(157, L, 300), mask2=m2.reshape(157, L, 300))
    for precision in ("fp32", "tf32"):
        mode = _lib.MODES[precision]
        with torch.no_grad():
            for n in (1, big.shape[0]):
                out = ops.news_encoder(_t(big[:n], dev), *w, mode=mode, ln=lnw)
                err = rel_l2_rows(out.cpu().numpy(), ref_big[:n])
                assert err < TOL_VEC[precision], (L, precision, n, err)
                _worst[(precision, ln)] = max(_worst.get((precision, ln), 0.0), err)
            tb = _t(table, dev)
            dense = ops.news_encoder(tb[_t(sel, dev)], *w, dropout_p=p, seed=seed, offset=offset, mode=mode, ln=lnw)
            rows = ops.news_encoder(tb, *w, dropout_p=p, seed=seed, offset=offset, mode=mode, ln=lnw,
                                    news_rows=_t(sel, dev))
        err = rel_l2_rows(rows.cpu().numpy(), ref_train)
        assert err < TOL_VEC[precision], (L, precision, "train", err)
        _worst[(precision, ln, "train")] = max(_worst.get((precision, ln, "train"), 0.0), err)
        assert torch.equal(dense, rows), (L, precision)
    print(f"worst relative L2 so far: { {str(k): f'{v:.2e}' for k, v in _worst.items()} }")


# ---- GPU: backward ----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ln", [False, True], ids=["nrms", "ln"])
@pytest.mark.parametrize("p", [0.0, 0.2])
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("L", [1, 17, 30, 64])
def test_gradients_vs_oracle(dev, golden_sd, L, precision, p, ln):
    """Every gradient of the news encoder (touched embedding rows, Wqkv, bqkv, Wa, ba, qa, the LayerNorm pair) against
    encoder_backward in fp64, with train-mode dropout fed the restated masks."""
    from newsrecommendationsystem_b200 import ops, _lib
    mode = _lib.MODES[precision]
    P = _params(golden_sd, ln)
    w, lnw = _weights(P, dev)
    rng = np.random.default_rng(300 + L)
    n, seed, offset = 41, 0x5EED, 77
    toks = _texts(rng, n, L, golden_sd[O.EMB_KEY].shape[0])
    d_out = rng.standard_normal((n, 300)).astype(np.float32)
    m1, m2 = _masks(n * L, p, seed, offset) if p > 0 else (None, None)
    ref_out, cache = O.news_encoder_forward(P, toks, mask1=None if m1 is None else m1.reshape(n, L, 300),
                                            mask2=None if m2 is None else m2.reshape(n, L, 300))
    dx, gr = O.encoder_backward(d_out.astype(np.float64), cache, O.enc_params(P, O.NEWS), 15)
    if m1 is not None:
        dx = dx * m1.reshape(n, L, 300)
    dE = np.zeros_like(P[O.EMB_KEY])
    np.add.at(dE, toks.reshape(-1), dx.reshape(-1, 300))
    dE[0] = 0
    touched = np.unique(toks[toks > 0])
    ref = {"emb": dE[touched], "wqkv": np.concatenate([gr["Wq"], gr["Wk"], gr["Wv"]]),
           "bqkv": np.concatenate([gr["bq"], gr["bk"], gr["bv"]]), "wa": gr["Wa"], "ba": gr["ba"], "qa": gr["qa"]}
    if ln:
        ref["ln_g"], ref["ln_b"] = gr["ln_g"], gr["ln_b"]
    leaves = [x.detach().clone().requires_grad_(True) for x in w] + \
        ([x.detach().clone().requires_grad_(True) for x in lnw] if ln else [])
    out = ops.news_encoder(_t(toks, dev), *leaves[:6], dropout_p=p, seed=seed, offset=offset, mode=mode,
                           ln=tuple(leaves[6:]) if ln else None)
    assert rel_l2_rows(out.detach().cpu().numpy(), ref_out) < TOL_VEC[precision]
    got = torch.autograd.grad(out, leaves, _t(d_out, dev))
    got = dict(zip(["emb", "wqkv", "bqkv", "wa", "ba", "qa", "ln_g", "ln_b"], [g.cpu().numpy() for g in got]))
    assert not got["emb"][0].any()
    untouched = np.setdiff1d(np.arange(1, dE.shape[0]), touched)
    assert not got["emb"][untouched].any()
    got["emb"] = got["emb"][touched]
    gtol = {"fp32": 3e-4, "tf32": 5e-3}[precision] if ln else GTOL[precision]
    floor = 1e-6 * max(float(np.abs(v).max()) for v in ref.values())
    worst = 0.0
    for k, r in ref.items():
        sc = float(np.abs(r).max()) + 1e-12
        err = float(np.abs(got[k] - r).max())
        assert err <= gtol * sc + floor, (L, k, err, sc)
        worst = max(worst, err / sc)
    print(f"L = {L} [{precision}, p = {p}{', LayerNorm' if ln else ''}]: worst gradient error / largest entry {worst:.2e}")


# ---- GPU: bitwise identities ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("form", ["dense", "ln", "rows"])
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("L", [20, 50])
def test_text_pair_equals_news_encoder_entries(lib, dev, golden_sd, L, precision, form):
    """At 20 and 50 the new pair runs what nrms_news_encoder_{,ln_,rows_}fwd / bwd run: output and stash bitwise, every
    gradient up to the order of its atomic accumulations (the embedding scatter and the split-K weight contractions add
    into their outputs with fp32 atomics, so two runs of the same entry differ in the last bits too)."""
    from newsrecommendationsystem_b200 import _lib
    mode = _lib.MODES[precision]
    P = _params(golden_sd, form == "ln")
    w, lnw = _weights(P, dev)
    rng = np.random.default_rng(L + 7)
    table = _t(_texts(rng, 200, L, golden_sd[O.EMB_KEY].shape[0]), dev)
    rows = _t(rng.integers(0, 200, size=150), dev) if form == "rows" else None
    d_out = _t(rng.standard_normal((150 if rows is not None else 200, 300)).astype(np.float32), dev)
    res = {}
    for entry in ("text", "news"):
        out, stash = _abi_fwd(lib, dev, entry, table, rows, w, lnw, L, mode, 0.2, 5, 9)
        g = _abi_bwd(lib, dev, entry, table, rows, w, lnw, L, mode, 0.2, 5, 9, stash, d_out)
        res[entry] = dict(out=out, stash=stash, **g)
    for k in ("out", "stash"):
        assert torch.equal(res["text"][k], res["news"][k]), k
    for k in res["text"]:
        a, b = res["text"][k], res["news"][k]
        assert float((a - b).abs().max()) <= 1e-5 * float(b.abs().max()), k


@pytest.mark.gpu
def test_i32_and_chunked_inference(dev, golden_sd):
    """At 30 tokens: ops.news_encoder_i32 equals ops.news_encoder on int64 ids; an inference pass that crosses a chunk
    equals single calls over the same rows (with dropout: the second call's offset shifted by its first row x 75)."""
    from newsrecommendationsystem_b200 import ops, _lib
    L = 30
    P = _params(golden_sd, False)
    w, _ = _weights(P, dev)
    rng = np.random.default_rng(30)
    n = INFER_CHUNK_ROWS // L + 40
    toks = _t(_texts(rng, n, L, golden_sd[O.EMB_KEY].shape[0]), dev)
    with torch.no_grad():
        a = ops.news_encoder_i32(toks.int(), *w)
        b = ops.news_encoder(toks, *w, mode=_lib.MODE_TF32)
        assert torch.equal(a, b)
        cut = INFER_CHUNK_ROWS // L
        for precision in ("fp32", "tf32"):
            mode = _lib.MODES[precision]
            for p, off in ((0.0, 0), (0.2, 1001)):
                whole = ops.news_encoder(toks, *w, dropout_p=p, seed=11, offset=off, mode=mode)
                first = ops.news_encoder(toks[:cut], *w, dropout_p=p, seed=11, offset=off, mode=mode)
                rest = ops.news_encoder(toks[cut:], *w, dropout_p=p, seed=11, offset=off + cut * L * 75, mode=mode)
                assert torch.equal(whole, torch.cat([first, rest])), (precision, p)


# ---- GPU: NRMS at 30-token titles -------------------------------------------------------------------------------------
def _nrms(golden_sd, dev, precision, L=30):
    from newsrecommendationsystem_b200 import NRMS

    class Cfg(_Cfg):
        num_words_title = L
    m = NRMS(Cfg)
    sd = {k: golden_sd[k] for k in m.state_dict()}
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.to(dev).eval().set_precision(precision)
    return m, sd


class _Recorder:
    """Wraps ops.news_encoder and keeps (tokens, news_rows, dropout_p, seed, offset) of every call."""

    def __init__(self, monkeypatch):
        from newsrecommendationsystem_b200 import ops
        self.calls, inner = [], ops.news_encoder

        def wrapped(tokens, *a, **kw):
            rows = kw.get("news_rows")
            self.calls.append((tokens.detach().cpu().numpy(), None if rows is None else rows.cpu().numpy(),
                               kw.get("dropout_p", 0.0), kw.get("seed", 0), kw.get("offset", 0)))
            return inner(tokens, *a, **kw)
        monkeypatch.setattr(ops, "news_encoder", wrapped)

    def masks(self, i):
        toks, rows, p, seed, offset = self.calls[i]
        n, L = (toks.shape if rows is None else (rows.size, toks.shape[1]))
        m1, m2 = _masks(n * L, p, seed, offset)
        return m1.reshape(n, L, 300), m2.reshape(n, L, 300)


@pytest.mark.gpu
@pytest.mark.parametrize("precision,ltol", [("fp32", 1e-5), ("tf32", 2e-3)])
def test_nrms_step_rows_at_30_tokens(dev, golden_sd, precision, ltol, monkeypatch):
    """TrainStep.step_rows with num_words_title = 30 and dropout 0.2: loss and every gradient against
    oracle.nrms_backward fed the restated masks."""
    from newsrecommendationsystem_b200 import synthetic
    from newsrecommendationsystem_b200.train import TrainStep
    m, sd = _nrms(golden_sd, dev, precision)
    m.train()
    rec = _Recorder(monkeypatch)
    ntok = synthetic.make_news(300, num_words=401, title_len=30, seed=31)
    rng = np.random.default_rng(32)
    cand = rng.integers(0, 300, size=(16, 5))
    hist = rng.integers(0, 300, size=(16, 50))
    ts = TrainStep(m)
    loss = float(ts.step_rows(_t(ntok, dev), torch.from_numpy(cand), torch.from_numpy(hist)))
    assert len(rec.calls) == 1 and rec.calls[0][2] == 0.2
    sd64 = {k: v.astype(np.float64) for k, v in sd.items()}
    logits, cache = O.nrms_forward(sd64, ntok[cand], ntok[hist], masks=rec.masks(0))
    loss_ref, dlogits = O.cross_entropy_label0(logits)
    grads = O.nrms_backward(dlogits, cache, sd64)
    assert abs(loss - float(loss_ref)) < ltol, (loss, loss_ref)
    for k, p in m.named_parameters():
        ref = grads[k]
        sc = float(np.abs(ref).max()) + 1e-12
        err = float(np.abs(p.grad.cpu().numpy() - ref).max())
        assert err <= GTOL[precision] * sc + 1e-8, (k, err, sc)


@pytest.mark.gpu
def test_nrms_three_adam_steps_at_30_tokens(dev, golden_sd):
    """Three FusedAdam steps (FP32 mode, eval-mode dropout) with num_words_title = 30 against oracle.train_step."""
    from newsrecommendationsystem_b200 import synthetic
    from newsrecommendationsystem_b200.train import TrainStep
    m, sd = _nrms(golden_sd, dev, "fp32")
    ntok = synthetic.make_news(300, num_words=401, title_len=30, seed=41)
    cand, clicked = synthetic.make_train_batch(8, ntok, k_neg=4, history=50, seed=42)
    ts = TrainStep(m)
    titles = torch.from_numpy(np.concatenate([cand, clicked], axis=1))
    params, state = {k: v.astype(np.float64) for k, v in sd.items()}, {}
    lr = 1e-4
    for step in range(1, 4):
        loss = float(ts.step_tokens(titles, cand.shape[1]))
        loss_ref, _, _, params, state = O.train_step(params, state, cand, clicked, step=step)
        assert abs(loss - float(loss_ref)) < 2e-5, (step, loss, loss_ref)
    for k, p in m.named_parameters():
        if k.endswith("W_K.bias"):
            continue        # zero gradient in exact arithmetic: Adam turns each side's rounding noise into +-lr steps
        d = np.abs(p.detach().cpu().numpy() - params[k])
        # the additive blocks' bias gradients cancel to a small fraction of their terms (test_history_length.py), so Adam
        # scales both sides' rounding noise there too: those take the bound on the largest step only
        cancels = k.endswith("additive_attention.linear.bias")
        assert d.max() <= 6 * lr and (cancels or d.mean() <= 0.02 * lr), (k, float(d.max()), float(d.mean()))


def _golden_data_at(tmp_path, L):
    """A copy of tests/golden/data whose titles are re-padded (right, with 0) to L tokens."""
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "data")
    dst = tmp_path / "data"
    shutil.copytree(src, dst)
    path = dst / "news_parsed.tsv"
    with open(path, newline="") as f:
        reader = csv.DictReader(f, delimiter="\t", quoting=csv.QUOTE_NONE)
        fields, rows = reader.fieldnames, list(reader)
    for r in rows:
        t = json.loads(r["title"])[:L]
        r["title"] = json.dumps(t + [0] * (L - len(t)))
    with open(path, "w", newline="") as f:
        w = csv.DictWriter(f, fieldnames=fields, delimiter="\t", quoting=csv.QUOTE_NONE, escapechar="\\",
                           lineterminator="\n")
        w.writeheader()
        w.writerows(rows)
    return str(dst)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_evaluate_directory_at_30_tokens(dev, golden_sd, tmp_path, precision):
    """evaluate(model, directory) on titles of 30 tokens against oracle.evaluate_pipeline: metrics to 3 decimals and
    the news table within 1e-3."""
    from newsrecommendationsystem_b200 import data, evaluate as E
    directory = _golden_data_at(tmp_path, 30)
    m, sd = _nrms(golden_sd, dev, precision)
    means = E.evaluate(m, directory)
    news = data.load_news_parsed(os.path.join(directory, "news_parsed.tsv"))
    assert news.title.shape[1] == 30
    ev = data.load_behaviors(os.path.join(directory, "behaviors.tsv"), news, num_clicked=50)
    owner = E.first_occurrence_rows(news.ids)
    hist = np.where(ev.hist_rows >= 0, owner[np.maximum(ev.hist_rows, 0)], -1)
    sd64 = {k: v.astype(np.float64) for k, v in sd.items()}
    ref = O.evaluate_pipeline(sd64, news.title, hist, ev.cand_offsets, owner[ev.cand_rows], ev.labels)
    assert np.abs(np.asarray(means) - ref[0]).max() < 1e-3, (means, ref[0])
    inp = E.EvalInputs(news.title, ev.hist_rows, ev.cand_offsets, ev.cand_rows, ev.labels, news_ids=news.ids, device=dev)
    _, det = E.evaluate_tensors(m, inp, return_details=True)
    table = det["table"][:len(news.ids), :300].float().cpu().numpy()
    nv, _ = O.news_encoder_forward(sd64, news.title)
    assert np.abs(table - nv).max() < 1e-3


@pytest.mark.gpu
def test_recommend_at_30_tokens(dev, golden_sd, tmp_path):
    """Recommender.from_directory on titles of 30 tokens: the news table against the oracle; recommend and top_k rank
    by that table (scores against oracle.recommend_user on it)."""
    from newsrecommendationsystem_b200 import data
    from newsrecommendationsystem_b200.recommend import Recommender
    directory = _golden_data_at(tmp_path, 30)
    m, sd = _nrms(golden_sd, dev, "fp32")
    rec = Recommender.from_directory(m, directory)
    news = data.load_news_parsed(os.path.join(directory, "news_parsed.tsv"))
    sd64 = {k: v.astype(np.float64) for k, v in sd.items()}
    nv, _ = O.news_encoder_forward(sd64, news.title)
    table = rec.table.cpu().numpy().astype(np.float64)
    for nid, r in rec.row_of.items():
        assert rel_l2_rows(table[r][None], nv[news.row_of[nid]][None]) < TOL_VEC["fp32"], nid
    rng = np.random.default_rng(5)
    ids = list(rec.row_of)
    clicked = [ids[i] for i in rng.choice(len(ids), 4, replace=False)]
    cand = [ids[i] for i in rng.choice(len(ids), min(40, len(ids)), replace=False)]
    hist = rec.history_rows(clicked)
    _, y_ref, _ = O.recommend_user(sd64, table, hist, [rec.row_of[c] for c in cand])
    got_ids, y = rec.recommend(clicked, cand)
    idx = [cand.index(c) for c in got_ids]
    assert sorted(idx) == list(range(len(cand)))
    assert np.abs(np.asarray(y) - y_ref[idx]).max() < 1e-5
    assert np.all(np.diff(np.asarray(y)) <= 0)                        # ranked by the table's scores
    top_ids, y_top = rec.top_k(clicked, 5)
    _, y_all, _ = O.recommend_user(sd64, table, hist, list(range(table.shape[0] - 1)))
    y_all[[rec.row_of[c] for c in clicked]] = -np.inf
    assert np.abs(np.asarray(y_top) - np.sort(y_all)[::-1][:5]).max() < 1e-5
    assert np.abs(y_all[[rec.row_of[c] for c in top_ids]] - np.asarray(y_top)).max() < 1e-5


# ---- GPU: Exp1 --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("lt,la", [(30, 64), (20, 37)])
def test_exp1_train_at_other_lengths(dev, lt, la, precision, monkeypatch):
    """Exp1 (title and abstract) with num_words_title = lt and num_words_abstract = la in train mode (dropout 0.2): the
    loss and every gradient against the fp64 restatement fed the restated masks."""
    from newsrecommendationsystem_b200 import Exp1, ops
    from exp1_weights import make_state
    from test_exp1_recommend import ATTRS_A, _cfg
    from test_exp1_abstract_train import EXP1_TOL, _items, _named, exp1_fp64

    B, n_cand, T = 5, 3, 13

    class Cfg(_cfg(ATTRS_A)):
        num_words_title = lt
        num_words_abstract = la
        num_clicked_news_a_user = T - n_cand
    m = Exp1(Cfg)
    sd = make_state({k: tuple(v.shape) for k, v in m.state_dict().items()}, 103)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.to(dev).train().set_precision(precision)
    rng = np.random.default_rng(lt + la)
    news = {"title": rng.integers(1, 401, size=(B, T, lt)), "abstract": rng.integers(1, 401, size=(B, T, la)),
            "category": rng.integers(0, 31, size=(B, T)), "subcategory": rng.integers(0, 31, size=(B, T))}
    news["title"][:, :, lt * 2 // 3:] = 0
    news["abstract"][:, :, la * 2 // 3:] = 0
    news["abstract"][:, ::5] = 0
    news = {k: v.astype(np.int64) for k, v in news.items()}
    rec = _Recorder(monkeypatch)
    logits = m(_items(news, ATTRS_A)[:n_cand], _items(news, ATTRS_A)[n_cand:])
    loss = ops.cross_entropy_label0(logits)
    m.zero_grad()
    loss.backward()
    masks = {}
    for i, (toks, _, p, _, _) in enumerate(rec.calls):
        assert p == 0.2
        masks["title" if toks.shape[1] == lt else "abstract"] = rec.masks(i)
    assert len(masks) == 2
    loss_ref, logits_ref, grads = exp1_fp64(_named(m, sd), news, n_cand, ATTRS_A, masks=masks)
    ltol, gtol = EXP1_TOL[precision]
    np.testing.assert_allclose(logits.detach().cpu().numpy(), logits_ref, atol=10 * ltol)
    assert abs(float(loss.detach()) - loss_ref) < ltol
    floor = 1e-6 * max(float(np.abs(v).max()) for v in grads.values())
    for k, p in m.named_parameters():
        ref = grads[k]
        sc = float(np.abs(ref).max()) + 1e-12
        err = float(np.abs(p.grad.detach().cpu().numpy() - ref).max())
        assert err <= gtol * sc + floor, (k, err, sc)
