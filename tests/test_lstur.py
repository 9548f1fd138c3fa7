"""LSTUR (reference src/model/LSTUR): the GRU user encoder nrms_gru_fwd / _bwd, the embedding rows nrms_rows_*, the
model and its training steps.

CPU part: the numpy restatement and the torch restatement of tests/lstur_reference.py agree (forward and every gradient,
ini and con); the left-pad quirk; the state_dict keys and shapes; the configuration rule; the ABI's shape rule.  GPU part
(`-m gpu`): the GRU alone, the model's logits, loss and every gradient with its dropout masks read back, the user mask's
statistics, and TrainStep.step == step_rows -- against the float64 torch restatement.
"""
import ctypes as C
import json
import os
import shutil

import numpy as np
import pytest
import torch

import lstur_reference as R
from test_text_length import dropout_mask, philox4x32_10, _M32

GRU_TOL = {"fp32": 1e-5, "tf32": 2e-3}           # GRU alone: max |err| over the tensor's largest entry (measured: DESIGN.md, LSTUR)
# GRU alone, last hidden state: worst row-wise relative L2.  Measured on a B200 at 2,049 sequences of 50 steps: 5.7e-7
# (FP32 mode) and 4.1e-4 (tensor mode, TF32 operands); see DESIGN.md, LSTUR.
GRU_ROW_TOL = {"fp32": 2e-6, "tf32": 1e-3}
GTOL = {"fp32": 2e-4, "tf32": 5e-3}              # the model's gradients, relative to the tensor's largest entry
LTOL = {"fp32": 1e-5, "tf32": 2e-3}              # logits / loss, relative to the largest logit
STREAM_EMB, STREAM_CTX, STREAM_ROW = 1, 2, 3


def _cfg(method="ini", p=0.2, masking=0.5, num_words=300, num_categories=20, num_users=40):
    from newsrecommendationsystem_b200.config import LSTURConfig

    class Cfg(LSTURConfig):
        pass
    Cfg.long_short_term_method = method
    Cfg.dropout_probability = p
    Cfg.masking_probability = masking
    Cfg.num_words = num_words
    Cfg.num_categories = num_categories
    Cfg.num_users = num_users
    return Cfg


def _lengths_mix(rng, B, T=50):
    base = [50, 0, 1, 25, 26]
    return np.array(base[:B] if B <= 5 else
                    base + list(rng.integers(0, T + 1, size=B - len(base))), dtype=np.int64)


# ---- CPU --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("method", ["ini", "con"])
def test_gru_restatements_agree(method):
    """numpy GRU (forward + written-out BPTT) == nn.GRU through pack_padded_sequence (autograd), float64."""
    rng = np.random.default_rng(1)
    P = R.random_params(rng, method)
    H = 900 if method == "ini" else 450
    B, T = 7, 50
    lengths = np.array([0, 1, 25, 26, 50, 13, 38])
    x = rng.standard_normal((B, T, 900))
    h0 = rng.standard_normal((B, H)) if method == "ini" else None
    w = [P[k] for k in R.GRU_KEYS]
    eff = np.maximum(lengths, 1)                # pack_padded_sequence takes lengths >= 1
    h, cache = R.gru_forward(*w, x, eff, h0)
    d_out = rng.standard_normal((B, H))
    g = R.gru_backward(w[0], w[1], x, eff, cache, d_out)
    tp = R.TorchLSTUR(P, method)
    xt = torch.tensor(x, requires_grad=True)
    h0t = None if h0 is None else torch.tensor(h0, requires_grad=True)
    ht = R.torch_gru(tp.gru, xt, eff, h0t)
    (ht * torch.as_tensor(d_out)).sum().backward()
    np.testing.assert_allclose(h, ht.detach().numpy(), atol=1e-12)
    np.testing.assert_allclose(g["x"], xt.grad.numpy(), atol=1e-11)
    if h0 is not None:
        np.testing.assert_allclose(g["h0"], h0t.grad.numpy(), atol=1e-11)
    for k, name in zip(R.GRU_KEYS, ("w_ih", "w_hh", "b_ih", "b_hh")):
        np.testing.assert_allclose(g[name], tp.P[k].grad.numpy(), atol=1e-10, err_msg=k)


@pytest.mark.parametrize("method", ["ini", "con"])
def test_model_restatements_agree(method):
    """LSTUR.forward: numpy == torch restatement (logits), with title masks and a user mask."""
    rng = np.random.default_rng(2)
    P = R.random_params(rng, method)
    B, K, N, L = 3, 2, 50, 20
    news = _news(rng, B, K + N, L)
    user = np.array([0, 5, 39])
    lengths = np.array([0, 26, 50])
    umask = np.array([2.0, 0.0, 2.0])
    ref = R.lstur_forward(P, method, user, lengths, news, K, user_mask=umask)
    got = R.TorchLSTUR(P, method).forward(user, lengths, news, K, user_mask=umask).detach().numpy()
    np.testing.assert_allclose(ref, got, atol=1e-9 * np.abs(ref).max())


@pytest.mark.parametrize("method", ["ini", "con"])
def test_user_encoder_restatements_agree_gradients(method):
    """The user side, every gradient: numpy (GRU BPTT written out, the user row's gradient from d_h0 (ini) or from the
    concatenated half (con)) == torch autograd through nn.GRU and F.embedding, lengths 0 (read as 1), 1, 25, 26, 50."""
    rng = np.random.default_rng(7)
    P = R.random_params(rng, method)
    H = 900 if method == "ini" else 450
    lengths = np.array([0, 1, 25, 26, 50])
    user = np.array([3, 0, 9, 3, 17])
    x = rng.standard_normal((5, 50, 900))
    d_out = rng.standard_normal((5, 900))
    U = P["user_embedding.weight"]
    eff = np.maximum(lengths, 1)
    u = U[user]
    w = [P[k] for k in R.GRU_KEYS]
    h, cache = R.gru_forward(*w, x, eff, u if method == "ini" else None)
    d_h = d_out if method == "ini" else d_out[:, :H]
    g = R.gru_backward(w[0], w[1], x, eff, cache, d_h)
    d_u = g["h0"] if method == "ini" else d_out[:, H:]
    d_U = np.zeros_like(U)
    np.add.at(d_U, user, d_u)
    d_U[0] = 0                                           # padding_idx
    tp = R.TorchLSTUR(P, method)
    xt = torch.tensor(x, requires_grad=True)
    out = tp.user(tp.user_rows(user), lengths, xt)
    np.testing.assert_allclose(R.user_forward(P, method, u, lengths, x), out.detach().numpy(), atol=1e-12)
    (out * torch.as_tensor(d_out)).sum().backward()
    np.testing.assert_allclose(g["x"], xt.grad.numpy(), atol=1e-11)
    np.testing.assert_allclose(d_U, tp.P["user_embedding.weight"].grad.numpy(), atol=1e-11)
    for k, name in zip(R.GRU_KEYS, ("w_ih", "w_hh", "b_ih", "b_hh")):
        np.testing.assert_allclose(g[name], tp.P[k].grad.numpy(), atol=1e-10, err_msg=k)


@pytest.mark.parametrize("method", ["ini", "con"])
@pytest.mark.parametrize("n", [0, 1, 12, 25])
def test_left_pad_quirk(method, n):
    """The history is left-padded and the GRU reads rows [0, n): with n <= 25 clicks it sees only padding, so the user
    vector does not depend on which news were clicked (the reference's behaviour, reproduced)."""
    rng = np.random.default_rng(3)
    P = R.random_params(rng, method)
    tp = R.TorchLSTUR(P, method)
    user = np.array([7])
    out = []
    for seed in (4, 5):
        hist = np.zeros((1, 50, 900))               # PADDED_NEWS rows, then the n clicks
        hist[0, 50 - n:] = np.random.default_rng(seed).standard_normal((n, 900))
        out.append(tp.user(tp.user_rows(user), np.array([n]), torch.as_tensor(hist)).detach().numpy())
    np.testing.assert_array_equal(out[0], out[1])
    if n == 25:       # with 26 clicks row 24, the first click, is read: two histories differing only there differ
        moved = []
        for first_click in (0.5, -0.5):
            hist = np.zeros((1, 50, 900))
            hist[0, 24:] = np.random.default_rng(6).standard_normal((26, 900))
            hist[0, 24] = first_click
            moved.append(tp.user(tp.user_rows(user), np.array([26]), torch.as_tensor(hist)).detach().numpy())
        assert np.abs(moved[0] - moved[1]).max() > 1e-6


def test_state_dict_keys_and_shapes():
    from newsrecommendationsystem_b200 import LSTUR
    from newsrecommendationsystem_b200.config import LSTURConfig
    want = {"news_encoder.word_embedding.weight": (70976, 300), "news_encoder.category_embedding.weight": (275, 300),
            "news_encoder.title_CNN.weight": (300, 1, 3, 300), "news_encoder.title_CNN.bias": (300,),
            "news_encoder.title_attention.linear.weight": (200, 300), "news_encoder.title_attention.linear.bias": (200,),
            "news_encoder.title_attention.attention_query_vector": (200,),
            "user_encoder.gru.weight_ih_l0": (2700, 900), "user_encoder.gru.weight_hh_l0": (2700, 900),
            "user_encoder.gru.bias_ih_l0": (2700,), "user_encoder.gru.bias_hh_l0": (2700,),
            "user_embedding.weight": (50001, 900)}
    sd = LSTUR(LSTURConfig).state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == want
    assert sum(v.numel() for v in sd.values()) == 71_572_300
    con = LSTUR(_cfg("con", num_words=70976, num_categories=275, num_users=50001)).state_dict()
    assert tuple(con["user_encoder.gru.weight_ih_l0"].shape) == (1350, 900)
    assert tuple(con["user_encoder.gru.weight_hh_l0"].shape) == (1350, 450)
    assert tuple(con["user_embedding.weight"].shape) == (50001, 450)
    assert sum(v.numel() for v in con.values()) == 46_031_650
    # the torch restatement reads the same keys
    assert set(R.random_params(np.random.default_rng(0), "ini")) == set(want)
    assert float(sd["user_embedding.weight"][0].abs().max()) == 0.0


@pytest.mark.parametrize("name,value", [("num_filters", 400), ("window_size", 5), ("query_vector_dim", 100),
                                        ("long_short_term_method", "sum")])
def test_configuration_rule(name, value):
    from newsrecommendationsystem_b200 import LSTUR
    cfg = _cfg()
    setattr(cfg, name, value)
    with pytest.raises(RuntimeError, match=name if name != "long_short_term_method" else "long_short_term_method"):
        LSTUR(cfg)


@pytest.fixture(scope="module")
def lib():
    from newsrecommendationsystem_b200 import _lib
    try:
        return _lib.load()
    except ImportError as e:
        pytest.skip(str(e))


@pytest.mark.parametrize("I,H", [(300, 300), (900, 300), (900, 451), (450, 450), (900, 1800)])
def test_gru_refuses_other_shapes(lib, I, H):
    """Any (I, H) but (900, 900) and (900, 450) returns NRMS_E_UNSUPPORTED before any other check or CUDA call (every
    pointer here is NULL)."""
    lengths = (C.c_int32 * 4)(1, 2, 3, 4)
    assert lib.nrms_gru_fwd(None, 8, None, 4, 2, I, H, lengths, None, None, None, None, None, None, None, None, 0, 1,
                            None) == 2
    assert lib.nrms_gru_bwd(None, None, 4, 2, I, H, lengths, None, None, None, None, None, None, None, None, None, None,
                            0, 1, None) == 2


def test_gru_sizes(lib):
    for H in (900, 450):
        assert lib.nrms_gru_stash_bytes(128, 50, 900, H) > 128 * 50 * 5 * H * 4
        assert lib.nrms_gru_fwd_workspace_bytes(128, 50, 128 * 50, 900, H) > 128 * 50 * 3 * H * 4
        assert lib.nrms_gru_bwd_workspace_bytes(128, 50, 900, H, 1) > lib.nrms_gru_bwd_workspace_bytes(128, 50, 900, H, 0)


def test_lengths_are_not_written():
    from newsrecommendationsystem_b200.model.LSTUR.user_encoder import gru_lengths
    given = torch.tensor([0, 3, 0, 50])
    got = gru_lengths(given, 50)
    assert given.tolist() == [0, 3, 0, 50] and got.tolist() == [1, 3, 1, 50]
    with pytest.raises(ValueError):
        gru_lengths(torch.tensor([51]), 50)


# ---- GPU --------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda")


def _news(rng, B, T, L, num_words=300, num_categories=20):
    t = rng.integers(1, num_words, size=(B, T, L))
    keep = rng.integers(1, L + 1, size=(B, T))
    return {"category": rng.integers(0, num_categories, size=(B, T)),
            "subcategory": rng.integers(0, num_categories, size=(B, T)),
            "title": np.where(np.arange(L)[None, None] < keep[..., None], t, 0).astype(np.int64)}


def _torch_gru_ref(P, method, x, lengths, h0, d_out, device):
    """float64 nn.GRU through pack_padded_sequence on `device`; sequences of length 0 run no step (h = h0)."""
    H = P["user_encoder.gru.weight_hh_l0"].shape[1]
    gru = torch.nn.GRU(900, H).double().to(device)
    with torch.no_grad():
        for k in R.GRU_KEYS:
            getattr(gru, k.rsplit(".", 1)[1]).copy_(torch.as_tensor(P[k]))
    xt = torch.tensor(x, dtype=torch.float64, device=device, requires_grad=True)
    h0t = None if h0 is None else torch.tensor(h0, dtype=torch.float64, device=device, requires_grad=True)
    run = np.nonzero(lengths > 0)[0]
    out = torch.zeros((x.shape[0], H), dtype=torch.float64, device=device) if h0t is None else h0t * 1.0
    if run.size:
        idx = torch.as_tensor(run, device=device)
        hr = R.torch_gru(gru, xt[idx], lengths[run], None if h0t is None else h0t[idx])
        out = out.index_copy(0, idx, hr)
    (out * torch.as_tensor(d_out, device=device)).sum().backward()
    g = {"x": xt.grad.cpu().numpy(), "h0": None if h0t is None else h0t.grad.cpu().numpy()}
    for k in R.GRU_KEYS:
        g[k] = getattr(gru, k.rsplit(".", 1)[1]).grad.cpu().numpy()
    return out.detach().cpu().numpy(), g


def _close(got, ref, tol, what):
    den = max(float(np.abs(ref).max()), 1e-12)
    err = float(np.abs(np.asarray(got, np.float64) - ref).max()) / den
    assert err <= tol, f"{what}: {err:.3g} > {tol}"
    return err


def _rel_rows(got, ref):
    got = np.asarray(got, np.float64)
    n = np.linalg.norm(ref, axis=1)
    keep = n > 0
    return float((np.linalg.norm(got - ref, axis=1)[keep] / n[keep]).max()) if keep.any() else 0.0


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("method", ["ini", "con"])
@pytest.mark.parametrize("n_seq", [1, 7, 128, 2049])
def test_gru_vs_oracle(dev, precision, method, n_seq):
    """The GRU alone (ini with h0, con without): last hidden state, d_x, d_h0 and the four parameter gradients."""
    from newsrecommendationsystem_b200 import ops, _lib
    rng = np.random.default_rng(n_seq)
    P = R.random_params(rng, method)
    H = 900 if method == "ini" else 450
    T = 50
    lengths = _lengths_mix(rng, n_seq)
    x = rng.standard_normal((n_seq, T, 900)).astype(np.float32)
    h0 = rng.standard_normal((n_seq, H)).astype(np.float32) * 0.5 if method == "ini" else None
    d_out = rng.standard_normal((n_seq, H)).astype(np.float32)
    ref, g = _torch_gru_ref(P, method, x.astype(np.float64), lengths, None if h0 is None else h0.astype(np.float64),
                            d_out.astype(np.float64), dev)
    w = [torch.tensor(P[k], dtype=torch.float32, device=dev, requires_grad=True) for k in R.GRU_KEYS]
    xt = torch.tensor(x, device=dev, requires_grad=True)
    h0t = None if h0 is None else torch.tensor(h0, device=dev, requires_grad=True)
    out = ops.gru(xt, torch.from_numpy(lengths), h0t, *w, mode=_lib.MODES[precision])
    (out * torch.from_numpy(d_out).to(dev)).sum().backward()
    tol = GRU_TOL[precision]
    assert _rel_rows(out.detach().cpu().numpy(), ref) < GRU_ROW_TOL[precision]
    _close(out.detach().cpu().numpy(), ref, tol, "h")
    _close(xt.grad.cpu().numpy(), g["x"], tol, "d_x")
    if h0 is not None:
        _close(h0t.grad.cpu().numpy(), g["h0"], tol, "d_h0")
    for k, wk in zip(R.GRU_KEYS, w):
        _close(wk.grad.cpu().numpy(), g[k], tol, k)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("method", ["ini", "con"])
def test_gru_indexed_equals_dense(dev, precision, method):
    """The table form (input projection over the table, rows gathered per step) == the dense form over gathered rows."""
    from newsrecommendationsystem_b200 import ops, _lib
    rng = np.random.default_rng(11)
    P = R.random_params(rng, method)
    H = 900 if method == "ini" else 450
    table = torch.tensor(rng.standard_normal((300, 900)), dtype=torch.float32, device=dev)
    table[299] = 0                                   # PADDED_NEWS
    rows = torch.tensor(rng.integers(0, 300, size=(333, 50)), device=dev)
    lengths = torch.from_numpy(_lengths_mix(rng, 333))
    h0 = torch.tensor(rng.standard_normal((333, H)), dtype=torch.float32, device=dev) if method == "ini" else None
    w = [torch.tensor(P[k], dtype=torch.float32, device=dev) for k in R.GRU_KEYS]
    mode = _lib.MODES[precision]
    a = ops.gru_indexed(table, rows, lengths, h0, *w, mode=mode)
    with torch.no_grad():
        b = ops.gru(table[rows], lengths, h0, *w, mode=mode)
    assert _rel_rows(a.cpu().numpy(), b.cpu().numpy().astype(np.float64)) < (1e-6 if precision == "fp32" else 1e-3)


def user_mask(n, p, seed, offset):
    """The whole-row mask of nrms_rows_fwd: row i keeps (scale 1 / (1 - p)) iff lane x of Philox((i + offset, 3, 0),
    seed) * 2^-32 >= p."""
    c = np.arange(n, dtype=np.uint64) + np.uint64(offset)
    r = philox4x32_10(c & _M32, c >> np.uint64(32), np.full_like(c, STREAM_ROW), np.zeros_like(c),
                      np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32))
    u = np.asarray(r[0]).astype(np.uint32).astype(np.float32) * np.float32(2.0 ** -32)
    return np.where(u >= np.float32(p), np.float32(1) / (np.float32(1) - np.float32(p)), np.float32(0))


@pytest.mark.gpu
def test_user_mask_statistics(dev):
    """Keep-rate ~ 1 - p, whole rows, survivors scaled by exactly 2 at p = 0.5, and the numpy restatement's mask."""
    from newsrecommendationsystem_b200 import ops
    rng = np.random.default_rng(5)
    W = torch.tensor(rng.standard_normal((50, 450)) + 3.0, dtype=torch.float32, device=dev)
    idx = torch.tensor(rng.integers(1, 50, size=20000), device=dev)
    out = ops.embedding_rows(idx, W, dropout_p=0.5, seed=99, offset=17)
    ratio = (out / W[idx]).cpu().numpy()
    assert np.all((ratio == 0) | (ratio == 2))
    assert np.all(ratio.min(axis=1) == ratio.max(axis=1))            # whole rows
    keep = float((ratio[:, 0] == 2).mean())
    assert abs(keep - 0.5) < 0.02
    np.testing.assert_array_equal(ratio[:, 0], user_mask(20000, 0.5, 99, 17))
    # the backward: gradient of sum(out * G) = scatter of G * mask into the rows, padding row untouched
    Wg = W.clone().requires_grad_(True)
    idx2 = torch.tensor([0, 3, 3, 7], device=dev)
    o = ops.embedding_rows(idx2, Wg, padding_idx=0, dropout_p=0.5, seed=1, offset=0)
    G = torch.randn_like(o)
    (o * G).sum().backward()
    m = torch.from_numpy(user_mask(4, 0.5, 1, 0)).to(dev)
    ref = torch.zeros_like(W)
    ref.index_add_(0, idx2[1:], G[1:] * m[1:, None])
    assert torch.allclose(Wg.grad, ref, atol=1e-6)


def _model(cfg, P, dev, precision):
    from newsrecommendationsystem_b200 import LSTUR
    m = LSTUR(cfg)
    m.load_state_dict({k: torch.from_numpy(v.astype(np.float32)) for k, v in P.items()})
    return m.to(dev).set_precision(precision)


def _masks(model, cfg, n_texts, L, n_users):
    ne = model.news_encoder
    p = cfg.dropout_probability
    title = (dropout_mask(n_texts * L, p, 0x5EED, ne._dropout_calls, STREAM_EMB),
             dropout_mask(n_texts * L, p, 0x5EED, ne._dropout_calls, STREAM_CTX))
    return title, user_mask(n_users, cfg.masking_probability, model.dropout_seed, model._masking_calls)


def _grads(model):
    return {k: v.grad.detach().cpu().numpy().copy() for k, v in model.named_parameters()}


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("method", ["ini", "con"])
@pytest.mark.parametrize("form", ["forward", "forward_rows"])
def test_model_training_vs_torch(dev, precision, method, form):
    """Logits, loss and every gradient in train mode (title dropout 0.2, user masking 0.5), with the masks restated
    from Philox and fed to the float64 torch restatement."""
    from newsrecommendationsystem_b200 import ops
    cfg = _cfg(method)
    rng = np.random.default_rng(21)
    P = R.random_params(rng, method)
    model = _model(cfg, P, dev, precision).train()
    B, K, N, L = 8, 4, 50, 20
    news = _news(rng, B, 1 + K + N, L)
    user = rng.integers(0, 40, size=B)
    lengths = np.array([0, 1, 25, 26, 50, 40, 33, 49])
    title_m, user_m = _masks(model, cfg, B * (1 + K + N), L, B)
    if form == "forward":
        cand = [{a: torch.from_numpy(np.ascontiguousarray(v[:, i])) for a, v in news.items()} for i in range(1 + K)]
        clicked = [{a: torch.from_numpy(np.ascontiguousarray(v[:, i])) for a, v in news.items()}
                   for i in range(1 + K, 1 + K + N)]
        logits = model(torch.from_numpy(user), torch.from_numpy(lengths), cand, clicked)
    else:
        flat = {a: v.reshape(B * (1 + K + N), *v.shape[2:]) for a, v in news.items()}
        table = {a: torch.from_numpy(np.concatenate([v, np.zeros((1,) + v.shape[1:], np.int64)])).to(dev)
                 for a, v in flat.items()}
        rows = np.arange(B * (1 + K + N)).reshape(B, 1 + K + N)
        logits = model.forward_rows(table, torch.from_numpy(rows[:, :1 + K]), torch.from_numpy(rows[:, 1 + K:]),
                                    torch.from_numpy(user), torch.from_numpy(lengths))
    loss = ops.cross_entropy_label0(logits)
    loss.backward()
    ref_logits, ref_loss, ref_g = R.TorchLSTUR(P, method).loss_and_grads(user, lengths, news, 1 + K, title_m, user_m)
    _close(logits.detach().cpu().numpy(), ref_logits, LTOL[precision], "logits")
    assert abs(float(loss.detach()) - ref_loss) <= LTOL[precision] * max(1.0, abs(ref_loss))
    g = _grads(model)
    for k, r in ref_g.items():
        if k == "news_encoder.word_embedding.weight":
            assert np.abs(g[k][0]).max() == 0.0
        _close(g[k], r, GTOL[precision], k)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_step_equals_step_rows(dev, precision):
    """TrainStep.step (reference minibatch) and step_rows (index-only) give the same loss and gradients for LSTUR."""
    from newsrecommendationsystem_b200.train import TrainStep
    cfg = _cfg("ini")
    rng = np.random.default_rng(31)
    P = R.random_params(rng, "ini")
    B, K, N, L = 8, 4, 50, 20
    news = _news(rng, B, 1 + K + N, L)
    user = torch.from_numpy(rng.integers(0, 40, size=B))
    lengths = torch.from_numpy(rng.integers(0, 51, size=B))
    out = []
    for form in ("step", "step_rows"):
        model = _model(cfg, P, dev, precision).train()
        ts = TrainStep(model, lr=1e-4)
        if form == "step":
            cand = [{a: torch.from_numpy(np.ascontiguousarray(v[:, i])) for a, v in news.items()} for i in range(1 + K)]
            clicked = [{a: torch.from_numpy(np.ascontiguousarray(v[:, i])) for a, v in news.items()}
                       for i in range(1 + K, 1 + K + N)]
            loss = ts.step(cand, clicked, user=user, clicked_news_length=lengths)
        else:
            flat = {a: v.reshape(B * (1 + K + N), *v.shape[2:]) for a, v in news.items()}
            table = {a: torch.from_numpy(v).to(dev) for a, v in flat.items()}
            rows = torch.arange(B * (1 + K + N)).view(B, 1 + K + N)
            loss = ts.step_rows(table, rows[:, :1 + K], rows[:, 1 + K:], user=user, clicked_news_length=lengths)
        out.append((float(loss), _grads(model)))
    assert abs(out[0][0] - out[1][0]) <= 1e-6 * max(1.0, abs(out[0][0]))
    for k in out[0][1]:
        _close(out[1][1][k], out[0][1][k].astype(np.float64), 1e-5, k)


# ---- readers and evaluate -------------------------------------------------------------------------------------------
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "data")


def test_train_rows_user_and_lengths():
    """TrainRows.user is the integer `user` column and clicked_news_length the number of (first 50) clicks."""
    from newsrecommendationsystem_b200 import data
    news = data.load_news_parsed(os.path.join(GOLDEN, "news_parsed.tsv"))
    tr = data.load_behaviors_parsed(os.path.join(GOLDEN, "behaviors_parsed.tsv"), news)
    with open(os.path.join(GOLDEN, "behaviors_parsed.tsv")) as f:
        rows = [line.rstrip("\n").split("\t") for line in f][1:]
    assert tr.user.tolist() == [int(r[0]) for r in rows]
    assert tr.clicked_news_length.tolist() == [min(len(r[1].split()), 50) for r in rows]
    assert (tr.hist_rows == len(news)).sum(axis=1).tolist() == [50 - n for n in tr.clicked_news_length]


def _lstur_eval_dir(tmp_path):
    """The golden news and behaviors plus three rows: U9 repeats U1's history (a different user, the same key), U7
    repeats U0's empty history, and UX is not in user2int.tsv.  -> (directory, user2int dict)."""
    d = tmp_path / "val"
    d.mkdir()
    shutil.copy(os.path.join(GOLDEN, "news_parsed.tsv"), d / "news_parsed.tsv")
    with open(os.path.join(GOLDEN, "behaviors.tsv")) as f:
        lines = [line.rstrip("\n").split("\t") for line in f]
    extra = [["7", "U9", "11/16/2019 9:06:00 AM", lines[1][3], "N101-1 N103-0 N104-0"],
             ["8", "U7", "11/16/2019 9:07:00 AM", "", "N105-0 N106-1"],
             ["9", "UX", "11/16/2019 9:08:00 AM", "N103 N104", "N100-1 N107-0 N113-0"]]
    with open(d / "behaviors.tsv", "w") as f:
        for r in lines + extra:
            f.write("\t".join(r) + "\n")
    user2int = {f"U{i}": i + 1 for i in range(10)}
    (tmp_path / "train").mkdir()
    with open(tmp_path / "train" / "user2int.tsv", "w") as f:
        f.write("user\tint\n" + "".join(f"{u}\t{i}\n" for u, i in user2int.items()))
    return str(d), user2int


def test_eval_rows_users_user2int_and_first_wins(tmp_path):
    from newsrecommendationsystem_b200 import data
    from newsrecommendationsystem_b200.evaluate import lstur_user_keys
    directory, want = _lstur_eval_dir(tmp_path)
    news = data.load_news_parsed(os.path.join(directory, "news_parsed.tsv"))
    ev = data.load_behaviors(os.path.join(directory, "behaviors.tsv"), news)
    assert ev.users == ["U0", "U1", "U2", "U3", "U4", "U5", "U9", "U7", "UX"]
    u2i = data.load_user2int(os.path.join(directory, "..", "train", "user2int.tsv"))
    assert u2i == want
    with pytest.raises(FileNotFoundError, match="nowhere"):
        data.load_user2int(os.path.join(directory, "nowhere", "user2int.tsv"))
    key_of, rows, users, lengths = lstur_user_keys(ev, u2i)
    # U9 shares U1's key and U7 shares U0's (empty history ' '): the first row's user wins
    assert key_of.tolist() == [0, 1, 2, 3, 4, 5, 1, 0, 6]
    assert rows.tolist() == [0, 1, 2, 3, 4, 5, 8]
    assert users.tolist() == [1, 2, 3, 4, 5, 6, 0]            # UX is missing: 0
    assert lengths.tolist() == [min(len(ev.clicked_news_strings[i].split()), 50) for i in rows.tolist()]
    assert lengths[0] == 0


def _reference_lstur_evaluate(P, method, directory, user2int):
    """A restatement of the reference's LSTUR evaluate walk in float64 numpy: news vectors of every news, user2vector
    filled in file order with first wins per clicked-news string (user id from user2int, 0 if missing; the history's first
    50 clicks, left-padded with a zero PADDED_NEWS row; length 0 read as 1), get_prediction per impression, the metrics of
    every impression, nanmean."""
    import csv
    from oracle import nrms_oracle as O
    with open(os.path.join(directory, "news_parsed.tsv"), newline="") as f:
        recs = list(csv.DictReader(f, delimiter="\t", quoting=csv.QUOTE_NONE))
    row_of = {}
    for i, r in enumerate(recs):
        row_of.setdefault(r["id"], i)
    news = {"category": np.array([int(r["category"]) for r in recs]),
            "subcategory": np.array([int(r["subcategory"]) for r in recs]),
            "title": np.array([json.loads(r["title"]) for r in recs], dtype=np.int64)}
    vec = R.news_forward(P, news)
    news2vector = {nid: vec[row_of[nid]] for nid in row_of}
    padded = np.zeros(900)
    user2vector = {}
    per = []
    with open(os.path.join(directory, "behaviors.tsv"), newline="") as f:
        rows = list(csv.reader(f, delimiter="\t", quoting=csv.QUOTE_NONE))
    for r in rows:
        clicked = r[3] if r[3] else " "
        if clicked not in user2vector:
            ids = clicked.split()[:50]
            hist = np.stack([padded] * (50 - len(ids)) + [news2vector[x] for x in ids])
            u = P["user_embedding.weight"][user2int.get(r[1], 0)]
            user2vector[clicked] = R.user_forward(P, method, u[None], np.array([len(ids)]), hist[None])[0]
    for r in rows:
        clicked = r[3] if r[3] else " "
        items = [x.split("-") for x in r[4].split()]
        cand = np.stack([news2vector[n] for n, _ in items])
        per.append(O.single_user_metric([int(y) for _, y in items], (cand @ user2vector[clicked]).tolist()))
    with np.errstate(all="ignore"):
        return np.nanmean(np.asarray(per, np.float64), axis=0)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("method", ["ini", "con"])
def test_evaluate_vs_reference_walk(dev, tmp_path, precision, method):
    """evaluate(model, directory) == the restated reference walk: a repeated history with different users, an empty
    history, a user missing from user2int.tsv.  Metrics to 1e-9 (FP32 mode), 3 decimals (tensor mode)."""
    from newsrecommendationsystem_b200.evaluate import evaluate
    directory, user2int = _lstur_eval_dir(tmp_path)
    rng = np.random.default_rng(41)
    P = R.random_params(rng, method, num_words=500, num_categories=275, num_users=12)
    model = _model(_cfg(method, num_words=500, num_categories=275, num_users=12), P, dev, precision)
    got = np.asarray(evaluate(model, directory))
    ref = _reference_lstur_evaluate(P, method, directory, user2int)
    np.testing.assert_allclose(got, ref, atol=1e-9 if precision == "fp32" else 1e-3)
    with pytest.raises(FileNotFoundError):
        evaluate(model, directory, user2int_path=os.path.join(directory, "missing.tsv"))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("method", ["ini", "con"])
def test_user_vectors_at_mind_small_size(dev, precision, method):
    """The table-projected GRU at MIND-small size (65,238 news + the zero PADDED_NEWS row, 73,152 left-padded
    histories of 0..50 clicks) against float64 nn.GRU on a sample of 64 users."""
    from newsrecommendationsystem_b200 import ops, _lib
    rng = np.random.default_rng(43)
    P = R.random_params(rng, method)
    H = 900 if method == "ini" else 450
    n_news, U = 65238, 73152
    table = torch.randn((n_news + 1, 900), device=dev) * 0.05
    table[n_news] = 0
    lengths = rng.integers(0, 51, size=U)
    hist = rng.integers(0, n_news, size=(U, 50))
    hist[np.arange(50)[None] < (50 - lengths)[:, None]] = n_news
    h0 = torch.randn((U, H), device=dev) if method == "ini" else None
    w = [torch.tensor(P[k], dtype=torch.float32, device=dev) for k in R.GRU_KEYS]
    eff = np.maximum(lengths, 1)
    out = ops.gru_indexed(table, torch.from_numpy(hist), torch.from_numpy(eff), h0, *w, mode=_lib.MODES[precision])
    sample = np.sort(rng.choice(U, size=64, replace=False))
    x = table[torch.from_numpy(hist[sample]).to(dev)].double().cpu().numpy()
    ref, _ = R.gru_forward(*(P[k] for k in R.GRU_KEYS), x, eff[sample],
                           None if h0 is None else h0[torch.from_numpy(sample).to(dev)].double().cpu().numpy())
    assert _rel_rows(out[torch.from_numpy(sample).to(dev)].cpu().numpy(), ref) < GRU_ROW_TOL[precision]


def test_gru_indexed_range_checks_host_rows():
    from newsrecommendationsystem_b200 import ops
    table = torch.zeros((10, 900))
    w = [torch.zeros(2700, 900), torch.zeros(2700, 900), torch.zeros(2700), torch.zeros(2700)]
    with pytest.raises(IndexError):
        ops.gru_indexed(table, torch.tensor([[0, 10]]), torch.tensor([2]), None, *w)
    with pytest.raises(IndexError):
        ops.gru_indexed(table, torch.tensor([[-1, 3]]), torch.tensor([2]), None, *w)


def test_score_width_rule(lib):
    """nrms_score_csr_width takes 300 or 900; any other width is NRMS_E_UNSUPPORTED before any other check."""
    for width in (450, 600, 0):
        assert lib.nrms_score_csr_width(None, None, None, None, 1, width, None, None) == 2


@pytest.mark.gpu
@pytest.mark.parametrize("width", [300, 900])
def test_score_csr_widths(dev, width):
    from newsrecommendationsystem_b200 import ops
    rng = np.random.default_rng(width)
    table = rng.standard_normal((500, width)).astype(np.float32)
    counts = rng.integers(1, 90, size=300)
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    rows = rng.integers(0, 500, size=int(offs[-1])).astype(np.int32)
    user = rng.standard_normal((300, width)).astype(np.float32)
    got = ops.score_csr(torch.from_numpy(table).to(dev), torch.from_numpy(rows).to(dev), torch.from_numpy(offs).to(dev),
                        torch.from_numpy(user).to(dev)).cpu().numpy()
    imp = np.repeat(np.arange(300), counts)
    ref = np.einsum("cd,cd->c", table[rows].astype(np.float64), user[imp].astype(np.float64))
    np.testing.assert_allclose(got, ref, atol=1e-4 * np.abs(ref).max())
