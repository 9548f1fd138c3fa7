"""NAML (reference src/model/NAML): the CNN text encoder nrms_cnn_text_fwd / _bwd, the model, its training steps,
evaluate and checkpoints.

CPU part: the numpy restatement and the torch port of tests/naml_reference.py agree; the model's state_dict keys and
shapes are the reference's; the length rule of the new pair; the configuration rule.  GPU part (`-m gpu`): the text
encoder, both dropout masks, every gradient, the model through TrainStep.step / step_rows and three FusedAdam steps, and
evaluate -- against the float64 torch port (autograd) / numpy restatement, with train-mode dropout fed the masks that
tests/test_text_length.py restates bit for bit.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import rel_l2_rows
from oracle import nrms_oracle as O
import naml_reference as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL_VEC = {"fp32": 2e-5, "tf32": 1e-3}          # max row-wise relative L2 (test_gpu_parity.py)
GTOL = {"fp32": 2e-4, "tf32": 5e-3}             # gradients, relative to the tensor's largest entry
STREAM_EMB, STREAM_CTX = 1, 2
INFER_CHUNK_ROWS = 2048 * 20                    # cnn_text.cu: rows per inference pass
ALL = ["category", "subcategory", "title", "abstract"]


def _cfg(attributes=ALL, lt=20, la=50, p=0.2, num_words=500, num_categories=30, clicks=6):
    from newsrecommendationsystem_b200.config import NAMLConfig

    class C(NAMLConfig):
        pass
    C.dataset_attributes = {"news": list(attributes), "record": []}
    C.num_words_title, C.num_words_abstract = lt, la
    C.dropout_probability = p
    C.num_words, C.num_categories = num_words, num_categories
    C.num_clicked_news_a_user = clicks
    return C


def _lengths(cfg):
    return {"title": cfg.num_words_title, "abstract": cfg.num_words_abstract}


# ---- CPU: the two restatements ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("attributes", [["title"], ["title", "abstract"], ALL])
@pytest.mark.parametrize("L", [1, 3, 20, 50])
def test_numpy_restatement_equals_torch_port(attributes, L):
    from newsrecommendationsystem_b200.model.NAML import NAML
    torch.manual_seed(L)
    cfg = _cfg(attributes, lt=L, la=L)
    params = R.model_params(NAML(cfg))
    rng = np.random.default_rng(L)
    B, T, n_cand = 2, 5, 2
    news = R.random_news(rng, B, T, attributes, _lengths(cfg), cfg.num_words, cfg.num_categories)
    masks = {a: tuple(rng.choice([0.0, 1.25], size=(B * T * L, 300), p=[0.2, 0.8]) for _ in range(2))
             for a in R.TEXTS if a in attributes}
    port = R.TorchNAML(params, attributes)
    for a in R.TEXTS:
        if a in attributes:
            ref = port.text(a, news[a].reshape(B * T, L), *masks[a]).detach().numpy()
            got = R.naml_text_encoder_forward(params, a, news[a].reshape(B * T, L), *masks[a])
            np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-12)
    ref = port.forward(news, n_cand, masks).detach().numpy()
    got = R.naml_forward(params, news, n_cand, attributes, masks)
    np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-12)


def test_conv_padding_is_zero_rows_not_token_0():
    """The conv's padding rows are zeros: with a nonzero embedding row 0 (a from_pretrained table), a text of one token
    sees only its own row through the middle tap."""
    rng = np.random.default_rng(0)
    E = rng.standard_normal((5, 300))
    W = rng.standard_normal((300, 1, 3, 300)) * 0.05
    b = rng.standard_normal(300) * 0.1
    pre = R.text_prefix("title")
    params = {f"{pre}.word_embedding.weight": E, f"{pre}.CNN.weight": W, f"{pre}.CNN.bias": b,
              f"{pre}.additive_attention.linear.weight": rng.standard_normal((200, 300)) * 0.05,
              f"{pre}.additive_attention.linear.bias": np.zeros(200),
              f"{pre}.additive_attention.attention_query_vector": rng.standard_normal(200)}
    got = R.naml_text_encoder_forward(params, "title", np.array([[3]]))
    np.testing.assert_allclose(got[0], np.maximum(W[:, 0, 1] @ E[3] + b, 0), rtol=1e-12)


def test_state_dict_keys_and_shapes():
    from newsrecommendationsystem_b200 import NAML, NAMLConfig
    m = NAML(NAMLConfig)
    sd = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    V, Ncat = NAMLConfig.num_words, NAMLConfig.num_categories
    want = {}
    for t in ("title", "abstract"):
        p = f"news_encoder.text_encoders.{t}"
        want.update({f"{p}.word_embedding.weight": (V, 300), f"{p}.CNN.weight": (300, 1, 3, 300), f"{p}.CNN.bias": (300,),
                     f"{p}.additive_attention.linear.weight": (200, 300), f"{p}.additive_attention.linear.bias": (200,),
                     f"{p}.additive_attention.attention_query_vector": (200,)})
    for e in ("category", "subcategory"):
        p = f"news_encoder.element_encoders.{e}"
        want.update({f"{p}.embedding.weight": (Ncat, 100), f"{p}.linear.weight": (300, 100), f"{p}.linear.bias": (300,)})
    for p in ("news_encoder.final_attention", "user_encoder.additive_attention"):
        want.update({f"{p}.linear.weight": (200, 300), f"{p}.linear.bias": (200,), f"{p}.attention_query_vector": (200,)})
    assert sd == want
    # the shared embeddings are one parameter each
    te = m.news_encoder.text_encoders
    assert te["title"].word_embedding is te["abstract"].word_embedding
    ee = m.news_encoder.element_encoders
    assert ee["category"].embedding is ee["subcategory"].embedding
    # the reference's default Conv2d init (the module is a real nn.Conv2d)
    assert isinstance(te["title"].CNN, torch.nn.Conv2d) and te["title"].CNN.padding == (1, 0)


def test_single_attribute_has_no_final_attention():
    from newsrecommendationsystem_b200 import NAML
    m = NAML(_cfg(["title"]))
    assert not hasattr(m.news_encoder, "final_attention")


@pytest.mark.parametrize("name,value", [("num_filters", 400), ("window_size", 5), ("word_embedding_dim", 200),
                                        ("query_vector_dim", 100), ("category_embedding_dim", 50)])
def test_configuration_rule(name, value):
    from newsrecommendationsystem_b200 import NAML
    cfg = _cfg()
    setattr(cfg, name, value)
    with pytest.raises(RuntimeError, match=name):
        NAML(cfg)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from newsrecommendationsystem_b200 import _lib
    return _lib.load()


def _cnn_calls(lib, L, news_rows=None):
    fwd = lambda: lib.nrms_cnn_text_fwd(None, 4, news_rows, 4, L, None, 10, None, None, None, None, None, None, None, None, 0,
                                        0.0, 0, 0, 0, None)
    bwd = lambda: lib.nrms_cnn_text_bwd(None, None, 4, news_rows, 4, L, 10, None, None, None, None, None, None, None, None,
                                        None, None, None, 0, 0.0, 0, 0, 0, None)
    return fwd, bwd


@pytest.mark.parametrize("L", [0, -1, 65, 100])
@pytest.mark.parametrize("form", ["dense", "rows"])
def test_cnn_pair_refuses_lengths_outside_1_to_64(lib, L, form):
    """NRMS_E_UNSUPPORTED before any pointer check (every pointer here is NULL) and before any CUDA call (this runs
    without a GPU)."""
    rows = C.c_void_p(16) if form == "rows" else None
    for call in _cnn_calls(lib, L, rows):
        assert call() == 2
        assert b"text length" in lib.nrms_last_error()


@pytest.mark.parametrize("L", [1, 20, 64])
def test_cnn_pair_takes_lengths_1_to_64(lib, L):
    """Inside 1..64 the length passes and the NULL pointers are what is refused (NRMS_E_INVALID)."""
    for call in _cnn_calls(lib, L):
        assert call() == 1


def test_cnn_sizes(lib):
    rows = 7 * 37
    a = lambda n: (n + 255) // 256 * 256
    assert lib.nrms_cnn_text_stash_bytes(7, 37) == 3 * a(rows * 1200) + a(rows * 800) + a(rows * 4)
    assert lib.nrms_cnn_text_fwd_workspace_bytes(7, 37, 1, 1) == a(900 * 1200) + a(rows * 3600)
    assert lib.nrms_cnn_text_bwd_workspace_bytes(7, 37, 0) > lib.nrms_cnn_text_stash_bytes(7, 37)
    assert lib.nrms_cnn_text_stash_bytes(0, 20) == 0


def test_width_rule():
    from newsrecommendationsystem_b200 import NAML
    m = NAML(_cfg(["title"], lt=30))
    with pytest.raises(RuntimeError, match="num_words_title = 30"):
        m.news_encoder.text_encoders["title"](torch.zeros((2, 31), dtype=torch.long))


# ---- GPU ----------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda")


def _mask(rows, p, seed, offset, stream):
    from test_text_length import dropout_mask
    return dropout_mask(rows, p, seed, offset, stream)


def _text_weights(rng, V, dev):
    E = rng.standard_normal((V, 300)).astype(np.float32)
    w = dict(emb=E, conv_w=(rng.standard_normal((300, 900)) * 0.035).astype(np.float32),
             conv_b=(rng.standard_normal(300) * 0.1).astype(np.float32),
             wa=(rng.standard_normal((200, 300)) * 0.06).astype(np.float32),
             ba=(rng.standard_normal(200) * 0.1).astype(np.float32),
             qa=rng.uniform(-0.1, 0.1, 200).astype(np.float32))
    return w, {k: torch.from_numpy(v).to(dev) for k, v in w.items()}


def _relu_on(out):
    """(relu(conv) > 0) as float64 [n * L, 300], read from the stash of the nrms_cnn_text_fwd call that produced `out`
    (H, the stash's second field; nrms_b200.h).  Read before the backward, which frees the stash."""
    tokens, stash = out.grad_fn.saved_tensors[0], out.grad_fn.saved_tensors[5]
    rows = out.shape[0] * tokens.shape[1]            # one row of `out` per text, L tokens each (dense or news_rows)
    a = (rows * 1200 + 255) // 256 * 256
    h = stash[a:a + rows * 1200].view(torch.float32).view(rows, 300)
    return (h > 0).double().cpu().numpy()


def _text_params(w):
    pre = R.text_prefix("title")
    return {f"{pre}.word_embedding.weight": w["emb"].astype(np.float64),
            f"{pre}.CNN.weight": w["conv_w"].astype(np.float64).reshape(300, 1, 3, 300),
            f"{pre}.CNN.bias": w["conv_b"].astype(np.float64),
            f"{pre}.additive_attention.linear.weight": w["wa"].astype(np.float64),
            f"{pre}.additive_attention.linear.bias": w["ba"].astype(np.float64),
            f"{pre}.additive_attention.attention_query_vector": w["qa"].astype(np.float64)}


def _tokens(rng, n, L, V):
    t = rng.integers(1, V, size=(n, L))
    keep = rng.integers(1, L + 1, size=n)
    return np.where(np.arange(L)[None] < keep[:, None], t, 0).astype(np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("L", [1, 2, 7, 20, 30, 50, 64])
@pytest.mark.parametrize("form", ["dense", "rows"])
@pytest.mark.parametrize("p", [0.0, 0.2])
def test_text_encoder_vs_oracle(dev, precision, L, form, p):
    from newsrecommendationsystem_b200 import ops, _lib
    mode = _lib.MODES[precision]
    rng = np.random.default_rng(L * 7 + int(p * 10))
    V = 300
    w, wt = _text_weights(rng, V, dev)
    n = 24
    if form == "dense":
        tok = _tokens(rng, n, L, V)
        call_tok, rows = torch.from_numpy(tok).to(dev), None
    else:
        table = _tokens(rng, 40, L, V)
        idx = rng.integers(0, 40, size=n)
        tok = table[idx]
        call_tok, rows = torch.from_numpy(table).to(dev), torch.from_numpy(idx).to(dev)
    seed, offset = 77, 1234
    out = ops.cnn_text_encoder(call_tok, wt["emb"], wt["conv_w"], wt["conv_b"], wt["wa"], wt["ba"], wt["qa"], dropout_p=p,
                               seed=seed, offset=offset, mode=mode, news_rows=rows)
    masks = (None, None)
    if p > 0:
        masks = (_mask(n * L, p, seed, offset, STREAM_EMB), _mask(n * L, p, seed, offset, STREAM_CTX))
    ref = R.naml_text_encoder_forward(_text_params(w), "title", tok, *masks)
    assert rel_l2_rows(out.cpu().numpy(), ref) < TOL_VEC[precision]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_chunked_inference(dev, precision):
    """A count that crosses an inference chunk: every row against the oracle, and the chunked pass equals single calls
    on the two halves."""
    from newsrecommendationsystem_b200 import ops, _lib
    mode = _lib.MODES[precision]
    rng = np.random.default_rng(5)
    L, V = 20, 400
    n = INFER_CHUNK_ROWS // L + 77
    w, wt = _text_weights(rng, V, dev)
    tok = _tokens(rng, n, L, V)
    t = torch.from_numpy(tok).to(dev)
    args = (wt["emb"], wt["conv_w"], wt["conv_b"], wt["wa"], wt["ba"], wt["qa"])
    with torch.no_grad():
        out = ops.cnn_text_encoder(t, *args, mode=mode)
        half = ops.cnn_text_encoder(t[-100:], *args, mode=mode)
    ref = R.naml_text_encoder_forward(_text_params(w), "title", tok)
    assert rel_l2_rows(out.cpu().numpy(), ref) < TOL_VEC[precision]
    assert torch.equal(out[-100:], half)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("L", [1, 7, 30, 64])
@pytest.mark.parametrize("form", ["dense", "rows"])
def test_masks_bit_for_bit(lib, dev, precision, L, form):
    """The stash holds X = emb[token] * mask1 and A = H * mask2 (H = relu(conv)): both masks equal the numpy Philox
    masks bit for bit."""
    from newsrecommendationsystem_b200 import _lib
    from newsrecommendationsystem_b200.ops import _bytes
    mode = _lib.MODES[precision]
    rng = np.random.default_rng(L)
    V, n, p, seed, offset = 200, 16, 0.3, 0xABC, 999
    w, wt = _text_weights(rng, V, dev)
    table = _tokens(rng, n + 5, L, V)
    idx = rng.permutation(n + 5)[:n] if form == "rows" else np.arange(n)
    tok = table[idx]
    rows = torch.from_numpy(idx).to(dev) if form == "rows" else None
    t = torch.from_numpy(table if form == "rows" else tok).to(dev)
    out = torch.empty((n, 300), device=dev)
    stash = _bytes(lib.nrms_cnn_text_stash_bytes(n, L), dev)
    ws = _bytes(lib.nrms_cnn_text_fwd_workspace_bytes(n, L, mode, 1), dev)
    P = lambda x: C.c_void_p(x.data_ptr()) if x is not None else None
    rc = lib.nrms_cnn_text_fwd(P(t), t.shape[0], P(rows), n, L, P(wt["emb"]), V, P(wt["conv_w"]), P(wt["conv_b"]),
                               P(wt["wa"]), P(wt["ba"]), P(wt["qa"]), P(out), P(stash), P(ws), ws.numel(), p, seed, offset,
                               mode, None)
    assert rc == 0, lib.nrms_last_error()
    torch.cuda.synchronize()
    rows_n = n * L
    a = lambda k: (k + 255) // 256 * 256
    raw = stash.cpu().numpy()
    f = lambda off, k: raw[off:off + k * 4].view(np.float32).reshape(-1, 300)
    X = f(0, rows_n * 300)
    H = f(a(rows_n * 1200), rows_n * 300)
    A = f(2 * a(rows_n * 1200), rows_n * 300)
    m1 = _mask(rows_n, p, seed, offset, STREAM_EMB)
    m2 = _mask(rows_n, p, seed, offset, STREAM_CTX)
    emb_rows = w["emb"][tok.reshape(-1)]
    assert np.array_equal(X.view(np.uint32), (emb_rows * m1).view(np.uint32))
    assert np.array_equal(A.view(np.uint32), (H * m2).view(np.uint32))
    assert (H >= 0).all() and (H > 0).mean() > 0.2


def _gclose(got, ref, tol, what):
    den = max(float(np.abs(ref).max()), 1e-6)
    err = float(np.abs(np.asarray(got, np.float64) - ref).max()) / den
    assert err <= tol, f"{what}: {err:.3g} > {tol}"


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("L", [1, 17, 20, 50, 64])
@pytest.mark.parametrize("p", [0.0, 0.2])
def test_text_encoder_gradients_vs_torch_port(dev, precision, L, p):
    """Every gradient of the text encoder (embedding with row 0 untouched, conv weight and bias, additive block) against
    float64 autograd of the torch port, for a loss sum(out * g).  The port's ReLU passes where the kernel's did (_relu_on):
    a pre-activation within rounding of 0 falls on either side in float64 and in the kernel, and its derivative is a whole
    d_a * W term of a dX row (measured: up to 10 % of the largest embedding-gradient entry in tensor mode)."""
    from newsrecommendationsystem_b200 import ops, _lib
    mode = _lib.MODES[precision]
    rng = np.random.default_rng(100 + L)
    V, n, seed, offset = 150, 48, 321, 77
    w, wt = _text_weights(rng, V, dev)
    tok = _tokens(rng, n, L, V)
    g = rng.standard_normal((n, 300)).astype(np.float32)
    leaves = {k: v.clone().requires_grad_(True) for k, v in wt.items()}
    out = ops.cnn_text_encoder(torch.from_numpy(tok).to(dev), leaves["emb"], leaves["conv_w"], leaves["conv_b"],
                               leaves["wa"], leaves["ba"], leaves["qa"], dropout_p=p, seed=seed, offset=offset, mode=mode)
    relu_on = _relu_on(out)
    (out * torch.from_numpy(g).to(dev)).sum().backward()
    masks = (None, None, relu_on)
    if p > 0:
        masks = (_mask(n * L, p, seed, offset, STREAM_EMB), _mask(n * L, p, seed, offset, STREAM_CTX), relu_on)
    params = _text_params(w)
    port = R.TorchNAML(params, ["title"])
    ref = port.text("title", tok, *masks)
    (ref * torch.from_numpy(g.astype(np.float64))).sum().backward()
    pre = R.text_prefix("title")
    pairs = {"emb": "word_embedding.weight", "conv_w": "CNN.weight", "conv_b": "CNN.bias",
             "wa": "additive_attention.linear.weight", "ba": "additive_attention.linear.bias",
             "qa": "additive_attention.attention_query_vector"}
    for k, name in pairs.items():
        got = leaves[k].grad.cpu().numpy()
        r = port.P[f"{pre}.{name}"].grad.numpy().reshape(got.shape)
        _gclose(got, r, GTOL[precision], k)
    assert not leaves["emb"].grad[0].any()          # padding_idx


def _naml(cfg, dev, precision, seed=0):
    from newsrecommendationsystem_b200 import NAML
    torch.manual_seed(seed)
    m = NAML(cfg)
    with torch.no_grad():                              # a nonzero pad row: the library must leave its gradient alone
        m.news_encoder.text_encoders["title"].word_embedding.weight[0].normal_()
    return m.to(dev).set_precision(precision)


class _ReluPatterns:
    """Records, per text length, the ReLU pattern (_relu_on) of every training call of ops.cnn_text_encoder, at forward
    time (the backward frees the stash)."""

    def __init__(self, monkeypatch):
        from newsrecommendationsystem_b200 import ops
        self.by_len = {}
        inner = ops.cnn_text_encoder

        def wrapped(tokens, *a, **kw):
            out = inner(tokens, *a, **kw)
            if out.grad_fn is not None:
                self.by_len[tokens.shape[-1]] = _relu_on(out)
            return out
        monkeypatch.setattr(ops, "cnn_text_encoder", wrapped)

    def add_to(self, masks, cfg):
        return {name: m + (self.by_len[_lengths(cfg)[name]],) for name, m in masks.items()}


def _model_masks(model, cfg, n_texts):
    from newsrecommendationsystem_b200.model.Exp1.news_encoder import DROPOUT_SEEDS
    p = cfg.dropout_probability
    out = {}
    for name, enc in model.news_encoder.text_encoders.items():
        rows = n_texts * _lengths(cfg)[name]
        out[name] = (_mask(rows, p, DROPOUT_SEEDS[name], enc._dropout_calls, STREAM_EMB),
                     _mask(rows, p, DROPOUT_SEEDS[name], enc._dropout_calls, STREAM_CTX))
    return out


def _model_grads(model):
    seen = {}
    for k, v in model.named_parameters(remove_duplicate=False):
        seen[k] = v.grad.detach().cpu().numpy().copy()
    return seen


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("form", ["step", "step_rows"])
def test_model_training_vs_torch_port(dev, precision, form, monkeypatch):
    """Three TrainStep steps with dropout.  At each step, against the float64 torch port at the model's current
    parameters: logits (step 0), loss and every parameter gradient (shared embeddings: the sum over their encoders; row 0
    of the word embedding untouched).  The FusedAdam transition is checked against O.adam_step in float64 on the GPU's
    own gradients.  The port's ReLUs pass where the kernels' did (_ReluPatterns; see the text-encoder gradient test)."""
    from newsrecommendationsystem_b200.train import TrainStep
    cfg = _cfg(ALL, lt=20, la=37, p=0.2)
    model = _naml(cfg, dev, precision)
    relu = _ReluPatterns(monkeypatch)
    lr = 1e-3
    ts = TrainStep(model, lr=lr)
    rng = np.random.default_rng(9)
    B, n_cand, N = 4, 3, cfg.num_clicked_news_a_user
    T = n_cand + N
    table = R.random_news(rng, 60, 1, ALL, _lengths(cfg), cfg.num_words, cfg.num_categories)
    table = {a: v[:, 0] for a, v in table.items()}
    dev_table = {a: torch.from_numpy(v).to(dev) for a, v in table.items()}
    names = [k for k, _ in model.named_parameters()]
    mom = {k: (0.0, 0.0) for k in names}
    for step in range(3):
        params = R.model_params(model)
        port = R.TorchNAML(params, ALL)
        idx = rng.integers(0, 60, size=(B, T))
        news = {a: v[idx] for a, v in table.items()}
        if form == "step":
            cand = [{a: torch.from_numpy(news[a][:, j]) for a in ALL} for j in range(n_cand)]
            hist = [{a: torch.from_numpy(news[a][:, j]) for a in ALL} for j in range(n_cand, T)]
            if step == 0:
                model.train()
                masks = _model_masks(model, cfg, B * T)
                with torch.no_grad():
                    logits = model(cand, hist)
                ref_logits = port.forward(news, n_cand, masks).detach().numpy()
                assert rel_l2_rows(logits.cpu().numpy(), ref_logits) < 10 * TOL_VEC[precision]
            masks = _model_masks(model, cfg, B * T)
            loss = ts.step(cand, hist)
        else:
            masks = _model_masks(model, cfg, B * T)
            loss = ts.step_rows(dev_table, torch.from_numpy(idx[:, :n_cand]), torch.from_numpy(idx[:, n_cand:]))
        _, ref_loss, ref_grads = port.loss_and_grads(news, n_cand, relu.add_to(masks, cfg))
        assert abs(float(loss) - ref_loss) <= 10 * TOL_VEC[precision] * max(1.0, abs(ref_loss))
        grads = _model_grads(model)
        for k, g in grads.items():
            _gclose(g, ref_grads[k], GTOL[precision], k)
        assert not grads["news_encoder.text_encoders.title.word_embedding.weight"][0].any()
        for k, v in model.named_parameters():
            g = grads[k].astype(np.float64)
            p_ref, m, s = O.adam_step(params[k], g, *mom[k], step + 1, lr=lr)
            mom[k] = (m, s)
            e = np.abs(v.detach().cpu().numpy().astype(np.float64) - p_ref)
            assert (e <= 2e-8 + 2 * np.spacing(np.abs(p_ref).astype(np.float32))).all(), (k, step, float(e.max()))


@pytest.mark.gpu
def test_evaluate_directory_vs_oracle(dev, tmp_path):
    """evaluate(model, 'tests/golden/data') in FP32 mode against the numpy pipeline (first occurrence of an id wins,
    PADDED_NEWS is a zero vector), metrics equal to three decimals; a checkpoint round trip keeps the result."""
    from newsrecommendationsystem_b200 import data
    from newsrecommendationsystem_b200.evaluate import evaluate, first_occurrence_rows
    from newsrecommendationsystem_b200.checkpoint import save_checkpoint, load_checkpoint
    from newsrecommendationsystem_b200.train import TrainStep
    d = os.path.join(ROOT, "tests", "golden", "data")
    news = data.load_news_parsed(os.path.join(d, "news_parsed.tsv"), attributes=ALL)
    lt, la = news.columns["title"].shape[1], news.columns["abstract"].shape[1]
    V = int(max(news.columns["title"].max(), news.columns["abstract"].max())) + 1
    Ncat = int(max(news.columns["category"].max(), news.columns["subcategory"].max())) + 1
    cfg = _cfg(ALL, lt=lt, la=la, num_words=V, num_categories=Ncat, clicks=50)
    model = _naml(cfg, dev, "fp32", seed=3)
    got = evaluate(model, d)
    params = R.model_params(model)
    ev = data.load_behaviors(os.path.join(d, "behaviors.tsv"), news, num_clicked=50)
    n = len(news)
    table = np.zeros((n + 1, 300))
    table[:n] = R.naml_news_encoder_forward(params, news.columns, ALL)
    own = first_occurrence_rows(news.ids)
    hist = np.where(ev.hist_rows < 0, n, own[np.maximum(ev.hist_rows, 0)])
    uv = R.naml_user_encoder_forward(params, table[hist])
    per = []
    for i in range(len(ev.cand_offsets) - 1):
        a, b = ev.cand_offsets[i], ev.cand_offsets[i + 1]
        per.append(O.single_user_metric(ev.labels[a:b], (table[own[ev.cand_rows[a:b]]] @ uv[i]).tolist()))
    with np.errstate(all="ignore"):
        ref = np.nanmean(np.asarray(per, np.float64), axis=0)
    np.testing.assert_allclose(got, ref, atol=5e-4)
    # checkpoint round trip in the reference's format
    ts = TrainStep(model)
    path = str(tmp_path / "naml.pt")
    save_checkpoint(path, model, ts.optimizer, 7, 0.5)
    other = _naml(cfg, dev, "fp32", seed=11)
    assert load_checkpoint(path, other) == (7, 0.5)
    ck = torch.load(path, weights_only=False)["model_state_dict"]
    assert set(ck) == set(model.state_dict())
    assert evaluate(other, d) == got
