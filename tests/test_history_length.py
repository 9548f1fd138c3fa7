"""Click histories of any length from 1 to 64 (config.num_clicked_news_a_user): the user encoder, training, evaluate and
the single-user path at lengths other than the compiled 20 and 50.

CPU part: the C-ABI's length rule (1..64 for every user-encoder entry point and for the standalone additive block) and
the workspace sizes at a run-time length.  GPU part (`-m gpu`): every result against the fp64 oracle (`oracle/`) or the
fp64 Exp1 restatement of test_exp1_abstract_train.py.
"""
import numpy as np
import pytest
import torch

from conftest import rel_l2_rows
from oracle import nrms_oracle as O

TOL_VEC = {"fp32": 2e-5, "tf32": 1e-3}          # test_gpu_parity.py: news / user vectors, max row-wise relative L2
GTOL = {"fp32": 2e-4, "tf32": 3e-3}             # gradients, relative to the tensor's largest entry
INFER_CHUNK_ROWS = 2048 * 20                    # encoder.cu: rows per inference pass


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from newsrecommendationsystem_b200 import _lib
    return _lib.load()


# ---- CPU ------------------------------------------------------------------------------------------------------------
def _user_calls(lib, S):
    """Every user-encoder entry point with null pointers (4 users, FP32 mode)."""
    n = None
    return {
        "fwd": lambda: lib.nrms_user_encoder_fwd(n, 0, n, 4, S, n, n, n, n, n, n, n, n, 0, 0, n),
        "ln_fwd": lambda: lib.nrms_user_encoder_ln_fwd(n, 0, n, 4, S, n, n, n, n, n, n, n, n, n, n, 0, 0, n),
        "bwd": lambda: lib.nrms_user_encoder_bwd(n, 4, S, n, n, n, n, n, n, n, n, n, n, n, 0, 0, n),
        "ln_bwd": lambda: lib.nrms_user_encoder_ln_bwd(n, 4, S, n, n, n, n, n, n, n, n, n, n, n, n, n, n, 0, 0, n),
        "table16_fwd": lambda: lib.nrms_user_encoder_table16_fwd(n, 10, n, 4, S, n, n, n, n, n, n, n, 0, n),
    }


@pytest.mark.parametrize("S", [0, -1, 65])
def test_user_encoder_refuses_lengths_outside_1_to_64(lib, S):
    for name, call in _user_calls(lib, S).items():
        assert call() == 2 and b"unsupported" in lib.nrms_last_error(), name


@pytest.mark.parametrize("S", [1, 37, 64])
def test_user_encoder_takes_lengths_1_to_64(lib, S):
    """Past the length check, the null pointers are what the call refuses."""
    for name, call in _user_calls(lib, S).items():
        assert call() == 1, (name, lib.nrms_last_error())


def test_additive_block_lengths(lib):
    n = None
    for S in (0, 65):
        assert lib.nrms_additive_fwd(n, 4, S, n, n, n, n, n, 0, 0, n) == 2 and b"unsupported" in lib.nrms_last_error()
        assert lib.nrms_additive_bwd(n, n, 4, S, n, n, n, n, n, n, n, n, 0, 0, n) == 2
        assert b"unsupported" in lib.nrms_last_error()
    for S in (1, 7, 64):
        assert lib.nrms_additive_fwd(n, 4, S, n, n, n, n, n, 0, 0, n) == 1
        assert lib.nrms_additive_bwd(n, n, 4, S, n, n, n, n, n, n, n, n, 0, 0, n) == 1


def _al(nbytes):
    return (nbytes + 255) // 256 * 256


def _stash(rows, ln=False):
    b = _al(rows * 300 * 4) + _al(rows * 900 * 4) + _al(rows * 300 * 4) + _al(rows * 200 * 4) + _al(rows * 4)
    return b + (_al(rows * 300 * 4) + _al(rows * 2 * 4) if ln else 0)


def test_sizes_at_a_run_time_length(lib):
    S, n = 37, 5000
    rows = n * S
    assert lib.nrms_encoder_stash_bytes(n, S) == _stash(rows)
    assert lib.nrms_encoder_ln_stash_bytes(n, S) == _stash(rows, True)
    chunk = INFER_CHUNK_ROWS // S                       # inference runs chunks of whole users, in both modes
    for mode in (0, 1):
        assert lib.nrms_encoder_fwd_workspace_bytes(n, S, mode, 0, 0) == _stash(chunk * S, True) + 256
        assert lib.nrms_encoder_fwd_workspace_bytes(n, S, mode, 0, 1000) == _stash(chunk * S, True) + 256
        assert lib.nrms_encoder_fwd_workspace_bytes(3, S, mode, 0, 0) == _stash(3 * S, True) + 256
    ldr = (rows + 3) // 4 * 4
    common = _al(rows * 300 * 4) + _al(rows * 200 * 4) + _al(rows * 900 * 4) + _al(rows * 300 * 4) + _al(296 * 900 * 4)
    assert lib.nrms_encoder_bwd_workspace_bytes(n, S, 0) == common + 256
    assert lib.nrms_encoder_bwd_workspace_bytes(n, S, 1) == \
        common + _al(ldr * 900 * 4) + _al(ldr * 300 * 4) + _al(900 * 300 * 4) + 256
    assert lib.nrms_user_encoder_table16_workspace_bytes(n, S, 1000) == _stash(chunk * S) + 256 > 0
    assert lib.nrms_user_encoder_table16_workspace_bytes(n, 65, 1000) == 0


# ---- GPU ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _user_params(golden_sd, ln, seed=7):
    """fp64 user-encoder parameters of the oracle (the golden weights; LayerNorm weight and bias drawn)."""
    p = {k: v.astype(np.float64) for k, v in O.enc_params(golden_sd, O.USER).items()}
    if ln:
        rng = np.random.default_rng(seed)
        p["ln_g"] = (1 + 0.2 * rng.standard_normal(300)).astype(np.float32).astype(np.float64)
        p["ln_b"] = (0.1 * rng.standard_normal(300)).astype(np.float32).astype(np.float64)
    return p


def _device_weights(p, dev):
    w = [np.concatenate([p["Wq"], p["Wk"], p["Wv"]]), np.concatenate([p["bq"], p["bk"], p["bv"]]), p["Wa"], p["ba"], p["qa"]]
    w = [_t(x.astype(np.float32), dev) for x in w]
    ln = (_t(p["ln_g"].astype(np.float32), dev), _t(p["ln_b"].astype(np.float32), dev)) if "ln_g" in p else None
    return w, ln


def _table(rng, n_rows):
    table = (rng.standard_normal((n_rows + 1, 300)) * 0.3).astype(np.float32)
    table[n_rows] = 0                                  # PADDED_NEWS
    return table


FWD_LENGTHS = [1, 2, 7, 16, 17, 30, 33, 49, 51, 63, 64]
_worst = {}


@pytest.mark.gpu
@pytest.mark.parametrize("ln", [False, True], ids=["nrms", "ln"])
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("S", FWD_LENGTHS)
def test_user_encoder_forward_vs_oracle(dev, golden_sd, S, precision, ln):
    """Dense, fp32-indexed and (tensor mode, plain NRMS) fp16-table forms, from 1 user to a count that crosses an
    inference chunk.  The dense and fp32-indexed forms read the same rows and agree bitwise."""
    from newsrecommendationsystem_b200 import ops, _lib
    mode = _lib.MODES[precision]
    p = _user_params(golden_sd, ln)
    w, lnw = _device_weights(p, dev)
    rng = np.random.default_rng(S)
    n_rows = 997
    table = _table(rng, n_rows)
    tb = _t(table, dev)
    for n_users in (1, INFER_CHUNK_ROWS // S + 2):
        rows = rng.integers(0, n_rows + 1, size=(n_users, S))
        rows[::5, : S // 2] = n_rows                       # left-padded histories
        ref, _ = O.encoder_forward(table[rows].astype(np.float64), p, 15)
        ix = _t(rows.astype(np.int32), dev)
        with torch.no_grad():
            dense = ops.user_encoder(_t(table[rows], dev), *w, mode=mode, ln=lnw)
            idx = ops.user_encoder_indexed(tb, ix, *w, mode=mode, ln=lnw)
        assert torch.equal(dense, idx), (S, n_users)
        err = rel_l2_rows(dense.cpu().numpy(), ref)
        assert err < TOL_VEC[precision], (S, n_users, err)
        _worst[(precision, ln)] = max(_worst.get((precision, ln), 0.0), err)
        if precision == "tf32" and not ln:
            with torch.no_grad():
                f16 = ops.user_encoder_table16(ops.pack_rows_f16(tb[:n_rows]), ix, *w)
            e16 = rel_l2_rows(f16.cpu().numpy(), ref)
            assert e16 < TOL_VEC["tf32"], (S, n_users, e16)
            _worst["table16"] = max(_worst.get("table16", 0.0), e16)
    print(f"worst relative L2 so far: { {str(k): f'{v:.2e}' for k, v in _worst.items()} }")


@pytest.mark.gpu
@pytest.mark.parametrize("ln", [False, True], ids=["nrms", "ln"])
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("S", [1, 17, 30, 64])
def test_user_encoder_gradients_vs_oracle(dev, golden_sd, S, precision, ln):
    """dX and every user-encoder parameter gradient against encoder_backward in fp64."""
    from newsrecommendationsystem_b200 import ops, _lib
    mode = _lib.MODES[precision]
    p = _user_params(golden_sd, ln)
    rng = np.random.default_rng(100 + S)
    n = 41
    x = (rng.standard_normal((n, S, 300)) * 0.4).astype(np.float32)
    x[3, : S // 2] = 0
    dout = rng.standard_normal((n, 300)).astype(np.float32)
    out_ref, cache = O.encoder_forward(x.astype(np.float64), p, 15)
    dx_ref, g_ref = O.encoder_backward(dout.astype(np.float64), cache, p, 15)
    g_ref["Wqkv"] = np.concatenate([g_ref.pop("Wq"), g_ref.pop("Wk"), g_ref.pop("Wv")])
    g_ref["bqkv"] = np.concatenate([g_ref.pop("bq"), g_ref.pop("bk"), g_ref.pop("bv")])
    w, lnw = _device_weights(p, dev)
    leaves = [v.requires_grad_() for v in w] + ([v.requires_grad_() for v in lnw] if lnw else [])
    xd = _t(x, dev).requires_grad_()
    out = ops.user_encoder(xd, *w, mode=mode, ln=tuple(leaves[5:]) if lnw else None)
    assert rel_l2_rows(out.detach().cpu().numpy(), out_ref) < TOL_VEC[precision]
    out.backward(_t(dout, dev))
    got = dict(zip(["Wqkv", "bqkv", "Wa", "ba", "qa", "ln_g", "ln_b"], [v.grad for v in leaves]), dX=xd.grad)
    g_ref["dX"] = dx_ref
    assert set(got) == set(g_ref)
    # d ba and (at long histories) d Wa are sums that cancel to a small fraction of their terms, so both sides hold
    # summation-order noise there: the floor is 1e-6 of the largest gradient entry, as in test_gpu_parity.py; the
    # LayerNorm variant takes that file's wider gradient bounds
    gtol = {"fp32": 3e-4, "tf32": 5e-3}[precision] if ln else GTOL[precision]
    floor = 1e-6 * max(float(np.abs(v).max()) for v in g_ref.values())
    worst = 0.0
    for k, ref in g_ref.items():
        sc = float(np.abs(ref).max()) + 1e-12
        err = float(np.abs(got[k].cpu().numpy() - ref).max())
        assert err <= gtol * sc + floor, (S, k, err, sc)
        worst = max(worst, err / sc)
    print(f"S = {S} [{precision}{', LayerNorm' if ln else ''}]: worst gradient error / largest entry {worst:.2e}")


class _Cfg30:
    num_words = 401
    word_embedding_dim = 300
    num_attention_heads = 15
    query_vector_dim = 200
    dropout_probability = 0.2
    num_words_title = 20
    num_clicked_news_a_user = 30


def _nrms(golden_sd, dev, precision, S=30, ln=False):
    """NRMS built for S clicks (the LayerNorm variant with drawn LayerNorm weights) -> (model, its fp32 state dict)."""
    from newsrecommendationsystem_b200 import NRMS

    class Cfg(_Cfg30):
        num_clicked_news_a_user = S
        use_layernorm = ln
    m = NRMS(Cfg)
    rng = np.random.default_rng(5)
    sd = {}
    for k, v in m.state_dict().items():
        if k in golden_sd:
            sd[k] = golden_sd[k]
        elif k.endswith("layer_norm.weight"):
            sd[k] = (1 + 0.2 * rng.standard_normal(tuple(v.shape))).astype(np.float32)
        else:
            sd[k] = (0.1 * rng.standard_normal(tuple(v.shape))).astype(np.float32)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.to(dev).eval().set_precision(precision)
    return m, sd


@pytest.mark.gpu
@pytest.mark.parametrize("precision,ltol", [("fp32", 1e-5), ("tf32", 2e-3)])
def test_nrms_step_rows_at_30_clicks(dev, golden_sd, precision, ltol):
    """TrainStep.step_rows with num_clicked_news_a_user = 30: loss and every gradient against oracle.nrms_backward."""
    from newsrecommendationsystem_b200 import synthetic
    from newsrecommendationsystem_b200.train import TrainStep
    m, sd = _nrms(golden_sd, dev, precision)
    ntok = synthetic.make_news(300, num_words=401, seed=31)
    rng = np.random.default_rng(32)
    cand = rng.integers(0, 300, size=(16, 5))
    hist = rng.integers(0, 300, size=(16, 30))
    sd64 = {k: v.astype(np.float64) for k, v in sd.items()}
    logits, cache = O.nrms_forward(sd64, ntok[cand], ntok[hist])
    loss_ref, dlogits = O.cross_entropy_label0(logits)
    grads = O.nrms_backward(dlogits, cache, sd64)
    ts = TrainStep(m)
    loss = float(ts.step_rows(_t(ntok, dev), torch.from_numpy(cand), torch.from_numpy(hist)))
    assert abs(loss - float(loss_ref)) < ltol, (loss, loss_ref)
    for k, p in m.named_parameters():
        ref = grads[k]
        sc = float(np.abs(ref).max()) + 1e-12
        err = float(np.abs(p.grad.cpu().numpy() - ref).max())
        assert err <= GTOL[precision] * sc + 1e-8, (k, err, sc)


@pytest.mark.gpu
def test_nrms_three_adam_steps_at_30_clicks(dev, golden_sd):
    """Three FusedAdam steps (FP32 mode) with num_clicked_news_a_user = 30 against oracle.train_step."""
    from newsrecommendationsystem_b200 import synthetic
    from newsrecommendationsystem_b200.train import TrainStep
    m, sd = _nrms(golden_sd, dev, "fp32")
    ntok = synthetic.make_news(300, num_words=401, seed=41)
    cand, clicked = synthetic.make_train_batch(8, ntok, k_neg=4, history=30, seed=42)
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
        assert d.max() <= 6 * lr and d.mean() <= 0.02 * lr, (k, float(d.max()), float(d.mean()))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_exp1_at_30_clicks_gradients_vs_fp64(dev, precision):
    """Exp1 (title and abstract) with num_clicked_news_a_user = 30: forward and every gradient against the fp64
    restatement."""
    from newsrecommendationsystem_b200 import Exp1, ops
    from exp1_weights import make_state
    from test_exp1_recommend import ATTRS_A, _cfg
    from test_exp1_abstract_train import EXP1_TOL, _items, _named, exp1_fp64

    class Cfg(_cfg(ATTRS_A)):
        num_clicked_news_a_user = 30
    m = Exp1(Cfg)
    sd = make_state({k: tuple(v.shape) for k, v in m.state_dict().items()}, 102)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.to(dev).eval().set_precision(precision)
    rng = np.random.default_rng(11)
    B, n_cand, T = 5, 3, 33
    news = {"title": rng.integers(1, 401, size=(B, T, 20)), "abstract": rng.integers(1, 401, size=(B, T, 50)),
            "category": rng.integers(0, 31, size=(B, T)), "subcategory": rng.integers(0, 31, size=(B, T))}
    news["title"][:, :, 12:] = 0
    news["abstract"][:, :, 35:] = 0
    news = {k: v.astype(np.int64) for k, v in news.items()}
    items = _items(news, ATTRS_A)
    logits = m(items[:n_cand], items[n_cand:])
    loss = ops.cross_entropy_label0(logits)
    m.zero_grad()
    loss.backward()
    loss_ref, logits_ref, grads = exp1_fp64(_named(m, sd), news, n_cand, ATTRS_A)
    ltol, gtol = EXP1_TOL[precision]
    np.testing.assert_allclose(logits.detach().cpu().numpy(), logits_ref, atol=10 * ltol)
    assert abs(float(loss.detach()) - loss_ref) < ltol
    floor = 1e-6 * max(float(np.abs(v).max()) for v in grads.values())
    for k, p in m.named_parameters():
        ref = grads[k]
        sc = float(np.abs(ref).max()) + 1e-12
        err = float(np.abs(p.grad.detach().cpu().numpy() - ref).max())
        assert err <= gtol * sc + floor, (k, err, sc)


@pytest.mark.gpu
@pytest.mark.parametrize("ln", [False, True], ids=["nrms", "ln"])
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("S", [30, 64])
def test_evaluate_at_other_lengths(dev, golden_sd, S, precision, ln):
    """evaluate_tensors over histories of S clicks against oracle.evaluate_pipeline: metrics to 3 decimals and every
    candidate's score."""
    from newsrecommendationsystem_b200 import synthetic
    from newsrecommendationsystem_b200.evaluate import EvalInputs, evaluate_tensors
    m, sd = _nrms(golden_sd, dev, precision, S=S, ln=ln)
    ntok = synthetic.make_news(400, num_words=401, seed=S)
    imp = synthetic.make_impressions(300, 400, history=S, seed=S + 1, single_class_every=17, max_cand=40)
    ref_means, _, ref_scores, _, ref_uv = O.evaluate_pipeline({k: v.astype(np.float64) for k, v in sd.items()}, ntok,
                                                              imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"],
                                                              imp["labels"])
    inp = EvalInputs(ntok, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"], device=dev)
    means, det = evaluate_tensors(m, inp, return_details=True)
    assert np.abs(np.asarray(means) - ref_means).max() < 1e-3, (means, ref_means)
    tol = TOL_VEC[precision] if not ln else 5 * TOL_VEC[precision]
    assert rel_l2_rows(det["user_vectors"].cpu().numpy(), ref_uv) < tol
    sc = det["scores"].cpu().numpy()
    assert np.abs(sc - ref_scores).max() < 10 * tol * np.abs(ref_scores).max()


@pytest.mark.gpu
def test_evaluate_directory_at_30_clicks(dev, golden_sd):
    """evaluate(model, directory) reads the model's history length from its config."""
    import os
    from newsrecommendationsystem_b200 import data, evaluate as E
    directory = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "data")
    m, sd = _nrms(golden_sd, dev, "fp32")
    means = E.evaluate(m, directory)
    news = data.load_news_parsed(os.path.join(directory, "news_parsed.tsv"))
    ev = data.load_behaviors(os.path.join(directory, "behaviors.tsv"), news, num_clicked=30)
    assert ev.hist_rows.shape[1] == 30
    from newsrecommendationsystem_b200.evaluate import first_occurrence_rows
    owner = first_occurrence_rows(news.ids)
    hist = np.where(ev.hist_rows >= 0, owner[np.maximum(ev.hist_rows, 0)], -1)
    ref = O.evaluate_pipeline(sd, news.title, hist, ev.cand_offsets, owner[ev.cand_rows], ev.labels)[0]
    np.testing.assert_allclose(means, ref, atol=1e-5)


def _recommender(golden_sd, dev, n_news=6000):
    from newsrecommendationsystem_b200.recommend import Recommender
    m, sd = _nrms(golden_sd, dev, "fp32")
    rng = np.random.default_rng(61)
    table = _table(rng, n_news)
    ids = [f"N{i}" for i in range(n_news)]
    return Recommender(m, ids, _t(table, dev)), sd, table, ids, rng


@pytest.mark.gpu
def test_recommend_at_30_clicks(dev, golden_sd):
    """Recommender.recommend with num_clicked_news_a_user = 30, on both sides of the 4,096-candidate limit: the user
    vector and scores against oracle.recommend_user; the order is exactly the stable descending order of the scores,
    and the oracle's order wherever the oracle's neighbouring scores are further apart than the FP32 error."""
    rec, sd, table, ids, rng = _recommender(golden_sd, dev)
    for n_clicked, n_cand in ((12, 300), (45, 5000)):
        clicked = [ids[i] for i in rng.choice(len(ids), n_clicked, replace=False)]
        cand = [ids[i] for i in rng.choice(len(ids), n_cand, replace=False)]
        hist = rec.history_rows(clicked)
        assert len(hist) == 30 and hist.count(rec.pad_row) == max(0, 30 - n_clicked)
        cand_rows = [rec.row_of[c] for c in cand]
        uv_ref, y_ref, order_ref = O.recommend_user(sd, table.astype(np.float64), hist, cand_rows)
        order, scores, uv = rec.recommend_rows(hist, cand_rows)
        order, scores = order.cpu().numpy(), scores.cpu().numpy()
        assert rel_l2_rows(uv.cpu().numpy()[None], uv_ref[None]) < TOL_VEC["fp32"]
        assert np.abs((scores.astype(np.float64) + 1) / 2 - y_ref).max() < 1e-5
        assert np.array_equal(order, np.argsort(-scores, kind="stable"))
        got_ids, y = rec.recommend(clicked, cand)
        assert list(got_ids) == [cand[i] for i in order] and np.array_equal(y, (scores[order].astype(np.float64) + 1) / 2)
        gaps = np.abs(np.diff(y_ref[order_ref]))
        sep = np.concatenate([[True], gaps > 1e-5]) & np.concatenate([gaps > 1e-5, [True]])
        assert np.array_equal(order[sep], order_ref[sep]), int((order[sep] != order_ref[sep]).sum())


@pytest.mark.gpu
def test_top_k_at_30_clicks(dev, golden_sd):
    """Recommender.top_k with num_clicked_news_a_user = 30 against ranking every news of the table."""
    rec, sd, table, ids, rng = _recommender(golden_sd, dev, n_news=3000)
    clicked = [ids[i] for i in rng.choice(len(ids), 20, replace=False)]
    got_ids, y = rec.top_k(clicked, 25)
    hist = rec.history_rows(clicked)
    uv, y_all, _ = O.recommend_user(sd, table.astype(np.float64), hist, list(range(len(ids))))
    y_all[[rec.row_of[c] for c in clicked]] = -np.inf
    order = np.argsort(-y_all, kind="stable")[:25]
    assert list(got_ids) == [ids[i] for i in order]
    assert np.abs(y - y_all[order]).max() < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("S", [1, 5, 37, 64])
def test_standalone_additive_attention(dev, golden_sd, S, precision):
    """AdditiveAttention at S candidates: forward and backward against oracle.additive_backward."""
    from newsrecommendationsystem_b200 import ops, _lib
    p = {k: v.astype(np.float64) for k, v in O.enc_params(golden_sd, O.USER).items()}
    rng = np.random.default_rng(70 + S)
    c = (rng.standard_normal((29, S, 300)) * 0.5).astype(np.float32)
    dout = rng.standard_normal((29, 300)).astype(np.float32)
    ref, cache = O.additive_forward(c.astype(np.float64), p)
    dc_ref, g_ref = O.additive_backward(dout.astype(np.float64), cache, p)
    cd = _t(c, dev).requires_grad_()
    w = [_t(p[k].astype(np.float32), dev).requires_grad_() for k in ("Wa", "ba", "qa")]
    out = ops.additive_attention(cd, *w, mode=_lib.MODES[precision])
    assert rel_l2_rows(out.detach().cpu().numpy(), ref) < TOL_VEC[precision]
    out.backward(_t(dout, dev))
    for name, got, want in (("c", cd.grad, dc_ref), ("Wa", w[0].grad, g_ref["Wa"]), ("ba", w[1].grad, g_ref["ba"]),
                            ("qa", w[2].grad, g_ref["qa"])):
        sc = float(np.abs(want).max()) + 1e-12
        err = float(np.abs(got.cpu().numpy() - want).max())
        assert err <= GTOL[precision] * sc, (S, name, err, sc)
