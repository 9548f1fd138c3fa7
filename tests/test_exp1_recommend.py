"""SURVEY 8 rows f2 / f3 / f4: index-only training minibatches, model/Exp1 and the single-user recommend path.

CPU part: the oracle's Exp1 / recommend restatements against fixtures generated from the LIVE reference modules
(tests/golden/make_golden_exp1.py).  GPU part (`-m gpu`): the CUDA path through the C-ABI against the same fixtures
and against the oracle.  Tolerances: FP32 mode 2e-5 (vectors, max row-wise relative L2), tensor mode 1e-3; gradients
2e-4 x the reference gradient's scale (FP32 mode); ranks exact, y to 1e-5.
"""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_l2_rows
from oracle import nrms_oracle as O

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from compact import expand_exp1, pinned  # noqa: E402
from exp1_weights import make_state  # noqa: E402

ATTRS = ['category', 'subcategory', 'title']
ATTRS_A = ['category', 'subcategory', 'title', 'abstract']


@pytest.fixture(scope="module")
def g1():
    return expand_exp1(np.load(os.path.join(ROOT, "tests", "golden", "exp1_golden.npz")))


def _cfg(attrs):
    from newsrecommendationsystem_b200.config import Exp1Config

    class Cfg(Exp1Config):
        num_words = 401
        num_categories = 31
        dataset_attributes = {"news": list(attrs), "record": []}
    return Cfg


def _exp1_state(attrs, seed):
    """The same seed-determined parameter values make_golden_exp1.py loaded into the reference module."""
    from newsrecommendationsystem_b200 import Exp1
    m = Exp1(_cfg(attrs))
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    return m, make_state(shapes, seed)


def _nrms_state(seed):
    from newsrecommendationsystem_b200 import NRMS, NRMSConfig

    class NCfg(NRMSConfig):
        num_words = 401
    m = NRMS(NCfg)
    return m, make_state({k: tuple(v.shape) for k, v in m.state_dict().items()}, seed)


# ---- CPU: oracle pinned against the live-reference fixtures ------------------------------------------------------
def test_oracle_exp1_forward(g1):
    _, sd = _exp1_state(ATTRS, 101)
    news = {a: g1["fwd/" + a] for a in ATTRS}
    nv = O.exp1_news_encoder_forward(sd, news, ATTRS)
    assert rel_l2_rows(nv, g1["fwd/news_vectors"]) < 2e-6
    pre = "news_encoder.element_encoders.category"
    ev = O.element_encoder_forward(sd[pre + ".embedding.weight"], sd[pre + ".linear.weight"], sd[pre + ".linear.bias"],
                                   news["category"])
    np.testing.assert_allclose(ev, g1["fwd/category_vectors"], atol=2e-6)
    uv = O.exp1_user_encoder_forward(sd, g1["fwd/user_input"])
    assert rel_l2_rows(uv, g1["fwd/user_vectors"]) < 2e-6
    tr = {a: g1["train/" + a] for a in ATTRS}
    logits = O.exp1_forward(sd, tr, int(g1["train/n_cand"]), ATTRS)
    np.testing.assert_allclose(logits, g1["train/logits"], atol=5e-6)
    loss, _ = O.cross_entropy_label0(logits)
    assert abs(float(loss) - float(g1["train/loss"])) < 1e-6


def test_oracle_exp1_abstract(g1):
    _, sd = _exp1_state(ATTRS_A, 102)
    news = {a: g1["fwda/" + a] for a in ATTRS_A}
    assert rel_l2_rows(O.exp1_news_encoder_forward(sd, news, ATTRS_A), g1["fwda/news_vectors"]) < 2e-6


def test_oracle_recommend(g1):
    _, sd = _nrms_state(103)
    table = g1["rec/table"]
    for case in range(int(g1["rec/n_cases"])):
        uv, y, order = O.recommend_user(sd, table, g1[f"rec/{case}/hist"], g1[f"rec/{case}/cand"])
        assert rel_l2_rows(uv[None], g1[f"rec/{case}/user"][None]) < 2e-6
        np.testing.assert_allclose(y, g1[f"rec/{case}/y"], atol=2e-6)
        # the order is a valid descending order of the reference's y (ties aside, it IS the reference's order)
        ry = g1[f"rec/{case}/y"]
        assert np.all(np.diff(ry[order]) <= 1e-6)
        assert sorted(order.tolist()) == list(range(len(ry)))


def test_exp1_state_dict_keys_match_reference_fixture(g1):
    m, _ = _exp1_state(ATTRS, 101)
    ref_keys = {k[5:] for k in g1 if k.startswith("grad/")}
    assert ref_keys == {k for k, _ in m.named_parameters()}


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _load(m, sd, dev, precision):
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.to(dev).eval()
    m.set_precision(precision)
    return m


TOL = {"fp32": 2e-5, "tf32": 1e-3}


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_exp1_forward_vs_reference(g1, dev, precision):
    m, sd = _exp1_state(ATTRS, 101)
    _load(m, sd, dev, precision)
    news = {a: torch.from_numpy(g1["fwd/" + a]) for a in ATTRS}
    with torch.no_grad():
        nv = m.get_news_vector(news).cpu().numpy()
        ev = m.news_encoder.element_encoders["category"](news["category"]).cpu().numpy()
        uv = m.get_user_vector(torch.from_numpy(g1["fwd/user_input"])).cpu().numpy()
    np.testing.assert_allclose(ev, g1["fwd/category_vectors"], atol=2e-6)          # fp32 in both modes
    assert rel_l2_rows(nv, g1["fwd/news_vectors"]) < TOL[precision]
    assert rel_l2_rows(uv, g1["fwd/user_vectors"]) < TOL[precision]
    assert rel_l2_rows(nv, O.exp1_news_encoder_forward(sd, {a: g1["fwd/" + a] for a in ATTRS}, ATTRS)) < TOL[precision]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_exp1_abstract_inference_vs_reference(g1, dev, precision):
    m, sd = _exp1_state(ATTRS_A, 102)
    _load(m, sd, dev, precision)
    news = {a: torch.from_numpy(g1["fwda/" + a]) for a in ATTRS_A}
    with torch.no_grad():
        nv = m.get_news_vector(news).cpu().numpy()
    assert rel_l2_rows(nv, g1["fwda/news_vectors"]) < TOL[precision]


@pytest.mark.gpu
def test_exp1_train_step_gradients_vs_reference(g1, dev):
    """Exp1.forward + CE(label 0) + backward in FP32 mode, eval-mode dropout (the fixture's setting): logits, loss and
    every parameter gradient against the live reference's autograd."""
    from newsrecommendationsystem_b200 import ops
    m, sd = _exp1_state(ATTRS, 101)
    _load(m, sd, dev, "fp32")
    K1 = int(g1["train/n_cand"])
    T = g1["train/title"].shape[1]
    items = [{a: torch.from_numpy(np.ascontiguousarray(g1["train/" + a][:, j])) for a in ATTRS} for j in range(T)]
    logits = m(items[:K1], items[K1:])
    loss = ops.cross_entropy_label0(logits)
    m.zero_grad()
    loss.backward()
    np.testing.assert_allclose(logits.detach().cpu().numpy(), g1["train/logits"], atol=2e-5)
    assert abs(float(loss) - float(g1["train/loss"])) < 1e-5
    for k, p in m.named_parameters():
        ref = g1["grad/" + k]
        got = p.grad.detach().cpu().numpy()
        got = pinned(got, 48)                      # make_golden_exp1.py stores the first 48 rows of a matrix
        scale = max(float(g1["absmax/grad/" + k]), float(g1["gradnorm/" + k]) / np.sqrt(max(p.numel(), 1)), 1e-12)
        err = float(np.abs(got - ref).max())
        assert err <= 2e-4 * scale + 1e-9, (k, err, scale)
        full_norm = float(torch.linalg.vector_norm(p.grad.double()))
        assert abs(full_norm - float(g1["gradnorm/" + k])) <= 2e-4 * float(g1["gradnorm/" + k]) + 1e-9, k


@pytest.mark.gpu
def test_additive_attention_standalone_backward(dev):
    """AdditiveAttention as a standalone trainable block (candidate sizes 3, 20, 50) against the oracle's backward."""
    from newsrecommendationsystem_b200 import ops, _lib
    rng = np.random.default_rng(3)
    for S in (3, 4, 20, 50):
        n = 11
        c = (rng.standard_normal((n, S, 300)) * 0.5).astype(np.float32)
        p = dict(Wa=rng.uniform(-0.1, 0.1, (200, 300)).astype(np.float32), ba=rng.uniform(-0.05, 0.05, 200).astype(np.float32),
                 qa=rng.uniform(-0.1, 0.1, 200).astype(np.float32))
        dout = rng.standard_normal((n, 300)).astype(np.float32)
        out_ref, cache = O.additive_forward(c, p)
        g_ref = O.additive_backward(dout, cache, p)
        tc, twa, tba, tqa = (torch.from_numpy(a).to(dev).requires_grad_(True) for a in (c, p["Wa"], p["ba"], p["qa"]))
        out = ops.additive_attention(tc, twa, tba, tqa, mode=_lib.MODE_FP32)
        out.backward(torch.from_numpy(dout).to(dev))
        assert rel_l2_rows(out.detach().cpu().numpy(), out_ref) < 2e-5
        dc_ref, grads = g_ref
        for got, ref in ((tc.grad, dc_ref), (twa.grad, grads["Wa"]), (tba.grad, grads["ba"]), (tqa.grad, grads["qa"])):
            ref = np.asarray(ref)
            assert float(np.abs(got.cpu().numpy() - ref).max()) <= 2e-4 * max(float(np.abs(ref).max()), 1e-12) + 1e-9


@pytest.mark.gpu
def test_recommend_user_vs_reference(g1, dev):
    """nrms_recommend_user (two cluster launches) against the reference's single-user arithmetic: user vector, y and the
    returned order; Recommender.recommend over id strings gives the same pair."""
    from newsrecommendationsystem_b200.recommend import Recommender
    m, sd = _nrms_state(103)
    _load(m, sd, dev, "fp32")
    table = torch.from_numpy(g1["rec/table"]).to(dev)
    ids = [f"N{i}" for i in range(table.shape[0] - 1)]
    rec = Recommender(m, ids, table)
    for case in range(int(g1["rec/n_cases"])):
        hist, cand = g1[f"rec/{case}/hist"], g1[f"rec/{case}/cand"]
        order, scores, user = rec.recommend_rows(hist, cand)
        ry = g1[f"rec/{case}/y"]
        assert rel_l2_rows(user.cpu().numpy()[None], g1[f"rec/{case}/user"][None]) < 2e-5
        y = (scores.cpu().numpy().astype(np.float64) + 1) / 2
        np.testing.assert_allclose(y, ry, atol=1e-5)
        order = order.cpu().numpy()
        assert sorted(order.tolist()) == list(range(len(ry)))
        # the kernel's order is exactly the stable descending order of ITS scores ...
        assert np.array_equal(order, np.argsort(-y, kind="stable"))
        # ... and equals the reference's order wherever the reference's scores are separated by more than fp32 noise
        ref_order = g1[f"rec/{case}/order"]
        gaps = np.abs(np.diff(ry[ref_order]))
        if len(gaps) == 0 or gaps.min() > 1e-5:
            assert np.array_equal(order, ref_order)
        else:
            assert np.all(np.abs(ry[order] - ry[ref_order]) <= 1e-5)
    # id-string API: left-padded first-50 history, 'id-label' impressions (recommend.py:117-124,301-332)
    hist0 = [f"N{i}" for i in g1["rec/4/hist"] if i != table.shape[0] - 1]
    imps = [f"N{i}-0" for i in g1["rec/4/cand"]]
    got_ids, got_y = rec.recommend(hist0, imps)
    ref_order = g1["rec/4/order"]
    np.testing.assert_allclose(got_y, g1["rec/4/y"][ref_order], atol=1e-5)
    assert sorted(got_ids.tolist()) == sorted(f"N{i}" for i in g1["rec/4/cand"])
    assert np.all(np.diff(got_y) <= 0)


@pytest.mark.gpu
def test_recommend_user_matches_batched_encoder(dev):
    """Full-size check: the latency kernels against the library's own batched FP32 user encoder + CSR scoring on a
    65k-row table (the two paths share no kernel), plus scores-only mode for a candidate list beyond the ranking limit."""
    from newsrecommendationsystem_b200 import NRMS, NRMSConfig, ops, _lib
    torch.manual_seed(0)
    m = NRMS(NRMSConfig).to(dev).eval().set_precision("fp32")
    n_rows = 65239
    table = torch.randn(n_rows, 300, device=dev) * 0.4
    table[-1] = 0
    rng = np.random.default_rng(0)
    hist = torch.from_numpy(rng.integers(0, n_rows, 50).astype(np.int32)).to(dev)
    ue = m.user_encoder
    w = (*ue.multihead_self_attention.packed(), ue.additive_attention.linear.weight, ue.additive_attention.linear.bias,
         ue.additive_attention.attention_query_vector)
    with torch.no_grad():
        uref = ops.user_encoder_indexed(table, hist.view(1, 50), *w, mode=_lib.MODE_FP32)
    for C in (300, 4096, 10000):
        cand = torch.from_numpy(rng.integers(0, n_rows, C).astype(np.int32)).to(dev)
        user, scores, order = ops.recommend_user(table, hist, cand, *w, rank=(C <= 4096))
        assert rel_l2_rows(user.cpu().numpy()[None], uref.cpu().numpy()) < 2e-5
        sref = (table[cand.long()].double() @ uref[0].double()).cpu().numpy()
        np.testing.assert_allclose(scores.cpu().numpy(), sref, atol=2e-5 * max(1.0, float(np.abs(sref).max())))
        if order is not None:
            s = scores.cpu().numpy()
            assert np.array_equal(order.cpu().numpy(), np.argsort(-s.astype(np.float64), kind="stable"))
    with pytest.raises(RuntimeError):
        ops.recommend_user(table, hist, torch.zeros(5000, dtype=torch.int32, device=dev), *w, rank=True)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_index_only_minibatch_equals_token_minibatch(golden_sd, dev, precision):
    """f2: TrainStep.step_rows (token table + news-row indices, gathered inside the embedding kernels) produces
    bit-identical parameters to TrainStep.step_tokens on the materialised token tensor (same dropout stream)."""
    from newsrecommendationsystem_b200 import NRMS
    from newsrecommendationsystem_b200.train import TrainStep
    from test_gpu_parity import Cfg

    def fresh():
        m = NRMS(Cfg)
        m.load_state_dict({k: torch.from_numpy(v) for k, v in golden_sd.items()})
        return m.to(dev).train().set_precision(precision)
    rng = np.random.default_rng(9)
    table = rng.integers(0, Cfg.num_words, size=(500, 20)).astype(np.int64)
    cand = rng.integers(0, 500, size=(16, 5)).astype(np.int64)
    hist = rng.integers(0, 500, size=(16, 50)).astype(np.int64)
    from newsrecommendationsystem_b200 import ops
    m1, m2 = fresh(), fresh()
    t_table = torch.from_numpy(table).to(dev)
    # one forward + backward through each form: same dropout stream, same arithmetic -> same loss and gradients (the
    # weight gradients go through fp32 atomics, so "same" is up to their summation order)
    l1 = ops.cross_entropy_label0(m1.forward_rows(t_table, torch.from_numpy(cand), torch.from_numpy(hist)))
    l1.backward()
    l2 = ops.cross_entropy_label0(m2.forward_tokens(torch.from_numpy(table[np.concatenate([cand, hist], axis=1)]), 5))
    l2.backward()
    assert abs(float(l1.detach()) - float(l2.detach())) < 1e-6
    for (k, a), (_, b) in zip(m1.named_parameters(), m2.named_parameters()):
        scale = max(float(b.grad.abs().max()), 1e-12)
        assert float((a.grad - b.grad).abs().max()) <= 2e-5 * scale + 1e-9, k
    # and the optimizer-step form runs on index-only minibatches (two steps, finite decreasing-or-equal loss scale)
    ts1 = TrainStep(fresh())
    losses = [float(ts1.step_rows(t_table, torch.from_numpy(cand), torch.from_numpy(hist))) for _ in range(2)]
    assert all(np.isfinite(losses)) and abs(losses[0] - float(l1.detach())) < 0.05
    with pytest.raises(IndexError):
        ts1.step_rows(t_table, torch.from_numpy(cand + 500), torch.from_numpy(hist))
