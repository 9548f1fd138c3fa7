"""GPU parity tests: the CUDA path (through the C-ABI) vs the numpy oracle and the committed
reference-generated golden fixtures.  Run on the B200 box: pytest -m gpu.

Tolerances (north_star): gathers / indexing bit-exact; news & user vectors <= 1e-3 max row-wise
relative L2 in TF32 mode (<= 2e-5 in FP32 mode); metrics equal to 3 decimals.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_l2_rows
from compact import expand_masked, pinned
from oracle import nrms_oracle as O

pytestmark = pytest.mark.gpu

TOL_VEC = {"fp32": 2e-5, "tf32": 1e-3}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib():
    from newsrecommendationsystem_b200 import _lib
    return _lib.load()


class Cfg:
    num_words = 401
    word_embedding_dim = 300
    num_attention_heads = 15
    query_vector_dim = 200
    dropout_probability = 0.2
    num_words_title = 20
    num_clicked_news_a_user = 50


def make_model(golden_sd, dev, precision, cfg=Cfg):
    from newsrecommendationsystem_b200 import NRMS
    m = NRMS(cfg)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in golden_sd.items()})   # reference keys/shapes
    m.to(dev).eval()
    m.set_precision(precision)
    return m


def t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


# ---------------------------------------------------------------------------------------------
def test_library_loaded_and_versioned(lib):
    assert lib.nrms_abi_version() == 2


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
@pytest.mark.parametrize("shape", [(128, 256, 32), (1000, 900, 300), (257, 200, 300), (61, 300, 900), (4096, 900, 300)])
def test_gemm_nt(dev, mode, shape):
    from newsrecommendationsystem_b200 import ops, _lib
    M, N, K = shape
    g = torch.Generator(device="cpu").manual_seed(M * 7 + N)
    a = torch.randn(M, K, generator=g).to(dev)
    b = (torch.randn(N, K, generator=g) * 0.1).to(dev)
    bias = torch.randn(N, generator=g).to(dev)
    c = ops.gemm_nt(a, b, bias, mode=_lib.MODES[mode])
    ref = (a.double() @ b.double().T + bias.double())
    err = (c.double() - ref).abs().max().item()
    scale = ref.abs().max().item()
    # TF32: operands rounded to 11-bit significands -> ~2^-11 relative per product, averaged over K
    tol = 2e-6 if mode == "fp32" else 2e-3
    assert err / scale < tol, (mode, shape, err, scale)


def test_gather_bit_exact(dev, lib, golden, golden_sd):
    """Embedding gather inside nrms_news_encoder_fwd (training stash X) is a bit-exact row copy."""
    from newsrecommendationsystem_b200._lib import ptr, stream_ptr, check, MODE_FP32
    from newsrecommendationsystem_b200 import ops
    toks = t(golden["fwd/tokens"], dev)
    n, L = toks.shape
    sd = {k: t(v, dev) for k, v in golden_sd.items()}
    p = O.enc_keys("news_encoder")
    wqkv = torch.cat([sd[p["Wq"]], sd[p["Wk"]], sd[p["Wv"]]]).contiguous()
    bqkv = torch.cat([sd[p["bq"]], sd[p["bk"]], sd[p["bv"]]]).contiguous()
    stash = torch.zeros(lib.nrms_encoder_stash_bytes(n, L), dtype=torch.uint8, device=dev)
    ws = torch.zeros(max(256, lib.nrms_encoder_fwd_workspace_bytes(n, L, MODE_FP32, 1, 0)), dtype=torch.uint8, device=dev)
    out = torch.empty(n, 300, device=dev)
    check(lib.nrms_news_encoder_fwd(ptr(toks), n, L, ptr(sd[O.EMB_KEY]), sd[O.EMB_KEY].shape[0], ptr(wqkv), ptr(bqkv),
                                    ptr(sd[p["Wa"]]), ptr(sd[p["ba"]]), ptr(sd[p["qa"]]), ptr(out), ptr(stash),
                                    ptr(ws), ws.numel(), 0.0, 0, 0, MODE_FP32, stream_ptr(dev)))
    torch.cuda.synchronize()
    x = stash[: n * L * 300 * 4].view(torch.float32).view(n, L, 300).cpu().numpy()
    assert np.array_equal(x.view(np.uint32), golden["fwd/gathered"].view(np.uint32))
    # the standalone gather entry point is bit-exact too
    g2 = ops.gather_rows(sd[O.EMB_KEY], toks.reshape(-1)).cpu().numpy().reshape(n, L, 300)
    assert np.array_equal(g2.view(np.uint32), golden["fwd/gathered"].view(np.uint32))


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_news_vectors_golden(dev, golden, golden_sd, precision):
    m = make_model(golden_sd, dev, precision)
    with torch.no_grad():
        nv = m.get_news_vector({"title": torch.from_numpy(golden["fwd/tokens"])})   # CPU input, like the DataLoader
    err = rel_l2_rows(nv.cpu().numpy(), golden["fwd/news_vectors"])
    assert err < TOL_VEC[precision], err


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_user_vectors_golden(dev, golden, golden_sd, precision):
    m = make_model(golden_sd, dev, precision)
    with torch.no_grad():
        uv = m.get_user_vector(t(golden["fwd/user_input"], dev))
    err = rel_l2_rows(uv.cpu().numpy(), golden["fwd/user_vectors"])
    assert err < TOL_VEC[precision], err


def test_scores_golden(dev, golden, golden_sd):
    m = make_model(golden_sd, dev, "fp32")
    nv, uv = t(golden["fwd/news_vectors"], dev), t(golden["fwd/user_vectors"], dev)
    with torch.no_grad():
        s = m.get_prediction(nv[:23], uv[0])
        sb = m.click_predictor(nv[:36].reshape(9, 4, 300), uv)
    np.testing.assert_allclose(s.cpu().numpy(), golden["fwd/scores_single"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(sb.cpu().numpy(), golden["fwd/scores_batched"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("n", [1, 6, 7, 130, 2049])
def test_news_encoder_vs_oracle_ragged_sizes(dev, golden_sd, precision, n):
    """Batch sizes around the tile boundaries (1 title, partial tiles, > one inference chunk)."""
    from newsrecommendationsystem_b200 import synthetic
    toks = synthetic.make_news(n, num_words=Cfg.num_words, seed=100 + n)
    if n > 6:
        toks[3] = 0          # all-pad title
    ref, _ = O.news_encoder_forward(golden_sd, toks)
    m = make_model(golden_sd, dev, precision)
    with torch.no_grad():
        nv = m.get_news_vector({"title": torch.from_numpy(toks)})
    assert rel_l2_rows(nv.cpu().numpy(), ref) < TOL_VEC[precision]


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("table_path", [0, 1])
def test_news_encoder_50_token_text(dev, lib, golden_sd, precision, table_path):
    """The text encoder at the other compiled length (50 tokens, e.g. an abstract: reference
    src/model/Exp1/news_encoder.py:10-34 is this same block): per-text projection and table path."""
    from newsrecommendationsystem_b200 import synthetic
    rng = np.random.default_rng(50)
    toks = rng.integers(1, Cfg.num_words, size=(333, 50)).astype(np.int64)
    toks[:, 37:] = 0
    toks[5] = 0
    ref, _ = O.news_encoder_forward(golden_sd, toks)
    m = make_model(golden_sd, dev, precision)
    lib.nrms_set_option(b"news_table_attn", table_path)
    try:
        with torch.no_grad():
            nv = m.get_news_vector({"title": torch.from_numpy(toks)})
    finally:
        lib.nrms_set_option(b"news_table_attn", 1)
    assert rel_l2_rows(nv.cpu().numpy(), ref) < TOL_VEC[precision]


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_user_encoder_indexed_equals_dense(dev, lib, golden_sd, precision):
    lib.nrms_set_option(b"user_table_attn", 0)      # per-user projection path (K1 v6): the gather is a pure copy
    try:
        _indexed_equals_dense(dev, golden_sd, precision)
    finally:
        lib.nrms_set_option(b"user_table_attn", 1)


def _indexed_equals_dense(dev, golden_sd, precision):
    rng = np.random.default_rng(5)
    table = rng.standard_normal((301, 300)).astype(np.float32) * 0.3
    table[300] = 0
    rows = rng.integers(0, 300, size=(67, 50))
    rows[4, :31] = 300
    rows[9] = 300
    ref, _ = O.user_encoder_forward(golden_sd, table[rows])
    m = make_model(golden_sd, dev, precision)
    tb = t(table, dev)
    with torch.no_grad():
        a = m.user_encoder.forward_indexed(tb, t(rows.astype(np.int32), dev))
        b = m.get_user_vector(tb[t(rows, dev)])
    assert rel_l2_rows(a.cpu().numpy(), ref) < TOL_VEC[precision]
    assert torch.equal(a, b)      # the in-library gather is a pure copy


@pytest.mark.parametrize("n_users,n_rows", [(1, 3), (13, 60), (67, 300), (200, 1000), (2500, 4001)])
def test_user_encoder_table_attention_path(dev, lib, golden_sd, n_users, n_rows):
    """K1g (tensor mode, indexed input): the table is projected once (q|k|v rows in fp16) and the attention runs on
    gathered rows.  Same numbers as the per-user projection within the 1e-3 tolerance: vs the oracle, and vs K1 v6."""
    rng = np.random.default_rng(n_users)
    table = (rng.standard_normal((n_rows + 1, 300)) * 0.3).astype(np.float32)
    table[n_rows] = 0                                     # PADDED_NEWS
    rows = rng.integers(0, n_rows, size=(n_users, 50))
    rows[0, :50 - min(49, n_users)] = n_rows              # left-padded history
    if n_users > 9:
        rows[9] = n_rows                                  # empty history
        rows[3] = rows[3, 0]                              # one news repeated 50 times
    assert n_users * 50 >= 8 * (n_rows + 1)               # well inside the size rule that selects the table path
    ref, _ = O.user_encoder_forward(golden_sd, table[rows])
    m = make_model(golden_sd, dev, "tf32")
    tb, ix = t(table, dev), t(rows.astype(np.int32), dev)
    with torch.no_grad():
        try:
            a = m.user_encoder.forward_indexed(tb, ix)
            lib.nrms_set_option(b"user_table_attn", 0)
            b = m.user_encoder.forward_indexed(tb, ix)
        finally:
            lib.nrms_set_option(b"user_table_attn", 1)
    assert rel_l2_rows(a.cpu().numpy(), ref) < TOL_VEC["tf32"]
    assert rel_l2_rows(b.cpu().numpy(), ref) < TOL_VEC["tf32"]
    assert not torch.equal(a, b)                          # two different kernels really ran
    assert rel_l2_rows(a.cpu().numpy(), b.cpu().numpy().astype(np.float64)) < TOL_VEC["tf32"]


@pytest.mark.parametrize("n_titles,num_words", [(2, 3), (37, 80), (777, 401), (6000, 2001)])
def test_news_encoder_table_attention_path(dev, lib, golden_sd, n_titles, num_words):
    """The news encoder over the projected EMBEDDING table (tensor mode, token rows >= 8 x vocabulary rows): same
    vectors as the per-title projection (K1 v6) within the 1e-3 tolerance, vs the oracle and vs each other."""
    from newsrecommendationsystem_b200 import synthetic
    sd = dict(golden_sd)
    rng = np.random.default_rng(num_words)
    emb = rng.standard_normal((num_words, 300)).astype(np.float32)
    emb[0] = 0
    sd["news_encoder.word_embedding.weight"] = emb

    class C2(Cfg):
        pass
    C2.num_words = num_words
    toks = synthetic.make_news(n_titles, num_words=num_words, seed=n_titles)
    if n_titles > 11:
        toks[11] = 0                                        # an all-padding title
    assert n_titles * 20 >= 8 * num_words
    ref, _ = O.news_encoder_forward(sd, toks)
    m = make_model(sd, dev, "tf32", cfg=C2)
    with torch.no_grad():
        a = m.get_news_vector({"title": torch.from_numpy(toks)})
        lib.nrms_set_option(b"news_table_attn", 0)
        try:
            b = m.get_news_vector({"title": torch.from_numpy(toks)})
        finally:
            lib.nrms_set_option(b"news_table_attn", 1)
    assert rel_l2_rows(a.cpu().numpy(), ref) < TOL_VEC["tf32"]
    assert rel_l2_rows(b.cpu().numpy(), ref) < TOL_VEC["tf32"]
    assert not torch.equal(a, b)                            # two different kernels really ran
    assert rel_l2_rows(a.cpu().numpy(), b.cpu().numpy().astype(np.float64)) < TOL_VEC["tf32"]


# ---------------------------------------------------------------------------------------------
def _train_once(golden, golden_sd, dev, precision, adamw=False, steps=1):
    from newsrecommendationsystem_b200.train import TrainStep
    m = make_model(golden_sd, dev, precision)
    m.eval()   # goldens were produced in eval mode (dropout = identity), grads still flow
    ts = TrainStep(m, lr=1e-4, adamw=adamw, weight_decay=0.01 if adamw else 0.0)
    cand, clicked = golden["train/cand"], golden["train/clicked"]
    titles = torch.from_numpy(np.concatenate([cand, clicked], axis=1))
    losses, grads = [], None
    for _ in range(steps):
        loss = ts.step_tokens(titles, cand.shape[1])
        losses.append(float(loss.item()))
        if grads is None:
            grads = {k: p.grad.detach().clone().cpu().numpy() for k, p in m.named_parameters()}
    return m, losses, grads


def test_train_step_fp32_matches_reference(dev, golden, golden_sd):
    m, losses, grads = _train_once(golden, golden_sd, dev, "fp32", steps=2)
    assert abs(losses[0] - float(golden["train/loss"])) < 1e-5
    assert abs(losses[1] - float(golden["train/loss2"])) < 2e-5
    for k, g in grads.items():
        ref = golden["train/grad/" + k]
        got = pinned(g, None if "embedding" in k else 48)
        scale = golden["absmax/train/grad/" + k] + 1e-12
        assert np.abs(got - ref).max() < 2e-4 * scale + 1e-8, (k, np.abs(got - ref).max(), scale)
    assert not grads[O.EMB_KEY][0].any()
    sd = {k: v.detach().cpu().numpy() for k, v in m.state_dict().items()}
    for k, v in sd.items():
        ref = golden["train/adam2/" + k]
        got = pinned(v, 48)
        gs = float(np.abs(golden["train/grad/" + k]).mean())
        d = np.abs(got.astype(np.float64) - ref)
        assert d.max() <= 2.5e-4, k                      # never more than ~2 lr per step off
        if gs >= 1e-5:                                    # tensors whose Adam update is well conditioned
            assert (d <= 1e-6).mean() >= 0.8 and d.mean() < 2e-6, (k, d.mean())


def test_train_step_tensor_mode_gradients(dev, golden, golden_sd):
    """Tensor mode: forward projections AND the four backward contractions (dX, dC, dWqkv, dWa: split-K, atomic and
    accumulate epilogues of the tcgen05 GEMM over transposed operand copies) run with TF32 operands.  Every gradient
    stays within 3e-3 of the reference's fp32 gradient (relative to the tensor's largest entry), the loss within 2e-3."""
    m, losses, grads = _train_once(golden, golden_sd, dev, "tf32", steps=1)
    assert abs(losses[0] - float(golden["train/loss"])) < 2e-3
    for k, g in grads.items():
        ref = golden["train/grad/" + k]
        got = pinned(g, None if "embedding" in k else 48)
        scale = golden["absmax/train/grad/" + k] + 1e-12
        assert np.abs(got - ref).max() < 3e-3 * scale + 1e-8, (k, np.abs(got - ref).max(), scale)
    assert not grads[O.EMB_KEY][0].any()


def test_train_logits_tf32(dev, golden, golden_sd):
    m = make_model(golden_sd, dev, "tf32")
    cand, clicked = golden["train/cand"], golden["train/clicked"]
    titles = torch.from_numpy(np.concatenate([cand, clicked], axis=1))
    with torch.no_grad():
        logits = m.forward_tokens(titles, cand.shape[1])
    np.testing.assert_allclose(logits.cpu().numpy(), golden["train/logits"], rtol=0, atol=2e-3)


def test_reference_list_of_dict_api(dev, golden, golden_sd):
    """model(candidate_news, clicked_news) with the reference's list-of-dict minibatch (train.py:202-203)."""
    m = make_model(golden_sd, dev, "fp32")
    cand, clicked = golden["train/cand"], golden["train/clicked"]
    cn = [{"title": torch.from_numpy(cand[:, i])} for i in range(cand.shape[1])]
    cl = [{"title": torch.from_numpy(clicked[:, i])} for i in range(clicked.shape[1])]
    with torch.no_grad():
        y = m(cn, cl)
    np.testing.assert_allclose(y.cpu().numpy(), golden["train/logits"], rtol=0, atol=2e-5)


def test_adam_kernel_elementwise(dev, golden, golden_sd):
    from newsrecommendationsystem_b200 import ops
    for k in golden_sd:
        if "embedding" in k:
            continue
        p0 = pinned(golden_sd[k], 48)
        g = golden["train/grad/" + k]
        for tag, kw in (("adam1", {}), ("adamw1", dict(weight_decay=0.01, decoupled=True))):
            p = t(p0.reshape(-1).copy(), dev)
            m_ = torch.zeros_like(p)
            v_ = torch.zeros_like(p)
            ops.adam_step_(p, t(g.reshape(-1).copy(), dev), m_, v_, 1, lr=1e-4, **kw)
            np.testing.assert_allclose(p.cpu().numpy().reshape(p0.shape), golden[f"train/{tag}/" + k], rtol=0,
                                       atol=2e-8, err_msg=k)


def test_ce_loss_and_score_backward_vs_oracle(dev):
    from newsrecommendationsystem_b200 import ops
    rng = np.random.default_rng(3)
    cand = rng.standard_normal((17, 5, 300)).astype(np.float32)
    user = rng.standard_normal((17, 300)).astype(np.float32)
    ct, ut = t(cand, dev).requires_grad_(), t(user, dev).requires_grad_()
    logits = ops.click_score(ct, ut)
    loss = ops.cross_entropy_label0(logits)
    loss.backward()
    lo = O.click_score(cand, user)
    l_ref, dl = O.cross_entropy_label0(lo)
    assert abs(float(loss.item()) - float(l_ref)) < 1e-4 * abs(float(l_ref))
    np.testing.assert_allclose(ct.grad.cpu().numpy(), dl[:, :, None] * user[:, None, :], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(ut.grad.cpu().numpy(), np.einsum("bc,bcx->bx", dl, cand), rtol=1e-4, atol=1e-5)


# ---------------------------------------------------------------------------------------------
def test_rank_metrics_golden(dev, golden):
    from newsrecommendationsystem_b200 import ops
    per, sums = ops.rank_metrics(t(golden["metric/scores"], dev), t(golden["metric/labels"], dev),
                                 t(golden["metric/offsets"], dev))
    per = per.cpu().numpy()
    offs = golden["metric/offsets"]
    for i in range(len(offs) - 1):
        a, b = offs[i], offs[i + 1]
        y, sc = golden["metric/labels"][a:b], golden["metric/scores"][a:b]
        want = O.single_user_metric(y.astype(np.int64), sc.tolist())
        if np.isnan(want).any():
            assert np.isnan(per[i]).all()
        else:
            np.testing.assert_allclose(per[i], want, rtol=1e-12)          # == oracle (reversed-stable ties)
            ref = golden["metric/results"][i]
            if len(np.intersect1d(sc[y == 1], sc[y == 0])) == 0:
                np.testing.assert_allclose(per[i], ref, rtol=1e-12)      # == reference, tie-free cases
            else:
                np.testing.assert_allclose(per[i][0], ref[0], rtol=1e-12)  # AUC is tie-order free
    s = sums.cpu().numpy()
    np.testing.assert_allclose(s[:4] / s[4:], np.nanmean(per, axis=0), rtol=1e-12)


def test_rank_metrics_long_impression_and_empty(dev):
    """C above the shared-memory staging cap (512) takes the global-memory path; n=0 is legal."""
    from newsrecommendationsystem_b200 import ops
    rng = np.random.default_rng(9)
    C_ = [700, 3, 513, 2]
    offs = np.concatenate([[0], np.cumsum(C_)]).astype(np.int64)
    sc = rng.standard_normal(offs[-1]).astype(np.float32)
    lb = (rng.random(offs[-1]) < 0.2).astype(np.int8)
    lb[offs[:-1]] = 1
    lb[offs[:-1] + 1] = 0
    per, _ = ops.rank_metrics(t(sc, dev), t(lb, dev), t(offs, dev))
    for i in range(4):
        a, b = offs[i], offs[i + 1]
        np.testing.assert_allclose(per[i].cpu().numpy(), O.single_user_metric(lb[a:b].astype(np.int64), sc[a:b].tolist()),
                                   rtol=1e-12)
    per0, s0 = ops.rank_metrics(t(sc[:0], dev), t(lb[:0], dev), t(offs[:1], dev))
    assert per0.shape == (0, 4) and float(s0.sum().item()) == 0.0


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_evaluate_pipeline_golden(dev, golden, golden_sd, precision):
    from newsrecommendationsystem_b200.evaluate import EvalInputs, evaluate_tensors
    m = make_model(golden_sd, dev, precision)
    inp = EvalInputs(golden["eval/news_tokens"], golden["eval/hist_rows"], golden["eval/cand_offsets"],
                     golden["eval/cand_rows"], golden["eval/labels"], news_ids=golden["eval/news_ids"], device=dev)
    means, det = evaluate_tensors(m, inp, max_count=int(golden["eval/max_count"]), return_details=True)
    ref_per = golden["eval/per_impression"]
    per = det["per_impression"].cpu().numpy()
    assert per.shape == ref_per.shape                       # max_count - 1 impressions (off-by-one kept)
    assert np.array_equal(np.isnan(per), np.isnan(ref_per))
    scores = det["scores"].cpu().numpy()
    np.testing.assert_allclose(scores, golden["eval/scores"], rtol=0, atol=5e-5 if precision == "fp32" else 3e-3)
    if precision == "fp32":
        # fp32 summation order differs from torch's: a near-tie can swap two ranks in an impression
        same = np.isclose(per, ref_per, rtol=1e-9, atol=1e-12, equal_nan=True)
        assert same.mean() >= 0.95, same.mean()
        assert np.nanmax(np.abs(per - ref_per)) < 0.05
    np.testing.assert_allclose(means, golden["eval/means"], atol=5e-4 if precision == "fp32" else 5e-3)


def test_evaluate_full_size_tensor_vs_fp32_mode(dev):
    """BASELINE configs[1] at FULL size (65,238 news, 73,152 impressions, 2.7 M candidates, 70,976-word vocabulary):
    the oracle would take minutes here, so the tensor-core pipeline (K1 v5 / K2, every tile shape and the chunked
    launches) is checked against the library's own FP32 CUDA-core mode -- which the small-size tests tie to the
    oracle and the reference goldens: every news vector within 1e-3 relative, metric means equal to 3 decimals,
    scores within 5e-3, and the run is deterministic (two passes are bit-identical)."""
    import bench
    from newsrecommendationsystem_b200 import NRMS, NRMSConfig, synthetic
    from newsrecommendationsystem_b200.evaluate import EvalHost, EvalInputs, evaluate_tensors
    sd = synthetic.init_state_dict(num_words=bench.NUM_WORDS, seed=0)
    news, imp = bench.make_data(1)
    host = EvalHost(news, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"])
    inp = EvalInputs.from_host(host, dev)
    out = {}
    for precision in ("fp32", "tf32"):
        m = NRMS(NRMSConfig)
        m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
        m.to(dev).eval().set_precision(precision)
        means, det = evaluate_tensors(m, inp, return_details=True)
        out[precision] = (np.asarray(means), det["table"].clone(), det["scores"].clone())
        if precision == "tf32":
            means2, det2 = evaluate_tensors(m, inp, return_details=True)
            assert torch.equal(det2["table"], det["table"]) and torch.equal(det2["scores"], det["scores"])
            assert np.array_equal(np.asarray(means2), np.asarray(means))
    (m32, t32, s32), (mtc, ttc, stc) = out["fp32"], out["tf32"]
    n = bench.NEWS_PER_GPU
    rel = (ttc[:n] - t32[:n]).norm(dim=1) / t32[:n].norm(dim=1)
    assert float(rel.max()) < 1e-3, float(rel.max())
    assert float(ttc[n:].abs().max()) == 0.0                      # PADDED_NEWS row stays exactly zero
    assert float((stc - s32).abs().max()) < 5e-3
    np.testing.assert_allclose(mtc, m32, atol=5e-4)


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_evaluate_pipeline_vs_oracle_medium(dev, golden_sd, precision):
    """3k news / 2k impressions: metric means agree with the oracle to 3 decimals."""
    from newsrecommendationsystem_b200 import synthetic
    from newsrecommendationsystem_b200.evaluate import EvalInputs, evaluate_tensors
    Nn, I = 3000, 2000
    ntok = synthetic.make_news(Nn, num_words=Cfg.num_words, seed=41)
    imp = synthetic.make_impressions(I, Nn, seed=42, single_class_every=50)
    ref_means, ref_per, ref_scores, ref_table, ref_uv = O.evaluate_pipeline(
        golden_sd, ntok, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"])
    m = make_model(golden_sd, dev, precision)
    inp = EvalInputs(ntok, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"], device=dev)
    means, det = evaluate_tensors(m, inp, return_details=True)
    assert rel_l2_rows(det["table"][:Nn].cpu().numpy(), ref_table[:Nn]) < TOL_VEC[precision]
    assert not det["table"][Nn].any()
    assert rel_l2_rows(det["user_vectors"].cpu().numpy(), ref_uv) < TOL_VEC[precision]
    np.testing.assert_allclose(means, ref_means, atol=5e-4)
    assert np.array_equal(np.isnan(det["per_impression"].cpu().numpy()), np.isnan(ref_per))


def test_dropout_determinism_and_scale(dev, golden_sd):
    """Train-mode dropout: same (seed, offset) -> same result; different offset -> different;
    backward regenerates the same masks (gradient of sum(out) wrt a scaled input is consistent)."""
    from newsrecommendationsystem_b200 import ops, _lib, synthetic
    sd = {k: t(v, dev) for k, v in golden_sd.items()}
    p = O.enc_keys("news_encoder")
    wqkv = torch.cat([sd[p["Wq"]], sd[p["Wk"]], sd[p["Wv"]]]).contiguous()
    bqkv = torch.cat([sd[p["bq"]], sd[p["bk"]], sd[p["bv"]]]).contiguous()
    toks = t(synthetic.make_news(64, num_words=Cfg.num_words, seed=77), dev)
    args = (sd[O.EMB_KEY], wqkv, bqkv, sd[p["Wa"]], sd[p["ba"]], sd[p["qa"]])
    a = ops.news_encoder(toks, *args, dropout_p=0.2, seed=11, offset=5, mode=_lib.MODE_FP32)
    b = ops.news_encoder(toks, *args, dropout_p=0.2, seed=11, offset=5, mode=_lib.MODE_FP32)
    c = ops.news_encoder(toks, *args, dropout_p=0.2, seed=11, offset=6, mode=_lib.MODE_FP32)
    e = ops.news_encoder(toks, *args, dropout_p=0.0, mode=_lib.MODE_FP32)
    assert torch.equal(a, b) and not torch.equal(a, c) and not torch.equal(a, e)
    # directional finite difference through the dropout path (masks fixed by seed/offset)
    emb = sd[O.EMB_KEY].clone().requires_grad_()
    out = ops.news_encoder(toks, emb, *args[1:], dropout_p=0.2, seed=11, offset=5, mode=_lib.MODE_FP32)
    w = torch.randn_like(out)
    (out * w).sum().backward()
    direction = torch.randn_like(emb)
    direction[0] = 0
    eps = 1e-2
    with torch.no_grad():
        f1 = (ops.news_encoder(toks, emb + eps * direction, *args[1:], dropout_p=0.2, seed=11, offset=5,
                               mode=_lib.MODE_FP32) * w).sum().double()
        f0 = (ops.news_encoder(toks, emb - eps * direction, *args[1:], dropout_p=0.2, seed=11, offset=5,
                               mode=_lib.MODE_FP32) * w).sum().double()
    fd = float((f1 - f0) / (2 * eps))
    an = float((emb.grad.double() * direction.double()).sum())
    assert abs(fd - an) < 2e-2 * max(1.0, abs(an)), (fd, an)


def test_unsupported_shape_and_cpu_inputs_fail_loudly(dev, golden_sd):
    from newsrecommendationsystem_b200 import ops
    m = make_model(golden_sd, dev, "fp32")
    with pytest.raises(RuntimeError):
        m.get_news_vector({"title": torch.zeros(4, 21, dtype=torch.long)})     # title length 21 not compiled
    with pytest.raises(RuntimeError):
        ops.click_score(torch.zeros(2, 3, 300), torch.zeros(2, 300))           # CPU tensors: no fallback


@pytest.mark.parametrize("seed", [1, 2])
def test_per_sequence_projection_kernel_agrees_with_oracle(dev, lib, golden_sd, seed):
    """K1 v6 (per-sequence projection on tcgen05: the path of dense input, small calls and the LayerNorm variant) stays
    inside the 1e-3 tolerance, news and users; unknown options / out-of-range values are refused."""
    from newsrecommendationsystem_b200 import synthetic
    lib.nrms_set_option(b"news_table_attn", 0)       # 777 titles over a 401-word vocabulary would take the table path
    try:
        m = make_model(golden_sd, dev, "tf32")
        toks = synthetic.make_news(777, num_words=Cfg.num_words, seed=500 + seed)
        toks[11] = 0
        ref_n, _ = O.news_encoder_forward(golden_sd, toks)
        rng = np.random.default_rng(seed)
        ux = (rng.standard_normal((93, 50, 300)) * 0.4).astype(np.float32)
        ux[5, :40] = 0
        ref_u, _ = O.user_encoder_forward(golden_sd, ux)
        with torch.no_grad():
            nv = m.get_news_vector({"title": torch.from_numpy(toks)})
            uv = m.get_user_vector(t(ux, dev))
        assert rel_l2_rows(nv.cpu().numpy(), ref_n) < TOL_VEC["tf32"]
        assert rel_l2_rows(uv.cpu().numpy(), ref_u) < TOL_VEC["tf32"]
    finally:
        lib.nrms_set_option(b"news_table_attn", 1)
    assert lib.nrms_set_option(b"table_ratio", 0) == 1 and lib.nrms_set_option(b"nope", 1) == 1
    assert lib.nrms_set_option(b"table_ratio", 4) == 0


def test_table_ratio_option_selects_the_path(dev, lib, golden_sd):
    """The size rule of the table path (gathered rows >= table_ratio x table rows): the same call run on both sides of
    the rule gives two different kernels' results, both inside the tolerance."""
    rng = np.random.default_rng(12)
    table = (rng.standard_normal((301, 300)) * 0.3).astype(np.float32)
    table[300] = 0
    rows = rng.integers(0, 300, size=(40, 50))            # 2,000 gathered rows over 301 table rows: ratio 6.6
    ref, _ = O.user_encoder_forward(golden_sd, table[rows])
    m = make_model(golden_sd, dev, "tf32")
    tb, ix = t(table, dev), t(rows.astype(np.int32), dev)
    with torch.no_grad():
        try:
            a = m.user_encoder.forward_indexed(tb, ix)                 # default ratio 4 -> table path
            assert lib.nrms_set_option(b"table_ratio", 8) == 0
            b = m.user_encoder.forward_indexed(tb, ix)                 # ratio 8 -> per-sequence projection
        finally:
            lib.nrms_set_option(b"table_ratio", 4)
    assert rel_l2_rows(a.cpu().numpy(), ref) < TOL_VEC["tf32"] and rel_l2_rows(b.cpu().numpy(), ref) < TOL_VEC["tf32"]
    assert not torch.equal(a, b)


def test_news_encoder_int32_tokens(dev, lib, golden_sd):
    """nrms_news_encoder_i32_fwd (evaluate's int32 token table): bit-identical to the int64 call, on both kernel paths."""
    from newsrecommendationsystem_b200 import synthetic
    m = make_model(golden_sd, dev, "tf32")
    for n in (5, 777):                                   # per-title projection (small call), table path
        toks = synthetic.make_news(n, num_words=Cfg.num_words, seed=n)
        with torch.no_grad():
            a = m.get_news_vector({"title": torch.from_numpy(toks)})
            b = m.get_news_vector({"title": torch.from_numpy(toks.astype(np.int32))})
        assert torch.equal(a, b)
    with pytest.raises(IndexError):
        m.get_news_vector({"title": torch.full((2, 20), Cfg.num_words, dtype=torch.int32)})


def test_user_encoder_fp16_table_form(dev, lib, golden_sd):
    """nrms_user_encoder_table16_fwd: the indexed user encoder fed with the caller's fp16 copy of the table (the form
    evaluate keeps between its stages) gives bit-identical vectors to the fp32-table call, on both kernel paths."""
    from newsrecommendationsystem_b200 import ops
    rng = np.random.default_rng(21)
    table = (rng.standard_normal((401, 300)) * 0.3).astype(np.float32)
    table[400] = 0
    rows = rng.integers(0, 401, size=(77, 50))
    rows[3, :20] = 400
    m = make_model(golden_sd, dev, "tf32")
    tb, ix = t(table, dev), t(rows.astype(np.int32), dev)
    ref, _ = O.user_encoder_forward(golden_sd, table[rows])
    with torch.no_grad():
        t16 = ops.pack_rows_f16(tb)
        assert t16.shape == (402, 320) and not t16[401].any() and float(t16[0, 300]) == 1.0
        for ratio in (4, 64):                                            # table path, then per-sequence projection
            try:
                lib.nrms_set_option(b"table_ratio", ratio)
                a = m.user_encoder.forward_indexed(tb, ix)
                b = m.user_encoder.forward_indexed(t16, ix)
            finally:
                lib.nrms_set_option(b"table_ratio", 4)
            assert torch.equal(a, b)
            assert rel_l2_rows(b.cpu().numpy(), ref) < TOL_VEC["tf32"]


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_standalone_l0_blocks(dev, golden_sd, precision):
    """MultiHeadSelfAttention.forward / AdditiveAttention.forward called on their own (reference L0 API)."""
    m = make_model(golden_sd, dev, precision)
    rng = np.random.default_rng(12)
    x = (rng.standard_normal((7, 20, 300)) * 0.5).astype(np.float32)
    p_ = O.enc_params(golden_sd, "news_encoder")
    ref_c, _ = O.mhsa_forward(x, p_, 15)
    ref_o, _ = O.additive_forward(ref_c, p_)
    att, add = m.news_encoder.multihead_self_attention, m.news_encoder.additive_attention
    att.precision = add.precision = precision
    with torch.no_grad():
        c = att(t(x, dev))
        o = add(t(ref_c, dev))
    tol = 2e-5 if precision == "fp32" else 1e-3
    assert rel_l2_rows(c.cpu().numpy(), ref_c) < tol
    assert rel_l2_rows(o.cpu().numpy(), ref_o) < tol
    with pytest.raises(NotImplementedError):
        with torch.no_grad():
            att(t(x, dev), K=t(x[:, :5], dev))          # cross-attention is not compiled


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_mhsa_length_mask(dev, precision):
    """MultiHeadSelfAttention.forward(Q, length=...) (multihead_self.py:60-68) against vectors produced by the live
    reference module (tests/golden/mhsa_masked_golden.npz) for both compiled sequence lengths."""
    import os
    from newsrecommendationsystem_b200.model.general.attention.multihead_self import MultiHeadSelfAttention
    g = expand_masked(np.load(os.path.join(GOLDEN, "mhsa_masked_golden.npz")))
    att = MultiHeadSelfAttention(300, 15)
    att.load_state_dict({f"W_{n.upper()}.{k}": torch.from_numpy(g[f"{'W' if k == 'weight' else 'b'}{n}"])
                         for n in "qkv" for k in ("weight", "bias")})
    att.to(dev).eval()
    att.precision = precision
    for S in (20, 50):
        with torch.no_grad():
            c = att(t(g[f"S{S}/x"], dev), length=torch.from_numpy(g[f"S{S}/length"]))
            c0 = att(t(g[f"S{S}/x"], dev))
        tol = 2e-5 if precision == "fp32" else 1e-3
        full = c.cpu().numpy()
        assert not full[g[f"S{S}/length"] == 0].any()          # the rows of the length-0 sequence are exactly zero
        ref = g[f"S{S}/ctx"].reshape(-1, 300)                  # the reference at the positions the fixture keeps
        got = full[:, g[f"S{S}/pos"]].reshape(-1, 300)
        keep = np.linalg.norm(ref, axis=1) > 0
        assert rel_l2_rows(got[keep], ref[keep]) < tol
        # every position against the oracle (pinned to the reference in test_oracle_golden.py)
        ora, _ = O.mhsa_forward(g[f"S{S}/x"], {k: g[k] for k in ("Wq", "bq", "Wk", "bk", "Wv", "bv")}, 15,
                                length=g[f"S{S}/length"])
        ora = ora.reshape(-1, 300)
        keep = np.linalg.norm(ora, axis=1) > 0
        assert rel_l2_rows(full.reshape(-1, 300)[keep], ora[keep]) < tol
        assert torch.equal(c[0], c0[0]) and torch.equal(c[5], c0[5])     # length >= S: the mask is a no-op


# ---------------------------------------------------------------------------------------------
# config-5 variant: LayerNorm(300) on the self-attention context of both encoders (builder-defined; the oracle's
# version of it is pinned against torch autograd in tests/test_oracle_golden.py)
# ---------------------------------------------------------------------------------------------
class CfgLN(Cfg):
    use_layernorm = True


def _ln_state_dict(golden_sd, seed=11):
    rng = np.random.default_rng(seed)
    sd = dict(golden_sd)
    for prefix in (O.NEWS, O.USER):
        sd[f"{prefix}.layer_norm.weight"] = (1 + 0.1 * rng.standard_normal(300)).astype(np.float32)
        sd[f"{prefix}.layer_norm.bias"] = (0.1 * rng.standard_normal(300)).astype(np.float32)
    return sd


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_layernorm_variant_vectors_and_evaluate(dev, golden_sd, precision):
    from newsrecommendationsystem_b200 import synthetic
    from newsrecommendationsystem_b200.evaluate import EvalInputs, evaluate_tensors
    sd = _ln_state_dict(golden_sd)
    m = make_model(sd, dev, precision, cfg=CfgLN)
    assert set(m.state_dict().keys()) == set(sd.keys())
    toks = synthetic.make_news(1500, num_words=Cfg.num_words, seed=77)
    toks[3] = 0
    ref_n, _ = O.news_encoder_forward(sd, toks)
    rng = np.random.default_rng(5)
    ux = (rng.standard_normal((131, 50, 300)) * 0.4).astype(np.float32)
    ux[2, :45] = 0
    ref_u, _ = O.user_encoder_forward(sd, ux)
    with torch.no_grad():
        nv = m.get_news_vector({"title": torch.from_numpy(toks)})
        uv = m.get_user_vector(t(ux, dev))
    tol = {"fp32": 3e-5, "tf32": 2e-3}[precision]       # the normalisation divides by the row spread
    assert rel_l2_rows(nv.cpu().numpy(), ref_n) < tol
    assert rel_l2_rows(uv.cpu().numpy(), ref_u) < tol
    imp = synthetic.make_impressions(600, 1500, seed=78, single_class_every=40)
    ref_means = O.evaluate_pipeline(sd, toks, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"])[0]
    inp = EvalInputs(toks, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"], device=dev)
    means = evaluate_tensors(m, inp)
    np.testing.assert_allclose(means, ref_means, atol=5e-4 if precision == "fp32" else 5e-3)


@pytest.mark.parametrize("precision,gtol", [("fp32", 3e-4), ("tf32", 5e-3)])
def test_layernorm_variant_train_step_gradients(dev, golden, golden_sd, precision, gtol):
    from newsrecommendationsystem_b200.train import TrainStep
    sd = _ln_state_dict(golden_sd)
    cand, clicked = golden["train/cand"][:16], golden["train/clicked"][:16]
    loss_ref, _, grads_ref, _, _ = O.train_step(sd, {}, cand, clicked, step=1)
    m = make_model(sd, dev, precision, cfg=CfgLN)
    ts = TrainStep(m, lr=1e-4, adamw=True, weight_decay=0.01)
    titles = torch.from_numpy(np.concatenate([cand, clicked], axis=1))
    loss = float(ts.step_tokens(titles, cand.shape[1]).item())
    # LayerNorm makes the logits large (loss ~ 18.8 at this init): the tensor-mode bound is relative, 2e-4 of the loss
    # (TF32 operands in the projections and in the title attention); FP32 mode stays absolute
    assert abs(loss - float(loss_ref)) < (1e-5 if precision == "fp32" else 2e-4 * max(1.0, abs(float(loss_ref))))
    grads = {k: p.grad.detach().cpu().numpy() for k, p in m.named_parameters()}
    assert set(grads) == set(grads_ref)
    # b_K's gradient is zero in exact arithmetic (a common shift of the scores of a row cancels in the softmax), so
    # both sides hold rounding noise there: the floor is 1e-6 of the largest gradient entry of the model
    floor = 1e-6 * max(float(np.abs(v).max()) for v in grads_ref.values())
    for k, g in grads.items():
        ref = grads_ref[k]
        scale = np.abs(ref).max() + 1e-12
        assert np.abs(g - ref).max() < gtol * scale + floor, (k, np.abs(g - ref).max(), scale)


def test_train_step_from_row_indices(dev, golden, golden_sd):
    """SURVEY 8 f2: index-only batches over a GPU-resident token table give the same step as token batches."""
    from newsrecommendationsystem_b200.train import TrainStep
    rng = np.random.default_rng(3)
    table = rng.integers(1, Cfg.num_words, size=(500, 20)).astype(np.int64)
    cand_rows = rng.integers(0, 500, size=(8, 5))
    hist_rows = rng.integers(0, 500, size=(8, 50))
    losses = []
    for mode in ("tokens", "rows"):
        m = make_model(golden_sd, dev, "fp32")
        ts = TrainStep(m, lr=1e-4)
        if mode == "tokens":
            titles = torch.from_numpy(np.concatenate([table[cand_rows], table[hist_rows]], axis=1))
            losses.append(float(ts.step_tokens(titles, 5).item()))
        else:
            losses.append(float(ts.step_rows(t(table, dev), torch.from_numpy(cand_rows), torch.from_numpy(hist_rows)).item()))
        w = m.user_encoder.additive_attention.linear.weight.detach().cpu().numpy()
        losses.append(w)
    assert losses[0] == losses[2] and np.array_equal(losses[1], losses[3])


def test_score_csr_f16_table(dev):
    """Tensor-mode scoring reads an fp16 copy of the news-vector table: same indexing as the fp32 kernel (bit-exact on
    fp16-representable rows), fp32 accumulation, rounding error of the copy within 1e-3 of |u||v|."""
    from newsrecommendationsystem_b200 import ops
    rng = np.random.default_rng(9)
    table = (rng.standard_normal((700, 300)) * 0.3).astype(np.float32)
    table[-1] = 0
    users = (rng.standard_normal((37, 300)) * 0.3).astype(np.float32)
    counts = rng.integers(1, 40, size=37)
    counts[5] = 301
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    rows = rng.integers(0, 700, size=offs[-1]).astype(np.int32)
    tb, ub = t(table, dev), t(users, dev)
    s32 = ops.score_csr(tb, t(rows, dev), t(offs, dev), ub).cpu().numpy()
    t16 = ops.pack_rows_f16(tb)
    assert t16.shape == (701, 320) and float(t16[:700, 300].float().min()) == 1.0 and not t16[700].any()
    s16 = ops.score_csr_f16(t16, t(rows, dev), t(offs, dev), ub).cpu().numpy()
    imp = np.repeat(np.arange(37), counts)
    bound = 1e-3 * np.linalg.norm(users[imp], axis=1) * np.linalg.norm(table[rows], axis=1)
    assert np.all(np.abs(s16 - s32) <= bound + 1e-6)
    exact = ops.score_csr(t16[:700, :300].float().contiguous(), t(rows, dev), t(offs, dev), ub).cpu().numpy()
    np.testing.assert_allclose(s16, exact, rtol=0, atol=2e-5)


def test_checkpoint_interchange_with_torch_adam(dev, golden, golden_sd, tmp_path):
    """SURVEY 8 f4: a checkpoint in the reference's layout (src/train.py:266-277) moves both ways between the fused
    optimizer and torch.optim.Adam: same parameters, same moments, and the NEXT step from the restored state agrees."""
    from newsrecommendationsystem_b200 import checkpoint as ck
    from newsrecommendationsystem_b200.train import TrainStep
    m, losses, _ = _train_once(golden, golden_sd, dev, "fp32", steps=2)
    ts = TrainStep(m, lr=1e-4)            # fresh optimizer over the same (already flat) parameters
    cand, clicked = golden["train/cand"], golden["train/clicked"]
    titles = torch.from_numpy(np.concatenate([cand, clicked], axis=1))
    ts.step_tokens(titles, cand.shape[1])
    path = str(tmp_path / "ckpt-3.pth")
    ck.save_checkpoint(path, m, ts.optimizer, step=3, early_stop_value=-0.5)
    raw = torch.load(path, weights_only=False)
    # the reference's four keys (train.py:266-277) + the position of the in-kernel dropout stream
    assert set(raw) == {"model_state_dict", "optimizer_state_dict", "step", "early_stop_value", "b200_dropout_state"}

    # -> torch.optim.Adam over plain CPU parameters with the reference's names
    params = {k: torch.nn.Parameter(v.clone()) for k, v in raw["model_state_dict"].items()}
    adam = torch.optim.Adam(list(params.values()), lr=1e-4)
    adam.load_state_dict(raw["optimizer_state_dict"])
    assert int(adam.state[list(params.values())[0]]["step"]) == 1
    grads = {k: p.grad.detach().cpu().clone() for k, p in m.named_parameters()}
    for k, p in params.items():
        p.grad = grads[k].clone()
    adam.step()                            # torch's step 2 from the restored moments
    ts.optimizer.step()                    # the fused kernel's step 2 on the same gradients
    for k, p in m.named_parameters():
        np.testing.assert_allclose(p.detach().cpu().numpy(), params[k].detach().numpy(), rtol=2.5e-7, atol=3e-8)  # 1 ulp

    # <- a checkpoint written from torch.optim.Adam restores the fused optimizer
    torch.save({"model_state_dict": {k: p.detach() for k, p in params.items()}, "optimizer_state_dict": adam.state_dict(),
                "step": 4, "early_stop_value": -0.6}, path)
    m2 = make_model(golden_sd, dev, "fp32")
    ts2 = TrainStep(m2, lr=1e-3)
    step, es = ck.load_checkpoint(path, m2, ts2.optimizer)
    assert (step, es) == (4, -0.6) and ts2.optimizer.step_count == 2 and ts2.optimizer.param_groups[0]["lr"] == 1e-4
    for k, p in m2.named_parameters():
        assert torch.equal(p.detach().cpu(), params[k].detach())
    st0 = adam.state[list(params.values())[0]]
    n0 = list(params.values())[0].numel()
    assert torch.equal(ts2.optimizer.exp_avg[:n0].cpu().view(-1), st0["exp_avg"].view(-1))


def test_training_attention_mma_vs_cuda_core(golden_sd, dev, lib):
    """Tensor-mode title attention on mma.sync TF32 tiles (attn_mma.cu) against the CUDA-core kernels it replaces: same
    stashed q|k|v rows, dropout 0.2 (same Philox stream), loss and every gradient within the tensor-mode tolerance; the
    two runs must differ somewhere (two kernels ran)."""
    from newsrecommendationsystem_b200 import ops
    rng = np.random.default_rng(21)
    titles = rng.integers(0, Cfg.num_words, size=(24, 55, 20)).astype(np.int64)
    titles[:, 40:, 10:] = 0
    res = []
    for use_mma in (0, 1):
        assert lib.nrms_set_option(b"train_attn_mma", use_mma) == 0
        m = make_model(golden_sd, dev, "tf32")
        m.train()
        loss = ops.cross_entropy_label0(m.forward_tokens(t(titles, dev), 5))
        loss.backward()
        res.append((float(loss.detach()), {k: p.grad.detach().cpu().numpy() for k, p in m.named_parameters()}))
    assert lib.nrms_set_option(b"train_attn_mma", 1) == 0
    (l0, g0), (l1, g1) = res
    assert abs(l0 - l1) < 2e-3
    differs = False
    # b_K's gradient is zero in exact arithmetic (both kernels hold rounding noise there): floor as in the LayerNorm test
    floor = 1e-6 * max(float(np.abs(v).max()) for v in g0.values())
    for k in g0:
        scale = max(float(np.abs(g0[k]).max()), 1e-12)
        err = float(np.abs(g0[k] - g1[k]).max())
        assert err <= 3e-3 * scale + floor, (k, err, scale)
        differs = differs or err > 0
    assert differs
