"""The kernels on state that outlives one call: parameters after optimizer steps, caches keyed on them, the Adam
moments, the in-place embedding-gradient sink, and the single-user ranking at its edges.

The reference trains, evaluates every so often and keeps training, then serves recommendations from the trained model.
Every check here is against an fp64 reference taken at the parameters live at that moment (the numpy oracle on the
model's `state_dict()` cast to float64), or against `np.argsort(-y, kind="stable")` for rankings.  Tolerances are those
of the rest of the suite: vectors 2e-5 (FP32 mode) / 1e-3 (tensor mode) max row-wise relative L2, metric means 5e-4.
"""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, rel_l2_rows
from oracle import nrms_oracle as O

pytestmark = pytest.mark.gpu

TOL_VEC = {"fp32": 2e-5, "tf32": 1e-3}
TOL_VEC_LN = {"fp32": 3e-5, "tf32": 2e-3}       # LayerNorm divides by the row spread (test_gpu_parity.py)
V = 401                                         # vocabulary of the golden parameters


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


class Cfg:
    num_words = V
    word_embedding_dim = 300
    num_attention_heads = 15
    query_vector_dim = 200
    dropout_probability = 0.2
    num_words_title = 20
    num_clicked_news_a_user = 50


class CfgLN(Cfg):
    use_layernorm = True


def _ln_state_dict(golden_sd, seed=11):
    rng = np.random.default_rng(seed)
    sd = dict(golden_sd)
    for prefix in (O.NEWS, O.USER):
        sd[f"{prefix}.layer_norm.weight"] = (1 + 0.1 * rng.standard_normal(300)).astype(np.float32)
        sd[f"{prefix}.layer_norm.bias"] = (0.1 * rng.standard_normal(300)).astype(np.float32)
    return sd


def _model(golden_sd, dev, precision, variant="nrms"):
    """NRMS on the golden parameters (variant "ln": the config-5 LayerNorm model), eval mode: dropout is the identity,
    gradients still flow."""
    from newsrecommendationsystem_b200 import NRMS
    sd = _ln_state_dict(golden_sd) if variant == "ln" else golden_sd
    m = NRMS(CfgLN if variant == "ln" else Cfg)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    return m.to(dev).eval().set_precision(precision)


def _live(m):
    """The parameters the model holds right now, in fp64."""
    return {k: v.detach().cpu().double().numpy() for k, v in m.state_dict().items()}


def _train_batch(rng, toks, lo=0, hi=None, B=8, K=4, pad_row=None):
    """Row indices of a training batch over the token table rows [lo, hi): candidates [B, 1+K], history [B, 50]
    left-padded with `pad_row` (an all-zero title)."""
    hi = toks.shape[0] if hi is None else hi
    cand = rng.integers(lo, hi, size=(B, 1 + K))
    hist = rng.integers(lo, hi, size=(B, 50))
    if pad_row is not None:
        hlen = rng.integers(1, 51, size=B)
        hist[np.arange(50)[None, :] < (50 - hlen)[:, None]] = pad_row
    return cand, hist


def _titles(toks, cand, hist):
    return torch.from_numpy(np.concatenate([toks[cand], toks[hist]], axis=1))


# ---- A: multi-step training, checked one step at a time ---------------------------------------------------------
STEPS, COSINE_T = 6, 8


def _two_vocabulary_table(seed):
    """Token table whose halves use disjoint words: rows [0, 300) words 1..199, rows [300, 600) words 201..399.  Rows 0
    and 300 are all-pad titles.  Steps alternate halves, so every word batch k-1 touched is untouched by batch k."""
    from newsrecommendationsystem_b200 import synthetic
    toks = synthetic.make_news(600, num_words=200, seed=seed)
    hi = toks[300:]
    hi[hi > 0] += 200
    toks[0] = 0
    toks[300] = 0
    return toks


@pytest.mark.parametrize("variant", ["nrms", "ln"])
@pytest.mark.parametrize("opt", ["adam", "adamw_cosine"])
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_training_steps_one_at_a_time_vs_oracle(dev, golden_sd, precision, opt, variant):
    """6 TrainStep steps (B = 8, K = 4), step_tokens and step_rows alternating over one optimizer, each step checked
    teacher-forced against the oracle at the parameters and moments the GPU held before it:
      - loss: 1e-5 (FP32), 2e-3 (tensor mode).  LayerNorm in tensor mode: 5e-4 of the loss -- its logits are large (loss
        11-19), test_layernorm_variant_train_step_gradients bounds the first step by 2e-4 of the loss, and two steps
        later the TF32 operands put 3.7e-4 of it between the GPU and the oracle;
      - every gradient within 2e-4 (FP32) / 3e-3 (tensor) of the tensor's largest reference entry, floor 1e-6 of the
        model's largest gradient entry (b_K).  LayerNorm: 3e-4 / 1e-2 -- the single-step test holds 5e-3 at the first
        step; at step 6 the news encoder's LayerNorm weight gradient was measured up to 5.8e-3 in tensor mode;
      - embedding row 0 and every word batch k does not touch -- all words batch k-1 used among them -- exactly zero;
      - the Adam transition p_k, g_k, m_k, v_k -> p_k+1, m_k+1, v_k+1 against O.adam_step in fp64 on the GPU's own fp32
        inputs (the hyperparameters too: the kernel takes fp32 betas, so its 1 - beta2 is 1 - fp32(0.999), 1.3e-5 away
        from 0.001): parameters within 2e-8 + 2 ulp of the result (the fp32 roundings of p itself: embedding entries
        reach 4.6), moments within 1e-6 of the magnitude of their terms.
    Largest errors on one B200 (1000 W), over the 8 cases: loss 6.9e-6 (FP32), 3.1e-5 (tensor), 5.8e-3 (tensor,
    LayerNorm, loss 15.3); gradient 0.02 (FP32) and 0.56 (tensor) of the bound; parameters 0.66 of 2e-8 + 2 ulp; moments
    1.7e-7 of their terms."""
    from newsrecommendationsystem_b200.train import TrainStep
    adamw = opt != "adam"
    wd = 0.01 if adamw else 0.0
    m = _model(golden_sd, dev, precision, variant)
    ts = TrainStep(m, lr=1e-4, adamw=adamw, weight_decay=wd, cosine_total_steps=COSINE_T if adamw else None)
    toks = _two_vocabulary_table(seed=51)
    toks_dev = torch.from_numpy(toks).to(dev)
    rng = np.random.default_rng(52)
    ln = variant == "ln"
    gtol = ({"fp32": 3e-4, "tf32": 1e-2} if ln else {"fp32": 2e-4, "tf32": 3e-3})[precision]
    names = [n for n, _ in m.named_parameters()]
    params = dict(m.named_parameters())
    err = dict(loss=0.0, grad=0.0, param=0.0, moment=0.0)
    prev_words = None
    for k in range(STEPS):
        half = k % 2
        cand, hist = _train_batch(rng, toks, lo=300 * half + 1, hi=300 * half + 300, pad_row=300 * half)
        # snapshot of what the GPU holds before step k
        P = {n: params[n].detach().cpu().numpy().copy() for n in names}
        st = ts.optimizer.state_dict()["state"]
        Mk = {n: st[i]["exp_avg"].cpu().numpy() if st else np.zeros_like(P[n]) for i, n in enumerate(names)}
        Vk = {n: st[i]["exp_avg_sq"].cpu().numpy() if st else np.zeros_like(P[n]) for i, n in enumerate(names)}
        lr = O.cosine_lr(1e-4, k, COSINE_T) if adamw else 1e-4
        # the hyperparameters as the kernel receives them: fp32 arguments of nrms_adam_step
        f32 = lambda x: float(np.float32(x))                            # noqa: E731
        hyper = dict(lr=f32(lr), beta1=f32(0.9), beta2=f32(0.999), eps=f32(1e-8), weight_decay=f32(wd),
                     decoupled=adamw)
        if k % 2 == 0:
            loss = float(ts.step_tokens(_titles(toks, cand, hist), cand.shape[1]).item())
        else:
            loss = float(ts.step_rows(toks_dev, torch.from_numpy(cand), torch.from_numpy(hist)).item())
        assert ts.optimizer.param_groups[0]["lr"] == lr
        P64 = {n: v.astype(np.float64) for n, v in P.items()}
        logits, cache = O.nrms_forward(P64, toks[cand], toks[hist])
        loss_ref, dl = O.cross_entropy_label0(logits)
        G = O.nrms_backward(dl, cache, P64)
        bound = 1e-5 if precision == "fp32" else (5e-4 * max(1.0, abs(float(loss_ref))) if ln else 2e-3)
        e = abs(loss - float(loss_ref))
        err["loss"] = max(err["loss"], e)
        assert e < bound, (k, "loss", loss, float(loss_ref))

        grads = {n: params[n].grad.detach().cpu().numpy().copy() for n in names}
        assert set(G) == set(grads)
        floor = 1e-6 * max(float(np.abs(v).max()) for v in G.values())
        for n in names:
            scale = float(np.abs(G[n]).max()) + 1e-12
            e = float(np.abs(grads[n] - G[n]).max())
            err["grad"] = max(err["grad"], e / (gtol * scale + floor))
            assert e < gtol * scale + floor, (k, n, e, scale)
        words = np.unique(np.concatenate([toks[cand].ravel(), toks[hist].ravel()]))
        untouched = np.setdiff1d(np.arange(V), words[words > 0])
        if prev_words is not None:
            assert np.intersect1d(untouched, prev_words).size > 100        # the check below covers last step's words
        prev_words = words[words > 0]
        g_emb = grads[O.EMB_KEY]
        assert not g_emb[untouched].any(), (k, "embedding rows outside batch k", np.flatnonzero(
            np.abs(g_emb[untouched]).max(axis=1)).size)

        st = ts.optimizer.state_dict()["state"]
        for i, n in enumerate(names):
            p_ref, m_ref, v_ref = O.adam_step(P64[n], grads[n].astype(np.float64), Mk[n].astype(np.float64),
                                              Vk[n].astype(np.float64), k + 1, **hyper)
            p_new = params[n].detach().cpu().numpy()
            e_p = np.abs(p_new - p_ref)
            tol_p = 2e-8 + 2 * np.spacing(np.abs(p_ref).astype(np.float32))
            err["param"] = max(err["param"], float((e_p / tol_p).max()))
            assert (e_p <= tol_p).all(), (k, n, "parameter", float(e_p.max()))
            g64 = grads[n].astype(np.float64)
            mag_m = 0.9 * np.abs(Mk[n]) + 0.1 * np.abs(g64)
            for got, ref, mag, what in ((st[i]["exp_avg"].cpu().numpy(), m_ref, mag_m, "exp_avg"),
                                        (st[i]["exp_avg_sq"].cpu().numpy(), v_ref, np.abs(v_ref), "exp_avg_sq")):
                e_m = np.abs(got - ref)
                err["moment"] = max(err["moment"], float((e_m / (mag + 1e-38)).max()))
                assert (e_m <= 1e-6 * mag + 1e-38).all(), (k, n, what, float(e_m.max()))
            assert int(float(st[i]["step"])) == k + 1
    key = f"{precision}-{opt}-{variant}"
    print(f"train[{key}]: loss {err['loss']:.2e}, gradient / bound {err['grad']:.2f}, parameter / (2e-8 + 2 ulp) "
          f"{err['param']:.2f}, moment / term magnitude {err['moment']:.2e}")


# ---- B: evaluate and no_grad forwards interleaved with training -------------------------------------------------
def _eval_data():
    from newsrecommendationsystem_b200 import synthetic
    ntok = synthetic.make_news(300, num_words=V, seed=61)
    imp = synthetic.make_impressions(64, 300, seed=62, single_class_every=16, max_cand=30)
    return ntok, imp


def _check_evaluate(m, inp, ntok, imp, precision, variant, tag):
    """evaluate_tensors against O.evaluate_pipeline at the live parameters -> largest vector error."""
    from newsrecommendationsystem_b200.evaluate import evaluate_tensors
    means, det = evaluate_tensors(m, inp, return_details=True)
    ref_means, ref_per, _, ref_table, ref_uv = O.evaluate_pipeline(
        _live(m), ntok, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"])
    tol = (TOL_VEC_LN if variant == "ln" else TOL_VEC)[precision]
    e_n = rel_l2_rows(det["table"][:300].cpu().numpy(), ref_table[:300])
    e_u = rel_l2_rows(det["user_vectors"].cpu().numpy(), ref_uv)
    assert e_n < tol, (tag, "news vectors", e_n)
    assert e_u < tol, (tag, "user vectors", e_u)
    # tensor mode: the bound of the existing evaluate tests (a near-tie can swap two ranks of a 64-impression set)
    e_m = float(np.abs(np.asarray(means) - ref_means).max())
    assert e_m < (5e-4 if precision == "fp32" else 5e-3), (tag, "metric means", means, ref_means)
    assert np.array_equal(np.isnan(det["per_impression"].cpu().numpy()), np.isnan(ref_per))
    return max(e_n, e_u)


@pytest.mark.parametrize("variant", ["nrms", "ln"])
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_evaluate_interleaved_with_training(dev, golden_sd, tmp_path, precision, variant):
    """evaluate; 1 step + no_grad validation forward; evaluate; 2 steps; evaluate; load the step-1 checkpoint;
    evaluate -- every evaluate's news table, user vectors and metric means against O.evaluate_pipeline, the validation
    logits against O.nrms_forward (2e-5 / 2e-3 of max(1, |logit|); LayerNorm 3e-5 / 4e-3), each at the parameters live
    at that moment.  The cached [W_Q;W_K;W_V] concatenation
    must follow every optimizer step.  Largest errors on one B200 (1000 W): vectors 7.1e-7 (FP32), 5.7e-4 (tensor);
    validation logits 2.4e-5 (FP32, LayerNorm, logits up to ~30) and 2.1e-2 (tensor, LayerNorm)."""
    from newsrecommendationsystem_b200 import checkpoint as ck
    from newsrecommendationsystem_b200.evaluate import EvalInputs
    from newsrecommendationsystem_b200.train import TrainStep
    m = _model(golden_sd, dev, precision, variant)
    ts = TrainStep(m, lr=1e-4)
    ntok, imp = _eval_data()
    inp = EvalInputs(ntok, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"], device=dev)
    rng = np.random.default_rng(63)
    worst = [0.0]

    def evaluate(tag):
        worst[0] = max(worst[0], _check_evaluate(m, inp, ntok, imp, precision, variant, tag))

    def step():
        cand, hist = _train_batch(rng, ntok)
        ts.step_tokens(_titles(ntok, cand, hist), cand.shape[1])

    evaluate("before training")
    step()
    vc, vh = _train_batch(rng, ntok)
    with torch.no_grad():
        logits = m.forward_tokens(_titles(ntok, vc, vh), vc.shape[1]).cpu().numpy()
    ref = O.nrms_forward(_live(m), ntok[vc], ntok[vh])[0]
    e_l = float(np.abs(logits - ref).max())
    # the logits bounds of test_gpu_parity.py (2e-5 / 2e-3), widened for LayerNorm as its vector bounds are
    bound = {("fp32", "nrms"): 2e-5, ("tf32", "nrms"): 2e-3, ("fp32", "ln"): 3e-5, ("tf32", "ln"): 4e-3}[
        (precision, variant)] * max(1.0, float(np.abs(ref).max()))
    assert e_l < bound, ("validation logits after step 1", e_l, bound)
    evaluate("after step 1")
    path = str(tmp_path / "step1.pth")
    ck.save_checkpoint(path, m, ts.optimizer, step=1, early_stop_value=0.0)
    at_step1 = _live(m)
    step()
    step()
    evaluate("after step 3")
    ck.load_checkpoint(path, m, ts.optimizer)
    assert all(np.array_equal(v, at_step1[k]) for k, v in _live(m).items())
    evaluate("after loading the step-1 checkpoint")
    print(f"evaluate-interleaved[{precision}-{variant}]: vectors {worst[0]:.2e}, validation logits {e_l:.2e}")


def _exp1_cfg():
    from newsrecommendationsystem_b200.config import Exp1Config

    class Cfg1(Exp1Config):
        num_words = 401
        num_categories = 31
        dataset_attributes = {"news": list(EXP1_ATTRS), "record": []}
    return Cfg1


EXP1_ATTRS = ["category", "subcategory", "title"]


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_exp1_no_grad_forward_after_step(dev, precision):
    """Exp1: a no_grad validation forward, then forward + CE(label 0) + backward as
    test_exp1_train_step_gradients_vs_reference drives them and one FusedAdam.step(), then the validation forward again
    -- each against O.exp1_forward at the live parameters: logits within 2e-5 (FP32) / 2e-3 (tensor) of
    max(1, |logit|).  Largest error on one B200 (1000 W): 9.7e-8 (FP32), 1.0e-4 (tensor)."""
    from compact import expand_exp1
    from exp1_weights import make_state
    from newsrecommendationsystem_b200 import Exp1, ops
    from newsrecommendationsystem_b200.optim import FusedAdam
    g1 = expand_exp1(np.load(os.path.join(GOLDEN, "exp1_golden.npz")))
    m = Exp1(_exp1_cfg())
    sd = make_state({k: tuple(v.shape) for k, v in m.state_dict().items()}, 101)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.to(dev).eval().set_precision(precision)
    opt = FusedAdam(m.parameters(), lr=1e-4)
    K1 = int(g1["train/n_cand"])
    T = g1["train/title"].shape[1]
    news = {a: g1["train/" + a] for a in EXP1_ATTRS}
    items = [{a: torch.from_numpy(np.ascontiguousarray(news[a][:, j])) for a in EXP1_ATTRS} for j in range(T)]
    errs = []

    def validate(tag):
        with torch.no_grad():
            logits = m(items[:K1], items[K1:]).cpu().numpy()
        ref = O.exp1_forward(_live(m), news, K1, EXP1_ATTRS)
        e = float(np.abs(logits - ref).max())
        errs.append(e)
        bound = (2e-5 if precision == "fp32" else 2e-3) * max(1.0, float(np.abs(ref).max()))
        assert e < bound, (tag, "Exp1 logits", e, bound)

    validate("before the step")
    loss = ops.cross_entropy_label0(m(items[:K1], items[K1:]))
    opt.zero_grad()
    loss.backward()
    opt.step()
    validate("after one step")
    print(f"exp1-validation[{precision}]: logits {max(errs):.2e}")


# ---- C: Recommender across training -----------------------------------------------------------------------------
def _topk_reference_check(mode, T, Uv, n_news, k, got_s, got_r, excl):
    """(score desc, row asc) top-k of the non-excluded rows against fp64 scores of the exact operands (the rule of
    tests/test_topk.py) -> largest score error relative to |row| |user|."""
    S = Uv @ T[:n_news].T
    worst = 0.0
    tn = np.linalg.norm(T[:n_news], axis=1)
    for u in range(S.shape[0]):
        rows = np.setdiff1d(np.arange(n_news), excl[u])
        s_all = S[u, rows]
        o = np.lexsort((rows, -s_all))
        rr, rs = rows[o][:k], s_all[o][:k]
        nv = len(rr)
        r, s = got_r[u], got_s[u]
        assert (r[nv:] == -1).all() and np.isneginf(s[nv:]).all()
        r, s = r[:nv], s[:nv]
        assert (r >= 0).all() and (r < n_news).all() and not np.isin(r, excl[u]).any()
        scale = tn[r] * np.linalg.norm(Uv[u]) + 1e-30
        e = np.abs(s - S[u, r])
        worst = max(worst, float((e / scale).max(initial=0.0)))
        assert all(s[j] > s[j + 1] or (s[j] == s[j + 1] and r[j] < r[j + 1]) for j in range(nv - 1))
        if mode == "fp32":
            assert (e <= 1e-5 * scale).all()
            sc = max(float(np.abs(rs).max(initial=0.0)), 1e-30)
            full = np.concatenate([[np.inf], rs, [-np.inf]])
            gap_ok = (full[1:-1] - full[2:] > 1e-6 * sc) & (full[:-2] - full[1:-1] > 1e-6 * sc)
            assert np.array_equal(r[gap_ok], rr[gap_ok])
        else:
            assert (e <= 1e-3 * scale).all()
            t2 = 2e-3 * float(tn.max(initial=0.0)) * np.linalg.norm(Uv[u])
            assert (S[u, r] >= rs[-1] - t2).all()
    return worst


@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_recommender_follows_training(dev, golden_sd, precision):
    """A Recommender built before training serves the parameters live at each call: recommend_rows (FP32 latency path
    in both modes) and top_k_rows (the model's mode), before and after one optimizer step.  User vectors against
    O.recommend_user (2e-5 FP32 / 1e-3 tensor mode), scores and order against fp64 dot products, the top-k against
    the (score desc, row asc) reference.  Largest errors on one B200 (1000 W): user vector 1.5e-7 (recommend_rows),
    3.2e-4 (top_k_rows, tensor mode); scores 1.7e-8 and top-k scores 7.2e-8 of |row| |user|."""
    from newsrecommendationsystem_b200 import synthetic
    from newsrecommendationsystem_b200.recommend import Recommender
    from newsrecommendationsystem_b200.train import TrainStep
    rng = np.random.default_rng(71)
    n = 300
    table = np.concatenate([rng.standard_normal((n, 300)) * 0.3, np.zeros((1, 300))]).astype(np.float32)
    m = _model(golden_sd, dev, precision)
    ts = TrainStep(m, lr=1e-4)
    rec = Recommender(m, [f"N{i}" for i in range(n)], torch.from_numpy(table).to(dev))
    hist = [n] * 10 + rng.integers(0, n, 40).tolist()
    cand = rng.integers(0, n, 200).tolist()
    toks = synthetic.make_news(400, num_words=V, seed=72)
    err = dict(user=0.0, score=0.0, topk_user=0.0, topk=0.0)
    for call in ("before training", "after one step"):
        if call == "after one step":
            c, h = _train_batch(rng, toks)
            ts.step_tokens(_titles(toks, c, h), c.shape[1])
        P = _live(m)
        order, scores, user = (x.cpu().numpy() for x in rec.recommend_rows(hist, cand))
        uv_ref, y_ref, order_ref = O.recommend_user(P, table, hist, cand)
        e = rel_l2_rows(user[None], uv_ref[None])
        err["user"] = max(err["user"], e)
        assert e < 2e-5, (call, "recommend_rows user vector", e)
        s_own = table[cand].astype(np.float64) @ user.astype(np.float64)
        rows_norm = np.linalg.norm(table[cand], axis=1) * np.linalg.norm(user)
        e = float((np.abs(scores - s_own) / rows_norm).max())
        err["score"] = max(err["score"], e)
        assert e < 1e-5, (call, "recommend_rows scores", e)
        s_ref = y_ref * 2 - 1
        assert float(np.abs(scores - s_ref).max()) < 2e-5 * max(1.0, float(np.abs(s_ref).max())), call
        assert np.array_equal(order, np.argsort(-scores.astype(np.float64), kind="stable")), call
        gaps = np.abs(np.diff(y_ref[order_ref]))                # ranks the fp32 rounding cannot swap must agree
        sep = np.concatenate([[True], gaps > 1e-4]) & np.concatenate([gaps > 1e-4, [True]])
        assert np.array_equal(order[sep], order_ref[sep]), call

        rows, tk_s, tk_u = (x.cpu() for x in rec.top_k_rows(np.array([hist], dtype=np.int32), 40))
        e = rel_l2_rows(tk_u.numpy(), uv_ref[None])
        err["topk_user"] = max(err["topk_user"], e)
        assert e < TOL_VEC[precision], (call, "top_k_rows user vector", e)
        if precision == "tf32":
            T, Uv = rec._table16[:, :300].double().cpu().numpy(), tk_u.half().double().numpy()
        else:
            T, Uv = table.astype(np.float64), tk_u.double().numpy()
        e = _topk_reference_check(precision, T, Uv, n, 40, tk_s.numpy(), rows.numpy(), np.array([hist]))
        err["topk"] = max(err["topk"], e)
    print(f"recommender-across-training[{precision}]: user {err['user']:.2e}, score / (|row||user|) "
          f"{err['score']:.2e}, top-k user {err['topk_user']:.2e}, top-k score {err['topk']:.2e}")


# ---- D: back-to-back recommend_rows while the stream is busy ----------------------------------------------------
def test_back_to_back_recommend_rows_behind_a_busy_stream(dev, golden_sd):
    """Two recommend_rows calls queued behind ~20 ms of device work: each call's indices reach the device intact (the
    pinned staging buffer is not rewritten while its copy is pending).  Both results against O.recommend_user, user
    vectors within 2e-5.  Largest error on one B200 (1000 W): 1.6e-7."""
    from newsrecommendationsystem_b200.recommend import Recommender
    rng = np.random.default_rng(81)
    n = 300
    table = np.concatenate([rng.standard_normal((n, 300)) * 0.3, np.zeros((1, 300))]).astype(np.float32)
    m = _model(golden_sd, dev, "fp32")
    rec = Recommender(m, [f"N{i}" for i in range(n)], torch.from_numpy(table).to(dev))
    calls = [([n] * 5 + rng.integers(0, n, 45).tolist(), rng.integers(0, n, 120).tolist()),
             (rng.integers(0, n, 50).tolist(), rng.integers(0, n, 37).tolist())]
    rec.recommend_rows(*calls[0])                  # builds the packed weights and staging buffers
    torch.cuda.synchronize()
    torch.cuda._sleep(40_000_000)                  # ~20 ms at B200 clocks: bounded
    got = [tuple(x.clone() for x in rec.recommend_rows(h, c)) for h, c in calls]
    torch.cuda.synchronize()
    P = _live(m)
    worst = 0.0
    for (h, c), (order, scores, user) in zip(calls, got):
        uv_ref, y_ref, _ = O.recommend_user(P, table, h, c)
        e = rel_l2_rows(user.cpu().numpy()[None], uv_ref[None])
        worst = max(worst, e)
        assert e < 2e-5, ("user vector", len(c), e)
        assert scores.numel() == len(c)
        s = scores.cpu().numpy()
        assert float(np.abs(s - (y_ref * 2 - 1)).max()) < 2e-5 * max(1.0, float(np.abs(y_ref * 2 - 1).max()))
        assert np.array_equal(order.cpu().numpy(), np.argsort(-s.astype(np.float64), kind="stable"))
    print(f"back-to-back recommend_rows: user vector {worst:.2e}")


# ---- E: edges of the single-user ranking ------------------------------------------------------------------------
RANK_C = [0, 1, 2, 3, 5, 7, 63, 64, 65, 4093, 4095, 4096, 4097]


def _edge_lists(C, rng, n_fin, special):
    """Candidate lists of length C: repeated rows (exact ties spread over the CTAs, the first and last position tied),
    and the same list with one row whose score is +inf, -inf or NaN."""
    if C == 0:
        return {"empty": np.zeros(0, np.int64)}
    base = rng.integers(0, max(1, min(n_fin, C // 3)), size=C)
    base[-1] = base[0]
    out = {"ties": base}
    for name, row in special.items():
        c = base.copy()
        c[rng.integers(0, C)] = row
        out[name] = c
    return out


def test_single_user_ranking_edges(dev, golden_sd):
    """ops.recommend_user(rank=True) (C <= 4,096) and Recommender.recommend_rows (both sides of the 4,096 limit) on
    C in {0, 1, 2, 3, 5, 7, 63, 64, 65, 4093, 4095, 4096, 4097}: every C mod 4 and mod 8, exact ties, +inf, -inf and
    NaN scores.  `order` is a permutation and equals np.argsort(-y, kind="stable") of the kernel's own scores in fp64
    (NaN last); finite scores within 2e-5 of the largest |score| of the fp64 dot product with the kernel's user vector.
    Largest finite-score error on one B200 (1000 W): 1.4e-7 of the largest |score|."""
    from newsrecommendationsystem_b200 import ops
    from newsrecommendationsystem_b200.recommend import Recommender
    rng = np.random.default_rng(91)
    n_fin = 5000
    fin = (rng.standard_normal((n_fin, 300)) * 0.3).astype(np.float32)
    hist = rng.integers(0, n_fin, 50)
    m = _model(golden_sd, dev, "fp32")
    ue = m.user_encoder
    a = ue.additive_attention
    with torch.no_grad():
        w = (*ue.multihead_self_attention.packed(), a.linear.weight, a.linear.bias, a.attention_query_vector)
    hist_t = torch.from_numpy(hist.astype(np.int32)).to(dev)
    probe = torch.from_numpy(np.concatenate([fin, np.zeros((1, 300), np.float32)])).to(dev)
    u0 = ops.recommend_user(probe, hist_t, hist_t[:1], *w, rank=False)[0].cpu().numpy()
    j_pos, j_neg = int(np.argmax(u0)), int(np.argmin(u0))
    assert u0[j_pos] > 0 > u0[j_neg]
    special = np.zeros((3, 300), np.float32)
    special[0, j_pos] = np.inf                 # score +inf
    special[1, j_neg] = np.inf                 # score -inf
    special[2, 7] = np.nan                     # score NaN
    table = np.concatenate([fin, special, np.zeros((1, 300), np.float32)])
    table_t = torch.from_numpy(table).to(dev)
    rows_special = {"+inf": n_fin, "-inf": n_fin + 1, "nan": n_fin + 2}
    rec = Recommender(m, [f"N{i}" for i in range(table.shape[0] - 1)], table_t)
    worst = 0.0
    failures = []
    for C in RANK_C:
        for name, cand in _edge_lists(C, rng, n_fin, rows_special).items():
            paths = {"recommend_rows": lambda: rec.recommend_rows(hist.tolist(), cand.tolist())}
            if C <= 4096:
                paths["ops.recommend_user"] = lambda: ops.recommend_user(
                    table_t, hist_t, torch.from_numpy(cand.astype(np.int32)).to(dev), *w, rank=True)
            for path, run in paths.items():
                res = run()
                order, scores, user = res if path == "recommend_rows" else (res[2], res[1], res[0])
                order, scores, user = order.cpu().numpy(), scores.cpu().numpy(), user.cpu().numpy()
                assert rel_l2_rows(user[None], u0[None].astype(np.float64)) < 1e-6     # same history as the probe
                s64 = scores.astype(np.float64)
                ref = table[cand].astype(np.float64) @ user.astype(np.float64)
                with np.errstate(invalid="ignore"):
                    assert np.array_equal(np.isnan(s64), np.isnan(ref)) and np.array_equal(s64[np.isinf(ref)],
                                                                                          ref[np.isinf(ref)])
                fm = np.isfinite(ref)
                if fm.any():
                    e = float(np.abs(s64[fm] - ref[fm]).max())
                    worst = max(worst, e / float(np.abs(ref[fm]).max()))
                    assert e <= 2e-5 * float(np.abs(ref[fm]).max()), (path, C, name, e)
                want = np.argsort(-s64, kind="stable")
                perm = sorted(order.tolist()) == list(range(C))
                if not (perm and np.array_equal(order, want)):
                    bad = np.flatnonzero(order != want) if order.shape == want.shape else []
                    failures.append(f"{path} C={C} {name}: permutation={perm}, first mismatch at "
                                    f"{bad[0] if len(bad) else '-'} (got {order[:8].tolist()}, want {want[:8].tolist()})")
    print(f"ranking-edges: finite score error / max |score| {worst:.2e}; {len(failures)} failing lists")
    assert not failures, "\n".join(failures)


# ---- F: the embedding-gradient sink belongs to the optimizer's parameters ----------------------------------------
def test_embedding_gradient_sink_is_per_optimizer(dev, golden_sd):
    """After model A gets a FusedAdam, a fresh FP32 model B whose embedding already holds a zero .grad (as after
    torch.optim.Adam.zero_grad(set_to_none=False)) gets its embedding gradient from torch.autograd.grad -- equal to the
    oracle's within 2e-4 of its largest entry -- and its .grad stays zero.  A's step still accumulates its embedding
    gradient in place, into the optimizer's flat buffer.  Largest error on one B200 (1000 W): 1.5e-6 of the scale."""
    from newsrecommendationsystem_b200 import ops
    from newsrecommendationsystem_b200.train import TrainStep
    from newsrecommendationsystem_b200 import synthetic
    toks = synthetic.make_news(400, num_words=V, seed=101)
    rng = np.random.default_rng(102)
    cand, hist = _train_batch(rng, toks)
    a = _model(golden_sd, dev, "fp32")
    ts = TrainStep(a, lr=1e-4)
    b = _model(golden_sd, dev, "fp32")
    emb_b = b.news_encoder.word_embedding.weight
    wv_b = b.news_encoder.multihead_self_attention.W_V.weight
    emb_b.grad = torch.zeros_like(emb_b)
    loss_b = ops.cross_entropy_label0(b.forward_tokens(_titles(toks, cand, hist), cand.shape[1]))
    g_emb, g_wv = torch.autograd.grad(loss_b, [emb_b, wv_b], allow_unused=True)
    P = _live(b)
    logits, cache = O.nrms_forward(P, toks[cand], toks[hist])
    G = O.nrms_backward(O.cross_entropy_label0(logits)[1], cache, P)
    assert g_emb is not None, "torch.autograd.grad returned no embedding gradient"
    assert not emb_b.grad.any(), "the embedding gradient was scattered into model B's .grad"
    worst = 0.0
    for got, name in ((g_emb, O.EMB_KEY), (g_wv, "news_encoder.multihead_self_attention.W_V.weight")):
        ref = G[name]
        e = float(np.abs(got.cpu().numpy() - ref).max())
        worst = max(worst, e / float(np.abs(ref).max()))
        assert e <= 2e-4 * float(np.abs(ref).max()), (name, e)
    # A: the step's embedding gradient lands in the optimizer's flat buffer; autograd is handed none for it
    emb_a = a.news_encoder.word_embedding.weight
    ts.step_tokens(_titles(toks, cand, hist), cand.shape[1])
    opt = ts.optimizer
    i = [p is emb_a for p in opt._params].index(True)
    assert emb_a.grad.data_ptr() == opt.flat_grad.data_ptr() + 4 * opt._offsets[i]
    e = float(np.abs(emb_a.grad.cpu().numpy() - G[O.EMB_KEY]).max())
    assert e <= 2e-4 * float(np.abs(G[O.EMB_KEY]).max()), ("A's embedding gradient", e)
    opt.zero_grad()
    loss_a = ops.cross_entropy_label0(a.forward_tokens(_titles(toks, cand, hist), cand.shape[1]))
    assert torch.autograd.grad(loss_a, [emb_a], allow_unused=True)[0] is None
    assert emb_a.grad.any()
    print(f"embedding-gradient sink: model B gradient / scale {worst:.2e}")
