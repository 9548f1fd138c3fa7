"""Generate golden fixtures by running the LIVE reference modules (torch CPU fp32).

Run in the build container only (needs /root/reference):
    python tests/golden/make_golden.py
Writes tests/golden/nrms_golden.npz.  Nothing at test/bench/smoke run time reads
/root/reference; the fixtures travel with the repo.

What is pinned (reference call sites):
  * NewsEncoder / UserEncoder / DotProductClickPredictor forward via
    NRMS.get_news_vector / get_user_vector / get_prediction (src/model/NRMS/__init__.py:50-84)
  * NRMS.forward + CrossEntropyLoss(label 0) + autograd + torch.optim.Adam(lr=1e-4), two
    steps (src/train.py:126-128,202-206,227-233), plus an AdamW(lr=1e-4, wd=0.01) step
  * calculate_single_user_metric (src/evaluate.py:160-168) on crafted (labels, scores)
    pairs incl. ties and single-class impressions
  * a tensor-level walk of evaluate() (src/evaluate.py:185-272) that calls the reference's
    get_* methods and metric function exactly as evaluate() does (UserDataset itself raises
    under pandas 3, SURVEY.md section 0).
"""
import os
import sys

import numpy as np
import torch

REF = "/root/reference/src"
sys.path.insert(0, REF)
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))

from config import NRMSConfig  # noqa: E402  (reference)
from model.NRMS import NRMS  # noqa: E402  (reference)
import evaluate as ref_eval  # noqa: E402  (reference)

from newsrecommendationsystem_b200 import synthetic  # noqa: E402
from compact import compact_nrms  # noqa: E402


class Cfg(NRMSConfig):
    num_words = 1 + 400          # small vocabulary keeps the fixture small
    dropout_probability = 0.2    # model is used in .eval() mode => identity


ROWS = 48   # 2-D tensors are pinned on their first ROWS rows (compact.compact_nrms keeps a sample of those)


def clip(a):
    a = np.asarray(a)
    return a[:ROWS].copy() if a.ndim == 2 else a.copy()


def main():
    torch.manual_seed(0)
    torch.set_num_threads(4)
    model = NRMS(Cfg)
    model.eval()
    out = {}
    sd0 = {k: v.detach().clone() for k, v in model.state_dict().items()}
    for k, v in sd0.items():
        out["sd/" + k] = v.numpy()

    rng = np.random.default_rng(7)
    # ---- forward goldens ------------------------------------------------------------
    toks = synthetic.make_news(37, num_words=Cfg.num_words, seed=11)
    toks[5] = 0  # an all-pad title (training-time history padding, dataset.py:47)
    with torch.no_grad():
        nv = model.get_news_vector({"title": torch.from_numpy(toks)})
        gathered = model.news_encoder.word_embedding(torch.from_numpy(toks))
    out["fwd/tokens"] = toks
    out["fwd/gathered"] = gathered.numpy()
    out["fwd/news_vectors"] = nv.numpy()
    ux = rng.standard_normal((9, 50, 300)).astype(np.float32) * 0.5
    ux[2, :17] = 0  # zero PADDED_NEWS rows (evaluate.py:203-204)
    ux[3] = 0       # empty history
    with torch.no_grad():
        uv = model.get_user_vector(torch.from_numpy(ux))
    out["fwd/user_input"] = ux
    out["fwd/user_vectors"] = uv.numpy()
    with torch.no_grad():
        sc = model.get_prediction(nv[:23], uv[0])
        sc_b = model.click_predictor(nv[:36].reshape(9, 4, 300), uv)
    out["fwd/scores_single"] = sc.numpy()
    out["fwd/scores_batched"] = sc_b.numpy()

    # ---- training goldens -----------------------------------------------------------
    news_tok = synthetic.make_news(64, num_words=Cfg.num_words, seed=12)
    cand, clicked = synthetic.make_train_batch(6, news_tok, k_neg=4, seed=13)
    out["train/cand"] = cand
    out["train/clicked"] = clicked

    def ref_step(m, opt):
        cn = [{"title": torch.from_numpy(cand[:, i])} for i in range(cand.shape[1])]
        cl = [{"title": torch.from_numpy(clicked[:, i])} for i in range(clicked.shape[1])]
        y_pred = m(cn, cl)
        y = torch.zeros(len(y_pred)).long()
        loss = torch.nn.CrossEntropyLoss()(y_pred, y)
        opt.zero_grad()
        loss.backward()
        grads = {k: p.grad.detach().clone().numpy() for k, p in m.named_parameters()}
        opt.step()
        return y_pred.detach().numpy(), float(loss.item()), grads

    opt = torch.optim.Adam(model.parameters(), lr=Cfg.learning_rate)
    logits, loss, grads = ref_step(model, opt)
    out["train/logits"] = logits
    out["train/loss"] = np.float32(loss)
    for k, g in grads.items():
        out["train/grad/" + k] = g if "embedding" in k else clip(g)
    for k, v in model.state_dict().items():
        out["train/adam1/" + k] = clip(v.detach().numpy())
    logits2, loss2, _ = ref_step(model, opt)
    out["train/loss2"] = np.float32(loss2)
    for k, v in model.state_dict().items():
        out["train/adam2/" + k] = clip(v.detach().numpy())

    # AdamW variant (config 5; torch defaults wd=0.01)
    model.load_state_dict(sd0)
    optw = torch.optim.AdamW(model.parameters(), lr=Cfg.learning_rate, weight_decay=0.01)
    ref_step(model, optw)
    for k, v in model.state_dict().items():
        out["train/adamw1/" + k] = clip(v.detach().numpy())
    model.load_state_dict(sd0)

    # ---- metric goldens -------------------------------------------------------------
    pairs = []
    mr = np.random.default_rng(21)
    for n in (2, 3, 5, 7, 12, 37, 120, 300):
        for _ in range(4):
            y = (mr.random(n) < 0.3).astype(np.int64)
            y[0], y[1] = 1, 0
            s = mr.standard_normal(n).astype(np.float32)
            pairs.append((y, s))
    # ties between a positive and a negative, repeated candidates with equal labels
    y = np.array([1, 0, 0, 1, 0, 0]); s = np.array([0.5, 0.5, 0.1, 0.9, 0.9, -1.0], np.float32)
    pairs.append((y, s))
    y = np.array([1, 1, 0, 0, 0]); s = np.array([0.3, 0.3, 0.2, 0.2, 0.2], np.float32)
    pairs.append((y, s))
    y = np.zeros(6, np.int64); s = mr.standard_normal(6).astype(np.float32)   # single class
    pairs.append((y, s))
    y = np.ones(4, np.int64); s = mr.standard_normal(4).astype(np.float32)
    pairs.append((y, s))
    offs = np.zeros(len(pairs) + 1, np.int64)
    np.cumsum([len(p[0]) for p in pairs], out=offs[1:])
    out["metric/offsets"] = offs
    out["metric/labels"] = np.concatenate([p[0] for p in pairs]).astype(np.int8)
    out["metric/scores"] = np.concatenate([p[1] for p in pairs])
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        res = [ref_eval.calculate_single_user_metric((p[0].tolist(), p[1].tolist())) for p in pairs]
    out["metric/results"] = np.array(res, dtype=np.float64)

    # ---- evaluate() walk ------------------------------------------------------------
    Nn, I = 90, 40
    ntok = synthetic.make_news(Nn, num_words=Cfg.num_words, seed=31)
    imp = synthetic.make_impressions(I, Nn, seed=32, single_class_every=7, max_cand=40)
    news_ids = [f"N{i}" for i in range(Nn)]
    news_ids[17] = news_ids[3]   # duplicate id: first occurrence wins (evaluate.py:197-201)
    with torch.no_grad():
        news2vector = {}
        for s0 in range(0, Nn, 32):   # batches, like the DataLoader at :186-191
            ids = news_ids[s0:s0 + 32]
            if any(i not in news2vector for i in ids):
                v = model.get_news_vector({"title": torch.from_numpy(ntok[s0:s0 + 32])})
                for i, vec in zip(ids, v):
                    if i not in news2vector:
                        news2vector[i] = vec
        news2vector["PADDED_NEWS"] = torch.zeros(list(news2vector.values())[0].size())
        hist_ids = [["PADDED_NEWS" if r < 0 else news_ids[r] for r in row] for row in imp["hist_rows"]]
        user2vector = {}
        for s0 in range(0, I, 16):
            mb = hist_ids[s0:s0 + 16]
            # evaluate.py:220-224 builds [50,B,300] then transposes; equivalent direct stack
            cv = torch.stack([torch.stack([news2vector[x] for x in nl], dim=0) for nl in mb], dim=0)
            uvv = model.get_user_vector(cv)
            for j, vec in enumerate(uvv):
                user2vector[s0 + j] = vec
        tasks, all_scores = [], []
        max_count = 36   # exercises the off-by-one at evaluate.py:247-249
        count = 0
        for i in range(I):
            count += 1
            if count == max_count:
                break
            a, b = imp["cand_offsets"][i], imp["cand_offsets"][i + 1]
            cvec = torch.stack([news2vector[news_ids[r]] for r in imp["cand_rows"][a:b]], dim=0)
            prob = model.get_prediction(cvec, user2vector[i])
            y_pred = prob.tolist()
            y_true = [int(x) for x in imp["labels"][a:b]]
            tasks.append((y_true, y_pred))
            all_scores.append(prob.numpy())
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        results = [ref_eval.calculate_single_user_metric(t) for t in tasks]
        aucs, mrrs, n5, n10 = np.array(results).T
        means = np.array([np.nanmean(aucs), np.nanmean(mrrs), np.nanmean(n5), np.nanmean(n10)])
    out["eval/news_tokens"] = ntok
    ids_int = np.arange(Nn, dtype=np.int64)
    ids_int[17] = 3
    out["eval/news_ids"] = ids_int
    for k, v in imp.items():
        out["eval/" + k] = v
    out["eval/max_count"] = np.int64(max_count)
    out["eval/scores"] = np.concatenate(all_scores)
    out["eval/per_impression"] = np.array(results, dtype=np.float64)
    out["eval/means"] = means

    path = os.path.join(HERE, "nrms_golden.npz")
    np.savez_compressed(path, **compact_nrms(out))
    print("wrote", path, os.path.getsize(path) // 1024, "KiB;", len(out), "arrays")
    print("loss", loss, loss2, "means", means)


if __name__ == "__main__":
    main()
