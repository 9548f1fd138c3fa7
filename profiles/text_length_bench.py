"""NRMS and Exp1 at title / abstract lengths other than the compiled 20 and 50 on one GPU (writes
profiles/text_length_bench_b200.json by default).

For L = num_words_title in {10, 20, 30, 50, 64}, in tensor (TF32) and FP32 mode:
  - evaluate_tensors over MIND-small-shaped synthetic data (65,238 news of L tokens from synthetic.make_news(...,
    title_len=L), 73,152 impressions of 50 clicks): the news stage and the whole pass, inputs resident on the device;
  - the NRMS training step (TrainStep.step_tokens, B = 128, 1 + 4 candidates, 50 clicked titles, dropout 0.2, Adam).
And the Exp1 training step (TrainStep.step_rows over a device-resident table, B = 128, 1 + 4 candidates, 50 clicks,
dropout 0.2; 'category', 'subcategory', 'title' of 20 tokens, 'abstract') with abstracts of 50 and 64 tokens.
L = 20 and 50 run the compiled paths; other lengths run gather -> GEMM -> run-time-length attention (dropout #2 inside)
-> GEMM -> additive, and inference takes the chunked path.  Times are CUDA events; the median over --windows passes.
"""
import argparse
import json
import os
import statistics
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from exp1_train_bench import gpu_info, make_cfg, timed, ATTRS_A, NUM_CATEGORIES  # noqa: E402
from newsrecommendationsystem_b200 import NRMS, Exp1, synthetic  # noqa: E402
from newsrecommendationsystem_b200.config import NRMSConfig  # noqa: E402
from newsrecommendationsystem_b200.evaluate import EvalHost, EvalInputs, evaluate_tensors  # noqa: E402
from newsrecommendationsystem_b200.train import TrainStep  # noqa: E402

N_NEWS, N_IMP, NUM_WORDS = 65238, 73152, 70976          # bench.py's MIND-small shape
LENGTHS = [10, 20, 30, 50, 64]
ABSTRACT_LENGTHS = [50, 64]


def model_for(L, sd, dev, precision, train=False):
    class Cfg(NRMSConfig):
        num_words = NUM_WORDS
        num_words_title = L
    m = NRMS(Cfg)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.to(dev).train(train).set_precision(precision)
    return m


def time_evaluate(m, inputs, windows):
    """(news stage ms, whole pass ms, metrics) medians over `windows` passes after one warm-up pass."""
    news, whole = [], []
    means = None
    for i in range(windows + 1):
        marks = {}

        def mark(name):
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            marks[name] = ev
        means = evaluate_tensors(m, inputs, mark=mark)
        torch.cuda.synchronize()
        if i:
            news.append(marks["start"].elapsed_time(marks["news"]))
            whole.append(marks["start"].elapsed_time(marks["metrics"]))
    return statistics.median(news), statistics.median(whole), means, news, whole


def time_train(m, titles, steps, windows):
    ts = TrainStep(m, lr=1e-4)
    for _ in range(3):
        ts.step_tokens(titles, 5)
    out = []
    for _ in range(windows):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            loss = ts.step_tokens(titles, 5)
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / steps)
    return statistics.median(out), float(loss), out


def exp1_step(La, dev, precision, windows):
    """Exp1 training step with abstracts of La tokens: (median ms, loss, windows)."""
    rng = np.random.default_rng(0)
    title = synthetic.make_news(N_NEWS + 1, num_words=NUM_WORDS, title_len=20, seed=1)
    abstract = synthetic.make_news(N_NEWS + 1, num_words=NUM_WORDS, title_len=La, seed=2)
    t = {"title": title, "abstract": abstract, "category": rng.integers(1, NUM_CATEGORIES, size=N_NEWS + 1),
         "subcategory": rng.integers(1, NUM_CATEGORIES, size=N_NEWS + 1)}
    for v in t.values():
        v[N_NEWS] = 0
    t = {k: torch.from_numpy(v.astype(np.int64)).to(dev) for k, v in t.items()}

    class Cfg(make_cfg(ATTRS_A)):
        num_words_abstract = La
    torch.manual_seed(0)
    m = Exp1(Cfg).to(dev).train().set_precision(precision)
    ts = TrainStep(m)
    cand = torch.from_numpy(rng.integers(0, N_NEWS, size=(128, 5)))
    hist = torch.from_numpy(rng.integers(0, N_NEWS + 1, size=(128, 50)))
    for _ in range(3):
        ts.step_rows(t, cand, hist)
    out = [timed(lambda: ts.step_rows(t, cand, hist), 1.0) for _ in range(windows)]
    loss = float(ts.step_rows(t, cand, hist))
    return statistics.median(out), loss, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "text_length_bench_b200.json"))
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--lengths", default=",".join(map(str, LENGTHS)))
    ap.add_argument("--abstract-lengths", default=",".join(map(str, ABSTRACT_LENGTHS)))
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    sd = synthetic.init_state_dict(num_words=NUM_WORDS, seed=0)
    imp = synthetic.make_impressions(N_IMP, N_NEWS, history=50, seed=1234)
    res = {"gpu_info": gpu_info(), "n_news": N_NEWS, "n_impressions": N_IMP, "windows": args.windows,
           "train_batch": 128, "train_k_neg": 4, "train_clicked": 50, "dropout": 0.2, "cases": [], "exp1": []}
    for L in [int(x) for x in args.lengths.split(",")]:
        news = synthetic.make_news(N_NEWS, num_words=NUM_WORDS, title_len=L, seed=1234)
        inputs = EvalInputs.from_host(EvalHost(news, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"]),
                                      dev)
        cand, clicked = synthetic.make_train_batch(128, news, k_neg=4, history=50, seed=1234)
        titles = torch.from_numpy(np.concatenate([cand, clicked], axis=1)).pin_memory()
        for precision in ("tf32", "fp32"):
            m = model_for(L, sd, dev, precision)
            news_ms, eval_ms, means, nw, ew = time_evaluate(m, inputs, args.windows)
            train_ms, loss, tw = time_train(model_for(L, sd, dev, precision, train=True), titles, args.train_steps,
                                            args.windows)
            case = {"L": L, "precision": precision, "evaluate_news_ms": news_ms, "evaluate_ms": eval_ms,
                    "news_per_s": N_NEWS / (news_ms / 1e3), "impressions_per_s": N_IMP / (eval_ms / 1e3),
                    "metrics": list(means), "train_step_ms": train_ms, "train_loss": loss,
                    "evaluate_news_ms_windows": nw, "evaluate_ms_windows": ew, "train_step_ms_windows": tw}
            print(json.dumps({k: v for k, v in case.items() if not k.endswith("windows")}), flush=True)
            res["cases"].append(case)
            del m
        del inputs
        torch.cuda.empty_cache()
    for La in [int(x) for x in args.abstract_lengths.split(",")]:
        for precision in ("tf32", "fp32"):
            ms, loss, w = exp1_step(La, dev, precision, args.windows)
            case = {"abstract_L": La, "title_L": 20, "precision": precision, "exp1_train_step_ms": ms, "train_loss": loss,
                    "exp1_train_step_ms_windows": w}
            print(json.dumps({k: v for k, v in case.items() if not k.endswith("windows")}), flush=True)
            res["exp1"].append(case)
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
