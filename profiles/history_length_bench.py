"""NRMS at click-history lengths other than the compiled 20 and 50 on one GPU (writes
profiles/history_length_bench_b200.json by default).

For S = num_clicked_news_a_user in {10, 20, 30, 50, 64}, in tensor (TF32) and FP32 mode:
  - evaluate_tensors over MIND-small-shaped synthetic data (65,238 news, 73,152 impressions, histories of S clicks from
    synthetic.make_impressions(..., history=S)): the users stage and the whole pass, inputs resident on the device;
  - the NRMS training step (TrainStep.step_tokens, B = 128, 1 + 4 candidates, S clicked titles, dropout 0.2, Adam);
  - Recommender.recommend_rows latency for one user and 300 candidates (host clock around the call and a device
    synchronise, so it includes the launches and the index copy).
S = 20 and 50 run the fused paths; the other lengths run gather -> GEMM -> run-time-length attention -> GEMM -> additive.
Evaluate and training times are CUDA events; the median over --windows passes is reported.
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from exp1_train_bench import gpu_info  # noqa: E402
from newsrecommendationsystem_b200 import NRMS, synthetic  # noqa: E402
from newsrecommendationsystem_b200.config import NRMSConfig  # noqa: E402
from newsrecommendationsystem_b200.evaluate import EvalHost, EvalInputs, encode_news_table, evaluate_tensors  # noqa: E402
from newsrecommendationsystem_b200.recommend import Recommender  # noqa: E402
from newsrecommendationsystem_b200.train import TrainStep  # noqa: E402

N_NEWS, N_IMP, NUM_WORDS = 65238, 73152, 70976          # bench.py's MIND-small shape
LENGTHS = [10, 20, 30, 50, 64]


def model_for(S, sd, dev, precision, train=False):
    class Cfg(NRMSConfig):
        num_words = NUM_WORDS
        num_clicked_news_a_user = S
    m = NRMS(Cfg)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    m.to(dev).train(train).set_precision(precision)
    return m


def time_evaluate(m, inputs, windows):
    """(users stage ms, whole pass ms, metrics) medians over `windows` passes after one warm-up pass."""
    users, whole = [], []
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
            users.append(marks["news"].elapsed_time(marks["users"]))
            whole.append(marks["start"].elapsed_time(marks["metrics"]))
    return statistics.median(users), statistics.median(whole), means, users, whole


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


def time_recommend(rec, hist, cand, calls):
    for _ in range(10):
        rec.recommend_rows(hist, cand)
    torch.cuda.synchronize()
    t = []
    for _ in range(calls):
        t0 = time.perf_counter()
        rec.recommend_rows(hist, cand)
        torch.cuda.synchronize()
        t.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(t), float(np.percentile(t, 90))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "history_length_bench_b200.json"))
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--recommend-calls", type=int, default=200)
    ap.add_argument("--lengths", default=",".join(map(str, LENGTHS)))
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    sd = synthetic.init_state_dict(num_words=NUM_WORDS, seed=0)
    news = synthetic.make_news(N_NEWS, num_words=NUM_WORDS, seed=1234)
    res = {"gpu_info": gpu_info(), "n_news": N_NEWS, "n_impressions": N_IMP, "windows": args.windows,
           "train_batch": 128, "train_k_neg": 4, "recommend_candidates": 300, "cases": []}
    rng = np.random.default_rng(7)
    for S in [int(x) for x in args.lengths.split(",")]:
        imp = synthetic.make_impressions(N_IMP, N_NEWS, history=S, seed=1234)
        inputs = EvalInputs.from_host(EvalHost(news, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"]),
                                      dev)
        cand, clicked = synthetic.make_train_batch(128, news, k_neg=4, history=S, seed=1234)
        titles = torch.from_numpy(np.concatenate([cand, clicked], axis=1)).pin_memory()
        for precision in ("tf32", "fp32"):
            m = model_for(S, sd, dev, precision)
            users_ms, eval_ms, means, uw, ew = time_evaluate(m, inputs, args.windows)
            with torch.no_grad():
                table = encode_news_table(m, torch.from_numpy(news).to(dev))[:N_NEWS + 1]
            rec = Recommender(m, [f"N{i}" for i in range(N_NEWS)], table)
            hist = rec.history_rows([f"N{i}" for i in rng.choice(N_NEWS, min(S, 40), replace=False)])
            rec_ms, rec_p90 = time_recommend(rec, hist, rng.choice(N_NEWS, 300, replace=False).tolist(),
                                             args.recommend_calls)
            train_ms, loss, tw = time_train(model_for(S, sd, dev, precision, train=True), titles, args.train_steps,
                                            args.windows)
            case = {"S": S, "precision": precision, "evaluate_users_ms": users_ms, "evaluate_ms": eval_ms,
                    "users_per_s": N_IMP / (users_ms / 1e3), "impressions_per_s": N_IMP / (eval_ms / 1e3),
                    "metrics": list(means), "train_step_ms": train_ms, "train_loss": loss,
                    "recommend_ms_median": rec_ms, "recommend_ms_p90": rec_p90,
                    "evaluate_users_ms_windows": uw, "evaluate_ms_windows": ew, "train_step_ms_windows": tw}
            print(json.dumps({k: v for k, v in case.items() if not k.endswith("windows")}), flush=True)
            res["cases"].append(case)
            del m, rec
        del inputs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
