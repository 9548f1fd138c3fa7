"""NAML on one GPU: news encoding, a training step and evaluate, each in both modes, against torch eager.

Workloads (MIND-small shapes):
  news     get_news_vector over 65,238 news (20-token titles, 50-token abstracts, category, subcategory)
  train    TrainStep.step_rows, B = 128, 1 + 4 candidates, 50 clicks (dropout 0.2, FusedAdam)
  evaluate evaluate_columns over 73,152 impressions of 37 candidates and 50 clicks on that table
torch eager runs the same arithmetic with stock modules in fp32 on the same GPU: F.embedding, nn.Conv2d's
F.conv2d (cuDNN), F.relu, the additive attention, torch.optim.Adam; torch.backends.cudnn.allow_tf32 /
torch.backends.cuda.matmul.allow_tf32 follow the mode.  Outputs are compared at the timed sizes (eval mode).  The conv's
FLOP count is 2 * rows * 900 * 300 per direction (shape-derived, below); achieved rates are over the whole timed call.

Usage: python profiles/naml_bench.py [--out profiles/naml_bench_b200.json] [--reps 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N_NEWS, LT, LA, N_CAT, V = 65238, 20, 50, 275, 70976
B, NEG, CLICKS = 128, 4, 50
N_IMP, CANDS = 73152, 37


def conv_flop(rows):
    """One conv forward: the [rows, 900] x [900, 300] contraction."""
    return 2.0 * rows * 900 * 300


def timed(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return dict(median_ms=float(np.median(ts)), min_ms=float(np.min(ts)), max_ms=float(np.max(ts)), reps=reps)


class Eager(torch.nn.Module):
    """NAML in stock torch modules sharing the B200 model's parameters (the reference's op sequence)."""

    def __init__(self, m):
        super().__init__()
        self.m = m

    def text(self, enc, t):
        x = F.dropout(F.embedding(t, enc.word_embedding.weight, padding_idx=0), 0.2, self.training)
        c = enc.CNN(x.unsqueeze(1)).squeeze(3)
        a = F.dropout(F.relu(c), 0.2, self.training).transpose(1, 2)
        return self.add(a, enc.additive_attention)

    @staticmethod
    def add(c, p):
        t = torch.tanh(F.linear(c, p.linear.weight, p.linear.bias))
        w = F.softmax(torch.matmul(t, p.attention_query_vector), dim=1)
        return torch.bmm(w.unsqueeze(1), c).squeeze(1)

    def news(self, cols):
        ne = self.m.news_encoder
        v = [self.text(ne.text_encoders[a], cols[a]) for a in ne.text_encoders] + \
            [F.relu(e.linear(e.embedding(cols[a]))) for a, e in ne.element_encoders.items()]
        return self.add(torch.stack(v, dim=1), ne.final_attention)

    def forward(self, cols, rows, n_cand):
        Bn, T = rows.shape
        vec = self.news({a: c[rows.reshape(-1)] for a, c in cols.items()}).view(Bn, T, -1)
        user = self.add(vec[:, n_cand:], self.m.user_encoder.additive_attention)
        return torch.bmm(vec[:, :n_cand], user.unsqueeze(-1)).squeeze(-1)


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float(((a - b).norm(dim=-1) / b.norm(dim=-1).clamp_min(1e-12)).max())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "naml_bench_b200.json"))
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("naml_bench needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    import __graft_entry__ as ge
    ge.build()
    from newsrecommendationsystem_b200 import NAML, NAMLConfig
    from newsrecommendationsystem_b200.evaluate import EvalHost, evaluate_columns
    from newsrecommendationsystem_b200.train import TrainStep
    dev = torch.device("cuda")
    rng = np.random.default_rng(0)

    def texts(n, L):
        t = rng.integers(1, V, size=(n, L))
        keep = rng.integers(1, L + 1, size=n)
        return np.where(np.arange(L)[None] < keep[:, None], t, 0)
    host_cols = dict(title=texts(N_NEWS, LT), abstract=texts(N_NEWS, LA),
                     category=rng.integers(1, N_CAT, N_NEWS), subcategory=rng.integers(1, N_CAT, N_NEWS))
    cols = {a: torch.as_tensor(v, dtype=torch.int64, device=dev) for a, v in host_cols.items()}
    pad_cols = {a: torch.cat([c, torch.zeros_like(c[:1])]) for a, c in cols.items()}     # row N_NEWS: the pad
    hist = rng.integers(0, N_NEWS, size=(N_IMP, CLICKS))
    short = rng.integers(0, CLICKS + 1, size=N_IMP)
    hist = np.where(np.arange(CLICKS)[None] < (CLICKS - short)[:, None], -1, hist)
    offs = np.arange(N_IMP + 1, dtype=np.int64) * CANDS
    cand = rng.integers(0, N_NEWS, size=N_IMP * CANDS)
    labels = (rng.random(N_IMP * CANDS) < 0.05).astype(np.int8)
    host = EvalHost(host_cols["title"], hist, offs, cand, labels)
    rows_news = N_NEWS * (LT + LA)
    result = dict(gpu=smi, workload=dict(n_news=N_NEWS, title=LT, abstract=LA, batch=B, candidates=1 + NEG, clicks=CLICKS,
                                         impressions=N_IMP, candidates_per_impression=CANDS), modes={})
    for precision in ("fp32", "tf32"):
        torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = precision == "tf32"
        torch.manual_seed(0)
        cfg = type("Cfg", (NAMLConfig,), dict(num_words=V, num_categories=N_CAT))
        model = NAML(cfg).to(dev).set_precision(precision)
        eager = Eager(model)
        r = {}
        # news encoding
        model.eval()
        eager.eval()
        with torch.no_grad():
            ours = model.get_news_vector(cols)
            ref = eager.news(cols)
            r["news"] = dict(ours=timed(lambda: model.get_news_vector(cols), args.reps),
                             eager=timed(lambda: eager.news(cols), args.reps), max_rel_l2_vs_eager=rel_l2(ours, ref))
        r["news"]["conv_flop"] = conv_flop(rows_news)
        r["news"]["conv_tflops_over_call"] = conv_flop(rows_news) / (r["news"]["ours"]["median_ms"] * 1e-3) / 1e12
        # training step
        cand_rows = torch.as_tensor(rng.integers(0, N_NEWS, size=(B, 1 + NEG)))
        hist_rows = torch.as_tensor(rng.integers(0, N_NEWS + 1, size=(B, CLICKS)))
        rows_all = torch.cat([cand_rows, hist_rows], 1).to(dev)
        with torch.no_grad():
            lo = model.forward_rows(pad_cols, cand_rows.to(dev), hist_rows.to(dev))
            le = eager(pad_cols, rows_all, 1 + NEG)
        model.train()
        eager.train()
        ts = TrainStep(model, lr=1e-4)
        opt = torch.optim.Adam(eager.parameters(), lr=1e-4)

        def eager_step():
            loss = F.cross_entropy(eager(pad_cols, rows_all, 1 + NEG), torch.zeros(B, dtype=torch.long, device=dev))
            opt.zero_grad()
            loss.backward()
            opt.step()
        rows_train = B * (1 + NEG + CLICKS) * (LT + LA)
        r["train_step"] = dict(ours=timed(lambda: ts.step_rows(pad_cols, cand_rows, hist_rows), args.reps),
                               eager=timed(eager_step, args.reps), logits_max_rel_l2_vs_eager=rel_l2(lo, le),
                               conv_flop=3 * conv_flop(rows_train))
        r["train_step"]["conv_tflops_over_call"] = 3 * conv_flop(rows_train) / (r["train_step"]["ours"]["median_ms"] * 1e-3) / 1e12
        # evaluate
        model.eval()
        eager.eval()
        hist_d = torch.as_tensor(np.where(hist < 0, N_NEWS, hist), device=dev)
        cand_d = torch.as_tensor(cand, device=dev)
        imp_of = torch.repeat_interleave(torch.arange(N_IMP, device=dev), CANDS)

        @torch.no_grad()
        def eager_eval():
            table = torch.cat([eager.news(cols), torch.zeros((1, 300), device=dev)])
            user = eager.add(table[hist_d], model.user_encoder.additive_attention)
            return (table[cand_d] * user[imp_of]).sum(-1)
        t0 = time.perf_counter()
        means = evaluate_columns(model, cols, host)
        first_call_s = time.perf_counter() - t0
        r["evaluate"] = dict(ours=timed(lambda: evaluate_columns(model, cols, host), max(3, args.reps // 4)),
                             eager_news_users_scores=timed(eager_eval, max(3, args.reps // 4)),
                             metric_means=list(means), first_call_s=first_call_s)
        result["modes"][precision] = r
        print(precision, json.dumps({k: (v["ours"]["median_ms"], v.get("eager", v.get("eager_news_users_scores"))["median_ms"])
                                     for k, v in r.items()}), flush=True)
        del model, eager, ts, opt
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["gpu"]))


if __name__ == "__main__":
    main()
