"""LSTUR on the B200: the GRU user encoder (forward + backward) and the training step, against torch eager of the same
model on the same GPU (nn.GRU on packed input, i.e. cuDNN; F.conv2d; TF32 on in tensor mode and off in FP32 mode).

Writes profiles/lstur_bench_b200.json (or the path given as argv[1]).  CUDA events around each call, warm-up first, then
the median over windows of >= 0.5 s.  Also the GRU's error at 2,049 sequences against float64 nn.GRU, and evaluate at
MIND-small shape with its user stage on its own.  The GPU's name, power limit and SM clock are read in the same run."""
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from newsrecommendationsystem_b200 import LSTUR, ops, _lib  # noqa: E402
from newsrecommendationsystem_b200.config import LSTURConfig  # noqa: E402
from newsrecommendationsystem_b200.train import TrainStep  # noqa: E402

B, K, N, L, T = 128, 4, 50, 20, 50
NUM_NEWS = 65238


def timed(fn, min_window_s=0.5, windows=5):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    fn()
    e.record()
    torch.cuda.synchronize()
    per = max(s.elapsed_time(e), 1e-3)
    reps = max(1, int(min_window_s * 1000 / per))
    out = []
    for _ in range(windows):
        s.record()
        for _ in range(reps):
            fn()
        e.record()
        torch.cuda.synchronize()
        out.append(s.elapsed_time(e) / reps)
    return float(np.median(out))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else torch.cuda.get_device_name()


def cfg_for(method):
    class C(LSTURConfig):
        pass
    C.long_short_term_method = method
    C.num_words = 70976
    C.dropout_probability = 0.2
    C.masking_probability = 0.5
    return C


def bench_gru(method, precision, lengths, dev):
    H = 900 if method == "ini" else 450
    gru = nn.GRU(900, H).to(dev)
    w = [p.detach().clone().requires_grad_(True) for p in gru.parameters()]   # weight_ih, weight_hh, bias_ih, bias_hh
    x = torch.randn(B, T, 900, device=dev, requires_grad=True)
    h0 = torch.randn(B, H, device=dev, requires_grad=True) if method == "ini" else None
    g = torch.randn(B, H, device=dev)
    mode = _lib.MODES[precision]
    lt = torch.as_tensor(lengths)

    def ours():
        ops.gru(x, lt, h0, *w, mode=mode).backward(g)

    def cudnn():
        packed = nn.utils.rnn.pack_padded_sequence(x, lt, batch_first=True, enforce_sorted=False)
        _, h = gru(packed) if h0 is None else gru(packed, h0.unsqueeze(0))
        h.squeeze(0).backward(g)
    torch.backends.cudnn.allow_tf32 = precision == "tf32"
    torch.backends.cuda.matmul.allow_tf32 = precision == "tf32"
    t_ours, t_ref = timed(ours), timed(cudnn)
    rows = int(lengths.sum())
    flop = 3 * rows * 2 * H * 3 * H            # forward step GEMM + the backward's dh and dW_hh contractions
    return dict(method=method, precision=precision, ms=t_ours, cudnn_ms=t_ref, speedup=t_ref / t_ours,
                sum_lengths=rows, recurrence_tflops_per_s=flop / (t_ours * 1e-3) / 1e12)


class EagerLSTUR(nn.Module):
    """The reference's LSTUR in torch eager (stock modules), for the baseline."""

    def __init__(self, cfg):
        super().__init__()
        H = 900 if cfg.long_short_term_method == "ini" else 450
        self.cfg = cfg
        self.word = nn.Embedding(cfg.num_words, 300, padding_idx=0)
        self.cat = nn.Embedding(cfg.num_categories, 300, padding_idx=0)
        self.cnn = nn.Conv2d(1, 300, (3, 300), padding=(1, 0))
        self.att = nn.Linear(300, 200)
        self.q = nn.Parameter(torch.empty(200).uniform_(-0.1, 0.1))
        self.gru = nn.GRU(900, H)
        self.user_emb = nn.Embedding(cfg.num_users, H, padding_idx=0)

    def news(self, c, s, t):
        x = F.dropout(self.word(t), 0.2, self.training)
        a = F.dropout(F.relu(self.cnn(x.unsqueeze(1)).squeeze(3)), 0.2, self.training).transpose(1, 2)
        w = F.softmax(torch.tanh(self.att(a)) @ self.q, dim=1)
        return torch.cat([self.cat(c), self.cat(s), torch.bmm(w.unsqueeze(1), a).squeeze(1)], dim=1)

    def forward(self, user, lengths, c, s, t):
        Bn, Tn = t.shape[:2]
        vec = self.news(c.reshape(-1), s.reshape(-1), t.reshape(Bn * Tn, -1)).view(Bn, Tn, -1)
        u = F.dropout2d(self.user_emb(user).unsqueeze(0), p=0.5, training=self.training).squeeze(0)
        lengths = lengths.clone()
        lengths[lengths == 0] = 1
        packed = nn.utils.rnn.pack_padded_sequence(vec[:, 1 + K:], lengths, batch_first=True, enforce_sorted=False)
        if self.cfg.long_short_term_method == "ini":
            _, h = self.gru(packed, u.unsqueeze(0))
            uv = h.squeeze(0)
        else:
            _, h = self.gru(packed)
            uv = torch.cat([h.squeeze(0), u], dim=1)
        return torch.bmm(vec[:, :1 + K], uv.unsqueeze(-1)).squeeze(-1)


def bench_train(method, precision, dev, rng):
    cfg = cfg_for(method)
    title = torch.from_numpy(rng.integers(1, cfg.num_words, size=(NUM_NEWS + 1, L))).to(dev)
    title[NUM_NEWS] = 0
    table = {"title": title,
             "category": torch.from_numpy(rng.integers(1, 275, size=NUM_NEWS + 1)).to(dev),
             "subcategory": torch.from_numpy(rng.integers(1, 275, size=NUM_NEWS + 1)).to(dev)}
    cand = torch.from_numpy(rng.integers(0, NUM_NEWS, size=(B, 1 + K)))
    lengths = torch.from_numpy(rng.integers(0, N + 1, size=B))
    hist = torch.from_numpy(rng.integers(0, NUM_NEWS, size=(B, N)))
    hist[torch.arange(N)[None] < (N - lengths)[:, None]] = NUM_NEWS          # left padding
    user = torch.from_numpy(rng.integers(1, cfg.num_users, size=B))
    model = LSTUR(cfg).to(dev).train().set_precision(precision)
    ts = TrainStep(model, lr=1e-4)
    t_ours = timed(lambda: ts.step_rows(table, cand, hist, user=user, clicked_news_length=lengths))
    torch.backends.cudnn.allow_tf32 = precision == "tf32"
    torch.backends.cuda.matmul.allow_tf32 = precision == "tf32"
    ref = EagerLSTUR(cfg).to(dev).train()
    opt = torch.optim.Adam(ref.parameters(), lr=1e-4)
    rows = torch.cat([cand, hist], dim=1).to(dev)
    user_d, len_d = user.to(dev), lengths

    def eager():
        logits = ref(user_d, len_d, table["category"][rows], table["subcategory"][rows], table["title"][rows])
        loss = F.cross_entropy(logits, torch.zeros(B, dtype=torch.long, device=dev))
        opt.zero_grad()
        loss.backward()
        opt.step()
    t_ref = timed(eager)
    return dict(method=method, precision=precision, ms=t_ours, eager_ms=t_ref, speedup=t_ref / t_ours)


def gru_accuracy(method, dev, n_seq=2049):
    """Tensor- and FP32-mode GRU at n_seq sequences of 50 steps (lengths 1..50) against float64 nn.GRU on the GPU: the
    worst row-wise relative L2 of the last state, and each gradient's max |error| over its largest entry."""
    H = 900 if method == "ini" else 450
    torch.manual_seed(5)
    ref = nn.GRU(900, H).double().to(dev)
    lengths = torch.randint(1, T + 1, (n_seq,))
    x = torch.randn(n_seq, T, 900, device=dev, dtype=torch.float64)
    h0 = torch.randn(n_seq, H, device=dev, dtype=torch.float64) if method == "ini" else None
    g = torch.randn(n_seq, H, device=dev, dtype=torch.float64)
    xr = x.clone().requires_grad_(True)
    h0r = None if h0 is None else h0.clone().requires_grad_(True)
    packed = nn.utils.rnn.pack_padded_sequence(xr, lengths, batch_first=True, enforce_sorted=False)
    _, hr = ref(packed) if h0r is None else ref(packed, h0r.unsqueeze(0))
    hr = hr.squeeze(0)
    hr.backward(g)
    want = {"h": hr.detach(), "dx": xr.grad, "dh0": None if h0r is None else h0r.grad}
    for name, p in ref.named_parameters():
        want[name] = p.grad
    out = {}
    for precision in ("tf32", "fp32"):
        w = [p.detach().float().clone().requires_grad_(True) for p in ref.parameters()]
        xo = x.float().requires_grad_(True)
        h0o = None if h0 is None else h0.float().requires_grad_(True)
        h = ops.gru(xo, lengths, h0o, *w, mode=_lib.MODES[precision])
        h.backward(g.float())
        got = {"h": h.detach(), "dx": xo.grad, "dh0": None if h0o is None else h0o.grad}
        for (name, _), p in zip(ref.named_parameters(), w):
            got[name] = p.grad
        row = ((got["h"].double() - want["h"]).norm(dim=1) / want["h"].norm(dim=1)).max().item()
        grads = {k: ((got[k].double() - want[k]).abs().max() / want[k].abs().max()).item()
                 for k in got if k != "h" and got[k] is not None}
        out[precision] = dict(worst_row_rel_l2_h=row, grad_max_err_over_max=grads)
    return dict(method=method, n_seq=n_seq, **out)


def bench_evaluate(method, precision, dev, rng, n_imp=73152, n_cand=37):
    """Evaluate at MIND-small shape: 65,238 news, 73,152 impressions x 37 candidates, one user per impression (distinct
    histories), histories of 0..50 clicks, left-padded.  Ours: LSTUR's evaluate pipeline after the files are read
    (news table, table-projected GRU, scoring, metrics); the user stage alone next to cuDNN's GRU over the same users
    (histories gathered from the same table, packed).  Eager: get_news_vector, cuDNN GRU, scoring, no metrics."""
    from newsrecommendationsystem_b200.data import EvalRows
    from newsrecommendationsystem_b200.evaluate import lstur_user_vectors
    cfg = cfg_for(method)
    cfg.num_users = 50001
    model = LSTUR(cfg).to(dev).eval().set_precision(precision)
    cols = {"title": torch.from_numpy(rng.integers(1, cfg.num_words, size=(NUM_NEWS, L))).to(dev),
            "category": torch.from_numpy(rng.integers(1, 275, size=NUM_NEWS)).to(dev),
            "subcategory": torch.from_numpy(rng.integers(1, 275, size=NUM_NEWS)).to(dev)}
    lengths = rng.integers(0, N + 1, size=n_imp)
    hist = rng.integers(0, NUM_NEWS, size=(n_imp, N))
    hist[np.arange(N)[None] < (N - lengths)[:, None]] = -1
    keys = [" ".join(map(str, h[h >= 0])) + f"#{i}" for i, h in enumerate(hist)]       # distinct histories
    ev = EvalRows(hist, np.arange(0, (n_imp + 1) * n_cand, n_cand, dtype=np.int64),
                  rng.integers(0, NUM_NEWS, size=n_imp * n_cand), rng.integers(0, 2, size=n_imp * n_cand).astype(np.int8),
                  list(range(n_imp)), keys, [f"U{i % 50000}" for i in range(n_imp)])
    user2int = {f"U{i}": i + 1 for i in range(50000)}
    offs = torch.from_numpy(ev.cand_offsets).to(dev)
    cand32 = torch.from_numpy(ev.cand_rows.astype(np.int32)).to(dev)
    labels = torch.from_numpy(ev.labels).to(dev)

    def ours():
        uv = lstur_user_vectors(model, cols, ev, user2int)
        s = ops.score_csr(uv.table, cand32, offs, uv.per_impression)
        ops.rank_metrics(s, labels, offs)
    torch.backends.cudnn.allow_tf32 = precision == "tf32"
    torch.backends.cuda.matmul.allow_tf32 = precision == "tf32"
    with torch.no_grad():
        uv = lstur_user_vectors(model, cols, ev, user2int)
        table = uv.table
        user_rows = model._user(torch.from_numpy(uv.users), False)
        lens = torch.from_numpy(np.maximum(uv.lengths, 1))
        hist_dev = torch.from_numpy(np.where(hist < 0, NUM_NEWS, hist)).to(dev)
        ue = model.user_encoder

        def ours_users():
            ue.forward_indexed(user_rows, lens, table, hist_dev)
        gru = ue.gru

        def cudnn_users(chunk=8192):
            for s0 in range(0, n_imp, chunk):
                x = table[hist_dev[s0:s0 + chunk]]
                packed = nn.utils.rnn.pack_padded_sequence(x, lens[s0:s0 + chunk], batch_first=True,
                                                           enforce_sorted=False)
                h0 = user_rows[s0:s0 + chunk].unsqueeze(0) if method == "ini" else None
                gru(packed, h0) if h0 is not None else gru(packed)
        ref = EagerLSTUR(cfg).to(dev).eval()
        imp = torch.repeat_interleave(torch.arange(n_imp, device=dev), n_cand)
        cand64 = cand32.long()

        def eager():
            t = torch.cat([ref.news(cols["category"][s0:s0 + 8192], cols["subcategory"][s0:s0 + 8192],
                                    cols["title"][s0:s0 + 8192]) for s0 in range(0, NUM_NEWS, 8192)])
            t = torch.cat([t, torch.zeros(1, 900, device=dev)])
            us = []
            for s0 in range(0, n_imp, 8192):
                packed = nn.utils.rnn.pack_padded_sequence(t[hist_dev[s0:s0 + 8192]], lens[s0:s0 + 8192],
                                                           batch_first=True, enforce_sorted=False)
                u = ref.user_emb(torch.from_numpy(uv.users[s0:s0 + 8192]).to(dev))
                _, h = ref.gru(packed, u.unsqueeze(0)) if method == "ini" else ref.gru(packed)
                us.append(h.squeeze(0) if method == "ini" else torch.cat([h.squeeze(0), u], dim=1))
            uvec = torch.cat(us)
            (t[cand64] * uvec[imp]).sum(1)
        res = dict(method=method, precision=precision, evaluate_ms=timed(ours), user_stage_ms=timed(ours_users),
                   cudnn_user_stage_ms=timed(cudnn_users), eager_evaluate_ms=timed(eager))
    return res


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "lstur_bench_b200.json")
    dev = torch.device("cuda")
    rng = np.random.default_rng(0)
    lengths = rng.integers(1, T + 1, size=B)
    res = dict(gpu=gpu_info(), batch=B, steps=T, gru=[], train_step=[])
    for method in ("ini", "con"):
        for precision in ("tf32", "fp32"):
            res["gru"].append(bench_gru(method, precision, lengths, dev))
            print(res["gru"][-1], flush=True)
    for method in ("ini", "con"):
        for precision in ("tf32", "fp32"):
            res["train_step"].append(bench_train(method, precision, dev, rng))
            print(res["train_step"][-1], flush=True)
    res["evaluate"] = []
    for method in ("ini", "con"):
        for precision in ("tf32", "fp32"):
            res["evaluate"].append(bench_evaluate(method, precision, dev, rng))
            print(res["evaluate"][-1], flush=True)
    res["accuracy_2049"] = [gru_accuracy(m, dev) for m in ("ini", "con")]
    print(res["accuracy_2049"], flush=True)
    res["gpu_after"] = gpu_info()
    res["datasheet_floor_note"] = ("dense TF32 data-sheet rate 1,125 TFLOP/s for one B200 at 1,000 W: a floor, not "
                                   "a rate reached")
    with open(out_path, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
