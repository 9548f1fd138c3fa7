"""Exp1 training with the abstract encoder on one GPU (writes profiles/exp1_train_bench_b200.json by default).

  - The Exp1 training step (TrainStep.step_rows over a device-resident news table: forward, CE(label 0), backward,
    fused Adam) at the reference's shape, B = 128, 1 + 4 candidates, 50 clicked news, tensor mode, with and without the
    abstract ('category', 'subcategory', 'title' [+ 'abstract']).
  - The 50-token news-encoder training pass (forward + backward with dropout 0.2) over the 7,040 abstracts of one such
    batch, with the mma.sync attention (attn_mma.cu) and with the CUDA-core attention_*_kernel<50,5>, switched through
    nrms_set_option("train_attn_mma") and alternated in one process.
  - With --profile, a torch.profiler pass (a separate run: tracing slows the host) gives the per-kernel device time of
    the attention kernels under both settings and the kernel split of the abstract training step.
Times are CUDA events over windows of at least --min-s seconds after warm-up; the working set of the encoder pass
(about 4 GB of stash and workspace) is larger than the L2, so it is read from HBM in every pass.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from newsrecommendationsystem_b200 import Exp1, _lib  # noqa: E402
from newsrecommendationsystem_b200.config import Exp1Config  # noqa: E402
from newsrecommendationsystem_b200.train import TrainStep  # noqa: E402

B, N_CAND, N_CLICKED = 128, 5, 50
NUM_WORDS, NUM_CATEGORIES, N_NEWS = 70976, 300, 65238
ATTRS = ['category', 'subcategory', 'title']
ATTRS_A = ATTRS + ['abstract']


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:          # the number is still labelled with the GPU name
        info["power_limit"] = f"unavailable ({e})"
    return info


def timed(fn, min_s):
    """ms per call from CUDA events over a window of at least min_s seconds."""
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    once = max(time.perf_counter() - t0, 1e-6)
    n = max(3, int(min_s / once) + 1)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def make_cfg(attrs):
    class Cfg(Exp1Config):
        num_words = NUM_WORDS
        num_categories = NUM_CATEGORIES
        dataset_attributes = {"news": list(attrs), "record": []}
    return Cfg


def news_table(dev, seed=0):
    """A synthetic pre-tokenised table of N_NEWS news + the pad row: titles of 8..20 tokens, abstracts of 0..50."""
    rng = np.random.default_rng(seed)
    title = rng.integers(1, NUM_WORDS, size=(N_NEWS + 1, 20))
    title[np.arange(20)[None] >= rng.integers(8, 21, size=(N_NEWS + 1, 1))] = 0
    abstract = rng.integers(1, NUM_WORDS, size=(N_NEWS + 1, 50))
    abstract[np.arange(50)[None] >= rng.integers(0, 51, size=(N_NEWS + 1, 1))] = 0
    t = {"title": title, "abstract": abstract, "category": rng.integers(1, NUM_CATEGORIES, size=N_NEWS + 1),
         "subcategory": rng.integers(1, NUM_CATEGORIES, size=N_NEWS + 1)}
    for v in t.values():
        v[N_NEWS] = 0
    return {k: torch.from_numpy(v.astype(np.int64)).to(dev) for k, v in t.items()}


def batch_rows(rng):
    cand = torch.from_numpy(rng.integers(0, N_NEWS, size=(B, N_CAND)))
    hist = torch.from_numpy(rng.integers(0, N_NEWS + 1, size=(B, N_CLICKED)))
    return cand, hist


def train_step_fn(attrs, table, dev, warmup):
    torch.manual_seed(0)
    m = Exp1(make_cfg(attrs)).to(dev).train().set_precision("tf32")
    ts = TrainStep(m)
    t = {k: table[k] for k in attrs}
    rng = np.random.default_rng(1)
    cand, hist = batch_rows(rng)
    for _ in range(warmup):
        ts.step_rows(t, cand, hist)
    return lambda: ts.step_rows(t, cand, hist)


def encoder_fn(dev, table, warmup):
    """Forward + backward of the abstract encoder over the 7,040 abstracts of one batch (dropout 0.2)."""
    torch.manual_seed(0)
    m = Exp1(make_cfg(ATTRS_A)).to(dev).train().set_precision("tf32")
    enc = m.news_encoder.text_encoders["abstract"]
    rows = torch.from_numpy(np.random.default_rng(2).integers(0, N_NEWS + 1, size=B * (N_CAND + N_CLICKED))).to(dev)
    toks = table["abstract"][rows].contiguous()
    g = torch.randn((toks.shape[0], 300), device=dev)
    params = [p for p in enc.parameters()]

    def fn():
        out = enc(toks)
        torch.autograd.grad(out, params, g)
    for _ in range(warmup):
        fn()
    return fn


def set_mma(lib, on):
    assert lib.nrms_set_option(b"train_attn_mma", 1 if on else 0) == 0


def profile_split(fn, match):
    from torch.profiler import profile, ProfilerActivity
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
    split = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t and any(s in e.key for s in match):
            split[e.key.split("(")[0][:120]] = round(t / 5, 2)            # us per call
    return dict(sorted(split.items(), key=lambda kv: -kv[1]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "exp1_train_bench_b200.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--min-s", type=float, default=0.5)
    ap.add_argument("--profile", action="store_true", help="per-kernel split with torch.profiler (a separate run)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    dev = torch.device("cuda:0")
    lib = _lib.load()
    res = dict(gpu_info(), batch=dict(B=B, candidates=N_CAND, clicked=N_CLICKED, abstracts=B * (N_CAND + N_CLICKED),
                                      num_words=NUM_WORDS, n_news=N_NEWS, precision="tf32", dropout=0.2))
    table = news_table(dev)
    enc = encoder_fn(dev, table, a.warmup)
    if a.profile:
        res["profile_us_per_call"] = {}
        attn = ("attn50_", "attention_fwd_kernel", "attention_bwd_kernel")
        for on in (1, 0):
            set_mma(lib, on)
            res["profile_us_per_call"][f"abstract_encoder_fwd_bwd_train_attn_mma={on}"] = profile_split(enc, attn)
        set_mma(lib, 1)
        step = train_step_fn(ATTRS_A, table, dev, a.warmup)
        res["profile_us_per_call"]["exp1_step_with_abstract"] = profile_split(step, ("",))
    else:
        set_mma(lib, 1)
        steps = {"without_abstract": train_step_fn(ATTRS, table, dev, a.warmup),
                 "with_abstract": train_step_fn(ATTRS_A, table, dev, a.warmup)}
        t_enc = {0: [], 1: []}
        t_step = {k: [] for k in steps}
        for r in range(a.rounds):                       # alternated: the two settings see the same machine state
            for on in ((1, 0) if r % 2 == 0 else (0, 1)):
                set_mma(lib, on)
                t_enc[on].append(timed(enc, a.min_s))
            set_mma(lib, 1)
            for k, fn in steps.items():
                t_step[k].append(timed(fn, a.min_s))
        set_mma(lib, 1)
        res["abstract_encoder_fwd_bwd_ms"] = {f"train_attn_mma={on}": dict(median=statistics.median(v),
                                                                           all=[round(x, 4) for x in v])
                                              for on, v in t_enc.items()}
        res["exp1_train_step_ms"] = {k: dict(median=statistics.median(v), all=[round(x, 4) for x in v])
                                     for k, v in t_step.items()}
    print(json.dumps(res), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
