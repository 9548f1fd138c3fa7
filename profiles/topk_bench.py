"""Top-k news over the whole table (ops.topk_news, tensor mode) against a chunked PyTorch baseline.

    python profiles/topk_bench.py --out profiles/topk_bench_b200.json [--quick]

For each (users U, news n_news, k) with the users' 50 history rows as exclusions:
  - fused: nrms_topk_news (users -> fp16, tcgen05 score pass with the selecting epilogue, merge).  Device time from CUDA
    events around replays of a CUDA graph of one call (so that host launch overhead does not pad the window at U = 1),
    plus the same with events around eager calls;
  - baseline: fp16 torch.mm over chunks of 2,048 users, the history rows set to -inf, torch.topk; eager, CUDA events;
  - the two are timed alternately (three rounds each, windows of >= 0.5 s; the median round is reported), then compared
    on their outputs (row overlap, largest difference of the sorted top-k scores);
  - a torch.profiler pass (separate from the timed windows) splits the fused call's device time by kernel.
Counts kept with the benchmark (not measured): useful FLOPs = 2 U n_news 300; the score pass reads the fp16 table
(640 B per row) once per 128-user block, ceil(U / 128) n_news 640 bytes of L2 reads.  Rates are over the measured time;
the share of peak is over the 2,250 TFLOP/s dense fp16 figure of the B200 data sheet (a data-sheet figure, not reached).
The table (41.8 MB at 65,238 rows in fp16) fits the 126 MB L2, so repeated calls read it from there after the first.
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

from newsrecommendationsystem_b200 import ops, _lib  # noqa: E402

PEAK_F16 = 2250e12
CHUNK = 2048


def gpu_info():
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info["power_limit"], info["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:          # the number is still labelled with the GPU name
        info["power_limit"] = f"unavailable ({e})"
    return info


def timed(fn, min_s=0.5):
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
    return a.elapsed_time(b) / n, n


def baseline(t16, n_news, users, hist, k):
    tv = t16[:n_news, :300]
    U = users.shape[0]
    out_s = torch.empty((U, k), dtype=torch.float32, device=users.device)
    out_r = torch.empty((U, k), dtype=torch.int64, device=users.device)
    for c0 in range(0, U, CHUNK):
        u16 = users[c0:c0 + CHUNK].half()
        s = torch.mm(u16, tv.t()).float()
        h = hist[c0:c0 + CHUNK].long()
        valid = (h >= 0) & (h < n_news)
        ri = torch.arange(h.shape[0], device=h.device)[:, None].expand_as(h)
        s[ri[valid], h[valid]] = -float("inf")
        v, i = torch.topk(s, k, dim=1)
        out_s[c0:c0 + CHUNK], out_r[c0:c0 + CHUNK] = v, i
    return out_s, out_r


def kernel_split(fn):
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
        if t and ("topk" in e.key or "users_to_f16" in e.key):
            name = e.key.split("(")[0].split("::")[-1]
            split[name] = round(t / 5 / 1000, 4)            # ms per call
    return split


def case(U, n_news, k, rounds, min_s, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    dev = torch.device("cuda:0")
    table = torch.randn(n_news, 300, device=dev, generator=g) * 0.1
    t16 = ops.pack_rows_f16(table)
    del table
    users = torch.randn(U, 300, device=dev, generator=g)
    hist = torch.randint(-1, n_news, (U, 50), device=dev, generator=g, dtype=torch.int32)
    fused = lambda: ops.topk_news(t16, n_news, users, k, exclude_rows=hist, mode=_lib.MODE_TF32)  # noqa: E731
    fused()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fused()
        with torch.cuda.graph(graph):
            g_out = fused()
    torch.cuda.current_stream().wait_stream(s)
    base = lambda: baseline(t16, n_news, users, hist, k)  # noqa: E731
    f_ms, f_eager_ms, b_ms = [], [], []
    for _ in range(rounds):
        f_ms.append(timed(graph.replay, min_s)[0])
        b_ms.append(timed(base, min_s)[0])
        f_eager_ms.append(timed(fused, min_s)[0])
    # output check between the two
    graph.replay()
    fs, fr = g_out
    bs, br = base()
    torch.cuda.synchronize()
    m = min(U, 512)
    fs, fr, bs, br = (x[:m].cpu().numpy() for x in (fs, fr, bs, br))
    overlap = float(np.mean([len(np.intersect1d(fr[i], br[i])) / k for i in range(m)]))
    fin = np.isfinite(fs) & np.isfinite(bs)
    score_diff = float(np.abs(fs - bs)[fin].max(initial=0.0))
    split = kernel_split(graph.replay)
    fm, bm, fe = statistics.median(f_ms), statistics.median(b_ms), statistics.median(f_eager_ms)
    flops = 2.0 * U * n_news * 300
    return {
        "users": U, "n_news": n_news, "k": k, "n_exclude": 50,
        "fused_ms": round(fm, 4), "fused_ms_rounds": [round(x, 4) for x in f_ms],
        "fused_eager_ms": round(fe, 4),
        "fused_users_per_s": round(U / (fm * 1e-3), 1),
        "fused_useful_tflops": round(flops / (fm * 1e-3) / 1e12, 2),
        "fused_fraction_of_datasheet_f16_dense": round(flops / (fm * 1e-3) / PEAK_F16, 4),
        "fused_kernel_ms_per_call": split,
        "baseline_ms": round(bm, 4), "baseline_ms_rounds": [round(x, 4) for x in b_ms],
        "baseline_users_per_s": round(U / (bm * 1e-3), 1),
        "baseline_useful_tflops": round(flops / (bm * 1e-3) / 1e12, 2),
        "speedup_vs_baseline": round(bm / fm, 2),
        "score_pass_l2_read_bytes_count": int((U + 127) // 128 * n_news * 640),
        "check_users": m, "check_row_overlap": round(overlap, 5), "check_max_sorted_score_diff": score_diff,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--quick", action="store_true", help="one small case (a rehearsal of the script)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--min-s", type=float, default=0.5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "topk_bench needs a GPU"
    res = {"what": "nrms_topk_news tensor mode vs chunked fp16 torch.mm + torch.topk", **gpu_info(),
           "datasheet_f16_dense_tflops": PEAK_F16 / 1e12, "cases": []}
    if a.quick:
        grid = [(1000, 20000, 10)]
    else:
        grid = [(U, n, k) for n in (65238, 161013) for U in (73152, 8192, 1) for k in (10, 100)]
    for U, n, k in grid:
        r = case(U, n, k, a.rounds, a.min_s)
        print(json.dumps(r), flush=True)
        res["cases"].append(r)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
