"""Cross-attention and other lengths in the standalone MultiHeadSelfAttention on one GPU (writes
profiles/mha_cross_bench_b200.json by default).

  - Forward + backward of the module (gradients of every input and the six parameters) over 7,040 sequences, in tensor
    (TF32) and FP32 mode, at:
      (Sq, Sk) = (5, 50) with K = V (candidates attending over a history);
      (50, 20) with K != V;  (20, 20) with K = V != Q;
      self-attention at 30 and at 64 tokens, without a mask and with uniform random lengths in [1, S].
  - The baseline: the reference's op sequence (multihead_self.py:15-23,46-76: three nn.Linear, exp of the scaled
    scores, times the mask, over (sum + 1e-8), times V) in torch eager on the same GPU, with TF32 matmuls allowed in
    tensor mode and disallowed in FP32 mode.
  - With --profile, a torch.profiler pass (a separate run: tracing slows the host) gives the per-kernel device time of
    every case in tensor mode.
Times are CUDA events over windows of at least --min-s seconds after warm-up; the median of --windows windows is
reported, the two sides alternated.  The inputs of every case (at least 85 MB) are not all L2-resident between passes.
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

from exp1_train_bench import gpu_info, timed  # noqa: E402
from newsrecommendationsystem_b200.model.general.attention.multihead_self import MultiHeadSelfAttention  # noqa: E402

N_SEQ = 7040
# (name, Sq, Sk, form, mask): form kv = K != V, k=v = K is V (not Q), self = K is V is Q
CASES = [("cand5_hist50", 5, 50, "k=v", "none"), ("q50_kv20", 50, 20, "kv", "none"), ("q20_kv20", 20, 20, "k=v", "none"),
         ("self30", 30, 30, "self", "none"), ("self30_masked", 30, 30, "self", "random"),
         ("self64", 64, 64, "self", "none"), ("self64_masked", 64, 64, "self", "random")]


def reference_eager(m, q, k, v, length):
    """The reference block in torch eager."""
    n, sq, _ = q.shape
    sk = k.shape[1]
    h = [lin(x).view(n, x.shape[1], 15, 20).transpose(1, 2) for lin, x in ((m.W_Q, q), (m.W_K, k), (m.W_V, v))]
    e = torch.exp(h[0] @ h[1].transpose(-1, -2) / np.sqrt(20.0))
    if length is not None:
        e = e * (torch.arange(sk, device=q.device).view(1, 1, 1, sk) < length.view(n, 1, 1, 1)).float()
    attn = e / (e.sum(-1, keepdim=True) + 1e-8)
    return (attn @ h[2]).transpose(1, 2).reshape(n, sq, 300)


def make_case(dev, sq, sk, form, mask):
    gen = torch.Generator(device=dev).manual_seed(1000 * sq + sk)
    x = torch.randn((N_SEQ, sq, 300), device=dev, generator=gen).requires_grad_(True)
    if form == "self":
        q = k = v = x
    else:
        q = x
        k = torch.randn((N_SEQ, sk, 300), device=dev, generator=gen).requires_grad_(True)
        v = k if form == "k=v" else torch.randn((N_SEQ, sk, 300), device=dev, generator=gen).requires_grad_(True)
    G = torch.randn((N_SEQ, sq, 300), device=dev, generator=gen)
    length = torch.randint(1, sk + 1, (N_SEQ,), device=dev, generator=gen, dtype=torch.int32) if mask == "random" else None
    return q, k, v, G, length


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mha_cross_bench_b200.json"))
    ap.add_argument("--min-s", type=float, default=0.3)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m = MultiHeadSelfAttention(300, 15).to(dev)
    res = {"gpu_info": gpu_info(), "n_seq": N_SEQ, "windows": args.windows, "min_window_s": args.min_s, "cases": []}
    for name, sq, sk, form, mask in CASES:
        q, k, v, G, length = make_case(dev, sq, sk, form, mask)
        leaves = [t for i, t in enumerate((q, k, v)) if all(t is not u for u in (q, k, v)[:i])]
        for precision in ("tf32", "fp32"):
            m.precision = precision
            torch.backends.cuda.matmul.allow_tf32 = precision == "tf32"

            def clear():
                for t in leaves + list(m.parameters()):
                    t.grad = None

            def ours():
                clear()
                m(q, K=k, V=v, length=length).backward(G)

            def eager():
                clear()
                reference_eager(m, q, k, v, length).backward(G)

            a, b = [], []
            for _ in range(args.windows):            # alternated, so that both see the same clocks
                a.append(timed(ours, args.min_s))
                b.append(timed(eager, args.min_s))
            case = {"case": name, "Sq": sq, "Sk": sk, "form": form, "mask": mask, "precision": precision,
                    "ms_b200": statistics.median(a), "ms_torch_eager": statistics.median(b), "ms_b200_windows": a,
                    "ms_torch_eager_windows": b}
            case["speedup"] = case["ms_torch_eager"] / case["ms_b200"]
            print(json.dumps(case), flush=True)
            res["cases"].append(case)
    torch.backends.cuda.matmul.allow_tf32 = False
    if args.profile:
        from torch.profiler import profile, ProfilerActivity
        m.precision = "tf32"
        res["profile_tf32"] = {}
        for name, sq, sk, form, mask in CASES:
            q, k, v, G, length = make_case(dev, sq, sk, form, mask)
            for _ in range(3):
                m(q, K=k, V=v, length=length).backward(G)
            torch.cuda.synchronize()
            reps = 10
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(reps):
                    m(q, K=k, V=v, length=length).backward(G)
                torch.cuda.synchronize()
            split = {}
            for e in prof.key_averages():
                t = getattr(e, "device_time_total", None)
                if t is None:
                    t = e.cuda_time_total
                if t > 0:
                    split[e.key[:120]] = round(t / reps, 1)
            split = dict(sorted(split.items(), key=lambda kv: -kv[1]))
            res["profile_tf32"][name] = {"us_per_iteration": split}
            print(f"{name}:", json.dumps(split), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
