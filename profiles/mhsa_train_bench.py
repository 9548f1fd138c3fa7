"""Training the standalone MultiHeadSelfAttention on one GPU (writes profiles/mhsa_train_bench_b200.json by default).

  - Forward + backward of the module (gradients of x and the six parameters) over 7,040 sequences of 20 and of 50
    tokens, without a mask and with uniform random lengths in [1, S], in tensor (TF32) and FP32 mode.
  - The baseline: the reference's op sequence (multihead_self.py:15-23,46-76: three nn.Linear, exp of the scaled
    scores, times the mask, over (sum + 1e-8), times V) in torch eager on the same GPU, with TF32 matmuls allowed in
    tensor mode and disallowed in FP32 mode.
  - With --profile, a torch.profiler pass (a separate run: tracing slows the host) gives the per-kernel device time of
    the masked and the unmasked backward in tensor mode.
Times are CUDA events over windows of at least --min-s seconds after warm-up; the median of --windows windows is
reported.  The inputs alone (x and the incoming gradient, 169 MB at S = 20, 422 MB at S = 50) are larger than the L2,
so every pass reads them from HBM.
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


def reference_eager(m, x, length):
    """The reference block in torch eager."""
    n, S, _ = x.shape
    h = [lin(x).view(n, S, 15, 20).transpose(1, 2) for lin in (m.W_Q, m.W_K, m.W_V)]
    e = torch.exp(h[0] @ h[1].transpose(-1, -2) / np.sqrt(20.0))
    if length is not None:
        e = e * (torch.arange(S, device=x.device).view(1, 1, 1, S) < length.view(n, 1, 1, 1)).float()
    attn = e / (e.sum(-1, keepdim=True) + 1e-8)
    return (attn @ h[2]).transpose(1, 2).reshape(n, S, 300)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mhsa_train_bench_b200.json"))
    ap.add_argument("--min-s", type=float, default=0.3)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--profile", action="store_true")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    m = MultiHeadSelfAttention(300, 15).to(dev)
    res = {"gpu_info": gpu_info(), "n_seq": N_SEQ, "windows": args.windows, "min_window_s": args.min_s, "cases": []}
    for S in (20, 50):
        gen = torch.Generator(device=dev).manual_seed(S)
        x = torch.randn((N_SEQ, S, 300), device=dev, generator=gen).requires_grad_(True)
        G = torch.randn((N_SEQ, S, 300), device=dev, generator=gen)
        rand_len = torch.randint(1, S + 1, (N_SEQ,), device=dev, generator=gen, dtype=torch.int32)
        for precision in ("tf32", "fp32"):
            m.precision = precision
            torch.backends.cuda.matmul.allow_tf32 = precision == "tf32"
            for mask in ("none", "random"):
                length = None if mask == "none" else rand_len

                def ours():
                    x.grad = None
                    for p in m.parameters():
                        p.grad = None
                    m(x, length=length).backward(G)

                def eager():
                    x.grad = None
                    for p in m.parameters():
                        p.grad = None
                    reference_eager(m, x, length).backward(G)

                a, b = [], []
                for _ in range(args.windows):            # alternated, so that both see the same clocks
                    a.append(timed(ours, args.min_s))
                    b.append(timed(eager, args.min_s))
                case = {"S": S, "precision": precision, "mask": mask, "ms_b200": statistics.median(a),
                        "ms_torch_eager": statistics.median(b), "ms_b200_windows": a, "ms_torch_eager_windows": b}
                case["speedup"] = case["ms_torch_eager"] / case["ms_b200"]
                print(json.dumps(case), flush=True)
                res["cases"].append(case)
    torch.backends.cuda.matmul.allow_tf32 = False
    if args.profile:
        from torch.profiler import profile, ProfilerActivity
        m.precision = "tf32"
        res["profile_tf32"] = {}
        for S in (20, 50):
            gen = torch.Generator(device=dev).manual_seed(S)
            x = torch.randn((N_SEQ, S, 300), device=dev, generator=gen).requires_grad_(True)
            G = torch.randn((N_SEQ, S, 300), device=dev, generator=gen)
            rand_len = torch.randint(1, S + 1, (N_SEQ,), device=dev, generator=gen, dtype=torch.int32)
            for mask, length in (("none", None), ("random", rand_len)):
                for _ in range(3):
                    m(x, length=length).backward(G)
                torch.cuda.synchronize()
                reps = 10
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(reps):
                        m(x, length=length).backward(G)
                    torch.cuda.synchronize()
                split = {}
                for e in prof.key_averages():
                    t = getattr(e, "device_time_total", None)
                    if t is None:
                        t = e.cuda_time_total
                    if t > 0:
                        split[e.key[:120]] = round(t / reps, 1)
                split = dict(sorted(split.items(), key=lambda kv: -kv[1]))
                res["profile_tf32"][f"S{S}_{mask}"] = {"us_per_iteration": split}
                print(f"S={S} mask={mask}:", json.dumps(split), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
