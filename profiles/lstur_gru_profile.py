"""torch.profiler run of the tensor-mode GRU forward + backward at B = 128, T = 50 (random lengths, the workload of
profiles/lstur_bench.py), in a run of its own: per-kernel device time and launch counts of one call, and the call's
wall time, written to the path given as argv[1] (default profiles/lstur_gru_profile_b200.txt)."""
import os
import sys

import numpy as np
import torch
import torch.nn as nn
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from newsrecommendationsystem_b200 import ops, _lib  # noqa: E402


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "lstur_gru_profile_b200.txt")
    dev = torch.device("cuda")
    lines = [torch.cuda.get_device_name()]
    lengths = torch.from_numpy(np.random.default_rng(0).integers(1, 51, size=128))
    for method, H in (("ini", 900), ("con", 450)):
        gru = nn.GRU(900, H).to(dev)
        w = [p.detach().clone().requires_grad_(True) for p in gru.parameters()]
        x = torch.randn(128, 50, 900, device=dev, requires_grad=True)
        h0 = torch.randn(128, H, device=dev, requires_grad=True) if method == "ini" else None
        g = torch.randn(128, H, device=dev)

        def call():
            ops.gru(x, lengths, h0, *w, mode=_lib.MODE_TF32).backward(g)
        for _ in range(5):
            call()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for _ in range(10):
                call()
            torch.cuda.synchronize()
        lines.append(f"\n== {method} (H = {H}), 10 calls, sum(lengths) = {int(lengths.sum())} ==")
        lines.append(prof.key_averages().table(sort_by="cuda_time_total", row_limit=20, max_name_column_width=60))
    with open(out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
