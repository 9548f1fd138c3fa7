#!/usr/bin/env python
"""bench.py -- NRMS hot-path benchmark on B200 (contract: see task brief / DESIGN.md section 5).

A "step" is ONE full evaluate pass (BASELINE.json configs[1]) over synthetic MIND-small-shaped data
per GPU: encode all 65,238 news, user vectors for 73,152 impressions, score every candidate, rank
metrics (AUC/MRR/nDCG@5/@10).  Weak scaling: every rank owns one MIND-small-shaped shard (N x news,
N x impressions in total); the news-vector table is all-gathered over NCCL, metric sums all-reduced.

The same JSON line also carries, at every N:
  mind_large  BASELINE configs[3]: the MIND-large-shaped evaluate (161,013 news / 376,471 impressions IN TOTAL) sharded
              over the N GPUs -- the strong-scaling curve of the north star;
  train       BASELINE configs[2]: training step, batch 128 per GPU, 1 + 4 candidates, Adam;
  train_ln    BASELINE configs[4]: the +LN +AdamW +cosine variant, data parallel;
  metrics_1rank / metrics_match_1rank (N > 1): rank 0 re-evaluates the whole workload alone, outside every timed region.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--precision tf32|fp32] [--impl reference] [--dump-outputs DIR]

Every timed loop (the headline evaluate, its end-to-end variant, the MIND-large and training side measurements) times
exactly K steps.  Prints ONE JSON line on rank 0.  `--impl reference` times the CPU restatement of the reference's
path (oracle/torch_port.py, PyTorch-CPU on all host cores) on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

# torch reads this when its CUDA allocator starts: VMM-mapped (2 MB page) segments, see _lib._prefer_large_page_segments
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NEWS_PER_GPU = 65238
IMPRESSIONS_PER_GPU = 73152
NUM_WORDS = 70976
MIND_LARGE = (161013, 376471)      # BASELINE configs[3]: news, impressions (strong scaling: fixed total)
# ---- algorithmic work per unit: SURVEY.md 8(d) (the figures `roofline.achieved` is computed from) ----
FLOP_PER_TITLE = 13_700_000
FLOP_PER_USER = 36_050_000
BYTES_PER_TITLE = 25_360           # 20 embedding rows x 1,200 B + 20 int64 ids + 1,200 B out
BYTES_PER_USER = 61_600            # 50 news vectors x 1,200 B + 50 x 8 B ids + 1,200 B out
BYTES_PER_CANDIDATE = 1212         # fp32 news vector + int64 index + fp32 score
BYTES_PER_IMPRESSION = 1208        # user vector + index
TRAIN_FLOP_PER_STEP = 303e9        # B = 128, K = 4: forward + backward ~ 3 x 101.1 GFLOP
ADAM_BYTES_PER_STEP = 7 * 21_955_400 * 4
# ---- bytes the kernels of THIS design move per unit (kept beside the 8(d) figure as frac_design_bytes) ----
K1G_BYTES_PER_USER = 50 * 2160 + 50 * 4 + 50 * 640        # gathered q|k|v rows (fp16, padded) + int32 rows + fp16 context rows out
K1G_BYTES_PER_TITLE = 20 * 2160 + 20 * 8 + 20 * 640
SCORE_BYTES_PER_CANDIDATE_F16 = 652                       # tensor mode: 640-byte fp16 row + int32 index + score


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained"),
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass
        # wait for the first sample: nvidia-smi takes ~1 s to initialise NVML (on every GPU of the box), and that
        # initialisation stalls kernel launches of ALL ranks -- started right in front of the timed loop it cost the
        # 8-GPU line 0.6 ms per step on the ranks that waited for rank 0 (e2e, timed later, was faster than resident)
        t0 = time.time()
        while self.p is not None and time.time() - t0 < 5.0:
            if os.path.getsize(self.f.name) > 0:
                break
            time.sleep(0.05)

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, pw, reasons = [], [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(min(sm)), "sm_max_mhz": float(max(mx)),
                "power_w_max": float(max(pw)), "reasons": sorted(reasons), "samples": len(sm)}


def workload_sizes(world, workload="small-per-gpu"):
    """(news, impressions) in total over all ranks."""
    if workload == "mind-large":
        return MIND_LARGE
    return NEWS_PER_GPU * world, IMPRESSIONS_PER_GPU * world


def make_data(world, workload="small-per-gpu"):
    from newsrecommendationsystem_b200 import synthetic
    n_news, n_imp = workload_sizes(world, workload)
    news = synthetic.make_news(n_news, num_words=NUM_WORDS, seed=1234)
    imp = synthetic.make_impressions(n_imp, n_news, seed=1234)
    return news, imp


# --------------------------------------------------------------------------------------------------
# CPU baseline: the torch-CPU port of the reference path on a bounded sample of the SAME workload
# --------------------------------------------------------------------------------------------------
def cpu_baseline(news, imp, n_users=4096, n_score=6000, train=True):
    """The reference's CPU path (oracle/torch_port.py: PyTorch-CPU, the reference's own arithmetic library and op
    order, all host cores) on a bounded sample of the MIND-small-shaped workload:
      news   get_news_vector over the WHOLE 65,238-title corpus in 2,048-title batches (evaluate.py:187) -- timed in full,
             and it gives the real news-vector table the next two legs read;
      users  get_user_vector for the first `n_users` impressions in 2,048-user batches gathered from that table by tensor
             indexing (the reference's dict / torch.stack loop, evaluate.py:220-224, is slower);
      score  get_prediction + .tolist() + calculate_single_user_metric per impression for the first `n_score`
             impressions (evaluate.py:245-265, :160-168);
      train  ONE step of the reference's training loop (train.py:202-233) at B = 128, K = 4.
    users and score are extrapolated to the 73,152 impressions; news is measured whole."""
    import torch
    from newsrecommendationsystem_b200 import synthetic
    from oracle import nrms_oracle as O
    from oracle import torch_port as TP
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = synthetic.init_state_dict(num_words=NUM_WORDS, seed=0)
    n_news, n_imp = NEWS_PER_GPU, IMPRESSIONS_PER_GPU
    news, hist_all = news[:n_news], imp["hist_rows"]
    TP.news_vectors(sd, news[:256])     # warm-up
    table = torch.zeros((n_news + 1, 300), dtype=torch.float32)
    t0 = time.perf_counter()
    for s in range(0, n_news, 2048):
        table[s:min(s + 2048, n_news)] = TP.news_vectors(sd, news[s:s + 2048])
    t_news_total = time.perf_counter() - t0
    hist = torch.from_numpy(np.where(hist_all[:n_users] < 0, n_news, hist_all[:n_users] % n_news))
    TP.user_vectors(sd, table[hist[:64]])
    t0 = time.perf_counter()
    uvs = []
    for s in range(0, n_users, 2048):
        uvs.append(TP.user_vectors(sd, table[hist[s:s + 2048]]))
    t_user = (time.perf_counter() - t0) / n_users
    uv = torch.cat(uvs)
    offs = imp["cand_offsets"]
    cand = torch.from_numpy(imp["cand_rows"][:int(offs[n_score])] % n_news)
    t0 = time.perf_counter()
    for i in range(n_score):
        a, b = int(offs[i]), int(offs[i + 1])
        y_pred = TP.prediction(table[cand[a:b]], uv[i % n_users])
        O.single_user_metric(imp["labels"][a:b], y_pred)
    t_score = (time.perf_counter() - t0) / n_score
    total = t_news_total + n_imp * t_user + n_imp * t_score
    out = dict(value=n_imp / total, unit="impressions/s", cores=cores, kind="port",
               sample=f"torch-CPU port of the reference op sequence: all {n_news} titles encoded (measured whole), "
                      f"{n_users} users from the real {n_news + 1}-row table and {n_score} impressions scored+ranked "
                      f"(extrapolated to {n_imp} impressions)",
               news_per_s=n_news / t_news_total, users_per_s=1.0 / t_user, scored_impressions_per_s=1.0 / t_score)
    if train:
        c, k = synthetic.make_train_batch(128, news, k_neg=4, seed=1234)
        t0 = time.perf_counter()
        TP.train_step(sd, c, k)
        dt = time.perf_counter() - t0
        out["train_samples_per_s"] = 128 / dt
        out["train_sample"] = "one reference training step (forward, CE, backward, Adam over 21,955,400 parameters) at B = 128, K = 4"
    return out


def run_reference(args, rank):
    if rank != 0:
        return
    news, imp = make_data(1)
    vals = []
    last = None
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        last = cpu_baseline(news, imp, n_users=2048, n_score=3000, train=False)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            vals.append((last["value"], dt))
    v = float(np.mean([x[0] for x in vals]))
    line = dict(impl="reference", metric="evaluate impressions/s", value=v, unit="impressions/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, ms_per_step=1e3 * IMPRESSIONS_PER_GPU / v,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                # the same `config` as the B200 arm prints (it names the WORKLOAD; this arm's own arithmetic is `dtype` f32 and
                # `cpu_baseline.kind`): the driver compares the two dictionaries
                config=workload_config(args.gpus, args.precision),
                cpu_baseline=dict(value=v, unit="impressions/s", cores=last["cores"], kind="port", sample=last["sample"]),
                e2e=dict(value=v, unit="impressions/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                # a step is a BOUNDED SAMPLE of the workload: `value` is the sample's rate, `ms_per_step` the time a full pass
                # would take at that rate (extrapolated), `sample_wall_s_per_step` what a step really took here
                extrapolated=True, sample_wall_s_per_step=float(np.mean([x[1] for x in vals])))
    print(json.dumps(line), flush=True)


DUMP_BYTES_PER_ARRAY = 12 << 20


def dump_outputs(out_dir, means, det, n_news):
    """--dump-outputs: what the last timed evaluate step returned (the metric means) and computed on the way (per-impression
    metrics, candidate scores, user vectors, news vectors) as float .npy files.  An array larger than DUMP_BYTES_PER_ARRAY
    is cut to a fixed sample of its rows (np.random.default_rng(0), sorted), so equal arguments give equal rows.
    per_impression holds the impressions whose metrics are defined: one with a single label class has no AUC (NaN in the
    reference, left out of its nanmean), and it is left out here too, so every value written is finite."""
    import torch

    def sample(a):
        rows = DUMP_BYTES_PER_ARRAY // (a[0].numel() * a.element_size())
        if a.shape[0] > rows:
            idx = np.sort(np.random.default_rng(0).choice(a.shape[0], rows, replace=False))
            a = a[torch.from_numpy(idx).to(a.device)]
        return a.cpu().numpy()

    per = det["per_impression"]
    per = per[~torch.isnan(per).any(dim=1)]
    arrays = dict(metrics=np.asarray(means, dtype=np.float64), per_impression=sample(per),
                  scores=sample(det["scores"]), user_vectors=sample(det["user_vectors"]),
                  news_vectors=sample(det["table"][:n_news]))
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        if not np.isfinite(a).all():
            raise RuntimeError(f"--dump-outputs: {name} of the last timed step is not finite")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config(world, precision, workload="small-per-gpu"):
    n_news, n_imp = workload_sizes(world, workload)
    name = ("NRMS evaluate pipeline, MIND-large-shaped in total, sharded over the GPUs (BASELINE configs[3])"
            if workload == "mind-large" else "NRMS evaluate pipeline, MIND-small-shaped per GPU (BASELINE configs[1])")
    return dict(workload=name, news_per_gpu=n_news / world, impressions_per_gpu=n_imp / world, vocab=NUM_WORDS,
                title_len=20, history=50, heads=15, dim=300, precision=precision,
                parallelism=f"dp{world}: news rows + impressions sharded, NCCL all-gather of the fp16 news table",
                l2="flushed between timed steps (256 MiB write); per-step CUDA events summed")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of every timed loop")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default="tf32", choices=["tf32", "fp32"])
    ap.add_argument("--workload", default="small-per-gpu", choices=["small-per-gpu", "mind-large"],
                    help="headline workload: small-per-gpu (default, weak scaling: one MIND-small-shaped shard per GPU) or "
                         "mind-large (strong scaling: 161,013 news / 376,471 impressions in total, BASELINE configs[3])")
    ap.add_argument("--no-train", action="store_true", help="skip the train-step side measurements")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-large", action="store_true", help="skip the MIND-large side measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed evaluate step computed to DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 evaluate pass (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from newsrecommendationsystem_b200 import NRMS, NRMSConfig, NRMSLNConfig, synthetic, _lib
    from newsrecommendationsystem_b200.evaluate import EvalHost, EvalInputs, evaluate_tensors
    from newsrecommendationsystem_b200.train import TrainStep

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback in the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    peaks = load_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sd = synthetic.init_state_dict(num_words=NUM_WORDS, seed=0)
    model = NRMS(NRMSConfig)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    model.to(dev).eval().set_precision(args.precision)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    # ---------------------------------------------------------------------------------------------------
    # one evaluate workload: resident loop (`value`), end-to-end loop (`e2e`), 1-rank cross-check
    # ---------------------------------------------------------------------------------------------------
    def run_eval(workload, steps, warmup, sample_clocks, dump_dir=None):
        news, imp = make_data(world, workload)
        host = EvalHost(news, imp["hist_rows"], imp["cand_offsets"], imp["cand_rows"], imp["labels"])
        inputs = EvalInputs.from_host(host, dev)
        n_imp_total = host.n_impressions
        stage = {}
        h2d = [host.nbytes()]

        def timed_eval(resident, record_stages=False, details=False):
            marks = []

            def mark(name):
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                marks.append((name, ev))
            flush_buf.fill_(1)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            inp = resident if resident is not None else EvalInputs.from_host(host, dev)
            h2d[0] = inp.h2d_bytes
            # ends with the D2H of 8 doubles
            out = evaluate_tensors(model, inp, mark=mark if record_stages else None, return_details=details)
            e1.record()
            torch.cuda.synchronize()
            if record_stages:
                for (n0, a), (n1, b) in zip(marks[:-1], marks[1:]):
                    stage.setdefault(n1, []).append(a.elapsed_time(b))
                # what the marks do not cover: up to the first mark, and from the last one to the end of the step (the
                # 8-double all-reduce, where a rank waits for the slowest one, and the read-back of the means)
                stage.setdefault("pre", []).append(e0.elapsed_time(marks[0][1]))
                stage.setdefault("allreduce_readback", []).append(marks[-1][1].elapsed_time(e1))
            return e0.elapsed_time(e1), out

        # the attention launches are bracketed with CUDA events in BOTH loops (same instrumentation; the events are
        # created and pooled during the warm-up)
        lib.nrms_set_option(b"time_k1", 1)
        # the clock sampler is up and past its NVML initialisation BEFORE the warm-up; it samples through the warm-up, the
        # timed resident loop and the timed e2e loop
        sampler = ClockSampler(local_rank) if (rank == 0 and sample_clocks and not os.environ.get("NRMS_BENCH_NO_SAMPLER")) else None
        barrier()
        for _ in range(warmup):
            timed_eval(inputs)
        barrier()
        lib.nrms_set_option(b"time_k1", 1)
        l0 = lib.nrms_launch_count()
        times, means = [], None
        for i in range(steps):
            # the last step also returns the arrays it computed on the way; in tensor mode that costs one fp32 copy of the
            # news table, so it is asked for only when they are dumped
            ms, means = timed_eval(inputs, record_stages=True, details=dump_dir is not None and i == steps - 1)
            times.append(ms)
        launches = int(lib.nrms_launch_count() - l0)
        if dump_dir is not None:
            means, det = means
            if rank == 0:
                dump_outputs(dump_dir, means, det, host.n_news)
            del det
        kstat = {k: tuple(lib.nrms_get_stat(f"{k}_{w}".encode()) for w in ("ms", "launches", "sequences"))
                 for k in ("k1", "k1n", "k1g", "k1gn")}
        lib.nrms_set_option(b"time_k1", 1)      # clears the records, stays on
        barrier()
        e2e_times = []
        for i in range(steps + 1):
            ms, _ = timed_eval(None)
            if i > 0:
                e2e_times.append(ms)
        lib.nrms_set_option(b"time_k1", 0)
        clocks = sampler.stop() if sampler else None
        total_ms = max_over_ranks(float(np.sum(times)))
        e2e_ms = max_over_ranks(float(np.sum(e2e_times)))
        rank_stage = None
        if world > 1:       # every rank's own stage means: names the rank / stage the others wait for
            mine = {k: round(float(np.mean(v)), 4) for k, v in stage.items()}
            for kk, (kms, kn, _) in kstat.items():
                if kn > 0:
                    mine[f"{kk}_us_per_launch"] = round(1e3 * kms / kn, 1)
            rank_stage = [None] * world
            dist.all_gather_object(rank_stage, mine)
        res = dict(workload=workload, n_news=int(host.n_news), n_impressions=int(n_imp_total),
                   n_candidates=int(host.cand_offsets_host[-1]), ms_per_step=total_ms / steps,
                   value=n_imp_total * steps / (total_ms / 1e3), e2e_ms_per_step=e2e_ms / steps,
                   e2e_value=n_imp_total * steps / (e2e_ms / 1e3), h2d_bytes=int(h2d[0]),
                   stage_ms={k: float(np.mean(v)) for k, v in stage.items()}, stage_ms_per_rank=rank_stage,
                   metrics=dict(zip(("auc", "mrr", "ndcg5", "ndcg10"), means)), launches=launches, kstat=kstat, clocks=clocks)
        if world > 1:
            # N ranks == 1 rank: rank 0 evaluates the WHOLE workload alone (outside every timed region)
            barrier()
            if rank == 0:
                full = EvalInputs.from_host(host, dev, shard=False, distributed=False)
                m1 = evaluate_tensors(model, full, distributed=False)
                res["metrics_1rank"] = dict(zip(("auc", "mrr", "ndcg5", "ndcg10"), m1))
                res["metrics_match_1rank"] = float(max(abs(a - b) for a, b in zip(m1, means)))
                del full
            barrier()
        del inputs, host
        torch.cuda.empty_cache()
        return res

    head = run_eval(args.workload, args.steps, args.warmup, sample_clocks=True, dump_dir=args.dump_outputs)
    large = None
    if args.workload != "mind-large" and not args.no_large:
        large = run_eval("mind-large", args.steps, 3, sample_clocks=False)

    # ---------------------------------------------------------------------------------------------------
    # rooflines of the headline workload, from SURVEY 8(d)'s algorithmic bytes / flops
    # ---------------------------------------------------------------------------------------------------
    tr_path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    tr = json.load(open(tr_path)) if os.path.exists(tr_path) else {}
    st = head["stage_ms"]
    kstat = head["kstat"]
    n_news_rank = head["n_news"] / world
    n_imp_rank = head["n_impressions"] / world
    cand_rank = head["n_candidates"] / world

    def attn_roof(kind, name, alg_bytes, design_bytes, flop_per_seq, traffic_key):
        ms, n, seqs = kstat[kind]
        if not (n > 0 and ms > 0):
            return None
        us = 1e3 * ms / n
        per_launch = seqs / n
        ach = per_launch * alg_bytes / (us * 1e-6) / 1e9
        t = tr.get(traffic_key) or {}
        return dict(bound="hbm", kernel=name, achieved=ach, peak=peaks["hbm_gbs"], unit="GB/s", frac=ach / peaks["hbm_gbs"],
                    traffic=t.get("dram_bytes_per_launch"), traffic_sequences_per_launch=t.get("sequences_per_launch"),
                    us_per_launch=us, launches=int(n), sequences_per_launch=per_launch,
                    algorithmic_bytes_per_sequence=alg_bytes,
                    frac_design_bytes=per_launch * design_bytes / (us * 1e-6) / 1e9 / peaks["hbm_gbs"],
                    design_bytes_per_sequence=design_bytes,
                    tensor_frac_reference_flops=per_launch * flop_per_seq / (us * 1e-6) / 1e12 / peaks["bf16_tflops"],
                    peak_source=f"{peaks['source']} HBM copy bandwidth (burst); algorithmic bytes = SURVEY 8(d) (fp32 rows "
                                f"in, vector out); design bytes = what this kernel moves (fp16 q|k|v rows gathered from a "
                                f"partly L2-resident projected table + fp16 context rows out)")

    roof = attn_roof("k1g", "k1g::seq_attn_kernel<50,int,false> (user encoder: q|k|v row gather + 15-head attention; <..,true> when the score bound asks for the row-shifted softmax)",
                     BYTES_PER_USER, K1G_BYTES_PER_USER, FLOP_PER_USER, "seq_attn_kernel<50>")
    roof_news = attn_roof("k1gn", "k1g::seq_attn_kernel<20,int,true> (news encoder: q|k|v row gather + 15-head attention, row-shifted softmax)",
                          BYTES_PER_TITLE, K1G_BYTES_PER_TITLE, FLOP_PER_TITLE, "seq_attn_kernel<20>")

    def tensor_roof(kind, name, flop_per_seq):
        ms, n, seqs = kstat[kind]
        if not (n > 0 and ms > 0):
            return None
        us = 1e3 * ms / n
        ach = (seqs / n) * flop_per_seq / (us * 1e-6) / 1e12
        return dict(bound="tensor", kernel=name, achieved=ach, peak=peaks["bf16_tflops"], unit="TFLOP/s",
                    frac=ach / peaks["bf16_tflops"], traffic=None, us_per_launch=us, launches=int(n),
                    sequences_per_launch=seqs / n, algorithmic_flop_per_sequence=flop_per_seq,
                    peak_source=f"{peaks['source']} dense bf16/fp16 burst (operands are fp16, fp32 accumulate)")

    if roof is None:      # fp32-table runs / small calls: the per-sequence projection kernel, bound by the tensor pipe
        roof = tensor_roof("k1", "k1v6::encoder_attn_tc6_kernel<50,64,2> (user encoder: gather+QKV+attention)",
                           FLOP_PER_USER - 6_050_000)
    if roof_news is None:
        roof_news = tensor_roof("k1n", "k1v6::encoder_attn_tc6_kernel<20,24,5> (news encoder: gather+QKV+attention)",
                                FLOP_PER_TITLE - 2_420_000)
    if roof is None:
        dominant = max(st, key=st.get) if st else "users"
        roof = dict(bound="hbm", kernel=f"{dominant} stage (FP32 mode: CUDA-core kernels)", achieved=None, peak=peaks["hbm_gbs"],
                    unit="GB/s", frac=None, traffic=None, peak_source=peaks["source"])
    score_s = st.get("score", float("nan")) / 1e3
    score_alg = cand_rank * BYTES_PER_CANDIDATE + n_imp_rank * BYTES_PER_IMPRESSION
    score_moved = cand_rank * (SCORE_BYTES_PER_CANDIDATE_F16 if args.precision == "tf32" else BYTES_PER_CANDIDATE) \
        + n_imp_rank * BYTES_PER_IMPRESSION
    roof_score = dict(bound="hbm", kernel="score_csr_f16_kernel" if args.precision == "tf32" else "score_csr_kernel",
                      achieved=score_alg / score_s / 1e9, peak=peaks["hbm_gbs"], unit="GB/s",
                      frac=score_alg / score_s / 1e9 / peaks["hbm_gbs"], algorithmic_bytes_per_candidate=BYTES_PER_CANDIDATE,
                      bytes_moved_gbs=score_moved / score_s / 1e9,
                      note="timed as the whole scoring stage (one launch).  Tensor mode reads 640-byte fp16 rows of a 42 MB "
                           "table that stays in L2: bytes_moved_gbs is an L2 rate, not DRAM traffic; `achieved` counts "
                           "SURVEY 8(d)'s 1,212 B per candidate and can exceed the HBM peak for that reason",
                      traffic=(tr.get("score_csr_f16_kernel") or {}).get("dram_bytes_per_launch"))

    # ---------------------------------------------------------------------------------------------------
    # training step side measurements (BASELINE configs[2] and configs[4])
    # ---------------------------------------------------------------------------------------------------
    news_small = None

    def run_train(cfg, adamw, cosine, label):
        nonlocal news_small
        if news_small is None:
            news_small = synthetic.make_news(NEWS_PER_GPU, num_words=NUM_WORDS, seed=1234)
        sdl = dict(sd)
        m = NRMS(cfg)
        missing = {k: v for k, v in m.state_dict().items() if k not in sdl}     # LayerNorm affine of the variant
        m.load_state_dict({**{k: torch.from_numpy(v) for k, v in sdl.items()}, **missing})
        m.to(dev).train().set_precision(args.precision)
        n_train = args.steps
        ts = TrainStep(m, lr=1e-4, adamw=adamw, weight_decay=0.01 if adamw else 0.0,
                       cosine_total_steps=(n_train + 3) if cosine else None)
        cand, clicked = synthetic.make_train_batch(128, news_small, k_neg=4, seed=1234 + rank)
        titles = torch.from_numpy(np.concatenate([cand, clicked], axis=1)).pin_memory()
        for _ in range(3):
            ts.step_tokens(titles, 5)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        lib.nrms_set_option(b"time_k1", 0)
        l0 = lib.nrms_launch_count()
        e0.record()
        for _ in range(n_train):
            loss = ts.step_tokens(titles, 5)
        loss_val = float(loss.item())            # D2H of the loss, like train.py:225
        e1.record()
        torch.cuda.synchronize()
        tms = max_over_ranks(e0.elapsed_time(e1))
        step_ms = tms / n_train
        out = dict(config=label, samples_per_s=128 * world * n_train / (tms / 1e3), ms_per_step=step_ms, batch_per_gpu=128,
                   k_neg=4, dropout=0.2, loss=loss_val, forward_precision=args.precision, backward_precision=args.precision,
                   gpu_launches_per_step=int(lib.nrms_launch_count() - l0) // n_train,
                   h2d_bytes_per_step=int(titles.numel() * titles.element_size()),
                   roofline=dict(bound="tensor", achieved=TRAIN_FLOP_PER_STEP / (step_ms / 1e3) / 1e12, unit="TFLOP/s",
                                 peak=peaks["bf16_tflops"], frac=TRAIN_FLOP_PER_STEP / (step_ms / 1e3) / 1e12 / peaks["bf16_tflops"],
                                 tf32_peak_measured=tf32_peak, frac_of_tf32_peak=(TRAIN_FLOP_PER_STEP / (step_ms / 1e3) / 1e12 / tf32_peak)
                                 if tf32_peak else None,
                                 algorithmic_flop_per_step=TRAIN_FLOP_PER_STEP,
                                 adam_floor_us=ADAM_BYTES_PER_STEP / (peaks["hbm_gbs"] * 1e9) * 1e6,
                                 note="whole step (forward + CE + backward + Adam over 21,955,400 parameters + loss D2H) against "
                                      "SURVEY 8(d)'s 303 GFLOP; the dense-Adam stream of 614.8 MB alone costs adam_floor_us at the "
                                      "measured HBM peak"))
        del ts, m
        torch.cuda.empty_cache()
        return out

    tf32_peak = None
    train = train_ln = None
    if not args.no_train:
        train = run_train(NRMSConfig, adamw=False, cosine=False, label="NRMS + Adam (BASELINE configs[2])")
        train_ln = run_train(NRMSLNConfig, adamw=True, cosine=True,
                             label="NRMS +LN +AdamW +cosine decay, data parallel (BASELINE configs[4]; builder-defined variant)")
        # (after the training runs: the 8192^3 burst pulls the clocks down for the next measurement)
        # TF32 tensor peak, measured like MEASURED_PEAKS.json measures bf16 (cuBLAS 8192^3, best of 10, CUDA events)
        a = torch.randn(8192, 8192, device=dev)
        b = torch.randn(8192, 8192, device=dev)
        old_flag = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        best = 1e9
        for i in range(12):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize()
            if i >= 2:
                best = min(best, e0.elapsed_time(e1))
        torch.backends.cuda.matmul.allow_tf32 = old_flag
        tf32_peak = 2 * 8192 ** 3 / (best / 1e3) / 1e12
        del a, b
        for t in (train, train_ln):
            r = t["roofline"]
            r["tf32_peak_measured"] = tf32_peak
            r["frac_of_tf32_peak"] = r["achieved"] / tf32_peak

    # ---------------------------------------------------------------------------------------------------
    # single-user latency path (SURVEY 8 f4, reference src/recommend.py:245-341): side measurement, one GPU
    # ---------------------------------------------------------------------------------------------------
    latency = None
    if rank == 0 and world == 1 and not args.no_train:
        from newsrecommendationsystem_b200.recommend import Recommender
        from newsrecommendationsystem_b200 import ops
        rng = np.random.default_rng(77)
        n_rows = NEWS_PER_GPU + 1
        table = torch.randn(n_rows, 300, device=dev) * 0.4
        table[-1] = 0
        rec = Recommender(model, [f"N{i}" for i in range(n_rows - 1)], table)
        hist = rng.integers(0, n_rows, 50).astype(np.int32)
        latency = dict(what="user vector from 50 cached news vectors + scores of C candidates + ranking, one user per call "
                            "(nrms_recommend_user: two cluster launches, FP32)", n_table_rows=n_rows)
        for Cn in (37, 300):
            cand = rng.integers(0, n_rows, Cn).astype(np.int32)
            hist_d, cand_d = torch.from_numpy(hist).to(dev), torch.from_numpy(cand).to(dev)
            ue = model.user_encoder
            w = (*ue.multihead_self_attention.packed(), ue.additive_attention.linear.weight, ue.additive_attention.linear.bias,
                 ue.additive_attention.attention_query_vector)

            def call_dev():
                return ops.recommend_user(table, hist_d, cand_d, *w)

            def call_host():
                return rec.recommend_rows(hist, cand)[0].cpu()       # host indices in, ranked positions back on the host

            def timed(fn, n, wall):
                for _ in range(10):
                    fn()
                torch.cuda.synchronize()
                if wall:
                    t0 = time.perf_counter()
                    for _ in range(n):
                        fn()
                    torch.cuda.synchronize()
                    return (time.perf_counter() - t0) / n * 1e6
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(n):
                    fn()
                b.record()
                torch.cuda.synchronize()
                return a.elapsed_time(b) * 1e3 / n
            side = torch.cuda.Stream()
            with torch.cuda.stream(side):
                for _ in range(3):
                    call_dev()
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                call_dev()
            latency[f"C={Cn}"] = dict(device_us_graph_replay=timed(graph.replay, 200, False),
                                      call_us_device_indices=timed(call_dev, 200, False),
                                      e2e_us_host_indices_to_host_ranking=timed(call_host, 200, True))
        del rec, table
        torch.cuda.empty_cache()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        news, imp = make_data(1)
        cpu = cpu_baseline(news, imp, train=not args.no_train)

    if rank == 0:
        def eval_extra(r):
            out = dict(n_gpus=world, news=r["n_news"], impressions=r["n_impressions"], candidates=r["n_candidates"],
                       ms_per_step=r["ms_per_step"], value=r["value"], unit="impressions/s",
                       e2e=dict(value=r["e2e_value"], ms_per_step=r["e2e_ms_per_step"], h2d_bytes_per_step=r["h2d_bytes"]),
                       stage_ms=r["stage_ms"], stage_ms_per_rank=r.get("stage_ms_per_rank"), metrics=r["metrics"])
            for k in ("metrics_1rank", "metrics_match_1rank"):
                if k in r:
                    out[k] = r[k]
            return out
        line = dict(metric="evaluate impressions/s", value=head["value"], unit="impressions/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=head["ms_per_step"], higher_is_better=True,
                    scaling="strong" if args.workload == "mind-large" else "weak",
                    vs_baseline=None, dtype="f16xf16->f32 (tcgen05 kind::f16; TF32-equivalent 11-bit significand)"
                    if args.precision == "tf32" else "f32", data="synthetic",
                    config=workload_config(world, args.precision, args.workload), clocks=head["clocks"],
                    e2e=dict(value=head["e2e_value"], unit="impressions/s", h2d_bytes_per_step=head["h2d_bytes"],
                             d2h_bytes_per_step=64, ms_per_step=head["e2e_ms_per_step"]),
                    gpu_launches=head["launches"], roofline=roof, roofline_news=roof_news, roofline_score=roof_score,
                    cpu_baseline=cpu, train=train, train_ln=train_ln, recommend_latency=latency, stage_ms=st,
                    stage_ms_per_rank=head.get("stage_ms_per_rank"), metrics=head["metrics"],
                    stage_note="news_encode = this rank's titles (incl. the embedding-table projection) + the fp16 pack; news = "
                               "what follows it in the news stage: the NCCL all-gather of the fp16 table and the pad rows",
                    news_per_s=head["n_news"] / ((st.get("news", float("nan")) + st.get("news_encode", 0.0)) / 1e3),
                    users_per_s=head["n_impressions"] / (st.get("users", float("nan")) / 1e3),
                    score_candidates_per_s=head["n_candidates"] / (st.get("score", float("nan")) / 1e3),
                    mind_large=eval_extra(large) if large else None)
        for k in ("metrics_1rank", "metrics_match_1rank"):
            if k in head:
                line[k] = head[k]
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
