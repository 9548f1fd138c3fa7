"""Device-resident evaluate pipeline (reference src/evaluate.py:171-272).

The reference walks Python dicts of GPU row views, stacks 102,400 tensors per user batch and
launches one bmm + .tolist() per impression.  Here the same semantics run on integer tables:

  stage A  news table  [N_news+1, 300]; last row = PADDED_NEWS zeros (evaluate.py:203-204);
           duplicate news ids resolve to their FIRST row (evaluate.py:197-201)
  stage B  user vectors from int32 history rows [I, S] (first S = num_clicked_news_a_user clicks, LEFT padded,
           evaluate.py:111-124), gathered inside the library
  stage C  CSR scoring (evaluate.py:245-260), `max_count` keeps the reference's off-by-one
           (:247-249 processes max_count-1 impressions)
  stage D  AUC / MRR / nDCG@5 / nDCG@10 per impression on the GPU + nanmean (:160-168,267-272)

With torch.distributed initialised (one process per GPU) the news rows and the impressions are
split into contiguous blocks per rank; the table is all-gathered (NCCL) and the eight metric
sums/counts are all-reduced.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops


def first_occurrence_rows(news_ids) -> np.ndarray:
    """owner[i] = first row whose id equals news_ids[i]  (evaluate.py:197-201 'if id not in')."""
    ids = np.asarray(news_ids)
    _, first_idx, inverse = np.unique(ids, return_index=True, return_inverse=True)
    return first_idx[inverse].astype(np.int64)


def build_history(clicked_rows_list, num_clicked=50, pad_row=-1) -> np.ndarray:
    """UserDataset.__getitem__ (evaluate.py:111-124): FIRST `num_clicked` clicks, LEFT padded."""
    out = np.full((len(clicked_rows_list), num_clicked), pad_row, dtype=np.int64)
    for i, h in enumerate(clicked_rows_list):
        h = list(h)[:num_clicked]
        if h:
            out[i, num_clicked - len(h):] = h
    return out


def _dist(distributed=True):
    """torch.distributed when it is initialised with more than one rank (and the caller wants it), else None."""
    import torch.distributed as dist
    if distributed and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist
    return None


# PADDED_NEWS is ONE vector in the reference (evaluate.py:203-204) and half of all history entries point at it (history
# lengths are uniform in 0..50).  As one table row it was an L2 hot spot for the row-gathering attention kernel: 1.8 M of the
# 3.7 M gathered rows of an evaluate pass hit the same 2,160 bytes, and the launch time moved between 417 and 762 us with
# the impression block (profiles/block_probe.py).  The table therefore carries PAD_REPLICAS identical zero rows and the pad
# references are spread over them on the host -- the same arithmetic (bit-identical user vectors), 488 / 564 -> 417 us.
PAD_REPLICAS = 64


def spread_pad_rows(hist: np.ndarray, n_news: int) -> None:
    """In place: history entries < 0 (PADDED_NEWS) -> n_news + r, r in [0, PAD_REPLICAS) by position."""
    pad = hist < 0
    idx = np.flatnonzero(pad.ravel())
    hist.ravel()[idx] = n_news + (idx * 7 + idx // hist.shape[-1]) % PAD_REPLICAS


def shard_range(n, rank, world):
    """Contiguous block [lo, hi) of rank `rank` (blocks of ceil(n/world))."""
    per = (n + world - 1) // world
    lo = min(rank * per, n)
    return lo, min(lo + per, n)


def shard_impressions_by_candidates(cand_offsets: np.ndarray, world: int):
    """Impression block boundaries [world+1] balancing the number of CANDIDATES per rank."""
    total = int(cand_offsets[-1])
    targets = (np.arange(1, world) * total) // world
    cuts = np.searchsorted(cand_offsets, targets, side="left")
    return np.concatenate([[0], cuts, [len(cand_offsets) - 1]]).astype(np.int64)


class EvalHost:
    """Evaluate inputs preprocessed on the host into the library's index formats, in pinned
    memory (when CUDA is available) so `EvalInputs.from_host` is a handful of async H2D copies.

    news_tokens  int64 [N_news, L]        hist_rows  int32 [I, S]   (pad -> N_news, the zero row)
    cand_rows    int32 [sumC]             cand_offsets int64 [I+1]   labels int8 [sumC]
    """

    def __init__(self, news_tokens, hist_rows, cand_offsets, cand_rows, labels, news_ids=None, num_words=None):
        n_news = int(news_tokens.shape[0])
        hist = np.asarray(hist_rows, dtype=np.int64).copy()
        cand = np.asarray(cand_rows, dtype=np.int64)
        if news_ids is not None:          # first occurrence wins
            owner = first_occurrence_rows(news_ids)
            valid = hist >= 0
            hist[valid] = owner[hist[valid]]
            cand = owner[cand]
        # the reference raises on an unknown id (KeyError in news2vector[...], evaluate.py:221,252; IndexError inside
        # nn.Embedding); the device kernels would clamp silently, so the ranges are checked here, once, on the host
        if hist.size and int(hist.max()) >= n_news:
            raise IndexError(f"history row {int(hist.max())} out of range for {n_news} news")
        if cand.size and (int(cand.min()) < 0 or int(cand.max()) >= n_news):
            raise IndexError(f"candidate rows must lie in [0, {n_news}), got [{int(cand.min())}, {int(cand.max())}]")
        tok = np.asarray(news_tokens)
        if num_words is not None and tok.size and (int(tok.min()) < 0 or int(tok.max()) >= int(num_words)):
            raise IndexError(f"token ids must lie in [0, {int(num_words)}), got [{int(tok.min())}, {int(tok.max())}]")
        spread_pad_rows(hist, n_news)     # PADDED_NEWS -> one of the PAD_REPLICAS all-zero rows that close the table
        self.n_news = n_news
        self.n_impressions = int(hist.shape[0])
        pin = torch.cuda.is_available()

        def t(a, dt):
            x = torch.as_tensor(np.ascontiguousarray(a), dtype=dt)
            return x.pin_memory() if pin else x
        # token ids travel as int32 when the vocabulary allows it (always, in practice): half the bytes of the reference's
        # LongTensor over PCIe; the tensor-mode news encoder reads them directly, every other path widens them on the device
        self.news_tokens = t(news_tokens, torch.int32 if (tok.size == 0 or int(tok.max()) < 2 ** 31) else torch.int64)
        self.hist_rows = t(hist, torch.int32)
        self.cand_rows = t(cand, torch.int32)
        self.cand_offsets = t(cand_offsets, torch.int64)
        self.labels = t(labels, torch.int8)
        self.cand_offsets_host = np.asarray(cand_offsets, dtype=np.int64)

    def nbytes(self):
        return sum(x.numel() * x.element_size() for x in
                   (self.news_tokens, self.hist_rows, self.cand_rows, self.cand_offsets, self.labels))


class EvalInputs:
    """Evaluate inputs resident on one device (the timed pipeline touches only these)."""

    def __init__(self, news_tokens, hist_rows, cand_offsets, cand_rows, labels, news_ids=None, device="cuda"):
        self._fill(EvalHost(news_tokens, hist_rows, cand_offsets, cand_rows, labels, news_ids), device)

    @classmethod
    def from_host(cls, host: EvalHost, device="cuda", shard=True, distributed=True):
        """`shard` (multi-rank only): copy just this rank's block of impressions (the block evaluate_tensors assigns it
        when `max_count` is None) instead of all of them -- the host-to-device traffic per rank stays constant as ranks
        are added."""
        self = cls.__new__(cls)
        self._fill(host, device, shard, distributed)
        return self

    def _fill(self, host, device, shard=False, distributed=True):
        self.device = torch.device(device)
        self.n_news, self.n_impressions = host.n_news, host.n_impressions
        self.cand_offsets_host = host.cand_offsets_host
        self._ready = None
        self.shard = None                # (lo, hi, c0, c1): the tensors below hold only impressions [lo, hi)
        dist = _dist(distributed)
        views = dict(hist_rows=host.hist_rows, cand_rows=host.cand_rows, cand_offsets=host.cand_offsets, labels=host.labels)
        if shard and dist is not None:
            bounds = shard_impressions_by_candidates(host.cand_offsets_host, dist.get_world_size())
            lo, hi = int(bounds[dist.get_rank()]), int(bounds[dist.get_rank() + 1])
            c0, c1 = int(host.cand_offsets_host[lo]), int(host.cand_offsets_host[hi])
            self.shard = (lo, hi, c0, c1)
            views = dict(hist_rows=host.hist_rows[lo:hi], cand_rows=host.cand_rows[c0:c1],
                         cand_offsets=host.cand_offsets[lo:hi + 1], labels=host.labels[c0:c1])
        tokens = host.news_tokens
        self.news_shard = None           # (lo, hi): news_tokens holds only the rows this rank encodes
        if shard and dist is not None:
            self.news_shard = shard_range(host.n_news, dist.get_rank(), dist.get_world_size())
            tokens = tokens[self.news_shard[0]:self.news_shard[1]]
        self.h2d_bytes = tokens.numel() * tokens.element_size() + sum(v.numel() * v.element_size() for v in views.values())
        if self.device.type != "cuda":
            self.news_tokens = tokens.to(self.device)
            for name, v in views.items():
                setattr(self, name, v.to(self.device))
            return
        # The news stage needs only the token table: it goes first on the caller's stream; the impression tables
        # follow on a copy stream and overlap the news encoders (evaluate_tensors waits on the event before stage B).
        main = torch.cuda.current_stream(self.device)
        self.news_tokens = tokens.to(self.device, non_blocking=True)
        side = _copy_stream(self.device)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            for name, v in views.items():
                t = v.to(self.device, non_blocking=True)
                t.record_stream(main)
                setattr(self, name, t)
            self._ready = torch.cuda.Event()
            self._ready.record(side)

    def wait_ready(self):
        """Make the caller's stream wait for the impression tables (no host sync)."""
        if self._ready is not None:
            torch.cuda.current_stream(self.device).wait_event(self._ready)
            self._ready = None


_copy_streams = {}


def _copy_stream(device):
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    if key not in _copy_streams:
        _copy_streams[key] = torch.cuda.Stream(device=device)
    return _copy_streams[key]


@torch.no_grad()
def encode_news_table(model, news_tokens: torch.Tensor, n_news=None, local_shard=None, distributed=True) -> torch.Tensor:
    """Stage A.  Returns [N_news+1, 300] with a zero last row.  Multi-rank: each rank encodes its
    contiguous row block straight into its slot of the (padded) table, then one all_gather."""
    dist = _dist(distributed)
    n = news_tokens.shape[0] if n_news is None else int(n_news)      # `local_shard`: news_tokens = rows [lo, hi) only
    dev = news_tokens.device
    was_training = model.training
    model.eval()
    try:
        if dist is None:
            table = torch.empty((n + PAD_REPLICAS, ops.D), dtype=torch.float32, device=dev)
            table[:n] = model.get_news_vector({"title": news_tokens})
            table[n:].zero_()
            return table
        world, rank = dist.get_world_size(), dist.get_rank()
        per = (n + world - 1) // world
        padded = torch.zeros((max(world * per, n + PAD_REPLICAS), ops.D), dtype=torch.float32, device=dev)
        lo, hi = shard_range(n, rank, world)
        # One encoder call per shard (the table path of the news encoder projects the embedding table once per CALL, and
        # needs >= 8 token rows per vocabulary row to be selected: splitting the shard to overlap the exchange with the
        # encoding cost more than the exchange itself -- measured at 2 GPUs: news 1.97 ms in three pieces), then one
        # all-gather of equal padded slots.
        if local_shard is not None and tuple(local_shard) != (lo, hi):
            raise RuntimeError(f"token rows were sharded for {tuple(local_shard)} but this rank encodes {(lo, hi)}")
        if hi > lo:
            padded[lo:hi] = model.get_news_vector({"title": news_tokens if local_shard is not None else news_tokens[lo:hi]})
        dist.all_gather_into_tensor(padded[:world * per].view(-1), padded[rank * per:(rank + 1) * per].reshape(-1).clone())
        table = padded[:n + PAD_REPLICAS]
        table[n:].zero_()
        return table
    finally:
        model.train(was_training)


@torch.no_grad()
def encode_news_table16(model, news_tokens: torch.Tensor, n_news=None, local_shard=None, want_fp32=False, distributed=True,
                        mark=None):
    """Stage A of the tensor-mode pipeline.  Returns (table16, table32): table16 = fp16 [N_news + PAD_REPLICAS + 1, 320] in
    `ops.pack_rows_f16`'s layout -- rows N_news .. N_news + PAD_REPLICAS - 1 are the PADDED_NEWS zero vector (evaluate.py:203-204; zeros with the 1.0 of the bias
    column), the row after it the all-zero closing row the kernels expect -- and table32 = the fp32 [N_news + 1, 300] table when `want_fp32`, else None.

    Nothing downstream of the news encoder reads fp32 rows in tensor mode: the user encoder projects the fp16 copy and the
    scoring kernel reads it, so the copy is made ONCE, by the rank that encoded the rows, straight into its slot of the
    gather buffer, and the NCCL all-gather moves 640-byte rows in place (no staging copy, half the bytes of fp32)."""
    dist = _dist(distributed)
    n = news_tokens.shape[0] if n_news is None else int(n_news)
    dev = news_tokens.device
    was_training = model.training
    model.eval()
    try:
        world, rank = (dist.get_world_size(), dist.get_rank()) if dist is not None else (1, 0)
        per = (n + world - 1) // world
        buf = torch.empty((max(world * per, n + PAD_REPLICAS) + 1, 320), dtype=torch.float16, device=dev)
        lo, hi = shard_range(n, rank, world)
        if local_shard is not None and tuple(local_shard) != (lo, hi):
            raise RuntimeError(f"token rows were sharded for {tuple(local_shard)} but this rank encodes {(lo, hi)}")
        vec = None
        if hi > lo:
            vec = model.get_news_vector({"title": news_tokens if (local_shard is not None or dist is None) else news_tokens[lo:hi]})
            ops.pack_rows_f16(vec, out=buf[lo:hi + 1])          # rows [lo, hi) + a zero row at hi
        if mark is not None:
            mark("news_encode")
        if dist is not None:
            if buf.is_cuda:       # NCCL gathers in place: every rank's slot already sits at rank * per
                dist.all_gather_into_tensor(buf[:world * per].view(-1), buf[rank * per:(rank + 1) * per].view(-1))
            else:                 # gloo (CPU tests of the plumbing)
                dist.all_gather_into_tensor(buf[:world * per].view(-1), buf[rank * per:(rank + 1) * per].reshape(-1).clone())
        buf[n:].zero_()           # the PADDED_NEWS rows, the closing row and the slot padding
        buf[n:n + PAD_REPLICAS, 300] = 1.0    # ... PADDED_NEWS is a zero VECTOR that still meets the biases (q = 0 W + b): its 1.0 column stays
        table32 = None
        if want_fp32:
            if dist is None:
                table32 = torch.zeros((n + 1, ops.D), dtype=torch.float32, device=dev)
                table32[:n] = vec
            else:
                padded = torch.zeros((world * per + 1, ops.D), dtype=torch.float32, device=dev)
                if hi > lo:
                    padded[lo:hi] = vec
                dist.all_gather_into_tensor(padded[:world * per].view(-1), padded[rank * per:(rank + 1) * per].reshape(-1).clone())
                table32 = padded[:n + 1]
                table32[n].zero_()
        return buf[:n + PAD_REPLICAS + 1], table32
    finally:
        model.train(was_training)


def _tensor_mode(model):
    from . import _lib
    from .config import resolve_mode
    ue = model.user_encoder
    return resolve_mode(ue.config, ue.precision) == _lib.MODE_TF32


@torch.no_grad()
def evaluate_tensors(model, inputs: EvalInputs, max_count=None, return_details=False, mark=None, distributed=True):
    """evaluate() on resident tensors -> (AUC, MRR, nDCG@5, nDCG@10) as Python floats.

    One D2H read (the 8 sums/counts) at the very end; no per-impression host work.
    `mark(name)` (optional) is called at stage boundaries (bench.py records CUDA events there).
    `distributed=False` evaluates everything on this rank even when torch.distributed is initialised (bench.py uses it
    to check that N ranks and one rank give the same metric means)."""
    dist = _dist(distributed)
    mark = mark or (lambda name: None)
    mark("start")
    # tensor mode (plain NRMS): one fp16 copy of the news vectors feeds the all-gather, the user encoder and the scoring
    f16_flow = _tensor_mode(model) and model.user_encoder.layer_norm is None
    table16 = None
    if f16_flow:
        table16, table = encode_news_table16(model, inputs.news_tokens, inputs.n_news, getattr(inputs, "news_shard", None),
                                             want_fp32=return_details, distributed=distributed, mark=mark)
    else:
        table = encode_news_table(model, inputs.news_tokens, inputs.n_news, getattr(inputs, "news_shard", None),
                                  distributed=distributed)
    mark("news")
    inputs.wait_ready()
    n_imp = inputs.n_impressions
    if max_count is not None:
        n_imp = max(0, min(n_imp, int(max_count) - 1))
    lo, hi = 0, n_imp
    if dist is not None:
        bounds = shard_impressions_by_candidates(inputs.cand_offsets_host[:n_imp + 1], dist.get_world_size())
        lo, hi = int(bounds[dist.get_rank()]), int(bounds[dist.get_rank() + 1])
    dev = inputs.device
    if hi > lo:
        c0, c1 = int(inputs.cand_offsets_host[lo]), int(inputs.cand_offsets_host[hi])
        shard = getattr(inputs, "shard", None)
        if shard is not None:            # the inputs hold only this rank's block: index relative to it
            if (lo, hi) != shard[:2]:
                raise RuntimeError(f"inputs were sharded for impressions {shard[:2]} but this call needs {(lo, hi)} "
                                   "(max_count or a different world size): build them with from_host(..., shard=False)")
            hist = inputs.hist_rows
            cand_rows, labels, offs = inputs.cand_rows, inputs.labels, (inputs.cand_offsets - c0).contiguous()
        else:
            hist = inputs.hist_rows[lo:hi]
            cand_rows, labels = inputs.cand_rows[c0:c1], inputs.labels[c0:c1]
            offs = (inputs.cand_offsets[lo:hi + 1] - c0).contiguous()
        user_vec = model.user_encoder.forward_indexed(table16 if f16_flow else table, hist)
        mark("users")
        if f16_flow:
            scores = ops.score_csr_f16(table16, cand_rows, offs, user_vec)
        elif _tensor_mode(model):
            # tensor mode (LayerNorm variant): candidates are read from an fp16 copy of the table
            scores = ops.score_csr_f16(ops.pack_rows_f16(table), cand_rows, offs, user_vec)
        else:
            scores = ops.score_csr(table, cand_rows, offs, user_vec)
        mark("score")
        per, sums = ops.rank_metrics(scores, labels, offs)
        mark("metrics")
    else:
        user_vec = torch.empty((0, ops.D), device=dev)
        scores = torch.empty((0,), device=dev)
        per = torch.empty((0, 4), dtype=torch.float64, device=dev)
        sums = torch.zeros((8,), dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(sums)
    s = sums.cpu().numpy()
    with np.errstate(all="ignore"):
        means = tuple(float(x) for x in (s[:4] / s[4:]))
    if return_details:
        return means, dict(table=table, user_vectors=user_vec, scores=scores, per_impression=per,
                           impression_range=(lo, hi))
    return means


def evaluate(model, directory, num_workers=0, max_count=None):
    """The reference's entry point (src/evaluate.py:171-272), same signature and return value: evaluate `model` on
    `directory` (which holds `behaviors.tsv` and `news_parsed.tsv`) -> (AUC, MRR, nDCG@5, nDCG@10).  The files are read once
    into integer tables (`data.py`); everything after that is the device-resident pipeline above.  `num_workers` (the
    reference's metric process pool) is accepted and unused: the metrics run on the GPU.  `max_count` as in the reference
    (`sys.maxsize` or None = all impressions)."""
    import os
    import sys
    from . import data
    news = data.load_news_parsed(os.path.join(directory, "news_parsed.tsv"))
    # the history length the model was built for (a model without a config: the reference's default, 50)
    num_clicked = int(getattr(getattr(model, "config", None), "num_clicked_news_a_user", 50))
    ev = data.load_behaviors(os.path.join(directory, "behaviors.tsv"), news, num_clicked=num_clicked)
    device = next(model.parameters()).device if hasattr(model, "parameters") else "cpu"
    inputs = EvalInputs(news.title, ev.hist_rows, ev.cand_offsets, ev.cand_rows, ev.labels, news_ids=news.ids, device=device)
    if max_count is not None and max_count >= sys.maxsize:
        max_count = None
    return evaluate_tensors(model, inputs, max_count=max_count)

