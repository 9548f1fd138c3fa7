"""One training iteration of the reference hot loop (src/train.py:202-206,227-233) on libnrms_b200.

    y_pred = model(candidate_news, clicked_news); loss = CrossEntropyLoss()(y_pred, zeros)
    optimizer.zero_grad(); loss.backward(); optimizer.step()

`TrainStep` keeps that exact order.  Data parallel (one process per GPU, torch.distributed/NCCL):
each rank runs its own batch of 128, the flat gradient is all-reduced once and scaled by
1/world inside the fused Adam kernel, so G ranks == one reference step on the concatenated
batch (CE mean over equal shards = mean of means).
"""
from __future__ import annotations

import torch

from . import ops
from .optim import FusedAdam, FusedAdamW, cosine_lr


class TrainStep:
    def __init__(self, model, lr=1e-4, weight_decay=0.0, adamw=False, cosine_total_steps=None):
        self.model = model
        self.base_lr = lr
        if adamw:
            self.optimizer = FusedAdamW(model.parameters(), lr=lr, weight_decay=weight_decay or 0.01)
        else:
            self.optimizer = FusedAdam(model.parameters(), lr=lr, weight_decay=weight_decay)
        self.cosine_total_steps = cosine_total_steps
        self.steps = 0

    def step_tokens(self, titles, n_cand):
        """titles: integer [B, 1+K+N, L] (host or device) -> loss (0-dim device tensor, no sync)."""
        if self.cosine_total_steps:
            self.optimizer.param_groups[0]["lr"] = cosine_lr(self.base_lr, self.steps, self.cosine_total_steps)
        logits = self.model.forward_tokens(titles, n_cand)
        loss = ops.cross_entropy_label0(logits)
        self.optimizer.zero_grad()
        loss.backward()
        scale = self.optimizer.allreduce_grads()
        self.optimizer.step(grad_scale=scale)
        self.steps += 1
        return loss.detach()

    def step_rows(self, token_table, cand_rows, hist_rows, user=None, clicked_news_length=None):
        """Index-only minibatch (SURVEY 8 f2): `token_table` is the pre-tokenised news table int64 [N_news, L]
        resident on the GPU, `cand_rows` [B, 1+K] and `hist_rows` [B, N] are news-row indices -- 55 x B x 8 bytes of
        H2D per step instead of the 55 token tensors the reference DataLoader ships (dataset.py:17-85,
        train.py:118-124).  The token rows are read through the indices inside the embedding gather / gradient scatter
        kernels (nrms_news_encoder_rows_fwd/bwd): no gathered token tensor is materialised.  user / clicked_news_length:
        the minibatch's `user` and `clicked_news_length` columns, passed on to a model that reads them (LSTUR)."""
        if self.cosine_total_steps:
            self.optimizer.param_groups[0]["lr"] = cosine_lr(self.base_lr, self.steps, self.cosine_total_steps)
        # a model with several news attributes (Exp1) takes a dict of device columns with one row per news
        n_rows = next(iter(token_table.values())).shape[0] if isinstance(token_table, dict) else token_table.shape[0]
        if not cand_rows.is_cuda and cand_rows.numel():
            lo = min(int(cand_rows.min()), int(hist_rows.min()))
            hi = max(int(cand_rows.max()), int(hist_rows.max()))
            if lo < 0 or hi >= n_rows:
                raise IndexError(f"news rows must lie in [0, {n_rows}), got [{lo}, {hi}]")
        if user is not None or clicked_news_length is not None:
            logits = self.model.forward_rows(token_table, cand_rows, hist_rows, user, clicked_news_length)
        else:
            logits = self.model.forward_rows(token_table, cand_rows, hist_rows)
        loss = ops.cross_entropy_label0(logits)
        self.optimizer.zero_grad()
        loss.backward()
        scale = self.optimizer.allreduce_grads()
        self.optimizer.step(grad_scale=scale)
        self.steps += 1
        return loss.detach()

    def step(self, candidate_news, clicked_news, user=None, clicked_news_length=None):
        """Reference minibatch format: lists of {"title": LongTensor[B, L]} (src/train.py:202-203), or of every
        attribute the model reads ({"title", "abstract", "category", ...}) for a model without forward_tokens (Exp1).
        user / clicked_news_length: the minibatch's columns of those names, for LSTUR, which the reference calls as
        model(minibatch["user"], minibatch["clicked_news_length"], candidate_news, clicked_news)."""
        if not hasattr(self.model, "forward_tokens"):
            if self.cosine_total_steps:
                self.optimizer.param_groups[0]["lr"] = cosine_lr(self.base_lr, self.steps, self.cosine_total_steps)
            if user is not None or clicked_news_length is not None:
                logits = self.model(user, clicked_news_length, candidate_news, clicked_news)
            else:
                logits = self.model(candidate_news, clicked_news)
            loss = ops.cross_entropy_label0(logits)
            self.optimizer.zero_grad()
            loss.backward()
            scale = self.optimizer.allreduce_grads()
            self.optimizer.step(grad_scale=scale)
            self.steps += 1
            return loss.detach()
        titles = torch.stack([x["title"] for x in candidate_news] + [x["title"] for x in clicked_news], dim=1)
        return self.step_tokens(titles, len(candidate_news))
