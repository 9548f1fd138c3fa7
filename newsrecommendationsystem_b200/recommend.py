"""Single-user recommendation path (SURVEY 8 row f4; reference src/recommend.py:197-341).

The reference's `evaluate(model, directory, ..., target_user_id)` (1) loads or builds the `news2vector.pt` cache
(:211-243), (2) stacks the target user's 50 clicked-news vectors and calls `model.get_user_vector` (:264-279), (3) stacks
the impression's candidate vectors and calls `model.get_prediction` (:301-315), and (4) returns the candidate ids and
`(score + 1) / 2` sorted by `np.argsort(-y)` (:338-340).  `Recommender` keeps the cache as a device table and runs steps
2-4 as `nrms_recommend_user`: two cluster launches, one 4-byte-per-candidate copy back (csrc/recommend.cu).
"""
from __future__ import annotations

import numpy as np
import torch

import csv
import ctypes as C
import os

from . import ops
from .checkpoint import news2vector_from_table, table_from_news2vector


def load_target_user(behaviors_path, target_user_id):
    """The FIRST row of `target_user_id` in a raw `behaviors.tsv` (the reference keeps `.iloc[[0]]` of the user's rows,
    src/recommend.py:100,159) -> (clicked news ids, impression strings).  An empty history is the reference's `' '`."""
    with open(behaviors_path, newline="") as f:
        for rec in csv.reader(f, delimiter="\t", quoting=csv.QUOTE_NONE):
            if rec[1] == target_user_id:
                return (rec[3] or " ").split(), rec[4].split()
    raise KeyError(f"user {target_user_id!r} not found in {behaviors_path}")


class Recommender:
    def __init__(self, model, news_ids, table):
        """model: NRMS (its user encoder and click predictor are used); news_ids: list of ids in table-row order;
        table: fp32 [N + 1, 300] on the model's device whose LAST row is PADDED_NEWS (zeros)."""
        self.model = model
        self.ids = list(news_ids)
        self.row_of = {}
        for i, nid in enumerate(self.ids):
            self.row_of.setdefault(nid, i)                 # first occurrence wins (src/evaluate.py:197-201)
        self.table = table.contiguous().float()
        self.pad_row = self.table.shape[0] - 1
        self.n_hist = int(model.config.num_clicked_news_a_user)

    @classmethod
    def from_news2vector(cls, model, news2vector, device):
        """From the reference's cache file content (dict id -> vector + 'PADDED_NEWS', src/recommend.py:211-243)."""
        ids, table = table_from_news2vector(news2vector, device=device)
        return cls(model, ids, table)

    @classmethod
    def from_directory(cls, model, directory, device=None, batch=2048):
        """`directory` as the reference's evaluate() takes it (src/recommend.py:197-243): `news2vector.pt` is loaded when it
        exists, else the news of `news_parsed.tsv` are encoded (`model.get_news_vector`, batches of 2,048 titles) and the
        cache is written in the reference's format (dict id -> vector + 'PADDED_NEWS')."""
        from . import data
        device = device or next(model.parameters()).device
        cache = os.path.join(directory, "news2vector.pt")
        if os.path.exists(cache):
            return cls.from_news2vector(model, torch.load(cache, map_location="cpu", weights_only=False), device)
        news = data.load_news_parsed(os.path.join(directory, "news_parsed.tsv"))
        was_training = model.training
        model.eval()
        with torch.no_grad():
            titles = torch.from_numpy(news.title)
            vec = torch.cat([model.get_news_vector({"title": titles[s:s + batch]}).float().cpu()
                             for s in range(0, len(news), batch)])
        model.train(was_training)
        table = torch.cat([vec, torch.zeros(1, vec.shape[1])])
        torch.save(news2vector_from_table(news.ids, table), cache)
        keep = [i for i, nid in enumerate(news.ids) if news.row_of[nid] == i]          # first occurrence of an id wins
        return cls(model, [news.ids[i] for i in keep], torch.cat([vec[keep], torch.zeros(1, vec.shape[1])]).to(device))

    def recommend_target_user(self, directory, target_user_id):
        """What the reference's recommend.evaluate(model, directory, ..., target_user_id) returns (:338-340) for the user's
        first behaviors row: (candidate ids by descending score, y = (score + 1) / 2 in that order)."""
        clicked, impressions = load_target_user(os.path.join(directory, "behaviors.tsv"), target_user_id)
        return self.recommend(clicked, impressions)

    def history_rows(self, clicked_news):
        """First num_clicked_news_a_user clicks, LEFT-padded with PADDED_NEWS (src/recommend.py:117-124 = evaluate.py:117-124)."""
        rows = [self.row_of[x] for x in list(clicked_news)[:self.n_hist]]
        return [self.pad_row] * (self.n_hist - len(rows)) + rows

    def _state(self):
        """Packed weights, workspace and pinned staging buffers, rebuilt only when a parameter is written."""
        ue = self.model.user_encoder
        a = ue.additive_attention
        ps = list(ue.multihead_self_attention.parameters()) + [a.linear.weight, a.linear.bias, a.attention_query_vector]
        key = tuple((p.data_ptr(), p._version) for p in ps)
        st = getattr(self, "_st", None)
        if st is None or st["key"] != key:
            from . import _lib
            lib = _lib.load()
            dev = self.table.device
            with torch.no_grad():
                wqkv, bqkv = ue.multihead_self_attention.packed()
                w = [t.detach().contiguous().float() for t in (wqkv, bqkv, a.linear.weight, a.linear.bias,
                                                                a.attention_query_vector)]
            st = {"key": key, "w": w, "lib": lib,
                  "ws": torch.empty(lib.nrms_recommend_workspace_bytes(), dtype=torch.uint8, device=dev),
                  "user": torch.empty(300, dtype=torch.float32, device=dev),
                  "idx_host": torch.empty(self.n_hist + 4096, dtype=torch.int32).pin_memory(),
                  "idx_dev": torch.empty(self.n_hist + 4096, dtype=torch.int32, device=dev),
                  "scores": torch.empty(4096, dtype=torch.float32, device=dev),
                  "order": torch.empty(4096, dtype=torch.int32, device=dev),
                  "copied": torch.cuda.Event()}        # recorded after each idx_host -> idx_dev copy
            self._st = st
        return st

    @torch.no_grad()
    def recommend_rows(self, hist_rows, cand_rows):
        """Row-index form: returns (order int32 [C], scores fp32 [C], user_vec fp32 [300]) on the device.
        Up to 4,096 candidates go through preallocated buffers (one pinned H2D copy of 50 + C indices, two launches);
        the returned tensors are views that the next call overwrites.  The host waits only when the previous call's
        index copy has not run yet, before it rewrites the pinned staging buffer; otherwise nothing syncs.
        Order: score descending, equal scores by ascending candidate position, NaN scores last (np.argsort(-y) on a
        stable sort), on both sides of the 4,096-candidate limit.  The cluster kernel is compiled for 50 history rows;
        other num_clicked_news_a_user take the indexed user encoder (FP32 mode) and a device sort, with fresh tensors."""
        from ._lib import check, ptr
        n_c = len(cand_rows)
        dev = self.table.device
        if self.n_hist != 50:
            return self._recommend_rows_any_length(hist_rows, cand_rows)
        if n_c > 4096:
            ue = self.model.user_encoder
            a = ue.additive_attention
            user, scores, _ = ops.recommend_user(self.table, torch.as_tensor(hist_rows, dtype=torch.int32).to(dev),
                                                 torch.as_tensor(cand_rows, dtype=torch.int32).to(dev),
                                                 *ue.multihead_self_attention.packed(), a.linear.weight, a.linear.bias,
                                                 a.attention_query_vector, rank=False)
            return torch.argsort(-scores, stable=True).int(), scores, user     # ascending sort puts NaN last
        st = self._state()
        st["copied"].synchronize()                 # the previous call's copy may still read idx_host
        h = st["idx_host"]
        h[:self.n_hist] = torch.as_tensor(hist_rows, dtype=torch.int32)
        h[self.n_hist:self.n_hist + n_c] = torch.as_tensor(cand_rows, dtype=torch.int32)
        d = st["idx_dev"]
        d[:self.n_hist + n_c].copy_(h[:self.n_hist + n_c], non_blocking=True)
        stream = torch.cuda.current_stream(dev)
        st["copied"].record(stream)
        w = st["w"]
        check(st["lib"].nrms_recommend_user(ptr(self.table), self.table.shape[0], ptr(d), ptr(d[self.n_hist:]), n_c,
                                            ptr(w[0]), ptr(w[1]), ptr(w[2]), ptr(w[3]), ptr(w[4]), ptr(st["user"]),
                                            ptr(st["scores"]), ptr(st["order"]), ptr(st["ws"]), st["ws"].numel(),
                                            C.c_void_p(stream.cuda_stream)), "nrms_recommend_user")
        return st["order"][:n_c], st["scores"][:n_c], st["user"]

    def _recommend_rows_any_length(self, hist_rows, cand_rows):
        """recommend_rows at a history length the cluster kernel is not compiled for (num_clicked_news_a_user != 50):
        the indexed user encoder in FP32 mode -- the arithmetic of the S = 50 latency path, which is FP32 too -- then
        score_csr over one impression and a stable descending sort (NaN last), as the > 4,096-candidate branch."""
        from . import _lib
        ue = self.model.user_encoder
        dev = self.table.device
        hist = torch.as_tensor(hist_rows, dtype=torch.int32).to(dev).view(1, -1)
        if hist.shape[1] != self.n_hist:
            raise RuntimeError(f"hist_rows must hold {self.n_hist} rows, got {hist.shape[1]}")
        cand = torch.as_tensor(cand_rows, dtype=torch.int32).to(dev).view(-1)
        user = ops.user_encoder_indexed(self.table, hist, *ue._weights(), mode=_lib.MODE_FP32, ln=ue._ln())
        offsets = torch.tensor([0, cand.numel()], dtype=torch.int64, device=dev)
        scores = ops.score_csr(self.table, cand, offsets, user)
        return torch.argsort(-scores, stable=True).int(), scores, user[0]

    @torch.no_grad()
    def top_k_rows(self, hist_rows, k, exclude_clicked=True):
        """The k best news of the whole table for each user, not only for candidates the caller already has.
        hist_rows: int32 [U, num_clicked_news_a_user] in `history_rows` form (pads = the table's last row), host or device.  Returns (rows int32
        [U, k], scores fp32 [U, k], user_vec fp32 [U, 300]) on the device, no sync: rows by descending score (equal scores
        by ascending row), the clicked rows left out when exclude_clicked; tail entries are row -1, score -inf.
        Arithmetic follows the user encoder's precision: tensor mode scores against an fp16 copy of the table, packed on
        the first call and kept."""
        from . import _lib
        from .config import resolve_mode
        ue = self.model.user_encoder
        dev = self.table.device
        hist = torch.as_tensor(hist_rows).to(device=dev, dtype=torch.int32).contiguous()
        if hist.dim() != 2 or hist.shape[1] != self.n_hist:
            raise RuntimeError(f"hist_rows must be [U, {self.n_hist}], got {tuple(hist.shape)}")
        user_vec = ue.forward_indexed(self.table, hist)
        mode = resolve_mode(ue.config, ue.precision)
        if mode == _lib.MODE_TF32:
            if getattr(self, "_table16", None) is None:
                self._table16 = ops.pack_rows_f16(self.table)
            table = self._table16
        else:
            table = self.table
        scores, rows = ops.topk_news(table, self.pad_row, user_vec, k, exclude_rows=hist if exclude_clicked else None,
                                     mode=mode)
        return rows, scores, user_vec

    def top_k(self, clicked_news, k, exclude_clicked=True):
        """Id form of `top_k_rows` for one user: clicked_news = list of news ids -> (news ids by descending score,
        y = (score + 1) / 2 in that order), the pair and convention of `recommend` (src/recommend.py:338-340) over the
        whole table.  Fewer than k ids come back when fewer news remain."""
        hist = torch.tensor([self.history_rows(clicked_news)], dtype=torch.int32)
        rows, scores, _ = self.top_k_rows(hist, k, exclude_clicked)
        rows = rows[0].cpu().numpy()
        scores = scores[0].cpu().numpy()
        keep = rows >= 0
        y = (scores[keep].astype(np.float64) + 1.0) / 2.0
        return np.array(self.ids, dtype=object)[rows[keep]].astype(str), y

    def recommend(self, clicked_news, impressions):
        """clicked_news: list of news ids; impressions: list of candidate ids, optionally 'id-label' strings
        (src/recommend.py:301-332) -> (candidate ids sorted by descending score, y = (score + 1) / 2 sorted), the pair
        the reference returns (:338-340)."""
        cand_ids = [c.split('-')[0] if c not in self.row_of else c for c in impressions]
        order, scores, _ = self.recommend_rows(self.history_rows(clicked_news), [self.row_of[c] for c in cand_ids])
        order = order.cpu().numpy()
        y = (scores.cpu().numpy().astype(np.float64) + 1.0) / 2.0      # python-float arithmetic of :338
        return np.array(cand_ids)[order], y[order]
