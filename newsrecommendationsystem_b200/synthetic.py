"""Synthetic MIND-shaped inputs (SURVEY.md section 8(d)); numpy only, deterministic.

Shapes follow the reference's data contracts:
  * news table   int64 [N_news, num_words_title]   right-padded with 0
    (`data_preprocess.py:115,132-139` truncates/pads titles to 20 tokens)
  * impressions  history = first <=50 clicks, LEFT-padded (`evaluate.py:111-124`),
    candidates as CSR (offsets, rows, labels) replacing the "N123-1 N456-0" strings
    (`evaluate.py:251-263`)
  * training batch  int64 [B, 1+K, L] candidates (column 0 = the positive,
    `data_preprocess.py:63-66`) and int64 [B, 50, L] clicked titles (L = the table's title width), left-padded with
    all-zero titles (`dataset.py:47,75-83`).
"""
from __future__ import annotations

import numpy as np

MIND_SMALL = dict(num_news=65238, num_impressions=73152)
MIND_LARGE = dict(num_news=161013, num_impressions=376471)


def make_news(num_news, num_words=70976, title_len=20, seed=1234):
    rng = np.random.default_rng(seed)
    lens = np.clip(np.rint(rng.normal(11, 4, size=num_news)), 1, title_len).astype(np.int64)
    toks = rng.integers(1, num_words, size=(num_news, title_len), dtype=np.int64)
    toks[np.arange(title_len)[None, :] >= lens[:, None]] = 0
    return toks


def make_impressions(num_impressions, num_news, history=50, seed=1234, single_class_every=1000,
                     max_cand=300):
    """Returns dict(hist_rows [I,history] int64 (-1 = PADDED_NEWS), cand_offsets [I+1] int64,
    cand_rows [sumC] int64, labels [sumC] int8)."""
    rng = np.random.default_rng(seed + 1)
    hlen = rng.integers(0, history + 1, size=num_impressions)
    hist = rng.integers(0, num_news, size=(num_impressions, history), dtype=np.int64)
    # left padding: positions [0, history-hlen) are pads
    hist[np.arange(history)[None, :] < (history - hlen)[:, None]] = -1
    C = np.clip(np.rint(rng.lognormal(3.3, 0.8, size=num_impressions)), 2, max_cand).astype(np.int64)
    offsets = np.zeros(num_impressions + 1, dtype=np.int64)
    np.cumsum(C, out=offsets[1:])
    total = int(offsets[-1])
    rows = rng.integers(0, num_news, size=total, dtype=np.int64)
    labels = (rng.random(total) < 0.04).astype(np.int8)
    # force one positive and one negative per impression ...
    labels[offsets[:-1]] = 1
    labels[offsets[:-1] + 1] = 0
    # ... except every `single_class_every`-th impression, left single-class (NaN path)
    if single_class_every:
        for i in range(single_class_every - 1, num_impressions, single_class_every):
            labels[offsets[i]:offsets[i + 1]] = 0
    return dict(hist_rows=hist, cand_offsets=offsets, cand_rows=rows, labels=labels)


def make_train_batch(batch, num_news_tokens, k_neg=4, history=50, seed=1234):
    """Index-free training batch as the reference's DataLoader would deliver it
    (already joined with the token table): cand [B,1+K,L], clicked [B,history,L]."""
    rng = np.random.default_rng(seed + 2)
    n = num_news_tokens.shape[0]
    L = num_news_tokens.shape[1]
    cand = num_news_tokens[rng.integers(0, n, size=(batch, 1 + k_neg))]
    hlen = rng.integers(1, history + 1, size=batch)
    clicked = num_news_tokens[rng.integers(0, n, size=(batch, history))].copy()
    pad = np.arange(history)[None, :] < (history - hlen)[:, None]
    clicked[pad] = np.zeros(L, dtype=np.int64)
    return cand, clicked


def init_state_dict(num_words=70976, dim=300, query_dim=200, seed=0, dtype=np.float32):
    """Random-init parameters with the reference's distributions (SURVEY.md Appendix B):
    embedding N(0,1) with row 0 zero (`news_encoder.py:15-17`), W_Q/K/V xavier_uniform
    (`multihead_self.py:41-44`), nn.Linear default biases/additive linear, query U(-0.1,0.1)
    (`additive.py:19-20`).  Same distributions, not the same stream as torch.manual_seed."""
    rng = np.random.default_rng(seed)
    sd = {}
    E = rng.standard_normal((num_words, dim)).astype(dtype)
    E[0] = 0
    sd["news_encoder.word_embedding.weight"] = E
    for enc in ("news_encoder", "user_encoder"):
        for w in ("W_Q", "W_K", "W_V"):
            a = np.sqrt(6.0 / (dim + dim))
            sd[f"{enc}.multihead_self_attention.{w}.weight"] = rng.uniform(-a, a, (dim, dim)).astype(dtype)
            b = 1 / np.sqrt(dim)
            sd[f"{enc}.multihead_self_attention.{w}.bias"] = rng.uniform(-b, b, dim).astype(dtype)
        b = 1 / np.sqrt(dim)
        sd[f"{enc}.additive_attention.linear.weight"] = rng.uniform(-b, b, (query_dim, dim)).astype(dtype)
        sd[f"{enc}.additive_attention.linear.bias"] = rng.uniform(-b, b, query_dim).astype(dtype)
        sd[f"{enc}.additive_attention.attention_query_vector"] = rng.uniform(-0.1, 0.1, query_dim).astype(dtype)
    return sd
