"""LSTUR NewsEncoder (reference src/model/LSTUR/news_encoder.py) on libnrms_b200.

news_vector = cat([category_embedding(category), category_embedding(subcategory), title_attention(relu(title_CNN(
dropout(word_embedding(title)))) after dropout)]): 900 wide.  The title path is NAML's CNN text encoder, one library
call (nrms_cnn_text_fwd / _bwd); the category rows are plain embedding rows (no linear, no ReLU) from one shared table,
and the three blocks are joined by strided row copies.  Sub-module names follow the reference, so state_dict keys are
identical."""
import torch.nn as nn

from ... import ops
from ...config import resolve_mode
from ..general.attention.additive import AdditiveAttention
from ..NRMS.news_encoder import check_text_width
from ..NAML.news_encoder import TextEncoder as _NAMLTextEncoder


def check_config(config):
    """The dimensions libnrms_b200 is compiled for; any other value raises a RuntimeError that names the setting."""
    rules = (("num_filters", ops.D), ("word_embedding_dim", ops.D), ("window_size", 3), ("query_vector_dim", ops.QD))
    for name, want in rules:
        got = getattr(config, name)
        if got != want:
            raise RuntimeError(f"libnrms_b200 is compiled for LSTUR with {name} = {want} (got {got})")
    method = getattr(config, "long_short_term_method")
    if method not in ("ini", "con"):
        raise RuntimeError(f"long_short_term_method must be 'ini' or 'con' (got {method!r})")


def _check_ids(ids, n, what):
    if not ids.is_cuda and ids.numel():
        lo, hi = int(ids.min()), int(ids.max())
        if lo < 0 or hi >= n:
            raise IndexError(f"{what} ids must lie in [0, {n}), got [{lo}, {hi}]")


class NewsEncoder(nn.Module):
    def __init__(self, config, pretrained_word_embedding):
        super().__init__()
        check_config(config)
        self.config = config
        if pretrained_word_embedding is None:
            self.word_embedding = nn.Embedding(config.num_words, config.word_embedding_dim, padding_idx=0)
        else:
            self.word_embedding = nn.Embedding.from_pretrained(pretrained_word_embedding, freeze=False, padding_idx=0)
        self.category_embedding = nn.Embedding(config.num_categories, config.num_filters, padding_idx=0)
        assert config.window_size >= 1 and config.window_size % 2 == 1
        self.title_CNN = nn.Conv2d(1, config.num_filters, (config.window_size, config.word_embedding_dim),
                                   padding=(int((config.window_size - 1) / 2), 0))
        self.title_attention = AdditiveAttention(config.query_vector_dim, config.num_filters)
        self.precision = None
        self._dropout_calls = 0
        self.dropout_seed = 0x5EED

    _seed = _NAMLTextEncoder._seed

    def _title(self, title, news_rows=None):
        """NAML's TextEncoder arithmetic over title_CNN / title_attention: [n, 300]."""
        check_text_width(title, self.config.num_words_title, "num_words_title")
        _check_ids(title, self.word_embedding.num_embeddings, "token")
        dev = self.word_embedding.weight.device
        title = title.to(dev, non_blocking=True)
        p = float(self.config.dropout_probability) if self.training else 0.0
        offset = 0
        if p > 0.0:
            offset = self._dropout_calls
            n_tok = title.numel() if news_rows is None else news_rows.numel() * title.shape[1]
            self._dropout_calls += (n_tok * ops.D) // 4 + 1
        a = self.title_attention
        return ops.cnn_text_encoder(title, self.word_embedding.weight, self.title_CNN.weight.view(ops.D, 3 * ops.D),
                                    self.title_CNN.bias, a.linear.weight, a.linear.bias, a.attention_query_vector,
                                    dropout_p=p, seed=self._seed(), offset=offset,
                                    mode=resolve_mode(self.config, self.precision), news_rows=news_rows)

    def _categories(self, category, subcategory):
        dev = self.category_embedding.weight.device
        n = self.category_embedding.num_embeddings
        _check_ids(category, n, "category")
        _check_ids(subcategory, n, "subcategory")
        w = self.category_embedding.weight
        return (ops.embedding_rows(category.to(dev, non_blocking=True), w),
                ops.embedding_rows(subcategory.to(dev, non_blocking=True), w))

    def forward(self, news):
        """news: {"category": B, "subcategory": B, "title": B x num_words_title} -> B x (num_filters * 3)"""
        category_vector, subcategory_vector = self._categories(news["category"], news["subcategory"])
        weighted_title_vector = self._title(news["title"])
        return ops.concat_rows(category_vector, subcategory_vector, weighted_title_vector)

    def forward_rows(self, news_table, rows):
        """news_table {"category": [N+1], "subcategory": [N+1], "title": [N+1, L]} device columns, rows int64 [m]
        (device) -> [m, 900].  The title tokens are read through the rows inside the CNN encoder's kernels."""
        category_vector, subcategory_vector = self._categories(news_table["category"][rows],
                                                               news_table["subcategory"][rows])
        weighted_title_vector = self._title(news_table["title"], news_rows=rows)
        return ops.concat_rows(category_vector, subcategory_vector, weighted_title_vector)
