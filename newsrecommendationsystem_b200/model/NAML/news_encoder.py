"""NAML NewsEncoder (reference src/model/NAML/news_encoder.py:9-115) on libnrms_b200.

TextEncoder (:9-40) is word embedding -> dropout -> Conv2d(1, num_filters, (window_size, word_embedding_dim),
padding=(1, 0)) -> ReLU -> dropout -> AdditiveAttention over a SHARED word embedding: one library call,
nrms_cnn_text_fwd / _bwd.  ElementEncoder is Exp1's (relu(linear(embedding(element))) over a shared category
embedding); the final AdditiveAttention pools the 2..4 vectors.  Sub-module names follow the reference so that
state_dict keys are identical."""
import torch.nn as nn

from ... import ops
from ...config import resolve_mode
from ..general.attention.additive import AdditiveAttention
from ..Exp1.news_encoder import DROPOUT_SEEDS, TEXT_LENGTHS, ElementEncoder, NewsEncoder as _Exp1NewsEncoder
from ..Exp1.news_encoder import TextEncoder as _Exp1TextEncoder
from ..NRMS.news_encoder import check_text_width


def check_config(config):
    """The dimensions libnrms_b200 is compiled for; any other value raises a RuntimeError that names the setting."""
    rules = (("num_filters", ops.D), ("word_embedding_dim", ops.D), ("window_size", 3), ("query_vector_dim", ops.QD),
             ("category_embedding_dim", 100))
    for name, want in rules:
        got = getattr(config, name)
        if got != want:
            raise RuntimeError(f"libnrms_b200 is compiled for NAML with {name} = {want} (got {got}); num_filters must "
                               f"equal word_embedding_dim = {ops.D} and window_size must be 3")


class TextEncoder(nn.Module):
    def __init__(self, word_embedding, word_embedding_dim, num_filters, window_size, query_vector_dim,
                 dropout_probability, dropout_seed=0x5EED, num_words=None):
        """num_words: (config attribute, value) of the text's configured length, as in Exp1's TextEncoder."""
        super().__init__()
        self.num_words = num_words
        self.word_embedding = word_embedding
        self.dropout_probability = dropout_probability
        self.CNN = nn.Conv2d(1, num_filters, (window_size, word_embedding_dim), padding=(int((window_size - 1) / 2), 0))
        self.additive_attention = AdditiveAttention(query_vector_dim, num_filters)
        self.precision = None
        self._dropout_calls = 0
        self.dropout_seed = dropout_seed

    # the per-text Philox key with the data-parallel rank folded in, as Exp1's text encoders draw it
    _seed = _Exp1TextEncoder._seed

    def forward(self, text, news_rows=None):
        """text: integer [n, L] (the configured num_words_title / num_words_abstract, any 1..64) -> fp32 [n, 300].
        With news_rows (int64 [m] on the device) `text` is the device-resident token column [N + 1, L] of the news table
        and the call encodes its rows news_rows, read through the indices inside the gather / scatter kernels."""
        if self.num_words is not None:
            check_text_width(text, self.num_words[1], self.num_words[0])
        dev = self.word_embedding.weight.device
        if not text.is_cuda and text.numel():
            lo, hi = int(text.min()), int(text.max())
            if lo < 0 or hi >= self.word_embedding.num_embeddings:
                raise IndexError(f"token ids must lie in [0, {self.word_embedding.num_embeddings}), got [{lo}, {hi}]")
        text = text.to(dev, non_blocking=True)
        p = float(self.dropout_probability) if self.training else 0.0
        offset = 0
        if p > 0.0:
            offset = self._dropout_calls
            n_tok = text.numel() if news_rows is None else news_rows.numel() * text.shape[1]
            self._dropout_calls += (n_tok * ops.D) // 4 + 1
        a = self.additive_attention
        return ops.cnn_text_encoder(text, self.word_embedding.weight, self.CNN.weight.view(ops.D, 3 * ops.D),
                                    self.CNN.bias, a.linear.weight, a.linear.bias, a.attention_query_vector,
                                    dropout_p=p, seed=self._seed(), offset=offset,
                                    mode=resolve_mode(None, self.precision), news_rows=news_rows)


class NewsEncoder(_Exp1NewsEncoder):
    """The reference's NAML NewsEncoder: the text encoders are CNN encoders; element encoders, the final attention,
    attribute order, precision switch and pooling are Exp1's (stack_vectors + final additive attention)."""

    def __init__(self, config, pretrained_word_embedding):
        nn.Module.__init__(self)
        self.config = config
        check_config(config)
        if pretrained_word_embedding is None:
            word_embedding = nn.Embedding(config.num_words, config.word_embedding_dim, padding_idx=0)
        else:
            word_embedding = nn.Embedding.from_pretrained(pretrained_word_embedding, freeze=False, padding_idx=0)
        assert len(config.dataset_attributes['news']) > 0
        text_names = sorted(set(config.dataset_attributes['news']) & {'title', 'abstract'})
        self.text_encoders = nn.ModuleDict({
            name: TextEncoder(word_embedding, config.word_embedding_dim, config.num_filters, config.window_size,
                              config.query_vector_dim, config.dropout_probability, DROPOUT_SEEDS[name],
                              num_words=(TEXT_LENGTHS[name][0], getattr(config, *TEXT_LENGTHS[name])))
            for name in text_names
        })
        category_embedding = nn.Embedding(config.num_categories, config.category_embedding_dim, padding_idx=0)
        element_names = sorted(set(config.dataset_attributes['news']) & {'category', 'subcategory'})
        self.element_encoders = nn.ModuleDict({
            name: ElementEncoder(category_embedding, config.category_embedding_dim, config.num_filters)
            for name in element_names
        })
        if len(config.dataset_attributes['news']) > 1:
            self.final_attention = AdditiveAttention(config.query_vector_dim, config.num_filters)
        self._precision = None
