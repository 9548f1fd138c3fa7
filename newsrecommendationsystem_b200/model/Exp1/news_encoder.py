"""Exp1 NewsEncoder (reference src/model/Exp1/news_encoder.py:10-111) on libnrms_b200.

TextEncoder (:10-34) is NRMS's news encoder (embedding gather, dropout, multi-head self-attention, dropout, additive
attention) with its own attention weights over a SHARED word embedding; ElementEncoder (:37-44) is
relu(linear(embedding(element))) over a shared category embedding; the final AdditiveAttention (:104-110) pools the
2..4 vectors.  Sub-module names follow the reference so that state_dict keys are identical."""
import torch
import torch.nn as nn

from ... import ops
from ...config import resolve_mode
from ..general.attention.multihead_self import MultiHeadSelfAttention
from ..general.attention.additive import AdditiveAttention
from ..NRMS.news_encoder import check_text_width


# Philox keys of the text encoders' dropout streams.  Both encoders start at offset 0 each step, so with one key element
# i of a title and element i of an abstract would drop together; the abstract gets its own key (the title keeps the
# key it always had, so title-only models draw the same masks as before).
DROPOUT_SEEDS = {"title": 0x5EED, "abstract": 0xAB57AC7}
# configured length of each text attribute: (config attribute, the reference's default)
TEXT_LENGTHS = {"title": ("num_words_title", 20), "abstract": ("num_words_abstract", 50)}


class TextEncoder(nn.Module):
    def __init__(self, word_embedding, word_embedding_dim, num_attention_heads, query_vector_dim, dropout_probability,
                 dropout_seed=0x5EED, num_words=None):
        """num_words: (config attribute, value) of the text's configured length, e.g. ("num_words_abstract", 50); texts
        of another width than that value, 20 and 50 are refused.  None: no width rule beyond the library's 1..64."""
        super().__init__()
        self.num_words = num_words
        self.word_embedding = word_embedding
        self.dropout_probability = dropout_probability
        self.multihead_self_attention = MultiHeadSelfAttention(word_embedding_dim, num_attention_heads)
        self.additive_attention = AdditiveAttention(query_vector_dim, word_embedding_dim)
        self.precision = None
        self._dropout_calls = 0
        self.dropout_seed = dropout_seed

    def _seed(self):
        import torch.distributed as dist
        rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
        return (int(self.dropout_seed) + 0x9E3779B97F4A7C15 * rank) & 0xFFFFFFFFFFFFFFFF

    def forward(self, text, news_rows=None):
        """text: integer [n, num_words_text] (num_words_title / num_words_abstract, any 1..64; training and inference)
        -> fp32 [n, 300].
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
        wqkv, bqkv = self.multihead_self_attention.packed()
        p = float(self.dropout_probability) if self.training else 0.0
        offset = 0
        if p > 0.0:
            offset = self._dropout_calls
            n_tok = text.numel() if news_rows is None else news_rows.numel() * text.shape[1]
            self._dropout_calls += (n_tok * ops.D) // 4 + 1
        a = self.additive_attention
        return ops.news_encoder(text, self.word_embedding.weight, wqkv, bqkv, a.linear.weight, a.linear.bias,
                                a.attention_query_vector, dropout_p=p, seed=self._seed(), offset=offset,
                                mode=resolve_mode(None, self.precision), news_rows=news_rows)


class ElementEncoder(nn.Module):
    def __init__(self, embedding, linear_input_dim, linear_output_dim):
        super().__init__()
        self.embedding = embedding
        self.linear = nn.Linear(linear_input_dim, linear_output_dim)

    def forward(self, element):
        """element: integer [n] -> fp32 [n, 300]"""
        dev = self.linear.weight.device
        if not element.is_cuda and element.numel():
            lo, hi = int(element.min()), int(element.max())
            if lo < 0 or hi >= self.embedding.num_embeddings:
                raise IndexError(f"element ids must lie in [0, {self.embedding.num_embeddings}), got [{lo}, {hi}]")
        return ops.element_encoder(element.to(dev, non_blocking=True), self.embedding.weight, self.linear.weight,
                                   self.linear.bias)


class NewsEncoder(nn.Module):
    def __init__(self, config, pretrained_word_embedding):
        super().__init__()
        self.config = config
        if (config.word_embedding_dim, config.num_attention_heads, config.query_vector_dim,
                config.category_embedding_dim) != (ops.D, ops.H, ops.QD, 100):
            raise RuntimeError("libnrms_b200 is compiled for word_embedding_dim=300, num_attention_heads=15, "
                               "query_vector_dim=200, category_embedding_dim=100 (reference src/config.py:33-45)")
        if pretrained_word_embedding is None:
            word_embedding = nn.Embedding(config.num_words, config.word_embedding_dim, padding_idx=0)
        else:
            word_embedding = nn.Embedding.from_pretrained(pretrained_word_embedding, freeze=False, padding_idx=0)
        assert len(config.dataset_attributes['news']) > 0
        # sorted (the reference iterates a set intersection, :64-70, whose order is not defined): the order only names
        # the rows of the final attention's input, and additive pooling is invariant to it
        text_names = sorted(set(config.dataset_attributes['news']) & {'title', 'abstract'})
        self.text_encoders = nn.ModuleDict({
            name: TextEncoder(word_embedding, config.word_embedding_dim, config.num_attention_heads,
                              config.query_vector_dim, config.dropout_probability, DROPOUT_SEEDS[name],
                              num_words=(TEXT_LENGTHS[name][0], getattr(config, *TEXT_LENGTHS[name])))
            for name in text_names
        })
        category_embedding = nn.Embedding(config.num_categories, config.category_embedding_dim, padding_idx=0)
        element_names = sorted(set(config.dataset_attributes['news']) & {'category', 'subcategory'})
        self.element_encoders = nn.ModuleDict({
            name: ElementEncoder(category_embedding, config.category_embedding_dim, config.word_embedding_dim)
            for name in element_names
        })
        if len(config.dataset_attributes['news']) > 1:
            self.final_attention = AdditiveAttention(config.query_vector_dim, config.word_embedding_dim)
        self._precision = None

    @property
    def precision(self):
        return self._precision

    @precision.setter
    def precision(self, name):
        self._precision = name
        for enc in self.text_encoders.values():
            enc.precision = name
        if hasattr(self, "final_attention"):
            self.final_attention.precision = name

    def attributes(self):
        return list(self.text_encoders.keys()) + list(self.element_encoders.keys())

    def forward(self, news):
        """news: {"category": B, "subcategory": B, "title": B x num_words_title, "abstract": B x num_words_abstract}
        -> B x word_embedding_dim"""
        all_vectors = [encoder(news[name]) for name, encoder in self.text_encoders.items()] + \
                      [encoder(news[name]) for name, encoder in self.element_encoders.items()]
        return self._pool(all_vectors)

    def forward_rows(self, news_table, rows):
        """news_table: {attribute: device column with N + 1 rows}, rows: int64 [m] on the device -> m x 300.  The text
        columns are read through the indices inside the gather / scatter kernels; the element ids are gathered first."""
        all_vectors = [encoder(news_table[name], news_rows=rows) for name, encoder in self.text_encoders.items()] + \
                      [encoder(news_table[name][rows]) for name, encoder in self.element_encoders.items()]
        return self._pool(all_vectors)

    def _pool(self, all_vectors):
        if len(all_vectors) == 1:
            return all_vectors[0]
        return self.final_attention(ops.stack_vectors(all_vectors))
