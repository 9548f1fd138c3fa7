"""NewsEncoder (reference src/model/NRMS/news_encoder.py:10-48) on libnrms_b200."""
import torch
import torch.nn as nn

from ... import ops
from ...config import resolve_mode
from ..._lib import MODE_TF32 as _TF32
from ..general.attention.multihead_self import MultiHeadSelfAttention
from ..general.attention.additive import AdditiveAttention


def check_text_width(text, configured, attr):
    """A text tensor is as wide as the configured length, or one of the compiled lengths; any other width is not a
    tokenisation of this model's data (the reference pads and truncates every text to the configured length)."""
    width = text.shape[-1] if text.dim() else 0
    if width != configured and width not in ops.TEXT_LENGTHS_COMPILED:
        raise RuntimeError(f"text of {width} tokens: this model is configured for {attr} = {configured} "
                           f"(texts of {configured} tokens, or of {' or '.join(map(str, ops.TEXT_LENGTHS_COMPILED))})")


class NewsEncoder(nn.Module):
    def __init__(self, config, pretrained_word_embedding):
        super().__init__()
        self.config = config
        if pretrained_word_embedding is None:
            self.word_embedding = nn.Embedding(config.num_words, config.word_embedding_dim, padding_idx=0)
        else:
            self.word_embedding = nn.Embedding.from_pretrained(pretrained_word_embedding, freeze=False,
                                                               padding_idx=0)
        self.multihead_self_attention = MultiHeadSelfAttention(config.word_embedding_dim,
                                                               config.num_attention_heads)
        self.additive_attention = AdditiveAttention(config.query_vector_dim, config.word_embedding_dim)
        # config-5 variant (builder-defined, DESIGN.md section 1): LayerNorm on the self-attention context
        self.layer_norm = nn.LayerNorm(config.word_embedding_dim) if getattr(config, "use_layernorm", False) else None
        self.precision = None          # None -> config.precision / $NRMS_B200_PRECISION / "tf32"
        self._dropout_calls = 0
        self.dropout_seed = 0x5EED     # base seed; data-parallel ranks draw from different streams (see _seed)

    def _check_dims(self):
        c = self.config
        if (c.word_embedding_dim, c.num_attention_heads, c.query_vector_dim) != (ops.D, ops.H, ops.QD):
            raise RuntimeError("libnrms_b200 is compiled for word_embedding_dim=300, num_attention_heads=15, "
                               "query_vector_dim=200 (reference src/config.py:33-45)")

    def _seed(self):
        """Philox key of this process: the base seed with the data-parallel rank folded in, so that G ranks apply G
        independent dropout masks (the reference's single process draws one mask for its whole batch)."""
        import torch.distributed as dist
        rank = dist.get_rank() if dist.is_available() and dist.is_initialized() else 0
        return (int(self.dropout_seed) + 0x9E3779B97F4A7C15 * rank) & 0xFFFFFFFFFFFFFFFF

    def encode_tokens(self, title, news_rows=None):
        """title: integer tensor [n, num_words_title] (any device) -> fp32 [n, 300].  With news_rows (int64 [m] on the
        device) `title` is the device-resident token table and the call encodes its rows news_rows (SURVEY 8 f2).
        The width is config.num_words_title (any 1..64; the reference's default 20), or one of the compiled 20 and 50."""
        self._check_dims()
        check_text_width(title, getattr(self.config, "num_words_title", 20), "num_words_title")
        dev = self.word_embedding.weight.device
        if not title.is_cuda and title.numel():
            # host input (the reference's DataLoader path): nn.Embedding would raise on an id outside the vocabulary; the
            # gather kernels do not check, so the check happens here while the ids are still on the host
            lo, hi = int(title.min()), int(title.max())
            if lo < 0 or hi >= self.word_embedding.num_embeddings:
                raise IndexError(f"token ids must lie in [0, {self.word_embedding.num_embeddings}), got [{lo}, {hi}]")
        title = title.to(dev, non_blocking=True)
        wqkv, bqkv = self.multihead_self_attention.packed()
        if (news_rows is None and title.dtype == torch.int32 and not self.training and not torch.is_grad_enabled() and self.layer_norm is None
                and resolve_mode(self.config, self.precision) == _TF32):
            # evaluate's pre-tokenised table ships int32 ids (half the H2D bytes of the reference's LongTensor)
            return ops.news_encoder_i32(title, self.word_embedding.weight, wqkv, bqkv, self.additive_attention.linear.weight,
                                        self.additive_attention.linear.bias, self.additive_attention.attention_query_vector)
        p = float(self.config.dropout_probability) if self.training else 0.0
        offset = 0
        if p > 0.0:
            # a fresh Philox offset per call (n*20*300/4 counters per dropout site)
            offset = self._dropout_calls
            n_tok = title.numel() if news_rows is None else news_rows.numel() * title.shape[1]
            self._dropout_calls += (n_tok * ops.D) // 4 + 1
        return ops.news_encoder(title, self.word_embedding.weight, wqkv, bqkv,
                                self.additive_attention.linear.weight, self.additive_attention.linear.bias,
                                self.additive_attention.attention_query_vector,
                                dropout_p=p, seed=self._seed(), offset=offset,
                                mode=resolve_mode(self.config, self.precision),
                                ln=None if self.layer_norm is None else (self.layer_norm.weight, self.layer_norm.bias),
                                news_rows=news_rows)

    def forward(self, news):
        """news: {"title": batch_size * num_words_title} -> batch_size, word_embedding_dim"""
        return self.encode_tokens(news["title"])
