"""UserEncoder (reference src/model/NRMS/user_encoder.py:6-26) on libnrms_b200."""
import torch
import torch.nn as nn

from ... import ops
from ...config import resolve_mode
from ..general.attention.multihead_self import MultiHeadSelfAttention
from ..general.attention.additive import AdditiveAttention


class UserEncoder(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        self.multihead_self_attention = MultiHeadSelfAttention(config.word_embedding_dim,
                                                               config.num_attention_heads)
        self.additive_attention = AdditiveAttention(config.query_vector_dim, config.word_embedding_dim)
        # config-5 variant (builder-defined, DESIGN.md section 1): LayerNorm on the self-attention context
        self.layer_norm = nn.LayerNorm(config.word_embedding_dim) if getattr(config, "use_layernorm", False) else None
        self.precision = None

    def _ln(self):
        return None if self.layer_norm is None else (self.layer_norm.weight, self.layer_norm.bias)

    def _weights(self):
        wqkv, bqkv = self.multihead_self_attention.packed()
        a = self.additive_attention
        return wqkv, bqkv, a.linear.weight, a.linear.bias, a.attention_query_vector

    def forward(self, user_vector):
        """user_vector: batch_size, num_clicked_news_a_user, word_embedding_dim -> batch_size, word_embedding_dim"""
        dev = self.additive_attention.linear.weight.device
        return ops.user_encoder(user_vector.to(dev), *self._weights(),
                                mode=resolve_mode(self.config, self.precision), ln=self._ln())

    def forward_indexed(self, table, rows):
        """Inference: history rows gathered from the news-vector table (int32 [B, S], S = num_clicked_news_a_user, 1..64).  `table` is the fp32 [n, 300]
        table, or (tensor mode, no LayerNorm) its fp16 copy [n + 1, 320] from `ops.pack_rows_f16`."""
        if table.dtype == torch.float16:
            from ... import _lib
            if self.layer_norm is not None or resolve_mode(self.config, self.precision) != _lib.MODE_TF32:
                raise RuntimeError("the fp16 table form of forward_indexed is the tensor-mode path of the plain NRMS encoder")
            return ops.user_encoder_table16(table, rows, *self._weights())
        return ops.user_encoder_indexed(table, rows, *self._weights(),
                                        mode=resolve_mode(self.config, self.precision), ln=self._ln())
