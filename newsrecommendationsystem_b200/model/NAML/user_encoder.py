"""NAML UserEncoder (reference src/model/NAML/user_encoder.py): AdditiveAttention(query_vector_dim, num_filters) over
the clicked news vectors, on libnrms_b200."""
import torch
import torch.nn as nn

from ... import ops
from ...config import resolve_mode
from ..general.attention.additive import AdditiveAttention


class UserEncoder(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.config = config
        self.additive_attention = AdditiveAttention(config.query_vector_dim, config.num_filters)
        self.precision = None

    def forward(self, clicked_news_vector):
        """clicked_news_vector: batch_size, num_clicked_news_a_user, num_filters -> batch_size, num_filters"""
        dev = self.additive_attention.linear.weight.device
        a = self.additive_attention
        return ops.additive_attention(clicked_news_vector.to(dev), a.linear.weight, a.linear.bias,
                                      a.attention_query_vector, mode=resolve_mode(self.config, self.precision))

    @torch.no_grad()
    def forward_indexed(self, table, rows):
        """Inference over rows of a news-vector table: table fp32 [n_rows, 300] on the device, rows integer [U, S] ->
        [U, 300].  The rows are gathered on the device, then pooled by the additive attention."""
        U, S = rows.shape
        x = ops.gather_rows(table, rows.reshape(-1)).view(U, S, ops.D)
        a = self.additive_attention
        return ops.additive_forward(x, a.linear.weight, a.linear.bias, a.attention_query_vector,
                                    mode=resolve_mode(self.config, self.precision))
