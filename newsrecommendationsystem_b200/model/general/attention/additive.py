"""AdditiveAttention parameter container.

Mirror of reference src/model/general/attention/additive.py:6-53: Linear(candidate_dim ->
query_dim), query vector ~ U(-0.1, 0.1).  `writer/tag/names` are accepted and ignored (NRMS
passes none: src/model/NRMS/news_encoder.py:24-25).
"""
import torch
import torch.nn as nn


class AdditiveAttention(nn.Module):
    def __init__(self, query_vector_dim, candidate_vector_dim, writer=None, tag=None, names=None):
        super().__init__()
        self.linear = nn.Linear(candidate_vector_dim, query_vector_dim)
        self.attention_query_vector = nn.Parameter(torch.empty(query_vector_dim).uniform_(-0.1, 0.1))
        self.writer = writer
        self.tag = tag
        self.names = names
        self.local_step = 1

    def forward(self, candidate_vector):
        """candidate_vector: batch_size, candidate_size, candidate_vector_dim -> batch_size, candidate_vector_dim.
        Standalone use (candidate_size 1..64; 2..4 is model/Exp1's final attention), forward and backward in
        libnrms_b200; inside the NRMS encoders this block is fused into the encoder kernels."""
        from .... import ops
        from ....config import resolve_mode
        dev = self.linear.weight.device
        return ops.additive_attention(candidate_vector.to(dev), self.linear.weight, self.linear.bias,
                                      self.attention_query_vector,
                                      mode=resolve_mode(None, getattr(self, "precision", None)))
