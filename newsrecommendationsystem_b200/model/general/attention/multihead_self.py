"""MultiHeadSelfAttention parameter container + standalone forward.

Mirror of reference src/model/general/attention/multihead_self.py:26-76: three nn.Linear
(W_Q, W_K, W_V; xavier_uniform weights, :41-44), no output projection.  Inside NewsEncoder /
UserEncoder the projections, the exp-softmax attention and the pooling run inside
libnrms_b200; this class owns the parameters so state_dict keys match the reference.
"""
import torch
import torch.nn as nn


class MultiHeadSelfAttention(nn.Module):
    def __init__(self, d_model, num_attention_heads):
        super().__init__()
        assert d_model % num_attention_heads == 0
        self.d_model = d_model
        self.num_attention_heads = num_attention_heads
        self.d_k = d_model // num_attention_heads
        self.d_v = d_model // num_attention_heads
        self.W_Q = nn.Linear(d_model, d_model)
        self.W_K = nn.Linear(d_model, d_model)
        self.W_V = nn.Linear(d_model, d_model)
        self._initialize_weights()

    def _initialize_weights(self):
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight, gain=1)

    def packed(self):
        """([W_Q;W_K;W_V] [3D,D], [b_Q;b_K;b_V] [3D]) -- autograd splits the gradients back.

        Without grad mode (inference: evaluate encodes thousands of batches with fixed parameters) the concatenation is
        cached and reused until a parameter is written (tensor version counters) or moved.  Every writer of the
        parameters must bump their version: torch's in-place ops do, and so does FusedAdam.step, whose kernel writes
        through raw pointers."""
        ps = (self.W_Q.weight, self.W_K.weight, self.W_V.weight, self.W_Q.bias, self.W_K.bias, self.W_V.bias)
        if torch.is_grad_enabled():
            return torch.cat(ps[:3], dim=0), torch.cat(ps[3:], dim=0)
        key = tuple((p.data_ptr(), p._version) for p in ps)
        cache = getattr(self, "_packed_cache", None)
        if cache is None or cache[0] != key:
            with torch.no_grad():
                cache = (key, torch.cat(ps[:3], dim=0), torch.cat(ps[3:], dim=0))
            self._packed_cache = cache
        return cache[1], cache[2]

    def forward(self, Q, K=None, V=None, length=None):
        """Standalone use (inference).  Inside NewsEncoder / UserEncoder this block is fused into the encoder
        kernels; NRMS never passes K, V or length (src/model/NRMS/news_encoder.py:41, user_encoder.py:23).  The
        `length` mask branch (reference :60-68: keys at positions >= length[b] are multiplied out of the exp-softmax)
        is compiled for the self-attention form; cross-attention (K or V different from Q) fails loudly."""
        if (K is not None and K is not Q) or (V is not None and V is not Q):
            raise NotImplementedError("libnrms_b200 compiles MultiHeadSelfAttention for K = V = Q (self-attention)")
        if torch.is_grad_enabled() and (Q.requires_grad or self.W_Q.weight.requires_grad):
            raise NotImplementedError("standalone MultiHeadSelfAttention.forward is inference-only; training goes "
                                      "through NewsEncoder / UserEncoder (use torch.no_grad() here)")
        from .... import ops
        from ....config import resolve_mode
        wqkv, bqkv = self.packed()
        return ops.mhsa_forward(Q.to(self.W_Q.weight.device), wqkv, bqkv,
                                mode=resolve_mode(None, getattr(self, "precision", None)), length=length)
