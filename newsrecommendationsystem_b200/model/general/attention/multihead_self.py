"""MultiHeadSelfAttention parameter container + standalone forward and backward.

Mirror of reference src/model/general/attention/multihead_self.py:26-76: three nn.Linear
(W_Q, W_K, W_V; xavier_uniform weights, :41-44), no output projection.  Inside NewsEncoder /
UserEncoder the projections, the exp-softmax attention and the pooling run inside
libnrms_b200; this class owns the parameters so state_dict keys match the reference.
Called on its own it trains too, with or without the `length` mask: self-attention at 20 and 50 tokens through
nrms_mhsa_*, and cross-attention or any other 1..64 queries and keys through nrms_mha_*.
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
        """Standalone use, in grad mode or not.  Inside NewsEncoder / UserEncoder this block is fused into the
        encoder kernels; NRMS never passes K, V or length (src/model/NRMS/news_encoder.py:41, user_encoder.py:23).
        K = None means K = Q and V = None means V = Q, as in the reference.
          - Self-attention (K and V None or `is Q`) at 20 or 50 tokens: nrms_mhsa_* (ops.mhsa).
          - Everything else with 1..64 queries Sq and 1..64 keys Sk, K and V of the same length: nrms_mha_* (ops.mha),
            cross-attention included.  An input used in two roles (`K is V`, ...) is projected once.
          - Other shapes raise NotImplementedError.
        The `length` mask branch (reference :60-68: keys at positions >= length[b] are multiplied out of the
        exp-softmax; `length` is a host or device integer tensor, one entry per sequence, and gets no gradient) is
        built from Q's length, so it exists where the reference's broadcast defines it: Sk == Sq (the key mask), or
        Sq == 1 (all keys kept iff length >= 1); any other Sq != Sk with a length raises NotImplementedError.
        Gradients reach Q, K, V and the six parameters (through torch.cat in packed())."""
        from .... import ops
        from ....config import resolve_mode
        K = Q if K is None else K
        V = Q if V is None else V
        mode = resolve_mode(None, getattr(self, "precision", None))
        if K is Q and V is Q and Q.dim() == 3 and Q.shape[1] in (20, 50):
            wqkv, bqkv = self.packed()
            return ops.mhsa(Q.to(self.W_Q.weight.device), wqkv, bqkv, mode=mode, length=length)
        ops.mha_check(Q, K, V, length)
        dev = self.W_Q.weight.device
        Qd = Q.to(dev)                                   # each distinct input moved once: aliases stay aliases
        Kd = Qd if K is Q else K.to(dev)
        Vd = Qd if V is Q else (Kd if V is K else V.to(dev))
        wqkv, bqkv = self.packed()
        return ops.mha(Qd, Kd, Vd, wqkv, bqkv, mode=mode, length=length)
