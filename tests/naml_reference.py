"""Two independent restatements of the reference's NAML (src/model/NAML/__init__.py:7-93, news_encoder.py:9-115,
user_encoder.py) -- TEST INFRASTRUCTURE ONLY, the checkers of model/NAML and nrms_cnn_text_*.

* numpy, float64: the conv written out as its sum over the three taps with explicit zero rows at both ends of every text
  (the padding of Conv2d(..., padding=(1, 0))); additive pooling and the element encoders are oracle/nrms_oracle.py's.
* torch (`TorchNAML`): stock torch ops -- F.embedding, F.conv2d (what nn.Conv2d.forward runs), F.relu, the additive
  attention of oracle/torch_port.py -- so that in float64 on the CPU its autograd supplies the reference gradients.

Dropout is given as explicit multiplicative masks (already scaled by 1 / (1 - p)): masks[name] = (mask1, mask2), both
[n * L, 300] over the rows text * L + i of the call, the layout the kernels draw them in; the torch port takes an optional
third entry, the ReLU pattern of TorchNAML.text.  tests/test_naml.py pins the two
restatements against each other on the CPU.
"""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import nrms_oracle as O
from oracle import torch_port as TP

TEXTS = ("title", "abstract")
ELEMENTS = ("category", "subcategory")


def text_prefix(name):
    return f"news_encoder.text_encoders.{name}"


def _add_p(params, prefix):
    return dict(Wa=params[f"{prefix}.linear.weight"], ba=params[f"{prefix}.linear.bias"],
                qa=params[f"{prefix}.attention_query_vector"])


# ---- numpy ------------------------------------------------------------------------------------------------------------
def naml_text_encoder_forward(params, name, text, mask1=None, mask2=None):
    """TextEncoder.forward (news_encoder.py:26-40): x = dropout(embedding(text)) (:33-35); c = CNN(x) with a zero row
    before and after each text (padding (1, 0), :20-24, :36); a = dropout(relu(c)) (:37-38); additive pooling (:39)."""
    pre = text_prefix(name)
    x = O.embedding_gather(params[f"{pre}.word_embedding.weight"], np.asarray(text)).astype(np.float64)
    n, L, D = x.shape
    if mask1 is not None:
        x = x * np.asarray(mask1, np.float64).reshape(n, L, D)
    W = np.asarray(params[f"{pre}.CNN.weight"], np.float64)[:, 0]          # [F, 3, D]
    xp = np.zeros((n, L + 2, D))
    xp[:, 1:L + 1] = x
    c = np.asarray(params[f"{pre}.CNN.bias"], np.float64) + sum(
        np.einsum("nld,fd->nlf", xp[:, w:w + L], W[:, w]) for w in range(3))
    a = np.maximum(c, 0.0)
    if mask2 is not None:
        a = a * np.asarray(mask2, np.float64).reshape(n, L, -1)
    out, _ = O.additive_forward(a, {k: np.asarray(v, np.float64) for k, v in _add_p(params, f"{pre}.additive_attention").items()})
    return out


def naml_news_encoder_forward(params, news, attributes, masks=None):
    """NewsEncoder.forward (news_encoder.py:93-115): text vectors, element vectors, one vector returned as is, else the
    final attention over their stack on dim 1."""
    masks = masks or {}
    vecs = [naml_text_encoder_forward(params, a, news[a], *masks.get(a, (None, None))) for a in TEXTS if a in attributes]
    for a in ELEMENTS:
        if a in attributes:
            pre = f"news_encoder.element_encoders.{a}"
            E, W, b = (np.asarray(params[f"{pre}.{k}"], np.float64) for k in ("embedding.weight", "linear.weight", "linear.bias"))
            vecs.append(O.element_encoder_forward(E, W, b, np.asarray(news[a])))
    if len(vecs) == 1:
        return vecs[0]
    p = {k: np.asarray(v, np.float64) for k, v in _add_p(params, "news_encoder.final_attention").items()}
    return O.additive_forward(np.stack(vecs, axis=1), p)[0]


def naml_user_encoder_forward(params, clicked_news_vector):
    """UserEncoder.forward (user_encoder.py): additive attention over the clicked news vectors."""
    p = {k: np.asarray(v, np.float64) for k, v in _add_p(params, "user_encoder.additive_attention").items()}
    return O.additive_forward(np.asarray(clicked_news_vector, np.float64), p)[0]


def naml_forward(params, news, n_cand, attributes, masks=None):
    """NAML.forward (__init__.py:24-50): news: {attribute: [B, 1+K+N, ...]} (candidates first) -> logits [B, 1+K]."""
    first = news[attributes[0]]
    B, T = first.shape[:2]
    flat = {a: np.asarray(news[a]).reshape(B * T, *np.asarray(news[a]).shape[2:]) for a in attributes}
    vec = naml_news_encoder_forward(params, flat, attributes, masks).reshape(B, T, -1)
    return O.click_score(vec[:, :n_cand], naml_user_encoder_forward(params, vec[:, n_cand:]))


# ---- torch ------------------------------------------------------------------------------------------------------------
class TorchNAML:
    """Float64 leaf tensors under the reference's state_dict keys; the two shared embeddings are one leaf each (their
    gradient is the sum over every encoder that reads them)."""

    def __init__(self, params, attributes):
        self.attributes = list(attributes)
        self.P = {}
        shared = {}
        for k, v in params.items():
            group = None
            if k.startswith("news_encoder.text_encoders.") and k.endswith(".word_embedding.weight"):
                group = "word_embedding"
            elif k.startswith("news_encoder.element_encoders.") and k.endswith(".embedding.weight"):
                group = "category_embedding"
            leaf = shared.get(group)
            if leaf is None:
                leaf = torch.tensor(np.asarray(v, np.float64), requires_grad=True)
                if group is not None:
                    shared[group] = leaf
            self.P[k] = leaf

    def text(self, name, text, mask1=None, mask2=None, relu_on=None):
        """relu_on ([n * L, 300], optional): where the ReLU passes, taken from another computation of the same conv (the
        kernel's relu(conv) > 0).  A pre-activation within rounding of 0 may fall on either side of the ReLU; its value is
        ~0 either way, but its derivative is 0 or 1, so gradients are compared at the pattern the kernel used."""
        pre = text_prefix(name)
        x = F.embedding(torch.as_tensor(np.asarray(text)), self.P[f"{pre}.word_embedding.weight"], padding_idx=0)
        n, L, D = x.shape
        if mask1 is not None:
            x = x * torch.as_tensor(np.asarray(mask1, np.float64)).view(n, L, D)
        c = F.conv2d(x.unsqueeze(1), self.P[f"{pre}.CNN.weight"], self.P[f"{pre}.CNN.bias"], padding=(1, 0)).squeeze(3)
        if relu_on is None:
            a = F.relu(c).transpose(1, 2)
        else:
            a = c.transpose(1, 2) * torch.as_tensor(np.asarray(relu_on, np.float64)).view(n, L, -1)
        if mask2 is not None:
            a = a * torch.as_tensor(np.asarray(mask2, np.float64)).view(n, L, -1)
        return TP.additive(a, {k: self.P[v] for k, v in
                               dict(Wa=f"{pre}.additive_attention.linear.weight", ba=f"{pre}.additive_attention.linear.bias",
                                    qa=f"{pre}.additive_attention.attention_query_vector").items()})

    def news(self, news, masks=None):
        masks = masks or {}
        vecs = [self.text(a, news[a], *masks.get(a, ())) for a in TEXTS if a in self.attributes]
        for a in ELEMENTS:
            if a in self.attributes:
                pre = f"news_encoder.element_encoders.{a}"
                e = F.embedding(torch.as_tensor(np.asarray(news[a])), self.P[f"{pre}.embedding.weight"], padding_idx=0)
                vecs.append(F.relu(F.linear(e, self.P[f"{pre}.linear.weight"], self.P[f"{pre}.linear.bias"])))
        if len(vecs) == 1:
            return vecs[0]
        pf = "news_encoder.final_attention"
        return TP.additive(torch.stack(vecs, dim=1), dict(Wa=self.P[f"{pf}.linear.weight"], ba=self.P[f"{pf}.linear.bias"],
                                                         qa=self.P[f"{pf}.attention_query_vector"]))

    def user(self, clicked):
        pu = "user_encoder.additive_attention"
        return TP.additive(clicked, dict(Wa=self.P[f"{pu}.linear.weight"], ba=self.P[f"{pu}.linear.bias"],
                                         qa=self.P[f"{pu}.attention_query_vector"]))

    def forward(self, news, n_cand, masks=None):
        first = np.asarray(news[self.attributes[0]])
        B, T = first.shape[:2]
        flat = {a: np.asarray(news[a]).reshape(B * T, *np.asarray(news[a]).shape[2:]) for a in self.attributes}
        vec = self.news(flat, masks).view(B, T, -1)
        return torch.bmm(vec[:, :n_cand], self.user(vec[:, n_cand:]).unsqueeze(-1)).squeeze(-1)

    def loss_and_grads(self, news, n_cand, masks=None):
        """CrossEntropyLoss against label 0 (src/train.py:126,205-206) and every key's gradient (shared leaves: the sum)."""
        for v in self.P.values():
            v.grad = None
        logits = self.forward(news, n_cand, masks)
        loss = F.cross_entropy(logits, torch.zeros(logits.shape[0], dtype=torch.long))
        loss.backward()
        return logits.detach().numpy(), float(loss), {k: v.grad.numpy().copy() for k, v in self.P.items()}


def model_params(model):
    """float64 numpy copies of a model's state_dict."""
    return {k: v.detach().cpu().double().numpy().copy() for k, v in model.state_dict().items()}


def random_news(rng, B, T, attributes, lengths, num_words, num_categories, zero_tail=True):
    """{attribute: [B, T, ...]} token / element ids; texts end in a run of padding (token 0), as the reference's
    tokeniser pads them (src/data_preprocess.py)."""
    out = {}
    for a in attributes:
        if a in TEXTS:
            L = lengths[a]
            t = rng.integers(1, num_words, size=(B, T, L))
            if zero_tail:
                keep = rng.integers(1, L + 1, size=(B, T))
                t = np.where(np.arange(L)[None, None] < keep[..., None], t, 0)
            out[a] = t.astype(np.int64)
        else:
            out[a] = rng.integers(0, num_categories, size=(B, T)).astype(np.int64)
    return out
