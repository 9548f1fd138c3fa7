"""Two independent restatements of the reference's LSTUR (src/model/LSTUR/__init__.py, news_encoder.py,
user_encoder.py) -- TEST INFRASTRUCTURE ONLY, the checkers of model/LSTUR and nrms_gru_*.

* numpy, float64: the GRU equations (torch's gate order r, z, n) with an explicit loop over each user's rows
  [0, length), and their backward written out step by step; the title path is tests/naml_reference.py's numpy CNN text
  encoder.
* torch (`TorchLSTUR`): stock torch pieces called the way the reference calls them -- F.embedding, F.conv2d, the additive
  attention of oracle/torch_port.py, and nn.GRU fed through pack_padded_sequence(..., batch_first=True,
  enforce_sorted=False) -- so that in float64 on the CPU its autograd supplies the reference gradients.

Dropout is given as explicit multiplicative masks: the title's two masks as in naml_reference ([n * L, 300] each, plus an
optional ReLU pattern), and the user-embedding mask as one factor per user row (0 or 1 / (1 - p)), which is what
F.dropout2d does to embedding(user).unsqueeze(0).  tests/test_lstur.py pins the two restatements against each other.
"""
import numpy as np
import torch
import torch.nn.functional as F

import naml_reference as NR
from oracle import torch_port as TP

GRU_KEYS = ("user_encoder.gru.weight_ih_l0", "user_encoder.gru.weight_hh_l0", "user_encoder.gru.bias_ih_l0",
            "user_encoder.gru.bias_hh_l0")


def _sig(x):
    return 1.0 / (1.0 + np.exp(-x))


# ---- numpy ------------------------------------------------------------------------------------------------------------
def gru_forward(w_ih, w_hh, b_ih, b_hh, x, lengths, h0=None):
    """Last hidden state of nn.GRU over rows [0, lengths[b]) of x [B, T, I], from h0 (None: zeros).  Also returns the
    per-step cache the backward reads."""
    w_ih, w_hh, b_ih, b_hh, x = (np.asarray(a, np.float64) for a in (w_ih, w_hh, b_ih, b_hh, x))
    B, T, _ = x.shape
    H = w_hh.shape[1]
    out = np.zeros((B, H)) if h0 is None else np.array(h0, np.float64)
    cache = []
    for b in range(B):
        h = out[b].copy()
        steps = []
        for t in range(int(lengths[b])):
            gi = w_ih @ x[b, t] + b_ih
            gh = w_hh @ h + b_hh
            r = _sig(gi[:H] + gh[:H])
            z = _sig(gi[H:2 * H] + gh[H:2 * H])
            n = np.tanh(gi[2 * H:] + r * gh[2 * H:])
            steps.append((h, r, z, n, gh[2 * H:]))
            h = (1 - z) * n + z * h
        out[b] = h
        cache.append(steps)
    return out, cache


def gru_backward(w_ih, w_hh, x, lengths, cache, d_out):
    """Gradients of sum(d_out * h_last) for gru_forward: d_x (zero past each length), d_h0, d_w_ih, d_w_hh, d_b_ih,
    d_b_hh."""
    w_ih, w_hh, x, d_out = (np.asarray(a, np.float64) for a in (w_ih, w_hh, x, d_out))
    B, T, I = x.shape
    H = w_hh.shape[1]
    g = dict(x=np.zeros((B, T, I)), h0=np.zeros((B, H)), w_ih=np.zeros((3 * H, I)), w_hh=np.zeros((3 * H, H)),
             b_ih=np.zeros(3 * H), b_hh=np.zeros(3 * H))
    for b in range(B):
        dh = d_out[b].copy()
        for t in range(int(lengths[b]) - 1, -1, -1):
            hp, r, z, n, ghn = cache[b][t]
            dnp = dh * (1 - z) * (1 - n * n)
            dzp = dh * (hp - n) * z * (1 - z)
            drp = dnp * ghn * r * (1 - r)
            dgi = np.concatenate([drp, dzp, dnp])
            dgh = np.concatenate([drp, dzp, dnp * r])
            g["w_ih"] += np.outer(dgi, x[b, t])
            g["b_ih"] += dgi
            g["w_hh"] += np.outer(dgh, hp)
            g["b_hh"] += dgh
            g["x"][b, t] = w_ih.T @ dgi
            dh = dh * z + w_hh.T @ dgh
        g["h0"][b] = dh
    return g


def _naml_title_params(params):
    pre = NR.text_prefix("title")
    ne = "news_encoder"
    return {f"{pre}.word_embedding.weight": params[f"{ne}.word_embedding.weight"],
            f"{pre}.CNN.weight": params[f"{ne}.title_CNN.weight"], f"{pre}.CNN.bias": params[f"{ne}.title_CNN.bias"],
            f"{pre}.additive_attention.linear.weight": params[f"{ne}.title_attention.linear.weight"],
            f"{pre}.additive_attention.linear.bias": params[f"{ne}.title_attention.linear.bias"],
            f"{pre}.additive_attention.attention_query_vector": params[f"{ne}.title_attention.attention_query_vector"]}


def news_forward(params, news, title_masks=(None, None)):
    """NewsEncoder.forward: cat([category_embedding(category), category_embedding(subcategory), title vector])."""
    E = np.asarray(params["news_encoder.category_embedding.weight"], np.float64)
    title = NR.naml_text_encoder_forward(_naml_title_params(params), "title", news["title"], *title_masks[:2])
    return np.concatenate([E[np.asarray(news["category"])], E[np.asarray(news["subcategory"])], title], axis=1)


def user_forward(params, method, user_vec, clicked_news_length, clicked_news_vector):
    """UserEncoder.forward: lengths of 0 read as 1, the GRU from user_vec (ini) or from zero then cat with it (con)."""
    lengths = np.maximum(np.asarray(clicked_news_length), 1)
    h, _ = gru_forward(*(params[k] for k in GRU_KEYS), clicked_news_vector, lengths,
                       user_vec if method == "ini" else None)
    return h if method == "ini" else np.concatenate([h, user_vec], axis=1)


def lstur_forward(params, method, user, clicked_news_length, news, n_cand, title_masks=(None, None), user_mask=None):
    """LSTUR.forward: news {attribute: [B, 1+K+N, ...]} (candidates first) -> logits [B, 1+K]."""
    B, T = np.asarray(news["title"]).shape[:2]
    flat = {a: np.asarray(v).reshape(B * T, *np.asarray(v).shape[2:]) for a, v in news.items()}
    vec = news_forward(params, flat, title_masks).reshape(B, T, -1)
    u = np.asarray(params["user_embedding.weight"], np.float64)[np.asarray(user)]
    if user_mask is not None:
        u = u * np.asarray(user_mask, np.float64)[:, None]
    uv = user_forward(params, method, u, clicked_news_length, vec[:, n_cand:])
    return np.einsum("bcd,bd->bc", vec[:, :n_cand], uv)


# ---- torch ------------------------------------------------------------------------------------------------------------
def torch_gru(gru, x, lengths, h0=None):
    """The reference's call: gru(pack_padded_sequence(x, lengths, batch_first=True, enforce_sorted=False), h0) -> h."""
    packed = torch.nn.utils.rnn.pack_padded_sequence(x, torch.as_tensor(np.asarray(lengths), dtype=torch.long),
                                                     batch_first=True, enforce_sorted=False)
    _, h = gru(packed) if h0 is None else gru(packed, h0.unsqueeze(0))
    return h.squeeze(0)


class TorchLSTUR:
    """Float64 leaf tensors under the reference's state_dict keys; the GRU is a float64 nn.GRU holding the GRU keys."""

    def __init__(self, params, method):
        self.method = method
        I, H = np.asarray(params["user_encoder.gru.weight_ih_l0"]).shape[1], np.asarray(
            params["user_encoder.gru.weight_hh_l0"]).shape[1]
        self.gru = torch.nn.GRU(I, H).double()
        with torch.no_grad():
            for k in GRU_KEYS:
                getattr(self.gru, k.rsplit(".", 1)[1]).copy_(torch.as_tensor(np.asarray(params[k], np.float64)))
        self.P = {k: torch.tensor(np.asarray(v, np.float64), requires_grad=True) for k, v in params.items()
                  if k not in GRU_KEYS}
        for k in GRU_KEYS:
            self.P[k] = getattr(self.gru, k.rsplit(".", 1)[1])

    def news(self, news, title_masks=()):
        pre = "news_encoder"
        E = self.P[f"{pre}.category_embedding.weight"]
        cat = F.embedding(torch.as_tensor(np.asarray(news["category"])), E, padding_idx=0)
        sub = F.embedding(torch.as_tensor(np.asarray(news["subcategory"])), E, padding_idx=0)
        x = F.embedding(torch.as_tensor(np.asarray(news["title"])), self.P[f"{pre}.word_embedding.weight"], padding_idx=0)
        n, L, D = x.shape
        m = list(title_masks) + [None] * (3 - len(title_masks))
        if m[0] is not None:
            x = x * torch.as_tensor(np.asarray(m[0], np.float64)).view(n, L, D)
        c = F.conv2d(x.unsqueeze(1), self.P[f"{pre}.title_CNN.weight"], self.P[f"{pre}.title_CNN.bias"],
                     padding=(1, 0)).squeeze(3)
        if m[2] is None:
            a = F.relu(c).transpose(1, 2)
        else:
            a = c.transpose(1, 2) * torch.as_tensor(np.asarray(m[2], np.float64)).view(n, L, -1)
        if m[1] is not None:
            a = a * torch.as_tensor(np.asarray(m[1], np.float64)).view(n, L, -1)
        pa = f"{pre}.title_attention"
        title = TP.additive(a, dict(Wa=self.P[f"{pa}.linear.weight"], ba=self.P[f"{pa}.linear.bias"],
                                    qa=self.P[f"{pa}.attention_query_vector"]))
        return torch.cat([cat, sub, title], dim=1)

    def user(self, user_vec, clicked_news_length, clicked_news_vector):
        lengths = torch.as_tensor(np.asarray(clicked_news_length)).clone()
        lengths[lengths == 0] = 1
        if self.method == "ini":
            return torch_gru(self.gru, clicked_news_vector, lengths, user_vec)
        return torch.cat([torch_gru(self.gru, clicked_news_vector, lengths), user_vec], dim=1)

    def user_rows(self, user, user_mask=None):
        u = F.embedding(torch.as_tensor(np.asarray(user)), self.P["user_embedding.weight"], padding_idx=0)
        if user_mask is not None:
            u = u * torch.as_tensor(np.asarray(user_mask, np.float64)).unsqueeze(1)
        return u

    def forward(self, user, clicked_news_length, news, n_cand, title_masks=(), user_mask=None):
        B, T = np.asarray(news["title"]).shape[:2]
        flat = {a: np.asarray(v).reshape(B * T, *np.asarray(v).shape[2:]) for a, v in news.items()}
        vec = self.news(flat, title_masks).view(B, T, -1)
        uv = self.user(self.user_rows(user, user_mask), clicked_news_length, vec[:, n_cand:])
        return torch.bmm(vec[:, :n_cand], uv.unsqueeze(-1)).squeeze(-1)

    def loss_and_grads(self, user, clicked_news_length, news, n_cand, title_masks=(), user_mask=None):
        """CrossEntropyLoss against label 0 and every key's gradient."""
        for v in self.P.values():
            v.grad = None
        logits = self.forward(user, clicked_news_length, news, n_cand, title_masks, user_mask)
        loss = F.cross_entropy(logits, torch.zeros(logits.shape[0], dtype=torch.long))
        loss.backward()
        return logits.detach().numpy(), float(loss.detach()), {k: v.grad.numpy().copy() for k, v in self.P.items()}


def random_params(rng, method, num_words=300, num_categories=20, num_users=40, scale_gru=1.0):
    """A float32-representable LSTUR state_dict in float64: torch's init ranges (nn.GRU uniform +-1/sqrt(H), embeddings
    N(0, 1) with row 0 zeroed)."""
    H = 900 if method == "ini" else 450
    k = 1 / np.sqrt(H)

    def f32(a):
        return np.asarray(a, np.float32).astype(np.float64)
    emb = rng.standard_normal((num_words, 300))
    emb[0] = 0
    cat = rng.standard_normal((num_categories, 300))
    cat[0] = 0
    usr = rng.standard_normal((num_users, H))
    usr[0] = 0
    return {
        "news_encoder.word_embedding.weight": f32(emb),
        "news_encoder.category_embedding.weight": f32(cat),
        "news_encoder.title_CNN.weight": f32(rng.standard_normal((300, 1, 3, 300)) * 0.035),
        "news_encoder.title_CNN.bias": f32(rng.choice([-4.0, 4.0], 300)),
        "news_encoder.title_attention.attention_query_vector": f32(rng.uniform(-0.1, 0.1, 200)),
        "news_encoder.title_attention.linear.weight": f32(rng.standard_normal((200, 300)) * 0.01),
        "news_encoder.title_attention.linear.bias": f32(rng.standard_normal(200) * 0.1),
        "user_encoder.gru.weight_ih_l0": f32(rng.uniform(-k, k, (3 * H, 900)) * scale_gru),
        "user_encoder.gru.weight_hh_l0": f32(rng.uniform(-k, k, (3 * H, H)) * scale_gru),
        "user_encoder.gru.bias_ih_l0": f32(rng.uniform(-k, k, 3 * H)),
        "user_encoder.gru.bias_hh_l0": f32(rng.uniform(-k, k, 3 * H)),
        "user_embedding.weight": f32(usr),
    }
