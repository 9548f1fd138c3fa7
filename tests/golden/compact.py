"""How the golden fixtures stay small: the layout the generators (make_golden*.py) save and the tests read back.

The generators draw parameters and inputs from seeded generators and run the reference modules on them.  A fixture
keeps the reference's outputs; the seeded arrays are rebuilt here (`expand_*`) and only the SHA-256 of the bytes the
generator saw is stored, so a rebuilt array is bit-identical to the original or the test fails.  Of the large
parameter-shaped reference outputs (gradients, optimizer steps) and of the masked self-attention output the fixtures
keep a fixed sample (`pinned`, `context_positions`), a sampled array with the largest |entry| of the whole one under
"absmax/" + key: the scale the tests' tolerances are relative to."""
import hashlib

import numpy as np

from newsrecommendationsystem_b200 import synthetic

EMB_KEY = "news_encoder.word_embedding.weight"


def digest(a):
    a = np.ascontiguousarray(a)
    return hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()


def pinned(a, rows=None):
    """The entries of a parameter-shaped reference array that a fixture keeps: a vector whole; of a matrix's first
    `rows` rows (all of them by default) every 6th row and every 4th column."""
    return a[:rows:6, ::4] if a.ndim == 2 else a


def context_positions(S):
    """The query positions of the masked self-attention output that the fixture keeps."""
    return np.array([0, 1, S // 2, S - 1])


def _pin(out, prefixes):
    kept = {}
    for k, v in out.items():
        if k.startswith(prefixes):
            kept["absmax/" + k] = np.float64(np.abs(v).max())
            v = pinned(v)
        kept[k] = v
    return kept


def _store_digests(out, keys):
    kept = {k: v for k, v in out.items() if k not in keys}
    kept.update({"sha256/" + k: np.array(digest(out[k])) for k in keys})
    return kept


def _rebuilt(z, arrays, what):
    """The fixture's arrays with `arrays` added, after checking them against the stored digests."""
    bad = [k for k, a in arrays.items() if digest(a) != str(z["sha256/" + k])]
    if bad:
        raise AssertionError(f"{what}: rebuilt arrays differ from the ones the fixture was generated with: {bad}")
    d = {k: z[k] for k in z.files if not k.startswith("sha256/")}
    d.update(arrays)
    return d


# ---- seeded parameters and inputs ----------------------------------------------------------------------------------
def nrms_state(num_words=401, dim=300, query_dim=200, seed=0):
    """The reference NRMS's parameters after torch.manual_seed(seed): the construction order and init rules of its
    modules (src/model/NRMS, src/model/general/attention) restated with stock torch.nn."""
    import torch
    import torch.nn as nn
    torch.manual_seed(seed)
    sd = {EMB_KEY: nn.Embedding(num_words, dim, padding_idx=0).weight}
    for enc in ("news_encoder", "user_encoder"):
        lin = {w: nn.Linear(dim, dim) for w in ("W_Q", "W_K", "W_V")}
        for w, m in lin.items():
            nn.init.xavier_uniform_(m.weight, gain=1)
            sd[f"{enc}.multihead_self_attention.{w}.weight"] = m.weight
            sd[f"{enc}.multihead_self_attention.{w}.bias"] = m.bias
        add = nn.Linear(dim, query_dim)
        sd[f"{enc}.additive_attention.attention_query_vector"] = torch.empty(query_dim).uniform_(-0.1, 0.1)
        sd[f"{enc}.additive_attention.linear.weight"] = add.weight
        sd[f"{enc}.additive_attention.linear.bias"] = add.bias
    return {k: v.detach().numpy().copy() for k, v in sd.items()}


def nrms_user_input():
    """make_golden.py's user-encoder input: 9 histories of 50 vectors, one partly padded, one empty."""
    ux = np.random.default_rng(7).standard_normal((9, 50, 300)).astype(np.float32) * 0.5
    ux[2, :17] = 0
    ux[3] = 0
    return ux


def _exp1_news(n, rng, abstract=False):
    d = {"title": synthetic.make_news(n, num_words=401, seed=int(rng.integers(1 << 30))),
         "category": rng.integers(0, 31, size=n), "subcategory": rng.integers(0, 31, size=n)}
    if abstract:
        t = rng.integers(1, 401, size=(n, 50))
        lens = rng.integers(1, 51, size=n)
        t[np.arange(50)[None, :] >= lens[:, None]] = 0
        d["abstract"] = t
    return d


def exp1_user_input_and_table():
    """make_golden_exp1.py's user-encoder input and recommend table: its draws from default_rng(5), replayed in order."""
    rng = np.random.default_rng(5)
    _exp1_news(29, rng)
    ux = (rng.standard_normal((7, 50, 300)) * 0.5).astype(np.float32)
    ux[2, :17] = 0
    for _ in range(3 + 50):
        _exp1_news(6, rng)
    _exp1_news(17, rng, abstract=True)
    table = (rng.standard_normal((301, 300)) * 0.4).astype(np.float32)
    table[-1] = 0
    return ux, table


def mhsa_masked_params_and_inputs():
    """make_golden_masked.py's MultiHeadSelfAttention(300, 15) parameters and inputs after torch.manual_seed(7)."""
    import torch
    import torch.nn as nn
    torch.manual_seed(7)
    lin = [nn.Linear(300, 300) for _ in range(3)]
    for m in lin:
        nn.init.xavier_uniform_(m.weight, gain=1)
    with torch.no_grad():
        for m in lin:
            m.bias.uniform_(-0.05, 0.05)
    out = {}
    for n, m in zip("qkv", lin):
        out[f"W{n}"] = m.weight.detach().numpy().copy()
        out[f"b{n}"] = m.bias.detach().numpy().copy()
    for S in (20, 50):
        out[f"S{S}/x"] = (torch.randn(6, S, 300) * 0.5).numpy()
    return out


# ---- nrms_golden.npz -----------------------------------------------------------------------------------------------
_NRMS_SEEDED = ("fwd/gathered", "fwd/user_input")
_NRMS_PINNED = ("train/grad/", "train/adam1/", "train/adam2/", "train/adamw1/")


def compact_nrms(out):
    out = _pin(out, _NRMS_PINNED)
    return _store_digests(out, [k for k in out if k.startswith("sd/")] + list(_NRMS_SEEDED))


def expand_nrms(z):
    sd = nrms_state()
    arrays = {"sd/" + k: v for k, v in sd.items()}
    arrays["fwd/gathered"] = sd[EMB_KEY][z["fwd/tokens"]]
    arrays["fwd/user_input"] = nrms_user_input()
    return _rebuilt(z, arrays, "nrms_golden.npz")


# ---- exp1_golden.npz -----------------------------------------------------------------------------------------------
def compact_exp1(out):
    out = _pin(out, ("grad/",))
    return _store_digests(out, ["fwd/user_input", "rec/table"])


def expand_exp1(z):
    ux, table = exp1_user_input_and_table()
    return _rebuilt(z, {"fwd/user_input": ux, "rec/table": table}, "exp1_golden.npz")


# ---- mhsa_masked_golden.npz ----------------------------------------------------------------------------------------
def compact_masked(out):
    out = dict(out)
    for S in (20, 50):
        out[f"S{S}/pos"] = context_positions(S)
        out[f"S{S}/ctx"] = out[f"S{S}/ctx"][:, out[f"S{S}/pos"]]
    return _store_digests(out, list(mhsa_masked_params_and_inputs()))


def expand_masked(z):
    return _rebuilt(z, mhsa_masked_params_and_inputs(), "mhsa_masked_golden.npz")
