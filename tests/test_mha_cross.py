"""The standalone MultiHeadSelfAttention beyond K = V = Q at 20 and 50 tokens: cross-attention (K and / or V other
inputs than Q) and any 1..64 queries and keys, forward and backward (nrms_mha_fwd / nrms_mha_bwd, ops.mha).

CPU part: a torch fp64 autograd transcription of the reference forward(Q, K, V, length) (src/model/general/attention/
multihead_self.py:15-23,46-76), pinned against the oracle on the inputs of mhsa_masked_golden.npz and on a hand-checked
Sq = 1 case; the ABI's argument errors, aliasing rule and workspace sizes; the Python shape rules.
GPU part (`-m gpu`): the forward and every gradient against the transcription over a grid of shapes and input forms in
both modes, the exact and bitwise properties, agreement with the 20 / 50-token path, and FusedAdam steps of a small
candidate-over-history model.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import nrms_oracle as O
from compact import expand_masked
from conftest import GOLDEN

GTOL = {"fp32": 2e-4, "tf32": 3e-3}       # gradients: of the largest entry of the reference gradient (test_mhsa_train.py)
FTOL = {"fp32": 2e-5, "tf32": 1.5e-3}     # forward: row-wise relative L2, max over all rows.  Tensor mode: TF32 projections
                                          # and attention; the worst of 450k rows at 7,040 sequences reached 1.1e-3
PNAMES = ("W_Q.weight", "W_Q.bias", "W_K.weight", "W_K.bias", "W_V.weight", "W_V.bias")


# ---- the fp64 transcription ----------------------------------------------------------------------------------------
def mha_ref(xq, xk, xv, Wq, bq, Wk, bk, Wv, bv, length=None):
    """multihead_self.py:15-23,46-76: e = exp(q k^T / sqrt 20) * mask, attn = e / (sum_j e + 1e-8), ctx = attn v.
    The mask is built from maxlen = Q.size(1): [B, H, Sq, Sq] of j < length[b], which multiplies the [B, H, Sq, Sk]
    scores where it broadcasts -- Sk == Sq (the key mask) or Sq == 1 ([B, H, 1, 1]: every key kept iff length >= 1)."""
    n, sq, _ = xq.shape
    sk = xk.shape[1]

    def heads(x, W, b):
        return torch.nn.functional.linear(x, W, b).view(n, x.shape[1], 15, 20).transpose(1, 2)
    q, k, v = heads(xq, Wq, bq), heads(xk, Wk, bk), heads(xv, Wv, bv)
    e = torch.exp(q @ k.transpose(-1, -2) / np.sqrt(20.0))
    if length is not None:
        L = torch.as_tensor(np.asarray(length), device=xq.device).view(n, 1, 1, 1)
        mask = (torch.arange(sq, device=xq.device).view(1, 1, 1, sq) < L).to(e.dtype)      # [B, 1, 1, Sq]
        if sq != sk and sq != 1:
            raise ValueError("the reference's mask does not broadcast")
        e = e * mask
    attn = e / (e.sum(-1, keepdim=True) + 1e-8)
    return (attn @ v).transpose(1, 2).reshape(n, sq, 300)


def _golden():
    import os
    return expand_masked(np.load(os.path.join(GOLDEN, "mhsa_masked_golden.npz")))


def test_transcription_pinned_against_oracle():
    """With K = V = Q the transcription equals the oracle's forward on the fixture's inputs, masked and unmasked."""
    g = _golden()
    P = {k: g[k].astype(np.float64) for k in ("Wq", "bq", "Wk", "bk", "Wv", "bv")}
    p = [torch.from_numpy(P[k]) for k in ("Wq", "bq", "Wk", "bk", "Wv", "bv")]
    for S in (20, 50):
        x = g[f"S{S}/x"].astype(np.float64)
        for length in (g[f"S{S}/length"], None):
            ref, _ = O.mhsa_forward(x, P, 15, length=length)
            xt = torch.from_numpy(x)
            got = mha_ref(xt, xt, xt, *p, length=length).numpy()
            np.testing.assert_allclose(got, ref, rtol=0, atol=1e-12)


def test_transcription_one_query_broadcast():
    """Sq = 1 < Sk: the reference's [B, H, 1, 1] mask keeps every key iff length >= 1 (not the first `length` keys).
    W_Q = W_K = 0 makes every score 0 and W_V = I makes v_j = xk_j, so ctx = sum_j xk_j / (Sk + 1e-8) or 0."""
    torch.manual_seed(0)
    n, sk = 4, 3
    xq = torch.randn(n, 1, 300, dtype=torch.float64)
    xk = torch.randn(n, sk, 300, dtype=torch.float64)
    z, zb = torch.zeros(300, 300, dtype=torch.float64), torch.zeros(300, dtype=torch.float64)
    eye = torch.eye(300, dtype=torch.float64)
    got = mha_ref(xq, xk, xk, z, zb, z, zb, eye, zb, length=[0, 1, 2, -1])
    full = xk.sum(1) / (sk + 1e-8)
    assert torch.equal(got[0, 0], torch.zeros(300, dtype=torch.float64))
    assert torch.equal(got[3, 0], torch.zeros(300, dtype=torch.float64))
    torch.testing.assert_close(got[1, 0], full[1], rtol=0, atol=1e-15)
    torch.testing.assert_close(got[2, 0], full[2], rtol=0, atol=1e-15)
    with pytest.raises(ValueError):
        mha_ref(xk[:, :2], xk, xk, z, zb, z, zb, eye, zb, length=[1, 1, 1, 1])


# ---- ABI -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from newsrecommendationsystem_b200 import _lib
    return _lib.load()


def _al(nbytes):
    return (nbytes + 255) // 256 * 256


def _fwd_ws(n, sq, sk):
    return _al(n * sq * 900 * 4) + 2 * _al(n * sk * 300 * 4)


def _bwd_ws(n, sq, sk, mode):
    ldr = (n * max(sq, sk) + 3) // 4 * 4
    b = _fwd_ws(n, sq, sk) + _al(296 * 900 * 4)
    if mode == 1:
        b += _al(ldr * 900 * 4) + _al(ldr * 300 * 4) + _al(900 * 300 * 4)
    return b


def test_mha_workspace_sizes(lib):
    for n in (1, 7, 7040):
        for sq, sk in ((1, 1), (5, 50), (50, 20), (64, 64), (33, 7)):
            assert lib.nrms_mha_fwd_workspace_bytes(n, sq, sk) == _fwd_ws(n, sq, sk)
            for mode in (0, 1):
                assert lib.nrms_mha_bwd_workspace_bytes(n, sq, sk, mode) == _bwd_ws(n, sq, sk, mode)
    assert lib.nrms_mha_fwd_workspace_bytes(0, 5, 5) == 0
    assert lib.nrms_mha_bwd_workspace_bytes(0, 5, 5, 1) == 0


A, B_, X3, G, W, F, WS, CT = (C.c_void_p((k + 1) << 24) for k in range(8))     # aligned, never dereferenced


def test_mha_fwd_arguments(lib):
    need = lib.nrms_mha_fwd_workspace_bytes(7, 5, 50)

    def call(xq=A, xk=B_, xv=B_, n=7, sq=5, sk=50, lengths=None, w=W, b=W, ctx=CT, ws=WS, ws_bytes=need, mode=1):
        return lib.nrms_mha_fwd(xq, xk, xv, n, sq, sk, lengths, w, b, ctx, ws, ws_bytes, mode, None)

    for sq, sk in ((0, 5), (5, 0), (65, 5), (5, 65), (-1, 5)):
        assert call(sq=sq, sk=sk) == 2 and b"unsupported" in lib.nrms_last_error(), (sq, sk)
    assert call(lengths=G) == 2                                     # 5 queries, 50 keys: the mask does not broadcast
    assert call(mode=7) == 1
    assert call(n=-1) == 1
    assert call(n=0, xq=None, xk=None, xv=None, ws=None) == 0      # nothing to do
    for k in ("xq", "xk", "xv", "w", "b", "ctx"):
        assert call(**{k: None}) == 1 and b"null" in lib.nrms_last_error(), k
    for k in ("xq", "xk", "xv", "w", "b", "ctx"):
        assert call(**{k: C.c_void_p((1 << 24) * 9 + 4)}) == 1 and b"aligned" in lib.nrms_last_error(), k
    assert call(sq=50, lengths=C.c_void_p((1 << 24) + 2)) == 1
    assert call(xk=A, xv=A) == 1                                    # Q's input as K's with 5 vs 50 rows
    assert call(ctx=A) == 1 and call(ctx=B_) == 1                   # ctx over an input
    assert call(ws_bytes=need - 1) == 3 and b"workspace" in lib.nrms_last_error()
    assert call(ws=None) == 3
    assert call(ws=C.c_void_p((8 << 24) + 8)) == 1 and b"aligned" in lib.nrms_last_error()
    # masks the reference defines: Sq == Sk, and Sq == 1; each is refused here for its workspace only
    assert call(sq=50, sk=50, lengths=G, ws_bytes=0) == 3
    assert call(sq=1, sk=50, lengths=G, ws_bytes=0) == 3


def test_mha_bwd_arguments_and_aliasing(lib):
    need = lib.nrms_mha_bwd_workspace_bytes(7, 20, 20, 1)

    def call(d_ctx=G, xq=A, xk=B_, xv=X3, n=7, sq=20, sk=20, lengths=None, w=W, fws=F, dq=C.c_void_p(10 << 24),
             dk=C.c_void_p(11 << 24), dv=C.c_void_p(12 << 24), dw=C.c_void_p(13 << 24), db=C.c_void_p(14 << 24), ws=WS,
             ws_bytes=need, mode=1):
        return lib.nrms_mha_bwd(d_ctx, xq, xk, xv, n, sq, sk, lengths, w, fws, dq, dk, dv, dw, db, ws, ws_bytes, mode, None)

    for sq, sk in ((0, 5), (65, 64), (64, 65)):
        assert call(sq=sq, sk=sk) == 2, (sq, sk)
    assert call(sq=5, lengths=G) == 2
    assert call(mode=2) == 1
    assert call(n=-1) == 1
    assert call(n=0, d_ctx=None, xq=None, ws=None) == 0
    for k in ("d_ctx", "xq", "xk", "xv", "w", "fws", "dw", "db"):
        assert call(**{k: None}) == 1 and b"null" in lib.nrms_last_error(), k
    for k in ("d_ctx", "xq", "xk", "xv", "w", "fws", "dw", "dq", "dk", "dv"):
        assert call(**{k: C.c_void_p((15 << 24) + 8)}) == 1 and b"aligned" in lib.nrms_last_error(), k
    D1, D2 = C.c_void_p(10 << 24), C.c_void_p(11 << 24)
    # the same input twice: one gradient buffer, or NULL for the alias (checked up to the workspace size)
    assert call(xk=A, dk=D1, ws_bytes=0) == 3
    assert call(xk=A, dk=None, ws_bytes=0) == 3
    assert call(xk=A, dq=None, dk=D1, ws_bytes=0) == 3
    assert call(xk=A, xv=A, dk=D1, dv=D1, ws_bytes=0) == 3
    assert call(xk=A, dk=D2) == 1 and b"gradient" in lib.nrms_last_error()
    assert call(xv=B_, dv=C.c_void_p(12 << 24)) == 1
    assert call(xk=A, xv=A, dk=None, dv=D2) == 1
    # distinct inputs: distinct buffers, none of them an input
    assert call(dk=D1) == 1 and b"distinct" in lib.nrms_last_error()
    assert call(dv=D2) == 1
    assert call(dq=A) == 1 and call(dk=X3) == 1 and call(dv=G) == 1
    assert call(ws_bytes=need - 1) == 3 and b"workspace" in lib.nrms_last_error()
    assert call(ws_bytes=lib.nrms_mha_bwd_workspace_bytes(7, 20, 20, 0)) == 3      # FP32-mode size in tensor mode
    assert call(dq=None, dk=None, dv=None, ws_bytes=0) == 3                      # no input gradient at all is fine
    assert call(ws=C.c_void_p((7 << 24) + 8)) == 1 and b"aligned" in lib.nrms_last_error()
    assert call(db=C.c_void_p((14 << 24) + 4)) == 1 and b"aligned" in lib.nrms_last_error()


def _cpu_module():
    from newsrecommendationsystem_b200.model.general.attention.multihead_self import MultiHeadSelfAttention
    torch.manual_seed(0)
    return MultiHeadSelfAttention(300, 15)


def test_python_shape_rules():
    """The shapes the reference leaves undefined or the library does not compile raise NotImplementedError before any
    device work; CPU tensors are refused (there is no CPU fallback)."""
    m = _cpu_module()
    x = torch.randn(3, 20, 300)
    y = torch.randn(3, 50, 300)
    with pytest.raises(NotImplementedError):
        m(x, K=x[:, :5])                                        # V = Q has 20 rows, K 5
    with pytest.raises(NotImplementedError):
        m(x, K=y, V=torch.randn(3, 49, 300))                    # K and V rows differ
    with pytest.raises(NotImplementedError):
        m(torch.randn(3, 65, 300))                              # above 64
    with pytest.raises(NotImplementedError):
        m(x, K=torch.randn(3, 65, 300), V=torch.randn(3, 65, 300))
    with pytest.raises(NotImplementedError):
        m(torch.randn(3, 0, 300))
    with pytest.raises(NotImplementedError):
        m(torch.randn(3, 5, 300), K=y, V=y, length=torch.tensor([1, 2, 3]))     # [B, 5] mask over 50 keys
    with pytest.raises(RuntimeError):
        m(x, K=torch.randn(2, 50, 300), V=torch.randn(2, 50, 300))            # batch differs
    for args in ((torch.randn(3, 5, 300), y, y), (torch.randn(3, 30, 300),), (torch.randn(3, 1, 300), y, y)):
        kw = {"K": args[1], "V": args[2]} if len(args) == 3 else {}
        with pytest.raises(RuntimeError, match="CUDA"):
            m(args[0], **kw)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.randn(3, 1, 300), K=y, V=y, length=torch.tensor([0, 1, 5]))
    from newsrecommendationsystem_b200 import ops
    wqkv, bqkv = m.packed()
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.mha(torch.randn(2, 5, 300), y[:2], y[:2], wqkv, bqkv)
    with pytest.raises(NotImplementedError):
        ops.mha(torch.randn(2, 5, 300), y[:2], None, wqkv, bqkv)        # V = Q: 5 rows against K's 50


def test_operands_follow_tensor_identity():
    """The library sees one pointer per tensor OBJECT: roles that are the same object share it, distinct objects never do,
    even when their copies would share storage (Q.detach(), a view of Q, a slice of a batch of one).  A pointer shared
    by distinct objects would fold one role's gradient into another's input."""
    from newsrecommendationsystem_b200.ops import _mha_operands
    x = torch.randn(3, 20, 300, requires_grad=True)
    h = torch.randn(1, 50, 300)

    def ptrs(q, k, v):
        return [t.data_ptr() for t in _mha_operands(q, k, v)]
    kv = x.detach()
    pq, pk, pv = ptrs(x, kv, kv)
    assert pq != pk and pk == pv
    kv = x[:]
    pq, pk, pv = ptrs(x, kv, kv)
    assert pq != pk and pk == pv
    pq, pk, pv = ptrs(h[:, :5], h, h)
    assert pq != pk and pk == pv
    pq, pk, pv = ptrs(x, x, x)
    assert pq == pk == pv
    pq, pk, pv = ptrs(x, x.detach(), x)
    assert pq == pv != pk
    pq, pk, pv = ptrs(x, x.detach(), x[:])
    assert len({pq, pk, pv}) == 3


# ---- GPU -----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def _module(dev, precision, seed=0):
    from newsrecommendationsystem_b200.model.general.attention.multihead_self import MultiHeadSelfAttention
    torch.manual_seed(seed)
    m = MultiHeadSelfAttention(300, 15)
    with torch.no_grad():                                   # nonzero biases, so that every bias gradient is exercised
        for lin in (m.W_Q, m.W_K, m.W_V):
            lin.bias.uniform_(-0.3, 0.3)
    m = m.to(dev)
    m.precision = precision
    return m


def _inputs(form, n, sq, sk, dev, seed):
    """(Q, K, V) as distinct leaf tensors in the roles `form` names: kv (three inputs), k=v (K is V), self (one input),
    q=k (K is Q), q=v (V is Q)."""
    gen = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn((n, sq, 300), device=dev, generator=gen)
    y = torch.randn((n, sk, 300), device=dev, generator=gen)
    z = torch.randn((n, sk, 300), device=dev, generator=gen)
    G = torch.randn((n, sq, 300), device=dev, generator=gen)
    roles = {"kv": (x, y, z), "k=v": (x, y, y), "self": (x, x, x), "q=k": (x, x, z), "q=v": (x, y, x)}[form]
    return roles, G


def _lengths(n, S):
    return np.resize(np.array([S, 1, 0, 3, S - 1, S + 5, -2], dtype=np.int64), n)


def _run(m, roles, G, length=None, need=(True, True, True)):
    """ctx and the gradients of sum(ctx * G): (ctx, [dQ, dK, dV] per role, {parameter: grad}).  Roles that are the same
    tensor share one leaf, so their entries are the same summed gradient."""
    for p in m.parameters():
        p.grad = None
    leaves = {}
    for t, nd in zip(roles, need):
        if id(t) not in leaves:
            leaves[id(t)] = t.detach().clone().requires_grad_(nd)
        elif nd:
            leaves[id(t)].requires_grad_(True)
    q, k, v = (leaves[id(t)] for t in roles)
    ctx = m(q, K=k, V=v, length=length)
    (ctx * G).sum().backward()
    return ctx.detach(), [t.grad for t in (q, k, v)], {k_: p.grad for k_, p in m.named_parameters() if p.grad is not None}


def _run64(m, roles, G, length=None):
    P = {k: p.detach().double().requires_grad_(True) for k, p in m.named_parameters()}
    leaves = {}
    for t in roles:
        leaves.setdefault(id(t), t.detach().double().requires_grad_(True))
    q, k, v = (leaves[id(t)] for t in roles)
    ctx = mha_ref(q, k, v, *(P[k_] for k_ in PNAMES), length=length)
    (ctx * G.double()).sum().backward()
    return ctx.detach(), [t.grad for t in (q, k, v)], {k_: v_.grad for k_, v_ in P.items()}


def _check(got, ref, tol, floor=0.0, what=""):
    scale = float(ref.abs().max()) + 1e-12
    err = float((got.double() - ref).abs().max())
    assert err <= tol * scale + floor, (what, err, scale)
    return err / scale


def _check_rows(got, ref, tol, what=""):
    """row-wise relative L2; rows whose reference is zero (length <= 0) must be exactly zero"""
    g, r = got.double().reshape(-1, 300), ref.reshape(-1, 300)
    nr = r.norm(dim=1)
    dead = nr == 0
    assert not g[dead].any(), what
    rel = float(((g - r).norm(dim=1)[~dead] / nr[~dead]).max()) if (~dead).any() else 0.0
    assert rel <= tol, (what, rel)
    return rel


def _compare(m, roles, G, length, precision, what):
    ctx, dx, grads = _run(m, roles, G, None if length is None else torch.from_numpy(length))
    ctx64, dx64, g64 = _run64(m, roles, G, length)
    tol = GTOL[precision]
    floor = 1e-6 * max(float(v.abs().max()) for v in list(g64.values()) + dx64)
    worst = {"ctx": _check_rows(ctx, ctx64, FTOL[precision], (what, "ctx"))}
    for name, a, b in zip("QKV", dx, dx64):
        worst["d" + name] = _check(a, b, tol, floor, (what, "d" + name))
    for k in PNAMES:
        worst[k] = _check(grads[k], g64[k], tol, floor, (what, k))
    assert all(torch.isfinite(v).all() for v in [ctx] + dx + list(grads.values()))
    return ctx, dx, grads, worst


SIZES = (1, 5, 20, 33, 50, 64)
WORST = {}


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("form", ["kv", "k=v", "self", "q=k", "q=v"])
def test_grid_vs_fp64(dev, form, precision):
    """Every (Sq, Sk) in {1, 5, 20, 33, 50, 64}^2 the form allows (K or V = Q needs Sq = Sk; self-attention at 20 and
    50 takes the other path), 7 sequences, with lengths {S, 1, 0, 3, S-1, S+5, -2} where the reference defines a mask
    (Sq = Sk, Sq = 1) and without."""
    m = _module(dev, precision, seed=1)
    worst = {}
    for sq in SIZES:
        for sk in SIZES:
            if form != "kv" and form != "k=v" and sq != sk:
                continue
            if form == "self" and sq in (20, 50):
                continue
            roles, G = _inputs(form, 7, sq, sk, dev, seed=100 * sq + sk)
            masks = [None] + ([_lengths(7, sk)] if sq == sk or sq == 1 else [])
            for length in masks:
                _, dx, _, w = _compare(m, roles, G, length, precision, (form, sq, sk, length is not None))
                if length is not None and sq == sk:
                    dead = torch.from_numpy(length <= 0).to(dev)
                    assert not dx[0][dead].any()               # length <= 0: zero d_xq
                for k, v in w.items():
                    worst[k] = max(worst.get(k, 0.0), v)
    print(f"{form} {precision}: " + " ".join(f"{k}={v:.1e}" for k, v in worst.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("shape", [(5, 50, "k=v"), (50, 20, "kv"), (64, 64, "self")])
@pytest.mark.parametrize("n", [1, 7, 130, 7040])
def test_batch_sizes_vs_fp64(dev, shape, precision, n):
    sq, sk, form = shape
    m = _module(dev, precision, seed=n)
    roles, G = _inputs(form, n, sq, sk, dev, seed=n + sq)
    masks = [None] + ([_lengths(n, sk)] if sq == sk else [np.resize(np.array([1, 0, 3, -1]), n)] if sq == 1 else [])
    for length in masks:
        _, _, _, w = _compare(m, roles, G, length, precision, (shape, n))
        print(f"{shape} {precision} n={n} mask={length is not None}: " + " ".join(f"{k}={v:.1e}" for k, v in w.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_one_query_mask(dev, precision):
    """Sq = 1 < Sk with a length: every key is kept iff length >= 1; length <= 0 gives zero context and zero d_xq."""
    m = _module(dev, precision, seed=4)
    roles, G = _inputs("k=v", 9, 1, 50, dev, seed=4)
    length = np.array([1, 0, 2, 50, 60, -3, 7, 1, 0])
    ctx, dx, _, _ = _compare(m, roles, G, length, precision, "one query")
    dead = torch.from_numpy(length <= 0).to(dev)
    assert not ctx[dead].any() and not dx[0][dead].any() and not dx[1][dead].any()
    live = ~dead
    full, _, _ = _run(m, roles, G, None)
    assert torch.equal(ctx[live], full[live])                # any length >= 1 is no mask at all


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("shape", [(33, 33), (64, 64), (20, 20)])
def test_exact_properties(dev, shape, precision):
    """Masked keys give exactly zero rows of d_xk / d_xv (K and V other inputs than Q); length <= 0 gives exactly zero
    context and d_xq; the context and input gradients of a sequence are bitwise the same alone and inside 7,040
    (parameter gradients come from atomics: to tolerance); grad-mode and no-grad forwards are bitwise equal."""
    sq, sk = shape
    m = _module(dev, precision, seed=2)
    n = 7
    roles, G = _inputs("kv", n, sq, sk, dev, seed=sq)
    length = _lengths(n, sk)
    ln_t = torch.from_numpy(length)
    ctx, dx, grads = _run(m, roles, G, ln_t)
    keymask = torch.arange(sk, device=dev).view(1, sk) < torch.from_numpy(length).to(dev).view(n, 1)
    assert not dx[1][~keymask].any() and not dx[2][~keymask].any()
    dead = torch.from_numpy(length <= 0).to(dev)
    assert not ctx[dead].any() and not dx[0][dead].any()
    # alone vs inside 7,040 (the first 7 sequences are the same)
    big_roles, big_G = _inputs("kv", 7040, sq, sk, dev, seed=sq + 1)
    big_roles = tuple(torch.cat([a, b[n:]]) for a, b in zip(roles, big_roles))
    big_G = torch.cat([G, big_G[n:]])
    big_len = torch.from_numpy(np.concatenate([length, _lengths(7040 - n, sk)]))
    bctx, bdx, bgrads = _run(m, big_roles, big_G, big_len)
    assert torch.equal(bctx[:n], ctx)
    for a, b in zip(bdx, dx):
        assert torch.equal(a[:n], b)
    # grad mode vs no grad, masked and not
    with torch.no_grad():
        assert torch.equal(m(roles[0], K=roles[1], V=roles[2], length=ln_t), ctx)
        nm = m(roles[0], K=roles[1], V=roles[2])
    assert torch.equal(nm, m(roles[0], K=roles[1], V=roles[2]).detach())
    # self-attention at a length the new path takes, masked: the same two properties
    if sq not in (20, 50):
        (x, _, _), Gs = _inputs("self", n, sq, sq, dev, seed=3)
        c, d, _ = _run(m, (x, x, x), Gs, ln_t)
        assert not c[dead].any() and not d[0][dead].any()
        with torch.no_grad():
            assert torch.equal(m(x, length=ln_t), c)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("S", [20, 50])
def test_agrees_with_self_attention_path(dev, S, precision):
    """K = Q.clone(), V = Q.clone() takes the new path (three inputs); its context, parameter gradients and
    dQ + dK + dV match the 20 / 50-token path (ops.mhsa) on Q alone."""
    m = _module(dev, precision, seed=S)
    gen = torch.Generator(device=dev).manual_seed(S)
    x = torch.randn((130, S, 300), device=dev, generator=gen)
    G = torch.randn((130, S, 300), device=dev, generator=gen)
    tol = GTOL[precision]
    for length in (None, _lengths(130, S)):
        ln_t = None if length is None else torch.from_numpy(length)
        ref_ctx, (ref_dx, _, _), ref_g = _run(m, (x, x, x), G, ln_t)
        ctx, dx, g = _run(m, (x, x.clone(), x.clone()), G, ln_t)
        _check_rows(ctx, ref_ctx.double(), FTOL[precision], "ctx")
        floor = 1e-6 * max(float(v.abs().max()) for v in list(ref_g.values()) + [ref_dx])
        _check(dx[0] + dx[1] + dx[2], ref_dx.double(), tol, floor, "dx")
        for k in PNAMES:
            _check(g[k], ref_g[k].double(), tol, floor, k)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_gradients_only_where_needed(dev, precision):
    """Each input alone, or the weights alone: what comes back equals the full run's, the rest gets no gradient; an
    input passed twice gets its summed gradient once."""
    m = _module(dev, precision, seed=6)
    roles, G = _inputs("kv", 9, 5, 33, dev, seed=6)
    _, dx, grads = _run(m, roles, G)
    for which in range(3):
        need = tuple(i == which for i in range(3))
        for p in m.parameters():
            p.requires_grad_(False)
        _, d, g = _run(m, roles, G, need=need)
        assert g == {}
        for i in range(3):
            assert (d[i] is None) != (i == which)
        assert torch.equal(d[which], dx[which])
        for p in m.parameters():
            p.requires_grad_(True)
    _, d, g = _run(m, roles, G, need=(False, False, False))
    assert all(t is None for t in d)
    floor = 1e-6 * max(float(v.abs().max()) for v in grads.values())
    for k in PNAMES:
        _check(g[k], grads[k].double(), 1e-5, floor, k)
    # K is V: one leaf, its gradient the sum over both roles
    roles2, G2 = _inputs("k=v", 9, 5, 33, dev, seed=7)
    _, d2, _ = _run(m, roles2, G2)
    _, d64, _ = _run64(m, roles2, G2)
    assert d2[1] is d2[2]
    _check(d2[1], d64[1], GTOL[precision], what="dK+dV")


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_candidate_over_history_fused_adam_steps(dev, precision):
    """Candidates attend over a click history: Q = [B, 5, 300], K = V = [B, 50, 300], a fixed linear loss, three
    FusedAdam steps.  Each step is checked teacher-forced at the parameters the GPU held before it: every gradient
    (parameters, Q and the history) against fp64 autograd, and the parameters after the step against fp64 Adam on the
    fp64 gradients (the tolerances of test_mhsa_train.py's FusedAdam test)."""
    from newsrecommendationsystem_b200.optim import FusedAdam
    n, lr = 64, 1e-3
    att = _module(dev, precision, seed=12)
    gen = torch.Generator(device=dev).manual_seed(13)
    cand = torch.randn((n, 5, 300), device=dev, generator=gen)
    hist = torch.randn((n, 50, 300), device=dev, generator=gen)
    wl = torch.randn((300,), device=dev, generator=gen)
    params = dict(att.named_parameters())
    opt = FusedAdam(list(params.values()), lr=lr)
    M = {k: torch.zeros_like(p, dtype=torch.float64) for k, p in params.items()}
    V = {k: torch.zeros_like(p, dtype=torch.float64) for k, p in params.items()}
    b1, b2, eps = 0.9, 0.999, 1e-8
    tol = GTOL[precision]
    loose = {k: torch.zeros_like(p, dtype=torch.bool) for k, p in params.items()}
    for step in range(1, 4):
        P = {k: p.detach().double().clone() for k, p in params.items()}
        Pr = {k: v.clone().requires_grad_(True) for k, v in P.items()}
        c64, h64 = cand.double().requires_grad_(True), hist.double().requires_grad_(True)
        (mha_ref(c64, h64, h64, *(Pr[k] for k in PNAMES)) @ wl.double()).sum().backward()
        g64 = {k: v.grad for k, v in Pr.items()}
        opt.zero_grad()
        c, h = cand.clone().requires_grad_(True), hist.clone().requires_grad_(True)
        (att(c, K=h, V=h) @ wl).sum().backward()
        floor = 1e-6 * max(float(v.abs().max()) for v in g64.values())
        for k, p in params.items():
            _check(p.grad, g64[k], tol, floor, (step, k))
        _check(c.grad, c64.grad, tol, floor, (step, "dQ"))
        _check(h.grad, h64.grad, tol, floor, (step, "dK+dV"))
        opt.step()
        for k, p in params.items():
            M[k] = b1 * M[k] + (1 - b1) * g64[k]
            V[k] = b2 * V[k] + (1 - b2) * g64[k] ** 2
            upd = lr * (M[k] / (1 - b1 ** step)) / ((V[k] / (1 - b2 ** step)).sqrt() + eps)
            err = (p.detach().double() - (P[k] - upd)).abs()
            scale = float(g64[k].abs().max()) + 1e-12
            loose[k] |= g64[k].abs() <= 100 * (tol * scale + floor)
            e_tight = float(err[~loose[k]].max()) if (~loose[k]).any() else 0.0
            assert e_tight <= 2e-2 * lr, (step, k, e_tight)
            assert float(err.max()) <= 3 * lr, (step, k, float(err.max()))
    with torch.no_grad():
        c_ng = att(cand, K=hist, V=hist)
    c64 = mha_ref(cand.double(), hist.double(), hist.double(), *(params[k].detach().double() for k in PNAMES))
    _check_rows(c_ng, c64, FTOL[precision], "no-grad forward after the steps")


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_shared_storage_inputs_vs_fp64(dev, precision):
    """Distinct tensor objects over one storage are distinct inputs: a stop-gradient memory over the block's own input
    (K = V = Q.detach()), a view that carries the gradient (K = V = Q[:]), and candidates sliced from a history of a batch
    of one (Q = h[:, :5], K = V = h).  The context and every gradient against the fp64 transcription of the same graph."""
    m = _module(dev, precision, seed=21)
    gen = torch.Generator(device=dev).manual_seed(21)
    tol = GTOL[precision]
    x0 = torch.randn((6, 20, 300), device=dev, generator=gen)
    G = torch.randn((6, 20, 300), device=dev, generator=gen)
    h0 = torch.randn((1, 50, 300), device=dev, generator=gen)
    Gh = torch.randn((1, 5, 300), device=dev, generator=gen)
    cases = {"detach": (x0, G, lambda x: (x, x.detach(), x.detach())),
             "view": (x0, G, lambda x: (x, x[:], x[:])),
             "batch-1 slice": (h0, Gh, lambda h: (h[:, :5], h, h))}
    for name, (base, g, roles) in cases.items():
        for p in m.parameters():
            p.grad = None
        xb = base.clone().requires_grad_(True)
        q, k, v = roles(xb)
        if name != "view":
            v = k                                             # K and V one object, as a caller passes a memory
        ctx = m(q, K=k, V=v)
        (ctx * g).sum().backward()
        P = {k_: p.detach().double().requires_grad_(True) for k_, p in m.named_parameters()}
        x64 = base.double().requires_grad_(True)
        q6, k6, v6 = roles(x64)
        ctx64 = mha_ref(q6, k6, v6, *(P[k_] for k_ in PNAMES))
        (ctx64 * g.double()).sum().backward()
        _check_rows(ctx.detach(), ctx64.detach(), FTOL[precision], (name, "ctx"))
        floor = 1e-6 * max(float(t.grad.abs().max()) for t in list(P.values()) + [x64])
        _check(xb.grad, x64.grad, tol, floor, (name, "dx"))
        for k_ in PNAMES:
            _check(dict(m.named_parameters())[k_].grad, P[k_].grad, tol, floor, (name, k_))
