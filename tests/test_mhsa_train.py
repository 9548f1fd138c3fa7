"""Training the standalone MultiHeadSelfAttention (K = V = Q), with and without its `length` key mask.

CPU part: a torch fp64 autograd restatement of the reference block (reference src/model/general/attention/
multihead_self.py:15-23,46-76: exp of the scaled scores, times the key mask, divided by (sum + 1e-8), no output
projection), pinned against the oracle -- itself pinned against the live reference in test_oracle_golden.py -- on the
inputs of mhsa_masked_golden.npz; the argument errors of nrms_mhsa_bwd and its workspace size.
GPU part (`-m gpu`): gradients of x and the six parameters against the fp64 restatement at S = 20 and 50 in both modes,
the exact-zero and bitwise properties of the mask, and a few FusedAdam steps of a small model built on the block.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import nrms_oracle as O
from compact import expand_masked
from conftest import GOLDEN

GTOL = {"fp32": 2e-4, "tf32": 3e-3}       # of the largest entry of the reference gradient, as the training parity tests


# ---- the fp64 restatement ------------------------------------------------------------------------------------------
def mhsa_ref(x, Wq, bq, Wk, bk, Wv, bv, length=None):
    """multihead_self.py:15-23,46-76 with K = V = Q: exp(QK^T / sqrt 20) * mask[b, j], over (sum_j + 1e-8), times V."""
    n, S, _ = x.shape
    h = [torch.nn.functional.linear(x, W, b).view(n, S, 15, 20).transpose(1, 2) for W, b in ((Wq, bq), (Wk, bk), (Wv, bv))]
    e = torch.exp(h[0] @ h[1].transpose(-1, -2) / np.sqrt(20.0))
    if length is not None:
        L = torch.as_tensor(np.asarray(length), device=x.device).view(n, 1, 1, 1)
        e = e * (torch.arange(S, device=x.device).view(1, 1, 1, S) < L).to(e.dtype)
    attn = e / (e.sum(-1, keepdim=True) + 1e-8)
    return (attn @ h[2]).transpose(1, 2).reshape(n, S, 300)


PNAMES = ("W_Q.weight", "W_Q.bias", "W_K.weight", "W_K.bias", "W_V.weight", "W_V.bias")


def _golden():
    import os
    return expand_masked(np.load(os.path.join(GOLDEN, "mhsa_masked_golden.npz")))


def test_restatement_pinned_against_oracle():
    """The restatement equals the oracle's forward on the fixture's inputs, with and without `length` (lengths S, 1, 0,
    S + 5 among them)."""
    g = _golden()
    p = [torch.from_numpy(g[k].astype(np.float64)) for k in ("Wq", "bq", "Wk", "bk", "Wv", "bv")]
    for S in (20, 50):
        x = g[f"S{S}/x"].astype(np.float64)
        for length in (g[f"S{S}/length"], None):
            ref, _ = O.mhsa_forward(x, {k: g[k].astype(np.float64) for k in ("Wq", "bq", "Wk", "bk", "Wv", "bv")}, 15,
                                    length=length)
            got = mhsa_ref(torch.from_numpy(x), *p, length=length).numpy()
            np.testing.assert_allclose(got, ref, rtol=0, atol=1e-12)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from newsrecommendationsystem_b200 import _lib
    return _lib.load()


def _al(nbytes):
    return (nbytes + 255) // 256 * 256


def _ws_bytes(n, S, mode):
    rows = n * S
    ldr = (rows + 3) // 4 * 4
    b = _al(rows * 900 * 4) + _al(296 * 900 * 4)
    if mode == 1:
        b += _al(ldr * 900 * 4) + _al(ldr * 300 * 4) + _al(900 * 300 * 4)
    return b


def test_mhsa_bwd_arguments_and_workspace(lib):
    """nrms_mhsa_bwd refuses bad arguments before any CUDA call; its workspace holds dQKV, the partial sums and, in
    tensor mode, the transposed operands of the weight and input contractions."""
    for n in (1, 7, 7040):
        for S in (20, 50):
            for mode in (0, 1):
                assert lib.nrms_mhsa_bwd_workspace_bytes(n, S, mode) == _ws_bytes(n, S, mode)
    assert lib.nrms_mhsa_bwd_workspace_bytes(0, 20, 1) == 0
    a = C.c_void_p(1 << 20)                                 # aligned, never dereferenced: every call below fails first
    need = lib.nrms_mhsa_bwd_workspace_bytes(7, 20, 1)

    def call(d_ctx=a, x=a, lengths=None, n=7, S=20, wqkv=a, fws=a, d_x=a, d_w=a, d_b=a, ws=a, ws_bytes=need, mode=1):
        return lib.nrms_mhsa_bwd(d_ctx, x, lengths, n, S, wqkv, fws, d_x, d_w, d_b, ws, ws_bytes, mode, None)

    for S in (19, 21, 30, 49, 51):
        assert call(S=S) == 2 and b"unsupported" in lib.nrms_last_error()
    assert call(mode=7) == 1
    assert call(n=-1) == 1
    assert call(n=0, d_ctx=None, x=None) == 0                # nothing to do
    for k in ("d_ctx", "x", "wqkv", "fws", "d_w", "d_b"):
        assert call(**{k: None}) == 1 and b"null" in lib.nrms_last_error(), k
    for k in ("d_ctx", "x", "wqkv", "fws", "d_w", "d_x"):
        assert call(**{k: C.c_void_p((1 << 20) + 4)}) == 1 and b"aligned" in lib.nrms_last_error(), k
    assert call(lengths=C.c_void_p((1 << 20) + 2)) == 1
    assert call(ws_bytes=need - 1) == 3 and b"workspace" in lib.nrms_last_error()
    assert call(ws=None) == 3
    assert call(ws_bytes=lib.nrms_mhsa_bwd_workspace_bytes(7, 20, 0), mode=1) == 3     # FP32-mode size in tensor mode


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


def _lengths(n, S):
    return np.resize(np.array([S, 1, 0, 3, S - 1, S + 5, -2], dtype=np.int64), n)


def _run(m, x, G, length=None, x_grad=True):
    """ctx and the gradients of sum(ctx * G) on the GPU: (ctx, dx, {parameter name: grad})."""
    for p in m.parameters():
        p.grad = None
    xr = x.clone().requires_grad_(x_grad)
    ctx = m(xr, length=length)
    (ctx * G).sum().backward()
    return ctx.detach(), (xr.grad if x_grad else None), {k: p.grad for k, p in m.named_parameters() if p.grad is not None}


def _run64(m, x, G, length=None):
    P = {k: p.detach().double().requires_grad_(True) for k, p in m.named_parameters()}
    x64 = x.double().requires_grad_(True)
    ctx = mhsa_ref(x64, *(P[k] for k in PNAMES), length=length)
    (ctx * G.double()).sum().backward()
    return ctx.detach(), x64.grad, {k: v.grad for k, v in P.items()}


def _check(got, ref, tol, floor=0.0, what=""):
    scale = float(ref.abs().max()) + 1e-12
    err = float((got.double() - ref).abs().max())
    assert err <= tol * scale + floor, (what, err, scale)
    return err / scale


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 7, 130, 2049, 7040])
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("S", [20, 50])
def test_gradients_vs_fp64(dev, S, precision, n):
    """dx and the six parameter gradients against the fp64 restatement, with lengths S, 1, 0, 3, S - 1, S + 5, -2
    (repeated over the batch) and without a mask.  b_K's gradient is zero in exact arithmetic (a common shift of a
    row's scores cancels in the softmax), so both sides hold rounding noise there: the floor is 1e-6 of the largest
    gradient entry, as in the training parity tests."""
    m = _module(dev, precision, seed=S + n)
    gen = torch.Generator(device=dev).manual_seed(7 * n + S)
    x = torch.randn((n, S, 300), device=dev, generator=gen)
    G = torch.randn((n, S, 300), device=dev, generator=gen)
    tol = GTOL[precision]
    for length in (_lengths(n, S), None):
        ln_t = None if length is None else torch.from_numpy(length)
        ctx, dx, grads = _run(m, x, G, ln_t)
        ctx64, dx64, g64 = _run64(m, x, G, length)
        floor = 1e-6 * max(float(v.abs().max()) for v in list(g64.values()) + [dx64])
        worst = {"ctx": _check(ctx, ctx64, tol, what="ctx"), "dx": _check(dx, dx64, tol, floor, "dx")}
        for k in PNAMES:
            worst[k] = _check(grads[k], g64[k], tol, floor, k)
        assert all(torch.isfinite(v).all() for v in [ctx, dx] + list(grads.values()))
        if length is not None:
            dead = torch.from_numpy(length <= 0).to(dev)
            assert not ctx[dead].any() and not dx[dead].any()          # length <= 0: no context, no input gradient
        print(f"S={S} {precision} n={n} mask={length is not None}: " +
              " ".join(f"{k}={v:.1e}" for k, v in worst.items()))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
@pytest.mark.parametrize("S", [20, 50])
def test_mask_exactness(dev, S, precision):
    """Bitwise properties of the mask:
      - a sequence of length 0 contributes nothing: its context and its dx rows are exactly zero, and the parameter
        gradients equal those of the batch without it (up to the atomic epilogue's summation order);
      - length = [S] * n gives the gradients of length = None bit for bit (one K split at 7 sequences: no atomics race);
      - the dx rows and the context of a sequence do not depend on the other sequences of the launch (bitwise);
      - the grad-mode forward equals the no-grad forward bit for bit."""
    m = _module(dev, precision, seed=3)
    gen = torch.Generator(device=dev).manual_seed(S)
    n = 7
    x = torch.randn((n, S, 300), device=dev, generator=gen)
    G = torch.randn((n, S, 300), device=dev, generator=gen)
    length = torch.from_numpy(_lengths(n, S))
    # length 0 alone and among others
    ctx, dx, grads = _run(m, x, G, length)
    assert not ctx[2].any() and not dx[2].any() and not ctx[6].any() and not dx[6].any()
    keep = [0, 1, 3, 4, 5]
    ctx_k, dx_k, grads_k = _run(m, x[keep], G[keep], length[keep])
    assert torch.equal(ctx_k, ctx[keep]) and torch.equal(dx_k, dx[keep])
    floor = 1e-6 * max(float(v.abs().max()) for v in grads.values())
    for k in PNAMES:
        _check(grads_k[k], grads[k].double(), 1e-5, floor, k)
    c0, d0, _ = _run(m, x[2:3], G[2:3], length[2:3])
    assert not c0.any() and not d0.any()
    # full length == no mask
    a = _run(m, x, G, torch.full((n,), S))
    b = _run(m, x, G, None)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for k in PNAMES:
        assert torch.equal(a[2][k], b[2][k]), k
    # launch independence: the first 7 sequences alone and inside a batch of 130
    xb = torch.cat([x, torch.randn((123, S, 300), device=dev, generator=gen)])
    Gb = torch.cat([G, torch.randn((123, S, 300), device=dev, generator=gen)])
    lb = torch.from_numpy(_lengths(130, S))
    big = _run(m, xb, Gb, lb)
    assert torch.equal(big[0][:n], ctx) and torch.equal(big[1][:n], dx)
    # grad mode vs no grad
    with torch.no_grad():
        assert torch.equal(m(x, length=length), ctx)
        assert torch.equal(m(x), b[0])


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_gradients_only_where_needed(dev, precision):
    """x alone, or the weights alone: the other side gets no gradient, and what comes back equals the full run's."""
    m = _module(dev, precision, seed=5)
    gen = torch.Generator(device=dev).manual_seed(5)
    x = torch.randn((9, 20, 300), device=dev, generator=gen)
    G = torch.randn((9, 20, 300), device=dev, generator=gen)
    length = torch.from_numpy(_lengths(9, 20)).to(dev)               # a device tensor this time
    _, dx, grads = _run(m, x, G, length)
    for p in m.parameters():
        p.requires_grad_(False)
    _, dx_only, g_none = _run(m, x, G, length)
    assert g_none == {} and torch.equal(dx_only, dx)
    for p in m.parameters():
        p.requires_grad_(True)
    _, no_dx, g_only = _run(m, x, G, length, x_grad=False)
    assert no_dx is None
    floor = 1e-6 * max(float(v.abs().max()) for v in grads.values())
    for k in PNAMES:
        _check(g_only[k], grads[k].double(), 1e-5, floor, k)          # the dW epilogue adds atomically
    with pytest.raises(NotImplementedError):
        m(x, K=x[:, :5])                                              # cross-attention is not compiled, in grad mode too


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "tf32"])
def test_small_model_fused_adam_steps(dev, precision):
    """MultiHeadSelfAttention (masked) -> standalone AdditiveAttention -> a fixed linear loss, three FusedAdam steps.
    Each step is checked teacher-forced at the parameters the GPU held before it: every gradient against fp64 autograd
    (tolerances as above), and the parameters after the step against fp64 Adam on the fp64 gradients, with moments
    carried in fp64.  Adam divides each entry by its own gradient's magnitude, so an entry whose fp64 gradient is within
    100 gradient tolerances of zero at some step (b_K's, zero in exact arithmetic, above all) may move by up to about lr
    either way; those entries are held to 3 lr, the others to 2 % of lr.  A no-grad forward after the steps sees the new weights."""
    from newsrecommendationsystem_b200.model.general.attention.additive import AdditiveAttention
    from newsrecommendationsystem_b200.optim import FusedAdam
    S, n, lr = 20, 64, 1e-3
    att = _module(dev, precision, seed=9)
    torch.manual_seed(10)
    add = AdditiveAttention(200, 300).to(dev)
    add.precision = precision
    gen = torch.Generator(device=dev).manual_seed(11)
    x = torch.randn((n, S, 300), device=dev, generator=gen)
    wl = torch.randn((300,), device=dev, generator=gen)
    length = torch.from_numpy(_lengths(n, S))
    params = {"att." + k: p for k, p in att.named_parameters()}
    params.update({"add." + k: p for k, p in add.named_parameters()})
    opt = FusedAdam(list(params.values()), lr=lr)
    M = {k: torch.zeros_like(p, dtype=torch.float64) for k, p in params.items()}
    V = {k: torch.zeros_like(p, dtype=torch.float64) for k, p in params.items()}
    b1, b2, eps = 0.9, 0.999, 1e-8
    tol = GTOL[precision]
    loose = {k: torch.zeros_like(p, dtype=torch.bool) for k, p in params.items()}
    for step in range(1, 4):
        P = {k: p.detach().double().clone() for k, p in params.items()}
        # fp64 reference gradients at the live parameters
        Pr = {k: v.clone().requires_grad_(True) for k, v in P.items()}
        c = mhsa_ref(x.double(), *(Pr["att." + k] for k in PNAMES), length=length.numpy())
        w = torch.softmax(torch.tanh(torch.nn.functional.linear(c, Pr["add.linear.weight"], Pr["add.linear.bias"])) @
                          Pr["add.attention_query_vector"], dim=1)
        ((w.unsqueeze(-1) * c).sum(1) @ wl.double()).sum().backward()
        g64 = {k: v.grad for k, v in Pr.items()}
        # the GPU step
        opt.zero_grad()
        (add(att(x, length=length)) @ wl).sum().backward()
        floor = 1e-6 * max(float(v.abs().max()) for v in g64.values())
        for k, p in params.items():
            _check(p.grad, g64[k], tol, floor, (step, k))
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
    # the no-grad path (cached packed weights) sees the stepped parameters
    with torch.no_grad():
        c_ng = att(x, length=length)
    c64 = mhsa_ref(x.double(), *(params["att." + k].detach().double() for k in PNAMES), length=length.numpy())
    _check(c_ng, c64, tol, what="no-grad forward after the steps")
    assert torch.equal(c_ng, att(x, length=length).detach())


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 5, 333, 7040])
def test_masked_attention50_kernel_vs_fp64(lib, dev, n):
    """The masked tensor-core backward at S = 50 on the q|k|v rows the forward left in its workspace: dQKV against the
    fp64 gradient of masked attention at those rows, including padding-only (length 0) and one-token sequences; masked
    keys get exactly zero dK and dV; the transposed copy equals dQKV bitwise."""
    from newsrecommendationsystem_b200 import _lib
    from newsrecommendationsystem_b200._lib import check, ptr
    S, rows = 50, n * 50
    gen = torch.Generator(device=dev).manual_seed(n)
    m = _module(dev, "tf32", seed=n)
    wqkv, bqkv = (t.detach().contiguous() for t in m.packed())
    x = torch.randn((n, S, 300), device=dev, generator=gen)
    length = torch.from_numpy(np.resize(np.array([0, 1, 50, 17, 49, 2, 60], dtype=np.int32), n)).to(dev)
    d_ctx = torch.randn((n, S, 300), device=dev, generator=gen)
    ctx = torch.empty_like(x)
    fws = torch.zeros(rows * 900 * 4, dtype=torch.uint8, device=dev)
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    check(lib.nrms_mhsa_masked_fwd(ptr(x), ptr(length), n, S, ptr(wqkv), ptr(bqkv), ptr(ctx), ptr(fws), fws.numel(),
                                   _lib.MODE_TF32, st), "nrms_mhsa_masked_fwd")
    ws = torch.zeros(int(lib.nrms_mhsa_bwd_workspace_bytes(n, S, _lib.MODE_TF32)), dtype=torch.uint8, device=dev)
    d_w, d_b = torch.zeros_like(wqkv), torch.zeros_like(bqkv)
    check(lib.nrms_mhsa_bwd(ptr(d_ctx), ptr(x), ptr(length), n, S, ptr(wqkv), ptr(fws), None, ptr(d_w), ptr(d_b), ptr(ws),
                            ws.numel(), _lib.MODE_TF32, st), "nrms_mhsa_bwd")
    torch.cuda.synchronize()
    qkv = fws.view(torch.float32).view(rows, 900)
    d_qkv = ws[:rows * 3600].view(torch.float32).view(rows, 900)
    ldr = (rows + 3) // 4 * 4
    o_t1 = _al(rows * 3600) + _al(296 * 3600)
    t1 = ws[o_t1:o_t1 + ldr * 3600].view(torch.float32).view(900, ldr)
    assert torch.equal(t1[:, :rows], d_qkv.T)
    q, k, v = (qkv[:, i * 300:(i + 1) * 300].double().view(n, S, 15, 20).transpose(1, 2).requires_grad_(True)
               for i in range(3))
    e = torch.exp(q @ k.transpose(-1, -2) / np.sqrt(20.0))
    keymask = (torch.arange(S, device=dev).view(1, S) < length.view(n, 1).long()).double()
    e = e * keymask.view(n, 1, 1, S)
    out = ((e / (e.sum(-1, keepdim=True) + 1e-8)) @ v).transpose(1, 2).reshape(rows, 300)
    assert _check(ctx.view(rows, 300), out.detach(), 3e-3, what="ctx") < 3e-3
    out.backward(d_ctx.double().view(rows, 300))
    ref = torch.cat([t.grad.transpose(1, 2).reshape(rows, 300) for t in (q, k, v)], dim=1)
    floor = 1e-5 * float(ref.abs().max())                  # a one-token sequence's dK is zero in exact arithmetic
    for i, name in enumerate("QKV"):
        _check(d_qkv[:, i * 300:(i + 1) * 300], ref[:, i * 300:(i + 1) * 300], 3e-3, floor, "d" + name)
    masked = (keymask.view(rows) == 0)
    assert not d_qkv[masked, 300:].any()                   # dK and dV of masked keys: exactly zero
    assert torch.isfinite(d_qkv).all()
