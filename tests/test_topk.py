"""Top-k news of the whole table per user (nrms_topk_news, ops.topk_news, Recommender.top_k / top_k_rows).

CPU part: argument errors come back as codes before any CUDA call, a dtype that does not match the mode is refused, and a
restatement of the host's split rule and the score kernel's work mapping visits every (user block, news tile) once.
GPU part (`-m gpu`): against an fp64 reference computed from the exact operands each mode consumes (fp32 table and users
in FP32 mode; the fp16-rounded table and users in tensor mode), with the (score desc, row asc) order; exclusions, ties,
NaN, launch independence, the padded evaluate table, and the Recommender against the candidate-ranking path.
"""
import os

import numpy as np
import pytest
import torch

from conftest import ROOT

SMS, BM, BN, FP32_NC = 148, 128, 256, 16384
E_INVALID, E_UNSUPPORTED = 1, 2


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from newsrecommendationsystem_b200 import _lib
    return _lib.load()


# ---- CPU ----------------------------------------------------------------------------------------------------------
def test_argument_errors_without_gpu(lib):
    p = 1 << 20                        # aligned, never dereferenced: every check runs before a CUDA call
    args = dict(table=p, n_news=1000, user=p, U=4, excl=p, ne=50, k=10, scores=p, rows=p, ws=p, wsb=1 << 40, mode=1)

    def call(**kw):
        a = dict(args, **kw)
        return lib.nrms_topk_news(a["table"], a["n_news"], a["user"], a["U"], a["excl"], a["ne"], a["k"], a["scores"],
                                  a["rows"], a["ws"], a["wsb"], a["mode"], None)
    for mode in (0, 1):
        assert call(k=0, mode=mode) == E_UNSUPPORTED and b"k = 0" in lib.nrms_last_error()
        assert call(k=257, mode=mode) == E_UNSUPPORTED
        assert call(ne=65, mode=mode) == E_UNSUPPORTED and b"n_exclude" in lib.nrms_last_error()
        for name in ("table", "user", "scores", "rows", "ws"):
            assert call(mode=mode, **{name: None}) == E_INVALID, name
        assert call(excl=None, mode=mode) == E_INVALID                     # n_exclude > 0 needs the array
        assert call(table=p + 8, mode=mode) == E_INVALID and b"misaligned" in lib.nrms_last_error()
        assert call(ws=p + 16, mode=mode) == E_INVALID
    assert call(mode=7) == E_INVALID
    assert lib.nrms_topk_workspace_bytes(4, 1000, 0, 0, 1) == 0 and lib.nrms_topk_workspace_bytes(4, 1000, 10, 65, 1) == 0


def test_workspace_does_not_grow_with_users_times_news(lib):
    for mode in (0, 1):
        small = lib.nrms_topk_workspace_bytes(73152, 65238, 100, 50, mode)
        large = lib.nrms_topk_workspace_bytes(73152, 161013, 100, 50, mode)
        assert 0 < small < 73152 * 65238 * 4 / 20 and large < 73152 * 161013 * 4 / 20
        assert lib.nrms_topk_workspace_bytes(1, 65238, 256, 64, mode) < 64 << 20


def test_mode_and_table_mismatch_is_refused():
    from newsrecommendationsystem_b200 import ops, _lib
    t32, t16 = torch.zeros(10, 300), torch.zeros(11, 320, dtype=torch.float16)
    u = torch.zeros(2, 300)
    with pytest.raises(RuntimeError, match="fp16"):
        ops.topk_news(t32, 10, u, 5, mode=_lib.MODE_TF32)
    with pytest.raises(RuntimeError, match="fp32"):
        ops.topk_news(t16, 10, u, 5, mode=_lib.MODE_FP32)
    with pytest.raises(RuntimeError, match="n_news"):
        ops.topk_news(t32, 11, u, 5, mode=_lib.MODE_FP32)


def _plan(U, n_news, sms=SMS):
    """Restatement of topk::make_plan (tensor mode)."""
    n_tiles = (n_news + BN - 1) // BN
    ublocks = (U + BM - 1) // BM
    s = max(1, min(n_tiles, sms // ublocks))
    tps = (n_tiles + s - 1) // s
    return ublocks, n_tiles, (n_tiles + tps - 1) // tps, tps


@pytest.mark.parametrize("U", [1, 127, 128, 129, 73152])
@pytest.mark.parametrize("n_news", [1, 255, 256, 257, 65238, 161013])
def test_work_mapping_covers_every_tile_once(U, n_news):
    """topk_score_kernel: CTA b takes items b, b + grid, ...; item w = (user block w // splits, split w % splits) and the
    split owns tiles [split * tps, min(n_tiles, (split + 1) * tps)).  Every (user block, news tile) exactly once, no
    split empty; one split when the user blocks fill the SMs, about one per SM for a single user."""
    ublocks, n_tiles, splits, tps = _plan(U, n_news)
    items = ublocks * splits
    grid = min(items, SMS)
    seen = np.zeros((ublocks, n_tiles), dtype=np.int64)
    for b in range(grid):
        my = (items - b + grid - 1) // grid
        for i in range(my):
            w = b + i * grid
            sp = w % splits
            t0, t1 = sp * tps, min(n_tiles, (sp + 1) * tps)
            assert t1 > t0
            seen[w // splits, t0:t1] += 1
    assert (seen == 1).all()
    if ublocks >= SMS:
        assert splits == 1
    if U == 1:
        assert splits == min(n_tiles, SMS) or tps == 1 or splits >= SMS // 2
    # FP32 mode: score blocks of FP32_NC rows cover [0, n_news) once
    n0 = np.arange(0, n_news, FP32_NC)
    assert n0[-1] < n_news <= n0[-1] + FP32_NC


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


MAX_ERR = {"fp32": 0.0, "tf32": 0.0}


def _operands(table32, users, mode):
    """-> (table argument, fp64 table rows, fp64 users): the exact operands the mode consumes."""
    from newsrecommendationsystem_b200 import ops
    if mode == "tf32":
        t16 = ops.pack_rows_f16(table32)
        return t16, t16[:, :300].double().cpu().numpy(), users.half().double().cpu().numpy()
    return table32, table32.double().cpu().numpy(), users.double().cpu().numpy()


def _reference(T, Uv, n_news, k, excl=None):
    """fp64 scores and the (score desc, row asc) top-k rows over the non-excluded rows of [0, n_news)."""
    S = Uv @ T[:n_news].T
    out = []
    for u in range(S.shape[0]):
        rows = np.arange(n_news)
        if excl is not None:
            rows = np.setdiff1d(rows, excl[u])
        s = S[u, rows]
        order = np.lexsort((rows, -s))
        out.append((rows[order][:k], s[order][:k]))
    return S, out


def _run(table, n_news, users, k, mode, excl=None):
    from newsrecommendationsystem_b200 import ops, _lib
    s, r = ops.topk_news(table, n_news, users, k, exclude_rows=excl, mode=_lib.MODES[mode])
    return s.cpu().numpy(), r.cpu().numpy()


def _check(mode, T, Uv, n_news, k, got_s, got_r, excl=None):
    S, ref = _reference(T, Uv, n_news, k, excl)
    tn = np.linalg.norm(T[:n_news], axis=1)
    for u in range(S.shape[0]):
        rr, rs = ref[u]
        nv = len(rr)
        r, s = got_r[u], got_s[u]
        assert (r[nv:] == -1).all() and np.isneginf(s[nv:]).all(), "tail must be -1 / -inf"
        r, s = r[:nv], s[:nv]
        assert (r >= 0).all() and (r < n_news).all()
        if excl is not None:
            assert not np.isin(r, excl[u]).any()
        scale = tn[r] * np.linalg.norm(Uv[u]) + 1e-30
        err = np.abs(s - S[u, r])
        MAX_ERR[mode] = max(MAX_ERR[mode], float((err / scale).max(initial=0.0)))
        # sorted: score descending, equal scores by ascending row
        assert all(s[j] > s[j + 1] or (s[j] == s[j + 1] and r[j] < r[j + 1]) for j in range(nv - 1))
        if mode == "fp32":
            assert (err <= 1e-5 * scale).all()
            sc = max(float(np.abs(rs).max(initial=0.0)), 1e-30)
            full = np.concatenate([[np.inf], rs, [-np.inf]])
            gap_ok = (full[1:-1] - full[2:] > 1e-6 * sc) & (full[:-2] - full[1:-1] > 1e-6 * sc)
            assert np.array_equal(r[gap_ok], rr[gap_ok])
        else:
            tol = 1e-3 * scale
            assert (err <= tol).all()
            t2 = 2 * 1e-3 * float(tn.max(initial=0.0)) * np.linalg.norm(Uv[u])
            kth = rs[-1]
            assert (S[u, r] >= kth - t2).all()
            cand = np.ones(n_news, bool)
            cand[r] = False
            if excl is not None:
                cand[excl[u][(excl[u] >= 0) & (excl[u] < n_news)]] = False
            if nv == k and cand.any():
                assert S[u, cand].max() <= s.min() + t2


SHAPES = [(1, 1, 1), (7, 127, 10), (7, 1, 256), (255, 129, 100), (256, 1, 256), (257, 1000, 10), (4097, 129, 256),
          (4097, 127, 1), (65238, 1, 100), (65238, 1000, 10)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_topk_matches_reference_over_shapes(dev, mode):
    g = torch.Generator(device="cpu").manual_seed(1)
    for n_news, U, k in SHAPES:
        table = (torch.randn(n_news + 5, 300, generator=g) * 0.3).to(dev)      # rows past n_news are never candidates
        table[n_news:] = 10.0
        users = torch.randn(U, 300, generator=g).to(dev)
        targ, T, Uv = _operands(table, users, mode)
        s, r = _run(targ, n_news, users, k, mode)
        _check(mode, T, Uv, n_news, k, s, r)
    print(f"topk[{mode}]: largest score error / (|row| |user|) = {MAX_ERR[mode]:.3e}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_all_equal_scores_return_rows_in_ascending_order(dev, mode):
    table = torch.zeros(1000, 300, device=dev)
    users = torch.randn(3, 300, device=dev)
    targ, _, _ = _operands(table, users, mode)
    s, r = _run(targ, 1000, users, 50, mode)
    assert (r == np.arange(50)[None]).all() and (s == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_exclusions(dev, mode):
    rng = np.random.default_rng(2)
    n_news, U, k = 5000, 200, 20
    table = torch.from_numpy(rng.standard_normal((n_news + 64, 300)).astype(np.float32) * 0.3).to(dev)
    users = torch.from_numpy(rng.standard_normal((U, 300)).astype(np.float32)).to(dev)
    targ, T, Uv = _operands(table, users, mode)
    S = Uv @ T[:n_news].T
    hist = rng.integers(0, n_news, size=(U, 50)).astype(np.int32)
    hist[:, :10] = np.argsort(-S, axis=1)[:, :10]              # the best rows are history: they must disappear
    hist[:, 10:15] = -1                                         # pads of both kinds
    hist[:, 15:20] = n_news + rng.integers(0, 64, size=(U, 5))
    hist[:, 20:25] = hist[:, :5]                                # duplicates
    s, r = _run(targ, n_news, users, k, mode, excl=hist)
    _check(mode, T, Uv, n_news, k, s, r, excl=hist)
    # on the device too, and an exclusion list that covers every row
    n_small = 40
    ex = np.concatenate([np.tile(np.arange(n_small, dtype=np.int32), (U, 1)), np.full((U, 10), -1, np.int32)], axis=1)
    s, r = _run(targ, n_small, users, 5, mode, excl=torch.from_numpy(ex).to(dev))
    assert (r == -1).all() and np.isneginf(s).all()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_nan_never_ranks_ahead_of_numbers(dev, mode):
    rng = np.random.default_rng(3)
    n_news = 3000
    table = torch.from_numpy(rng.standard_normal((n_news, 300)).astype(np.float32)).to(dev)
    table[17, 5] = float("nan")
    users = torch.from_numpy(rng.standard_normal((4, 300)).astype(np.float32)).to(dev)
    users[1, 7] = float("nan")
    targ, T, Uv = _operands(table, users, mode)
    s, r = _run(targ, n_news, users, 30, mode)
    assert not np.isnan(s).any()
    assert (r[1] == -1).all()                                   # every score of user 1 is NaN
    assert not (r == 17).any()
    Tf = T.copy()
    Tf[17] = 0.0                                                # the reference leaves row 17 out
    ok = [0, 2, 3]
    _check(mode, Tf, Uv[ok], n_news, 30, s[ok], r[ok], excl=np.full((3, 1), 17))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "tf32"])
def test_launch_independence(dev, mode):
    rng = np.random.default_rng(4)
    n_news, U, k = 65238, 1000, 100
    table = torch.from_numpy(rng.standard_normal((n_news, 300)).astype(np.float32) * 0.2).to(dev)
    users = torch.from_numpy(rng.standard_normal((U, 300)).astype(np.float32)).to(dev)
    hist = torch.from_numpy(rng.integers(-1, n_news, size=(U, 50)).astype(np.int32)).to(dev)
    targ, _, _ = _operands(table, users, mode)
    s, r = _run(targ, n_news, users, k, mode, excl=hist)
    s1, r1 = _run(targ, n_news, users[:500], k, mode, excl=hist[:500])
    s2, r2 = _run(targ, n_news, users[500:], k, mode, excl=hist[500:])
    assert np.array_equal(np.concatenate([r1, r2]), r)
    assert np.array_equal(np.concatenate([s1, s2]).view(np.uint32), s.view(np.uint32))
    s0, r0 = _run(targ, n_news, users[:1], k, mode, excl=hist[:1])
    assert np.array_equal(r0[0], r[0]) and np.array_equal(s0[0].view(np.uint32), s[0].view(np.uint32))


@pytest.mark.gpu
def test_padded_evaluate_table_never_returns_a_pad_row(dev):
    """evaluate's table16: n news, PAD_REPLICAS zero rows whose 1.0 bias column stays, and a closing zero row.  With
    every real score negative the zero-scored pads would lead the ranking if they were candidates."""
    from newsrecommendationsystem_b200 import ops
    from newsrecommendationsystem_b200.evaluate import PAD_REPLICAS
    n = 50
    real = -torch.rand(n, 300, device=dev) - 0.1
    table16 = ops.pack_rows_f16(torch.cat([real, torch.zeros(PAD_REPLICAS, 300, device=dev)]))
    users = torch.rand(8, 300, device=dev)
    s, r = _run(table16, n, users, 100, "tf32")
    assert (r[:, :n] >= 0).all() and (r[:, :n] < n).all() and (r[:, n:] == -1).all()
    assert (s[:, :n] < 0).all()


def _rec_case():
    from compact import expand_exp1
    from test_exp1_recommend import _nrms_state
    g1 = expand_exp1(np.load(os.path.join(ROOT, "tests", "golden", "exp1_golden.npz")))
    m, sd = _nrms_state(103)
    return g1, m, sd


@pytest.mark.gpu
def test_recommender_top_k_equals_ranking_all_candidates(dev):
    """On the 300-news fixture table: Recommender.top_k (FP32) gives the head of Recommender.recommend over all 300 ids
    (the path pinned to the reference's ranking), and with exclude_clicked the clicked ids are gone, the rest in order."""
    from newsrecommendationsystem_b200.recommend import Recommender
    from test_exp1_recommend import _load
    g1, m, sd = _rec_case()
    _load(m, sd, dev, "fp32")
    table = torch.from_numpy(g1["rec/table"]).to(dev)
    n = table.shape[0] - 1
    ids = [f"N{i}" for i in range(n)]
    rec = Recommender(m, ids, table)
    clicked = [f"N{i}" for i in g1["rec/4/hist"] if i != n]
    ref_ids, ref_y = rec.recommend(clicked, ids)

    def same_head(got_ids, got_y, want_ids, want_y):
        np.testing.assert_allclose(got_y, want_y, atol=1e-5)
        full = np.concatenate([[np.inf], want_y, [-np.inf]])
        sep = (full[1:-1] - full[2:] > 1e-5) & (full[:-2] - full[1:-1] > 1e-5)
        assert np.array_equal(np.asarray(got_ids)[sep], np.asarray(want_ids)[sep])

    got_ids, got_y = rec.top_k(clicked, 256, exclude_clicked=False)
    assert len(got_ids) == 256
    same_head(got_ids, got_y, ref_ids[:256], ref_y[:256])
    got_ids, got_y = rec.top_k(clicked, 256, exclude_clicked=True)
    keep = ~np.isin(ref_ids, clicked)
    want_ids, want_y = ref_ids[keep][:256], ref_y[keep][:256]
    assert len(got_ids) == min(256, int(keep.sum())) and not np.isin(got_ids, clicked).any()
    same_head(got_ids, got_y, want_ids, want_y)


@pytest.mark.gpu
def test_recommender_top_k_rows_tensor_mode(dev):
    """Tensor mode: batched users from the indexed encoder, scored against the cached fp16 table copy."""
    from newsrecommendationsystem_b200.recommend import Recommender
    from test_exp1_recommend import _load
    g1, m, sd = _rec_case()
    _load(m, sd, dev, "tf32")
    table = torch.from_numpy(g1["rec/table"]).to(dev)
    n = table.shape[0] - 1
    rec = Recommender(m, [f"N{i}" for i in range(n)], table)
    rng = np.random.default_rng(5)
    hist = rng.integers(0, n, size=(6, 50)).astype(np.int32)
    hist[:, :20] = n                                            # left pads = the table's last row
    rows, scores, user = rec.top_k_rows(hist, 40)
    rows, scores = rows.cpu().numpy(), scores.cpu().numpy()
    T = rec._table16[:, :300].double().cpu().numpy()
    _check("tf32", T, user.half().double().cpu().numpy(), n, 40, scores, rows, excl=hist)
