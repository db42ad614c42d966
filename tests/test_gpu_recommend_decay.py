"""Top-K recommendation ranked by a freshness decay per session (tcar_score_fwd_decay / tcar_recommend_decay /
Seq2SeqAttNN.recommend(decay=...) / recommend_split with recommend_half_life_h): the decayed GEMM maxima against
mode 1, mode 2 and fp64, the result against the fp64 reference minus the pinned penalty, against plain recommend at
rate 0 and against exclusion lists bit for bit, the edges of the age arithmetic, the margin of the selection on an
adversarial catalog, the host checks and main.py end to end."""
import datetime
import pickle

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from recommend_ref import GLOBO_N, check_topk, excluded_sets, make_lists, oracle_scores, own_order_ok  # noqa: E402
from test_gpu_parity import batch_for, build  # noqa: E402

I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def penalty(t_ref, rate, times):
    from tcar_b200.util import decay_penalty
    return decay_penalty(t_ref, rate, times)


# ------------------------------------------------------------------------------------------------ the decayed GEMM
def _operands(B, N, seed):
    from tcar_b200 import _native as nv
    g = torch.Generator(device="cuda").manual_seed(seed)
    n_pad = (N + 255) // 256 * 256
    Q = torch.zeros(nv.QROWS, nv.KEXT, device="cuda", dtype=torch.bfloat16)
    Q[:B] = (torch.randn(B, nv.KEXT, device="cuda", generator=g) * 0.5).bfloat16()
    I = torch.zeros(n_pad, nv.KEXT, device="cuda", dtype=torch.bfloat16)
    I[:N] = (torch.randn(N, nv.KEXT, device="cuda", generator=g) * 0.1).bfloat16()
    c = torch.randn(nv.QROWS, device="cuda", generator=g) * 0.3
    return Q, I, c, n_pad


def _maxima(Q, I, c, B, N, n_pad, mode, t=None, t_ref=None, rate=None, lo=None, hi=None):
    from tcar_b200 import _native as nv
    p = nv.ptr
    part = torch.full((n_pad // 128, nv.QROWS), float("nan"), device="cuda")
    cm = torch.full((nv.QROWS, n_pad // 8), float("nan"), device="cuda")
    tm = torch.full((nv.QROWS, n_pad // 128), float("nan"), device="cuda")
    if mode == 1:
        rc = nv.lib().tcar_score_fwd(p(Q), p(I), p(c), None, p(part), p(cm), p(tm), B, N, n_pad, 1, nv.CLUSTER_PAIR,
                                     nv.stream_ptr())
    elif mode == 2:
        rc = nv.lib().tcar_score_fwd_window(p(Q), p(I), p(c), p(part), p(cm), p(tm), p(t), p(lo), p(hi), B, N, n_pad,
                                            nv.stream_ptr())
    else:
        rc = nv.lib().tcar_score_fwd_decay(p(Q), p(I), p(cm), p(tm), p(t), p(t_ref), p(rate), p(lo), p(hi), B, N,
                                           n_pad, nv.stream_ptr())
    assert rc == 0
    torch.cuda.synchronize()
    return cm[:B], tm[:B]


@pytest.mark.parametrize("B", [1, 200, 512])
def test_decay_gemm_maxima(B):
    N = 7001                                            # not a multiple of 256: a partial last tile
    Q, I, c, n_pad = _operands(B, N, 31 + B)
    rs = np.random.RandomState(B + 3)
    t = np.zeros(n_pad, np.int32)
    t[:N] = rs.randint(0, 20000, N)
    t[N:] = 5
    t_ref = rs.randint(10000, 25000, B).astype(np.int32)    # some items lie in the future of every row
    zero = np.zeros(B, np.float32)
    cm1, tm1 = _maxima(Q, I, c, B, N, n_pad, 1)
    # rate 0: bit for bit the mode-1 maxima
    cm0, tm0 = _maxima(Q, I, c, B, N, n_pad, 3, dev(t), dev(t_ref), dev(zero))
    assert torch.equal(cm0, cm1) and torch.equal(tm0, tm1)
    # rate > 0: the maxima of s - p, against fp64 s minus the same fp32 penalty
    rate = (10.0 ** rs.uniform(-5, -2, B)).astype(np.float32)
    cmd, tmd = _maxima(Q, I, c, B, N, n_pad, 3, dev(t), dev(t_ref), dev(rate))
    assert torch.equal(tmd, cmd.view(B, -1, 16).max(-1).values)
    S = (Q[:B].double() @ I[:N].double().t()).cpu().numpy()
    R = S - penalty(t_ref, rate, t[:N]).astype(np.float64)
    R = np.concatenate([R, np.full((B, n_pad - N), -np.inf)], 1)
    ref = R.reshape(B, -1, 8).max(-1)
    got = cmd.cpu().numpy()
    assert np.isneginf(got[:, N // 8 + 1:]).all() and np.isneginf(ref[:, N // 8 + 1:]).all()
    live = np.isfinite(ref)
    np.testing.assert_allclose(got[live], ref[live], rtol=1e-6, atol=2e-3)
    assert (got <= cm1.cpu().numpy()).all(), "a penalty never raises a maximum"
    # with a window: the -inf pattern of mode 2, and at rate 0 its maxima bit for bit
    lo = rs.randint(-50, 15000, B).astype(np.int32)
    hi = (lo + rs.randint(100, 6000, B)).astype(np.int32)
    if B > 2:
        lo[1], hi[1] = 5, 4                             # an empty window
    w = (dev(lo), dev(hi))
    cm2, tm2 = _maxima(Q, I, c, B, N, n_pad, 2, dev(t), lo=w[0], hi=w[1])
    cmw0, tmw0 = _maxima(Q, I, c, B, N, n_pad, 3, dev(t), dev(t_ref), dev(zero), *w)
    assert torch.equal(cmw0, cm2) and torch.equal(tmw0, tm2)
    cmw, tmw = _maxima(Q, I, c, B, N, n_pad, 3, dev(t), dev(t_ref), dev(rate), *w)
    assert torch.equal(torch.isneginf(cmw), torch.isneginf(cm2))
    assert torch.equal(torch.isneginf(tmw), torch.isneginf(tm2))
    inw = (t[None, :N] >= lo[:, None]) & (t[None, :N] <= hi[:, None])
    refw = np.concatenate([np.where(inw, R[:, :N], -np.inf), np.full((B, n_pad - N), -np.inf)], 1).reshape(B, -1, 8)
    refw = refw.max(-1)
    live = np.isfinite(refw)
    np.testing.assert_allclose(cmw.cpu().numpy()[live], refw[live], rtol=1e-6, atol=2e-3)


# ------------------------------------------------------------------------------------------------ recommend(decay=)
def decay_setup(rs, N, B, S, kind):
    """Item times in minutes over ten days, t_ref near their end (some items in the future), and rates per session
    that make the penalty spread over the catalog `frac` times the session's score spread: negligible, comparable or
    dominant.  For "dominant", 300 items (more than K) are published exactly at t_ref: the list is the best of them."""
    times = rs.randint(0, 14400, N).astype(np.int32)
    t_ref = rs.randint(13000, 15000, B).astype(np.int64)
    frac = {"negligible": 1e-7, "moderate": 1.0, "dominant": 1e4}[kind]
    spread = S.max(1) - S.min(1)
    rate = (frac * spread / 14400).astype(np.float32)
    if kind == "dominant":
        newest = rs.choice(N, 300, replace=False)
        times[newest] = 20000
        t_ref[:] = 20000
    return times, t_ref, rate


@pytest.mark.parametrize("B,N,K,T,kind,ex", [(7, 30000, 1, 3, "moderate", "dup"),
                                             (64, 30000, 20, 4, "negligible", "clicked"),
                                             (512, 30000, 256, 20, "moderate", "clicked"),
                                             (40, 30000, 100, 2, "dominant", "lists"),
                                             (24, GLOBO_N, 20, 5, "moderate", "none"),
                                             (10, GLOBO_N, 256, 3, "dominant", "clicked"),
                                             (12, GLOBO_N, 100, 2, "negligible", "lists")])
def test_decay_matches_fp64_reference(B, N, K, T, kind, ex):
    from tcar_b200 import _native as nv
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=B + K + 7)
    S = oracle_scores(model, content, mwdhm, batch)
    rs = np.random.RandomState(K + 11)
    times, t_ref, rate = decay_setup(rs, N, B, S, kind)
    model.set_item_times(times)
    off = lst = None
    if ex == "dup":
        off, lst = make_lists(rs, N, [0, 1, 5, 37, 100, 3, 250], dup=True)
    elif ex == "lists":
        off, lst = make_lists(rs, N, rs.randint(0, nv.RECOMMEND_MAXX + 1, B).tolist())
    clicked = ex == "clicked"
    kw = dict(exclude_off=off, exclude_ids=lst, exclude_clicked=clicked, decay=(t_ref, rate))
    ids, sc = [x.clone() for x in model.recommend(bt, K, **kw)]
    ids2, sc2 = model.recommend(bt, K, **kw)
    torch.cuda.synchronize()
    assert torch.equal(ids, ids2) and torch.equal(sc, sc2), "a second run must be bit-identical"
    R = S - penalty(t_ref, rate, times).astype(np.float64)
    ex_sets = excluded_sets(B, off, lst, batch["seq"].numpy() if clicked else None)
    ids_h, sc_h = ids.cpu().numpy(), sc.cpu().numpy()
    check_topk(ids_h, sc_h, R, K, ex_sets)
    if kind == "dominant":
        # the newest articles only, ordered by score: with age 0 their decayed score is the score itself
        assert (times[ids_h] == 20000).all()
        for b in range(B):
            np.testing.assert_allclose(sc_h[b], S[b, ids_h[b]], rtol=1e-4, atol=1e-5)
    rescored = model.rec_rescored[:B].cpu().numpy()
    assert (rescored >= K).all() and rescored.mean() < N / 2, "the band stays narrow"


def test_zero_rate_equals_plain_and_window_equals_lists():
    """Rate 0: ids and scores torch.equal to plain recommend (with exclusions, with the clicks and with a window).
    Decay with a window: bit for bit decay with the out-of-window ids passed as an exclusion list."""
    from tcar_b200 import _native as nv
    N, B, T, K = 1500, 96, 3, 50
    model, _, mwdhm, _ = build(N, emb_scale=20.0)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=23)
    rs = np.random.RandomState(6)
    times = rs.randint(0, 1000, N).astype(np.int32)
    model.set_item_times(times)
    t_ref = rs.randint(500, 1200, B)
    off, lst = make_lists(rs, N, rs.randint(0, 40, B).tolist())
    for clicked in (False, True):
        a = [x.clone() for x in model.recommend(bt, K, off, lst, exclude_clicked=clicked)]
        na = model.rec_rescored[:B].clone()
        d = model.recommend(bt, K, off, lst, exclude_clicked=clicked, decay=(t_ref, 0.0))
        torch.cuda.synchronize()
        assert torch.equal(a[0], d[0]) and torch.equal(a[1], d[1]), clicked
        assert (model.rec_rescored[:B] >= na).all()
    lo = rs.randint(0, 450, B)
    hi = lo + rs.randint(420, 550, B)
    a = [x.clone() for x in model.recommend(bt, K, window=(lo, hi))]
    d = model.recommend(bt, K, window=(lo, hi), decay=(t_ref, np.zeros(B, np.float32)))
    torch.cuda.synchronize()
    assert torch.equal(a[0], d[0]) and torch.equal(a[1], d[1])
    out = [np.flatnonzero((times < lo[b]) | (times > hi[b])) for b in range(B)]
    assert max(len(o) for o in out) + T <= nv.RECOMMEND_MAXX
    woff = np.cumsum([0] + [len(o) for o in out]).astype(np.int32)
    wlst = np.concatenate(out).astype(np.int32)
    rate = (10.0 ** rs.uniform(-3, 0, B)).astype(np.float32)
    for clicked in (False, True):
        a = [x.clone() for x in model.recommend(bt, K, exclude_clicked=clicked, window=(lo, hi), decay=(t_ref, rate))]
        b_ = model.recommend(bt, K, woff, wlst, exclude_clicked=clicked, decay=(t_ref, rate))
        torch.cuda.synchronize()
        assert torch.equal(a[0], b_[0]) and torch.equal(a[1], b_[1]), clicked
    assert (a[0] >= 0).all()


def test_decay_int32_extremes_and_future_articles():
    """t_ref and item times at the int32 extremes (ages saturate at DECAY_MAX_AGE), articles after t_ref at age 0:
    the result against fp64 with the penalty of util.decay_penalty, and the returned scores are s - p exactly as
    the host computes p."""
    from tcar_b200 import _native as nv
    N, B, T, K = 4000, 6, 2, 64
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=5)
    S = oracle_scores(model, content, mwdhm, batch)
    rs = np.random.RandomState(8)
    times = rs.randint(-1000, 1000, N).astype(np.int64)
    times[:300] = I32_MIN
    times[300:600] = I32_MAX
    times[600:900] = I32_MAX - 5
    model.set_item_times(times)
    t_ref = np.array([I32_MAX, I32_MIN, 0, I32_MAX - 3, I32_MIN + 10, 500])
    rate = np.array([1e-6, 1.0, 0.01, 0.5, 2.0, 1e-3], np.float32)
    P = penalty(t_ref, rate, times)
    assert P[0, 0] == np.float32(rate[0]) * np.float32(nv.DECAY_MAX_AGE)           # saturated
    assert (P[1] == 0).all(), "t_ref = INT32_MIN: every article is at or after it"
    assert (P[3, 300:600] == 0).all() and P[3, 600] == np.float32(0.5) * 2
    ids, sc = model.recommend(bt, K, decay=(t_ref, rate))
    torch.cuda.synchronize()
    ids_h, sc_h = ids.cpu().numpy(), sc.cpu().numpy()
    check_topk(ids_h, sc_h, S - P.astype(np.float64), K, [set() for _ in range(B)])
    plain = model.recommend(bt, K)
    torch.cuda.synchronize()
    assert torch.equal(plain[0][1], ids[1]) and torch.equal(plain[1][1], sc[1]), "no penalty for session 1"
    # every returned score is fl(s - p) with the exact fp32 score s of plain recommend
    full = model.recommend(bt, nv.RECOMMEND_MAXK)
    torch.cuda.synchronize()
    for b in range(B):
        s32 = dict(zip(full[0][b].cpu().numpy().tolist(), full[1][b].cpu().numpy().tolist()))
        for j, r in zip(ids_h[b], sc_h[b]):
            if j in s32:
                assert np.float32(np.float32(s32[j]) - P[b, j]) == np.float32(r), (b, j)


# ------------------------------------------------------------------------------------------------ crafted catalogs
def _crafted(N, B, rs, item_rows=None):
    """A catalog whose exact scores are easy to steer: Tq = 0, content = 0, a_ic and item rows bf16-exact.  Returns
    the host arrays and the device buffers of tcar_score_fwd_decay / tcar_recommend_decay (cat_stats = the largest
    item row norm, 0: a valid error bound because nothing is rounded to bf16)."""
    from tcar_b200 import _native as nv
    H, HP, XW, NB = 250, 256, 500, 139
    n_pad = (N + 255) // 256 * 256
    items = item_rows if item_rows is not None else rs.randn(N, H).astype(np.float32)
    items = torch.from_numpy(items).bfloat16().float().numpy()
    q = torch.from_numpy(rs.randn(B, H).astype(np.float32)).bfloat16().float().numpy()
    item_tab = np.zeros((N + 1, HP), np.float32)
    item_tab[1:, :H] = items
    a_ic = np.zeros((B, XW), np.float32)
    a_ic[:, :H] = q
    Q = torch.zeros(nv.QROWS, nv.KEXT, dtype=torch.bfloat16)
    Q[:B, :H] = torch.from_numpy(q).bfloat16()
    I = torch.zeros(n_pad, nv.KEXT, dtype=torch.bfloat16)
    I[:N, :H] = torch.from_numpy(items).bfloat16()
    d = dict(Q=Q.cuda(), I=I.cuda(), a_ic=dev(a_ic), Tq=torch.zeros(B, NB, device="cuda"), item=dev(item_tab),
             content=torch.zeros(N + 1, HP, device="cuda"), mwdhm=torch.zeros(N, 5, device="cuda", dtype=torch.int32),
             stats=dev(np.array([np.linalg.norm(items, axis=1).max() * 1.01, 0.0], np.float32)))
    S = q.astype(np.float64) @ items.astype(np.float64).T
    return d, S, n_pad


def _run(d, B, N, n_pad, K, times, t_ref, rate, cm=None, tm=None):
    """tcar_score_fwd_decay (unless cm / tm are given) then tcar_recommend_decay; returns ids, scores, rescored."""
    from tcar_b200 import _native as nv
    p, lib, st = nv.ptr, nv.lib(), nv.stream_ptr()
    tt = torch.zeros(n_pad, device="cuda", dtype=torch.int32)
    tt[:N] = dev(times.astype(np.int32))
    tr, rr = dev(np.asarray(t_ref, np.int32)), dev(np.asarray(rate, np.float32))
    if cm is None:
        cm = torch.zeros(nv.QROWS, n_pad // 8, device="cuda")
        tm = torch.zeros(nv.QROWS, n_pad // 128, device="cuda")
        assert lib.tcar_score_fwd_decay(p(d["Q"]), p(d["I"]), p(cm), p(tm), p(tt), p(tr), p(rr), None, None, B, N,
                                        n_pad, st) == 0
    ws = torch.zeros(int(lib.tcar_recommend_ws_bytes(B)), device="cuda", dtype=torch.uint8)
    ids = torch.empty(B, K, device="cuda", dtype=torch.int32)
    sc = torch.empty(B, K, device="cuda")
    resc = torch.zeros(B, device="cuda", dtype=torch.int32)
    assert lib.tcar_recommend_decay(p(cm), p(tm), p(d["a_ic"]), p(d["Tq"]), p(d["item"]), p(d["content"]),
                                    p(d["mwdhm"]), p(d["stats"]), None, None, None, 1, B, N, n_pad, K, p(ws), p(ids),
                                    p(sc), p(resc), p(tt), p(tr), p(rr), None, None, st) == 0
    torch.cuda.synchronize()
    return ids.cpu().numpy(), sc.cpu().numpy(), resc.cpu().numpy()


def test_identical_rows_and_times_are_ordered_by_id():
    N, B, K = 5000, 8, 40
    rs = np.random.RandomState(1)
    rows = rs.randn(N, 250).astype(np.float32)
    twins = rs.choice(N, 12, replace=False)
    rows[twins] = rows[twins[0]] * 3.0                  # twelve identical rows, scoring near the top for most q
    times = rs.randint(0, 5000, N)
    times[twins] = 4000
    d, S, n_pad = _crafted(N, B, rs, rows)
    ids, sc, _ = _run(d, B, N, n_pad, K, times, np.full(B, 4500), np.full(B, 1e-3, np.float32))
    own_order_ok(ids, sc)
    for b in range(B):
        at = np.flatnonzero(np.isin(ids[b], twins))
        if len(at):
            assert (np.diff(at) == 1).all() and (len(at) == len(twins) or at[-1] == K - 1), "the twins are adjacent"
            assert (np.diff(ids[b, at]) > 0).all() and len(set(sc[b, at].tolist())) == 1, "ordered by id"
    assert sum(np.isin(ids[b], twins).any() for b in range(B)) >= 1


def test_selection_margin_covers_the_rounding_of_the_penalty():
    """Adversarial chunk maxima: with every item at the same age, p = 1000 and the session's error bound eps ~ 0
    (bf16-exact operands, cat_stats = 0), the decayed scores of the items sit on the fp32 grid of |r| ~ 1000.  The
    maxima are set one ulp BELOW the exact decayed score in many chunks -- what the GEMM's rounding of s_gemm - p may
    legitimately give.  A threshold of v - 2 eps would skip those chunks and lose items that tie with (and have lower
    ids than) the K-th best; the rounding term of the margin must re-score them."""
    from tcar_b200 import _native as nv
    N, B, K = 4096, 2, 20
    n_pad = N
    rs = np.random.RandomState(3)
    d, _, _ = _crafted(N, B, rs, np.zeros((N, 250), np.float32))
    d["a_ic"].zero_()
    d["a_ic"][:, 0] = 1.0                                # s = item[n, 0] exactly
    d["stats"].zero_()                                   # eps_b = 1e-30
    ulp = np.float32(2.0 ** -14)                         # fp32 spacing in [512, 1024)
    # decayed scores r = s - 1000 on a coarse grid of 64 levels: many exact ties
    level = rs.randint(0, 64, N)
    r = (np.float32(-1000.0) + level.astype(np.float32) * 4 * ulp).astype(np.float32)
    s = (r + np.float32(1000.0)).astype(np.float32)
    assert (np.float32(s - np.float32(1000.0)) == r).all()
    item = d["item"].cpu().numpy()
    item[1:, 0] = s
    d["item"] = dev(item)
    times, t_ref, rate = np.zeros(N, np.int64), np.full(B, 1000), np.ones(B, np.float32)
    # chunk maxima: the exact chunk maximum, one ulp lower in every other chunk (the lower-id half of each pair)
    cmax = r.reshape(-1, 8).max(1)
    low = np.arange(cmax.shape[0]) % 2 == 0
    cm_h = np.where(low, cmax - ulp, cmax).astype(np.float32)
    cm = torch.zeros(nv.QROWS, n_pad // 8, device="cuda")
    cm[:B] = dev(np.tile(cm_h, (B, 1)))
    tm = torch.zeros(nv.QROWS, n_pad // 128, device="cuda")
    tm[:B] = cm[:B].view(B, -1, 16).max(-1).values
    # the fixture is adversarial: the K-th largest maximum v, and chunks holding items of the exact top-K below v
    v = np.sort(cm_h)[::-1][K - 1]
    order = np.lexsort((np.arange(N), -r))
    top = order[:K]
    assert (cm_h[top // 8] < v).any(), "some top-K item sits in a chunk below v: v - 2 eps would miss it"
    ids, sc, resc = _run(d, B, N, n_pad, K, times, t_ref, rate, cm, tm)
    for b in range(B):
        assert ids[b].tolist() == top.tolist()
        assert (sc[b] == r[top]).all()
    assert (resc < N).all()


# ------------------------------------------------------------------------------------------------ checks
def test_decay_host_checks_launch_nothing():
    from tcar_b200 import _native as nv
    N, B, T = 500, 4, 2
    model, _, mwdhm, _ = build(N)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=1)
    before = nv.LAUNCHES["count"]
    with pytest.raises(ValueError, match="set_item_times"):
        model.recommend(bt, 5, decay=(np.zeros(B, int), 0.1))
    model.set_item_times(np.arange(N) - 10 ** 9)
    model.set_item_categories(np.arange(N) % 7)
    for decay, what in [((np.zeros(B - 1, int), 0.1), "t_ref must hold B = 4"),
                        ((np.zeros(B, float), 0.1), "integers"),
                        ((np.array([0, 0, 2 ** 31, 0]), 0.1), "session 2"),
                        ((np.zeros(B, int), np.ones(B + 1)), "B = 4 numbers"),
                        ((np.zeros(B, int), np.array([0.1, -1e-9, 0, 0])), "session 1: decay rate"),
                        ((np.zeros(B, int), np.array([0.1, 0, np.nan, 0])), "session 2: decay rate"),
                        ((np.zeros(B, int), np.array([0, 0, 0, np.inf])), "session 3: decay rate"),
                        ((np.zeros(B, int), 1e39), "overflows float32"),
                        ((np.full(B, 10 ** 9), np.array([0, 0, 1e32, 0])), "session 2: .*penalty"),
                        ((np.zeros(B, int), "x"), "numbers"), (np.zeros(B, int), "pair")]:
        with pytest.raises(ValueError, match=what):
            model.recommend(bt, 5, decay=decay)
    with pytest.raises(ValueError, match="categories"):
        model.recommend(bt, 5, decay=(np.zeros(B, int), 0.1), max_per_category=2)
    assert nv.LAUNCHES["count"] == before, "validation happens before any launch"
    # the C entry points refuse missing inputs, a window given by half and bad limits
    p, ps, st = nv.ptr, model.ps, nv.stream_ptr()
    buf = torch.zeros(ps.n_pad * 4, device=model.dev)
    lib = nv.lib()
    good = [p(buf)] * 7 + [None, None, B, N, ps.n_pad, st]
    for at, val in [(4, None), (5, None), (6, None), (7, p(buf)), (9, 0), (9, nv.QROWS + 1), (11, ps.n_pad + 128),
                    (10, ps.n_pad + 1)]:
        a = list(good)
        a[at] = val
        assert lib.tcar_score_fwd_decay(*a) == -1, at
    ws = torch.zeros(int(lib.tcar_recommend_ws_bytes(B)), device=model.dev, dtype=torch.uint8)
    base = [p(buf)] * 8 + [None, None, None, T, B, N, ps.n_pad, 5, p(ws), p(buf), p(buf), None, p(buf), p(buf),
                           p(buf), None, None, st]
    for at, val in [(20, None), (21, None), (22, None), (23, p(buf)), (15, 0), (15, nv.RECOMMEND_MAXK + 1),
                    (12, nv.QROWS + 1)]:
        a = list(base)
        a[at] = val
        assert lib.tcar_recommend_decay(*a) == -1, at
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ end to end
@pytest.mark.parametrize("max_age", [None, 48])
def test_recommend_split_with_half_life_end_to_end(tmp_path, monkeypatch, capsys, max_age):
    """main.py --recommend_k 20 --recommend_half_life_h 6 [--recommend_max_age_h 48] on a synthetic split whose test
    sessions were moved into the publication month: the written lists are ordered by the decayed score, mean_age_h is
    the mean age of the written articles, and a half-life brings the lists' mean age down against no decay."""
    from tcar_b200 import main as tmain, synth
    from tcar_b200.util import epoch_minutes
    N, n_test = 1500, 150
    monkeypatch.chdir(tmp_path)
    root = str(tmp_path) + "/synth/TCAR-mid/Normal/"
    synth.write_dataset(root, N=N, n_train=700, n_test=n_test, fold=0)
    load = lambda name: pickle.load(open(root + name, "rb"))
    tdict = load("session_time_dict_test0.pkl")
    rs = np.random.RandomState(9)
    t0 = datetime.datetime(2017, 10, 1)
    for key, clicks in tdict.items():                    # sessions from Nov 1-14 into Oct 3-29 (articles: Oct 1-30)
        shift = t0 + datetime.timedelta(days=int(rs.randint(2, 28)), seconds=int(rs.randint(0, 86400))) - \
            clicks[0]["click_t"]
        for c in clicks:
            c["click_t"] = c["click_t"] + shift
    pickle.dump(tdict, open(root + "session_time_dict_test0.pkl", "wb"))
    base = ["--datapath", str(tmp_path) + "/", "--dataset", "synth/TCAR-mid/", "--foldnum", "0", "--epoch", "1",
            "--batch_size", "64", "--recommend_k", "20"] + (["--recommend_max_age_h", str(max_age)] if max_age else [])
    model = tmain.main(tmain.build_parser().parse_args(base + ["--recommend_half_life_h", "6"]))
    got = model.last_recommend_metrics
    out = capsys.readouterr().out
    assert "mean age of the returned articles: {} h".format(got["mean_age_h"]) in out
    publish_dt, _ = load("publish_time_0.txt")
    item_dict = load("item_dict_0.txt")
    pub = epoch_minutes(publish_dt)
    t_req = {k: int(epoch_minutes([v[-2]["click_t"]])[0]) for k, v in tdict.items()}
    lines = open(tmp_path / "saved" / "recommend_0.txt").read().splitlines()
    assert len(lines) == n_test == got["sessions"]
    ages = []
    for line in lines:
        key, *pairs = line.split()
        key = int(key)
        arts = [a.rsplit(":", 1)[0] for a in pairs]
        scores = [float(a.rsplit(":", 1)[1]) for a in pairs]
        assert len(arts) <= 20 and len(set(arts)) == len(arts)
        assert scores == sorted(scores, reverse=True)
        for a in arts:
            age = t_req[key] - pub[item_dict[a] - 1]
            if max_age:
                assert 0 <= age <= 60 * max_age, (key, a)
            ages.append(max(age, 0))
    assert len(ages) > 10 * n_test
    np.testing.assert_allclose(got["mean_age_h"], np.mean(ages) / 60, rtol=1e-9)
    if max_age:
        assert "labels published outside their window" in out and "label_outside" in got
    # the same split without a half-life: older lists
    plain = tmain.main(tmain.build_parser().parse_args(base)).last_recommend_metrics
    assert "mean_age_h" not in plain
    old = []
    for line in open(tmp_path / "saved" / "recommend_0.txt").read().splitlines():
        key, *pairs = line.split()
        old += [max(t_req[int(key)] - pub[item_dict[a.rsplit(":", 1)[0]] - 1], 0) for a in pairs]
    assert np.mean(ages) < np.mean(old)
