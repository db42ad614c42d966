"""Top-K recommendation restricted to a publish-time window per session (tcar_score_fwd_window / tcar_recommend_window /
Seq2SeqAttNN.recommend(window=...) / recommend_split with recommend_max_age_h): the masked GEMM maxima against mode 1
and fp64, the result against the fp64 reference with out-of-window items excluded, against exclusion lists bit for
bit, and against no window at all."""
import datetime
import pickle

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from recommend_ref import GLOBO_N, check_topk, excluded_sets, make_lists, oracle_scores, own_order_ok  # noqa: E402
from test_gpu_parity import batch_for, build  # noqa: E402

I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1


# ------------------------------------------------------------------------------------------------ the windowed GEMM
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


def _gemm(Q, I, c, B, N, n_pad, window=None):
    """mode 1 (CTA pairs) when window is None, else tcar_score_fwd_window with window = (item_time, lo, hi)."""
    from tcar_b200 import _native as nv
    p = nv.ptr
    part = torch.full((n_pad // 128, nv.QROWS), float("nan"), device="cuda")
    cm = torch.full((nv.QROWS, n_pad // 8), float("nan"), device="cuda")
    tm = torch.full((nv.QROWS, n_pad // 128), float("nan"), device="cuda")
    if window is None:
        nv.call("tcar_score_fwd", p(Q), p(I), p(c), None, p(part), p(cm), p(tm), B, N, n_pad, 1, nv.CLUSTER_PAIR)
    else:
        t, lo, hi = window
        nv.call("tcar_score_fwd_window", p(Q), p(I), p(c), p(part), p(cm), p(tm), p(t), p(lo), p(hi), B, N, n_pad)
    torch.cuda.synchronize()
    return part, cm[:B], tm[:B]


@pytest.mark.parametrize("B", [1, 200, 512])
def test_window_gemm_masks_exactly(B):
    N = 7001                                            # not a multiple of 256: a partial last tile
    Q, I, c, n_pad = _operands(B, N, 11 + B)
    rs = np.random.RandomState(B)
    t = np.zeros(n_pad, np.int32)
    t[:N] = rs.randint(0, 1000, N)
    t[N:] = 500                                         # padding ids sit inside most windows: still never counted
    t[8 * 100: 8 * 104] = 2000                          # chunks 100..103 wholly outside every window below
    lo = rs.randint(-50, 900, B).astype(np.int32)
    hi = (lo + rs.randint(100, 600, B)).astype(np.int32)
    if B > 2:
        lo[0], hi[0] = I32_MIN, I32_MAX                 # row 0: everything
        lo[1], hi[1] = 5, 4                             # row 1: an empty window (lo > hi)
        lo[2], hi[2] = t[17], t[17]                     # row 2: one time value
    dev = lambda a: torch.from_numpy(a).cuda()
    part1, cm1, tm1 = _gemm(Q, I, c, B, N, n_pad)
    partw, cmw, tmw = _gemm(Q, I, c, B, N, n_pad, (dev(t), dev(lo), dev(hi)))
    # every tile maximum is the maximum of its 16 chunk maxima
    assert torch.equal(tmw, cmw.view(B, -1, 16).max(-1).values)
    valid = np.arange(n_pad) < N
    inw = (t[None, :] >= lo[:, None]) & (t[None, :] <= hi[:, None]) & valid[None, :]        # [B, n_pad]
    n_in = inw.reshape(B, -1, 8).sum(-1)
    n_valid = valid.reshape(-1, 8).sum(-1)[None, :].repeat(B, 0)
    g1, gw = cm1.cpu().numpy(), cmw.cpu().numpy()
    whole = (n_in == n_valid) & (n_valid > 0)
    assert (gw[whole].view(np.int32) == g1[whole].view(np.int32)).all(), "chunks wholly inside: mode-1 bits"
    assert np.isneginf(gw[n_in == 0]).all(), "chunks without an in-window item: -inf"
    if B > 2:
        assert np.isneginf(gw[1]).all()
    mixed = (n_in > 0) & (n_in < n_valid)
    assert mixed.sum() > 100, "fixture must have mixed chunks"
    assert (gw[mixed] <= g1[mixed]).all()
    S = (Q[:B].double() @ I.double().t()).cpu().numpy()
    ref = np.where(inw, S, -np.inf).reshape(B, -1, 8).max(-1)
    np.testing.assert_allclose(gw[mixed], ref[mixed], rtol=0, atol=2e-3)
    # the partial sums count in-window items only
    want = (np.exp(S - c[:B, None].double().cpu().numpy()) * inw).sum(1)
    got = partw[:, :B].double().sum(0).cpu().numpy()
    np.testing.assert_allclose(got, want, rtol=2e-3)
    # the whole int32 range is no window at all
    full = (dev(t), dev(np.full(B, I32_MIN, np.int32)), dev(np.full(B, I32_MAX, np.int32)))
    _, cmf, tmf = _gemm(Q, I, c, B, N, n_pad, full)
    assert torch.equal(cmf, cm1) and torch.equal(tmf, tm1)


# ------------------------------------------------------------------------------------------------ recommend(window=)
def make_windows(rs, times, B, K):
    """Per-session windows of five kinds: the whole range / ~10 % of it / K // 2 items (fewer than K: padding) / one
    item / no item.  The last three give their items times of their own: times [N] int32 in [0, 10000) is updated in
    place.  Returns (lo, hi, the one-item sessions' items)."""
    N = len(times)
    lo, hi = np.zeros(B, np.int64), np.zeros(B, np.int64)
    perm = rs.permutation(N)
    times[perm[:K // 2]] = 30000
    one = {}
    for b in range(B):
        kind = (b + 1) % 5 if B > 1 else 1
        if kind == 0:
            lo[b], hi[b] = 0, 9999
        elif kind == 1:
            lo[b] = rs.randint(0, 9000)
            hi[b] = lo[b] + 999
        elif kind == 2:
            lo[b] = hi[b] = 30000
        elif kind == 3:
            one[b] = j = int(perm[(K // 2 + b) % N])
            times[j] = 20000 + b
            lo[b] = hi[b] = 20000 + b
        else:
            lo[b], hi[b] = -100, -1
    return lo, hi, one


def in_window(times, lo, hi):
    return (times[None, :] >= lo[:, None]) & (times[None, :] <= hi[:, None])


@pytest.mark.parametrize("B,N,K,T,kind", [(1, 300, 1, 1, "plain"), (7, 2000, 20, 3, "dup"),
                                          (512, 9000, 256, 20, "clicked"), (64, 70000, 256, 2, "maxx"),
                                          (5, 300, 256, 4, "small"), (24, GLOBO_N, 20, 5, "plain"),
                                          (10, GLOBO_N, 256, 3, "clicked")])
def test_window_matches_fp64_reference(B, N, K, T, kind):
    from tcar_b200 import _native as nv
    model, content, mwdhm, _ = build(N, emb_scale=20.0)
    bt, batch = batch_for(model, N, B, T, 0, mwdhm, seed=B + K + 1)
    rs = np.random.RandomState(K + 5)
    times = rs.randint(0, 10000, N).astype(np.int32)
    lo, hi, one = make_windows(rs, times, B, K)
    model.set_item_times(times)
    off = lst = None
    clicked = kind in ("clicked", "small")
    if kind == "dup":
        off, lst = make_lists(rs, N, [0, 1, 5, 37, 100, 3, 250], dup=True)
    elif kind == "maxx":
        off, lst = make_lists(rs, N, [nv.RECOMMEND_MAXX] + rs.randint(0, nv.RECOMMEND_MAXX + 1, B - 1).tolist())
    elif kind == "small":
        off, lst = make_lists(rs, N, [40, 0, 100, 7, 60])
    kw = dict(exclude_off=off, exclude_ids=lst, exclude_clicked=clicked, window=(lo, hi))
    ids, sc = [x.clone() for x in model.recommend(bt, K, **kw)]
    ids2, sc2 = model.recommend(bt, K, **kw)
    torch.cuda.synchronize()
    assert torch.equal(ids, ids2) and torch.equal(sc, sc2), "a second run must be bit-identical"
    S = np.where(in_window(times, lo, hi), oracle_scores(model, content, mwdhm, batch), -np.inf)  # out of window
    ex = excluded_sets(B, off, lst, batch["seq"].numpy() if clicked else None)
    ids_h, sc_h = ids.cpu().numpy(), sc.cpu().numpy()
    check_topk(ids_h, sc_h, S, K, ex)
    got_t = np.where(ids_h >= 0, times[np.maximum(ids_h, 0)], lo[:, None])
    assert ((got_t >= lo[:, None]) & (got_t <= hi[:, None])).all(), "every returned item is in its window"
    if B >= 5:
        kinds = [(b + 1) % 5 for b in range(B)]
        assert all((ids_h[b] == -1).all() for b in range(B) if kinds[b] == 4), "no item in the window: all -1"
        assert all((ids_h[b] == -1).any() for b in range(B) if kinds[b] == 2), "fewer than K: padded"
        for b, j in one.items():                         # its item, unless one of its clicks excludes it
            assert ids_h[b, 0] in (j, -1) and (ids_h[b, 1:] == -1).all()
        assert np.isneginf(sc_h[ids_h == -1]).all()
        rescored = model.rec_rescored[:B].cpu().numpy()
        assert all(rescored[b] == 0 for b in range(B) if kinds[b] == 4), "an empty window re-scores nothing"


def test_window_equals_exclusion_lists_bit_for_bit():
    """Where the out-of-window ids fit in an exclusion list, a window and that list give the same result, ids and
    scores with torch.equal, with and without the clicks excluded as well."""
    from tcar_b200 import _native as nv
    N, B, T, K = 1500, 96, 3, 50
    model, _, mwdhm, _ = build(N, emb_scale=20.0)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=21)
    rs = np.random.RandomState(4)
    times = rs.randint(0, 1000, N).astype(np.int32)
    lo = rs.randint(0, 450, B)
    hi = lo + rs.randint(420, 550, B)
    model.set_item_times(times)
    out = [np.flatnonzero((times < lo[b]) | (times > hi[b])) for b in range(B)]
    assert max(len(o) for o in out) + T <= nv.RECOMMEND_MAXX
    off = np.cumsum([0] + [len(o) for o in out]).astype(np.int32)
    lst = np.concatenate(out).astype(np.int32)
    for clicked in (False, True):
        a = [x.clone() for x in model.recommend(bt, K, exclude_clicked=clicked, window=(lo, hi))]
        b_ = model.recommend(bt, K, off, lst, exclude_clicked=clicked)
        torch.cuda.synchronize()
        assert torch.equal(a[0], b_[0]) and torch.equal(a[1], b_[1]), clicked
    assert (a[0] >= 0).all()


def test_full_window_equals_no_window():
    N, B, T, K = 20000, 200, 4, 100
    model, _, mwdhm, _ = build(N, emb_scale=20.0)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=8)
    model.set_item_times(np.random.RandomState(2).randint(I32_MIN, I32_MAX, N, dtype=np.int64))
    full = (np.full(B, I32_MIN), np.full(B, I32_MAX))
    a = [x.clone() for x in model.recommend(bt, K, exclude_clicked=True)]
    na = model.rec_rescored[:B].clone()
    w = [x.clone() for x in model.recommend(bt, K, exclude_clicked=True, window=full)]
    nw = model.rec_rescored[:B].clone()
    w2 = model.recommend(bt, K, exclude_clicked=True, window=full)
    torch.cuda.synchronize()
    assert torch.equal(a[0], w[0]) and torch.equal(a[1], w[1]) and torch.equal(na, nw)
    assert torch.equal(w[0], w2[0]) and torch.equal(w[1], w2[1])
    own_order_ok(w[0].cpu().numpy(), w[1].cpu().numpy())


def test_window_host_checks_launch_nothing():
    from tcar_b200 import _native as nv
    N, B, T = 500, 4, 2
    model, _, mwdhm, _ = build(N)
    bt, _ = batch_for(model, N, B, T, 0, mwdhm, seed=1)
    before = nv.LAUNCHES["count"]
    with pytest.raises(ValueError, match="set_item_times"):
        model.recommend(bt, 5, window=(np.zeros(B, int), np.ones(B, int)))
    for times, what in [(np.zeros(N - 1, np.int32), f"N = {N}"), (np.full(N, 2 ** 31), "item 0"),
                        (np.zeros(N), "integers")]:
        with pytest.raises(ValueError, match=what):
            model.set_item_times(times)
    assert getattr(model, "_item_time", None) is None
    model.set_item_times(np.arange(N))
    for window, what in [((np.zeros(B - 1, int), np.ones(B, int)), "lo must hold B = 4"),
                         ((np.zeros(B, int), np.ones(B + 1, int)), "hi must hold B = 4"),
                         ((np.array([0, 0, -2 ** 31 - 1, 0]), np.ones(B, int)), "session 2"),
                         ((np.zeros(B, int), np.array([1, 1, 1, 2 ** 31])), "session 3"),
                         ((np.array([0, 9, 0, 0]), np.array([1, 8, 1, 1])), "session 1: window lo 9 > hi 8")]:
        with pytest.raises(ValueError, match=what):
            model.recommend(bt, 5, window=window)
    assert nv.LAUNCHES["count"] == before, "validation happens before any launch"
    # the C entry points refuse missing window inputs
    p, ps = nv.ptr, model.ps
    buf = torch.zeros(ps.n_pad * 4, device=model.dev)
    assert nv.lib().tcar_score_fwd_window(p(buf), p(buf), p(buf), p(buf), p(buf), p(buf), None, p(buf), p(buf), B, N,
                                          ps.n_pad, nv.stream_ptr()) == -1
    assert nv.lib().tcar_score_fwd_window(p(buf), p(buf), p(buf), p(buf), p(buf), p(buf), p(buf), p(buf), p(buf), B, N,
                                          ps.n_pad + 128, nv.stream_ptr()) == -1
    ws = torch.zeros(int(nv.lib().tcar_recommend_ws_bytes(B)), device=model.dev, dtype=torch.uint8)
    base = [p(buf)] * 8 + [None, None, None, T, B, N, ps.n_pad, 5, p(ws), p(buf), p(buf), None, p(buf), p(buf), p(buf),
                           nv.stream_ptr()]
    for at in (20, 21, 22):
        a = list(base)
        a[at] = None
        assert nv.lib().tcar_recommend_window(*a) == -1
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ end to end
def test_recommend_split_with_max_age_end_to_end(tmp_path, monkeypatch):
    """main.py --recommend_k 20 --recommend_max_age_h 24 on a synthetic split whose test sessions were moved into the
    publication month: every written article was published in its session's window, and label_outside counts the
    sessions whose label was not."""
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
    args = tmain.build_parser().parse_args(["--datapath", str(tmp_path) + "/", "--dataset", "synth/TCAR-mid/",
                                            "--foldnum", "0", "--epoch", "1", "--batch_size", "64",
                                            "--recommend_k", "20", "--recommend_max_age_h", "24"])
    model = tmain.main(args)
    got = model.last_recommend_metrics
    publish_dt, _ = load("publish_time_0.txt")
    item_dict, sdict = load("item_dict_0.txt"), load("session_dict_test_0.pkl")
    pub = epoch_minutes(publish_dt)
    t_req = {k: int(epoch_minutes([v[-2]["click_t"]])[0]) for k, v in tdict.items()}
    outside = sum(not (t_req[k] - 1440 <= pub[sdict[k][-1] - 1] <= t_req[k]) for k in sdict)
    assert got["label_outside"] == outside > 0
    lines = open(tmp_path / "saved" / "recommend_0.txt").read().splitlines()
    assert len(lines) == n_test == got["sessions"]
    n_pairs = 0
    for line in lines:
        key, *pairs = line.split()
        key = int(key)
        arts = [a.rsplit(":", 1)[0] for a in pairs]
        assert len(arts) <= 20 and len(set(arts)) == len(arts)
        for a in arts:
            assert t_req[key] - 1440 <= pub[item_dict[a] - 1] <= t_req[key], (key, a)
        n_pairs += len(arts)
    assert n_pairs > 10 * n_test, "windows must hold articles"
