"""Helpers shared by the top-K recommendation tests: the oracle's scores, the fp64 reference of recommend() (plain,
windowed through -inf scores, capped and filtered by category) and the checks of a result against it."""
import numpy as np

GLOBO_N = 364047


def oracle_scores(model, content, mwdhm, batch):
    """The oracle's softmax_input (model_combine.py:138) for the batch: [B, N] fp64 scores."""
    import torch
    from oracle import tcar_oracle as O
    from test_gpu_parity import oracle_inputs
    params, c64, m64 = oracle_inputs(model, content, mwdhm)
    with torch.no_grad():
        return O.forward(params, c64, m64, batch)["softmax_input"].numpy()


def topk_ref(S, K, excluded, C=None, cat=None, allowed=None):
    """fp64 greedy reference: per row walk the eligible items (finite score, allowed category, not excluded) by (score
    desc, id asc), drop an item that has C items of its category before it, stop at K kept.  C = None: no cap; cat =
    None: one category; allowed = None: every category (else one set or None per row).  Returns ids / scores padded
    with -1 / -inf and whether the scores that decide the walk (the first C + 1 of each category up to one item past
    its end; without a cap the first K + 1) are separated by more than 2e-5 |score| (the ids are then exact)."""
    B, N = S.shape
    C = K if C is None else C
    cat = np.zeros(N, np.int64) if cat is None else cat
    allowed = [None] * B if allowed is None else allowed
    ids = np.full((B, K), -1, np.int64)
    sc = np.full((B, K), -np.inf)
    margin = np.zeros(B, bool)
    for b in range(B):
        s = S[b].copy()
        if allowed[b] is not None:
            s[~np.isin(cat, np.asarray(sorted(allowed[b]), np.int64))] = -np.inf
        s[np.array(sorted(excluded[b]), np.int64)] = -np.inf
        order = np.lexsort((np.arange(N), -s))
        order = order[np.isfinite(s[order])]
        used, n, decide = {}, 0, []
        for j in order:
            g = int(cat[j])
            seen = used.get(g, 0)
            used[g] = seen + 1
            if seen <= C:
                decide.append(s[j])
            if n == K:
                break
            if seen < C:
                ids[b, n], sc[b, n] = j, s[j]
                n += 1
        head = np.array(decide)
        margin[b] = len(head) < 2 or bool((np.abs(np.diff(head)) > 2e-5 * np.abs(head).max()).all())
    return ids, sc, margin


def own_order_ok(ids, sc):
    """Every row is ordered exactly by (score desc, id asc) of its own fp32 scores, padding last."""
    for i_row, s_row in zip(ids, sc):
        n = int((i_row >= 0).sum())
        assert (i_row[n:] == -1).all() and np.isneginf(s_row[n:]).all()
        i, s = i_row[:n].astype(np.int64), s_row[:n].astype(np.float64)
        assert (np.lexsort((i, -s)) == np.arange(n)).all()
        assert len(set(i.tolist())) == n


def check_topk(ids, sc, S, K, excluded, C=None, cat=None, allowed=None):
    """A device result against topk_ref: its own order, padding where the reference has no eligible item, scores
    within fp32 error, ids exact on margin-checked rows, and on every row eligible items as good as the reference's,
    position by position.  With categories (cat given) also: only allowed categories and at most C per category.
    Returns the margin mask."""
    r_ids, r_sc, margin = topk_ref(S, K, excluded, C, cat, allowed)
    own_order_ok(ids, sc)
    valid = r_ids >= 0
    assert ((ids >= 0) == valid).all(), "padding where the reference has no eligible item"
    np.testing.assert_allclose(sc[valid], r_sc[valid], rtol=1e-4, atol=1e-5)
    assert (ids[margin] == r_ids[margin]).all(), "ids exact on margin-checked rows"
    for b in range(len(ids)):
        got = ids[b][ids[b] >= 0]
        assert not (set(got.tolist()) & excluded[b])
        if cat is not None:
            if allowed is not None and allowed[b] is not None:
                assert set(cat[got].tolist()) <= allowed[b]
            assert np.bincount(cat[got]).max(initial=0) <= (K if C is None else C), "at most C per category"
        np.testing.assert_allclose(S[b, got], r_sc[b, :len(got)], rtol=1e-4, atol=1e-5)
    return margin


def make_lists(rs, N, lens, dup=False):
    off = np.zeros(len(lens) + 1, dtype=np.int32)
    off[1:] = np.cumsum(lens)
    ids = rs.randint(0, N, int(off[-1])).astype(np.int32)
    if dup:
        for b, L in enumerate(lens):
            if L > 2:
                ids[off[b] + L - 1] = ids[off[b]]
                ids[off[b] + 1] = ids[off[b]]
    return off, ids


def excluded_sets(B, off, ids, seq=None):
    ex = [set() for _ in range(B)]
    if off is not None:
        for b in range(B):
            ex[b].update(ids[off[b]:off[b + 1]].tolist())
    if seq is not None:
        for b in range(B):
            ex[b].update((seq[b] - 1).tolist())
    return ex
