"""Host utilities mirroring the reference's util.py: data_partition (pickle loader, util.py:20-57), cau_metrics
(util.py:8-18), save_model (util.py:102-106; the reference version is broken -- stray `self`, wrong key)."""
import datetime
import os
import pickle
import time

import numpy as np

from ._native import CHUNK, DECAY_MAX_AGE, RECOMMEND_MAXG


def cau_metrics(preds, labels, cutoff=20):
    """util.py:8-18 on a materialised score matrix (used by tests / debugging; the hot path gets the rank from
    tcar_eval_topk_certified's n_greater instead)."""
    preds = np.asarray(preds)
    recall, mrr, ndcg = [], [], []
    for row, lab in zip(preds, labels):
        rank = int((row[lab] < row).sum()) + 1
        recall.append(rank <= cutoff)
        mrr.append(1 / rank if rank <= cutoff else 0.0)
        ndcg.append(1 / np.log2(rank + 1) if rank <= cutoff else 0.0)
    return recall, mrr, ndcg


IMPRESSION_SUMS = ("auc", "mrr", "ndcg5", "ndcg10", "sessions", "skipped")


def impression_sums(rank, auc, n_neg):
    """Per-session results of ranking impression lists (one positive each: rank = 1 + #negatives scoring above it,
    auc, n_neg = #negatives) -> float64 [6]: the sums of AUC, MRR = 1/rank (not truncated), nDCG@5 and nDCG@10
    (1/log2(1 + rank) when rank <= k, else 0) over the sessions with at least one negative, their number, and the
    number of sessions without a negative.  Sums add up across batches and ranks; impression_metrics averages them."""
    rank = np.asarray(rank, dtype=np.float64)
    auc = np.asarray(auc, dtype=np.float64)
    used = np.asarray(n_neg) > 0
    r, a = rank[used], auc[used]
    gain = 1.0 / np.log2(1.0 + r)
    return np.array([a.sum(), (1.0 / r).sum(), np.where(r <= 5, gain, 0.0).sum(), np.where(r <= 10, gain, 0.0).sum(),
                     used.sum(), (~used).sum()], dtype=np.float64)


def impression_metrics(sums):
    """impression_sums (possibly added up) -> {"auc", "mrr", "ndcg5", "ndcg10", "sessions", "skipped"}."""
    s = np.asarray(sums, dtype=np.float64)
    n = s[4]
    out = {k: float(s[i] / n) if n > 0 else float("nan") for i, k in enumerate(IMPRESSION_SUMS[:4])}
    out["sessions"], out["skipped"] = int(s[4]), int(s[5])
    return out


def label_positions(ids, labels):
    """1-based position of each session's label in its recommended list ids [B, K] (0 when absent)."""
    ids = np.asarray(ids)
    hit = ids == np.asarray(labels).reshape(-1, 1)
    return np.where(hit.any(1), hit.argmax(1) + 1, 0)


def topk_sums(rank):
    """Label positions in top-K lists (label_positions; 0 = not in the list) -> float64 [4]: the sums of HR@K (hit),
    MRR@K (1/rank) and nDCG@K (1/log2(1 + rank)), misses counting 0, and the number of sessions.  Sums add up across
    batches and ranks; topk_metrics averages them."""
    r = np.asarray(rank, dtype=np.float64)
    hit = r > 0
    rr = np.where(hit, r, 1.0)
    return np.array([hit.sum(), np.where(hit, 1.0 / rr, 0.0).sum(), np.where(hit, 1.0 / np.log2(1.0 + rr), 0.0).sum(),
                     len(r)], dtype=np.float64)


def topk_metrics(sums):
    """topk_sums (possibly added up) -> {"hr", "mrr", "ndcg", "sessions"}."""
    s = np.asarray(sums, dtype=np.float64)
    n = s[3]
    out = {k: float(s[i] / n) if n > 0 else float("nan") for i, k in enumerate(("hr", "mrr", "ndcg"))}
    out["sessions"] = int(n)
    return out


def recommend_line(key, ids, scores, reverse_item):
    """One line of a recommendation file: the session key, then `article:score` for every returned item (original
    article ids through reverse_item, 0-based item id -> article; the -1 padding of a small catalog is left out).
    Scores are printed with 9 significant digits, enough to read back the fp32 value exactly."""
    pairs = ["{}:{:.9g}".format(reverse_item[int(i)], float(s)) for i, s in zip(ids, scores) if i >= 0]
    return " ".join([str(key)] + pairs) + "\n"


def check_id_lists(off, ids, B, N, *, names, nouns, limit, limit_name, extra=0):
    """Validate B per-session id lists in CSR form (session b's ids are ids[off[b]:off[b + 1]]) before anything is
    launched: off holds B + 1 integer offsets from 0 to len(ids), never decreasing; a list's length plus `extra` (the
    session's clicks counted against the same limit) is at most `limit`; every id lies in [0, N).  The checks run in
    the caller's own integer type (min / max first: no int64 copy of a long list) and raise a ValueError that names the
    first offending session.  names = (offsets, ids) and nouns = (one id, the list's entries) word the messages, e.g.
    ("cand_off", "cand_ids") and ("candidate id", "candidates").
    Returns (the int32 host array [off | ids] the kernels read, the longest list's length; 0 when B = 0)."""
    off, ids = np.asarray(off).reshape(-1), np.asarray(ids).reshape(-1)
    if off.dtype.kind not in "iu" or (ids.size and ids.dtype.kind not in "iu"):
        raise ValueError(f"{names[0]} and {names[1]} must hold integers")
    if off.shape[0] != B + 1 or off[0] != 0 or off[-1] != ids.shape[0]:
        raise ValueError(f"{names[0]} must hold B + 1 = {B + 1} offsets from 0 to len({names[1]}) = {ids.shape[0]}")
    lens = np.diff(off.astype(np.int64))
    for bad, what in ((lens < 0, f"{names[0]} decreases"),
                      (lens + extra > limit, f"more than {limit_name} = {limit} {nouns[1]}" +
                       (f" with its {extra} clicks" if extra else ""))):
        if bad.any():
            raise ValueError(f"session {int(np.argmax(bad))}: {what}")
    if ids.size and (ids.min() < 0 or ids.max() >= N):
        j = int(np.argmax((ids < 0) | (ids >= N)))
        s = int(np.searchsorted(off, j, side="right")) - 1
        raise ValueError(f"session {s}: {nouns[0]} {int(ids[j])} outside [0, {N})")
    host = np.empty(B + 1 + ids.shape[0], dtype=np.int32)
    host[:B + 1], host[B + 1:] = off, ids
    return host, int(lens.max()) if B else 0


INT32_MIN, INT32_MAX = -2 ** 31, 2 ** 31 - 1
_EPOCH = datetime.datetime(1970, 1, 1)
_EPOCH_UTC = _EPOCH.replace(tzinfo=datetime.timezone.utc)
_MINUTE = datetime.timedelta(minutes=1)


def epoch_minutes(datetimes):
    """datetime objects -> int64 whole minutes since 1970-01-01 00:00 (floor: seconds are dropped, so a click and an
    article of the same minute compare equal).  Naive datetimes are read as UTC, aware ones converted."""
    return np.array([(d - (_EPOCH if d.tzinfo is None else _EPOCH_UTC)) // _MINUTE for d in datetimes],
                    dtype=np.int64)


def check_item_times(times, N):
    """Validate one time per item before anything is uploaded: N integers of any integer type, each within int32.
    Returns them as an int32 host array; raises ValueError naming the first bad item."""
    t = np.asarray(times).reshape(-1)
    if t.size and t.dtype.kind not in "iu":
        raise ValueError("item times must be integers")
    if t.shape[0] != N:
        raise ValueError(f"item times must hold N = {N} values, got {t.shape[0]}")
    if N and (t.min() < INT32_MIN or t.max() > INT32_MAX):
        n = int(np.argmax((t < INT32_MIN) | (t > INT32_MAX)))
        raise ValueError(f"item {n}: time {int(t[n])} outside int32")
    return t.astype(np.int32)


def check_windows(window, B):
    """Validate the publish-time windows (lo, hi) of B sessions before anything is launched: two host arrays of B
    integers each within int32, lo[b] <= hi[b].  Returns the int32 host array [lo | hi] the kernels read; raises
    ValueError naming the first bad session."""
    if not isinstance(window, (tuple, list)) or len(window) != 2:
        raise ValueError("window must be a pair (lo, hi) of arrays of B integers")
    lo, hi = (np.asarray(w).reshape(-1) for w in window)
    for name, w in (("lo", lo), ("hi", hi)):
        if w.size and w.dtype.kind not in "iu":
            raise ValueError(f"window {name} must hold integers")
        if w.shape[0] != B:
            raise ValueError(f"window {name} must hold B = {B} values, got {w.shape[0]}")
        if B and (w.min() < INT32_MIN or w.max() > INT32_MAX):
            b = int(np.argmax((w < INT32_MIN) | (w > INT32_MAX)))
            raise ValueError(f"session {b}: window {name} {int(w[b])} outside int32")
    if B and (lo.astype(np.int64) > hi.astype(np.int64)).any():
        b = int(np.argmax(lo.astype(np.int64) > hi.astype(np.int64)))
        raise ValueError(f"session {b}: window lo {int(lo[b])} > hi {int(hi[b])}")
    out = np.empty(2 * B, dtype=np.int32)
    out[:B], out[B:] = lo, hi
    return out


def decay_penalty(t_ref, rate, times):
    """The penalty p = rate * age of the freshness decay (DESIGN §4.10, csrc/decay.cuh) in float32, for session
    request times t_ref [B], rates [B] and item times [N] -> [B, N]: age = min(max(t_ref - t, 0), DECAY_MAX_AGE),
    exact in float32, then one float32 multiply.  The decayed score is s - p, one float32 subtract."""
    age = np.clip(np.asarray(t_ref, np.int64).reshape(-1, 1) - np.asarray(times, np.int64).reshape(1, -1), 0,
                  DECAY_MAX_AGE).astype(np.float32)
    return np.asarray(rate, np.float32).reshape(-1, 1) * age


def check_decay(decay, B, times):
    """Validate the freshness decay (t_ref, rate) of B sessions before anything is launched: t_ref holds B integers
    within int32 (the clock unit of the item times), rate is one number or B numbers, each finite and >= 0 (score
    units per clock unit), and every session's largest penalty over the catalog (item times `times`, int32 [N]) is
    finite in float32.  Returns the int32 host array [t_ref | the rates' float32 bits] the kernels read; raises
    ValueError naming the first bad session."""
    if not isinstance(decay, (tuple, list)) or len(decay) != 2:
        raise ValueError("decay must be a pair (t_ref, rate)")
    t_ref = np.asarray(decay[0]).reshape(-1)
    if t_ref.size and t_ref.dtype.kind not in "iu":
        raise ValueError("decay t_ref must hold integers")
    if t_ref.shape[0] != B:
        raise ValueError(f"decay t_ref must hold B = {B} values, got {t_ref.shape[0]}")
    if B and (t_ref.min() < INT32_MIN or t_ref.max() > INT32_MAX):
        b = int(np.argmax((t_ref < INT32_MIN) | (t_ref > INT32_MAX)))
        raise ValueError(f"session {b}: decay t_ref {int(t_ref[b])} outside int32")
    rate = np.asarray(decay[1])
    if rate.dtype.kind not in "iuf" or rate.ndim > 1 or (rate.ndim == 1 and rate.shape[0] != B):
        raise ValueError(f"decay rate must be one number or B = {B} numbers")
    rate = np.broadcast_to(rate.astype(np.float64), (B,))
    if B and not (np.isfinite(rate) & (rate >= 0)).all():
        b = int(np.argmax(~(np.isfinite(rate) & (rate >= 0))))
        raise ValueError(f"session {b}: decay rate {float(rate[b])} is not finite and >= 0")
    with np.errstate(over="ignore"):                   # an overflow is what the checks below look for
        r32 = rate.astype(np.float32)
        worst = decay_penalty(t_ref, r32, [np.asarray(times).min()])[:, 0] if len(times) else np.zeros(B)
    if B and not np.isfinite(r32).all():
        b = int(np.argmax(~np.isfinite(r32)))
        raise ValueError(f"session {b}: decay rate {float(rate[b])} overflows float32")
    if B and not np.isfinite(worst).all():
        b = int(np.argmax(~np.isfinite(worst)))
        raise ValueError(f"session {b}: decay rate {float(rate[b])} gives the penalty {worst[b]} for its oldest "
                         "item, not finite in float32")
    out = np.empty(2 * B, dtype=np.int32)
    out[:B], out[B:] = t_ref, r32.view(np.int32)
    return out


def session_request_times(keys, session_time_dict):
    """Request times t_req of a batch's sessions (keys in batch order) in epoch minutes: the click_t of the session's
    last input click (session_time_dict[key][-2], the click the sampler takes the request context from).  int64."""
    return epoch_minutes([session_time_dict[k][-2]["click_t"] for k in keys])


def session_windows(keys, session_time_dict, max_age_min):
    """Publish-time windows of a batch's sessions (keys in batch order) for recommend(window=...): [t_req - max_age_min,
    t_req] in epoch minutes, t_req = session_request_times.  Returns int64 arrays (lo, hi)."""
    hi = session_request_times(keys, session_time_dict)
    return hi - int(max_age_min), hi


def count_outside(times, lo, hi):
    """Number of sessions whose time (e.g. their label's publish time) lies outside their window [lo, hi]."""
    t = np.asarray(times, dtype=np.int64)
    return int(((t < np.asarray(lo)) | (t > np.asarray(hi))).sum())


def check_item_categories(codes, N, G=None):
    """Validate one category code per item before anything is uploaded: N integers in [0, G), G <= RECOMMEND_MAXG
    (G defaults to max(codes) + 1).  Returns (the codes as an int32 host array, G); raises ValueError."""
    c = np.asarray(codes).reshape(-1)
    if c.size and c.dtype.kind not in "iu":
        raise ValueError("item categories must be integers")
    if c.shape[0] != N:
        raise ValueError(f"item categories must hold N = {N} codes, got {c.shape[0]}")
    if G is None:
        G = max(int(c.max()) + 1, 1) if c.size else 1
    if isinstance(G, (bool, np.bool_)) or not isinstance(G, (int, np.integer)) or not 1 <= G <= RECOMMEND_MAXG:
        raise ValueError(f"the number of categories must be in [1, TCAR_RECOMMEND_MAXG = {RECOMMEND_MAXG}], got {G!r}")
    if c.size and (c.min() < 0 or c.max() >= G):
        n = int(np.argmax((c < 0) | (c >= G)))
        raise ValueError(f"item {n}: category {int(c[n])} outside [0, {G})")
    return c.astype(np.int32), int(G)


def category_layout(codes, G):
    """The catalog in category order for recommend(max_per_category / categories): codes = N ints in [0, G).
    Items are sorted by (code, id) and every category is padded to a multiple of CHUNK positions by repeating its last
    item, so that every chunk holds items of one category only and its maximum is the score of a real item.
    Returns (perm int32 [N'], cat_chunk_off int32 [G + 1], N'): perm[p] = the original id at position p, -1 on a pad
    (pad_sources gives the item a pad repeats); category g owns the chunks cat_chunk_off[g] .. cat_chunk_off[g + 1]
    (empty for an empty category); N' = CHUNK * cat_chunk_off[G] <= N + 7 G."""
    c = np.asarray(codes, dtype=np.int64).reshape(-1)
    order = np.argsort(c, kind="stable")                       # by (code, id)
    count = np.bincount(c, minlength=G)[:G]
    off = np.zeros(G + 1, dtype=np.int64)
    np.cumsum((count + CHUNK - 1) // CHUNK, out=off[1:])
    first = np.zeros(G + 1, dtype=np.int64)                    # first sorted index of each category
    np.cumsum(count, out=first[1:])
    n2 = int(off[G]) * CHUNK
    perm = np.full(n2, -1, dtype=np.int32)
    cat = c[order]
    perm[off[cat] * CHUNK + (np.arange(c.shape[0]) - first[cat])] = order
    return perm, off.astype(np.int32), n2


def pad_sources(perm):
    """The id whose row every position of a category_layout holds: perm[p], or on a pad the item it repeats (the
    last real position before it, which always lies in the same chunk and category).  int64 [N']."""
    perm = np.asarray(perm)
    last = np.where(perm >= 0, np.arange(perm.shape[0]), 0)
    return perm[np.maximum.accumulate(last)].astype(np.int64) if perm.size else np.zeros(0, dtype=np.int64)


def list_ild(cats):
    """Intra-list diversity of one list's category codes (model_combine.py:174-182 of the reference): the share of
    ordered pairs of distinct positions whose categories differ; 0 for a list of fewer than two items."""
    c = np.asarray(cats).reshape(-1)
    n = c.shape[0]
    return float((c[:, None] != c[None, :]).sum()) / (n * (n - 1)) if n > 1 else 0.0


def list_unexp(cats, clicked_cats):
    """Unexpectedness of one list (model_combine.py:184-194 of the reference): the share of (recommended, clicked)
    pairs whose categories differ; 0 for an empty list."""
    c, ci = np.asarray(cats).reshape(-1), np.asarray(clicked_cats).reshape(-1)
    if c.shape[0] == 0 or ci.shape[0] == 0:
        return 0.0
    return float((c[:, None] != ci[None, :]).sum()) / (c.shape[0] * ci.shape[0])


def diversity_sums(ids, clicked, cat):
    """Sums of list_ild and list_unexp over the returned lists ids [B, K] (the -1 padding dropped) of at least two
    items, and their number (test() averages over those lists); clicked[b] = the 0-based ids of session b's clicks,
    cat = the category code of every item.  float64 [3]; the sums add up across batches and ranks."""
    cat = np.asarray(cat)
    s = np.zeros(3)
    for row, cl in zip(np.asarray(ids), clicked):
        c = cat[row[row >= 0]]
        if len(c) > 1:
            s += (list_ild(c), list_unexp(c, cat[np.asarray(cl, dtype=np.int64)]), 1)
    return s


def _load(path):
    with open(path, "rb") as f:
        return pickle.load(f)


def data_partition(fname, foldnum, impression_path=None):
    """Same 7-tuple as util.data_partition.  `fname` = datapath + dataset + split_way.  The reference hard-codes
    /home/sansa/recsys/TCAR/data/mind/sess_impressions.mid (util.py:47); here `impression_path` (or
    <fname>sess_impressions.mid, else <fname>neighbor_<fold>.txt) supplies the neighbour dict."""
    f = str(foldnum)
    train = (_load(fname + "len_dict_train" + f + ".pkl"), _load(fname + "session_dict_train_" + f + ".pkl"),
             _load(fname + "session_time_dict_train" + f + ".pkl"))
    test = (_load(fname + "len_dict_test" + f + ".pkl"), _load(fname + "session_dict_test_" + f + ".pkl"),
            _load(fname + "session_time_dict_test" + f + ".pkl"))
    item_dict = _load(fname + "item_dict_" + f + ".txt")
    neighbor_dict = None
    for cand in (impression_path, fname + "sess_impressions.mid", fname + "neighbor_" + f + ".txt"):
        if cand and os.path.exists(cand):
            neighbor_dict = _load(cand)
            break
    if neighbor_dict is None:
        raise FileNotFoundError("no impression / neighbour file found (pass --impression_path)")
    content_emb = _load(fname + "content_weight_" + f + ".txt")
    publish_time = _load(fname + "publish_time_" + f + ".txt")
    return train, test, item_dict, neighbor_dict, content_emb, publish_time, None


def save_model(model, args, saver=None):
    """Checkpoint = parameters + Adam moments + step (torch.save)."""
    import torch
    suf = time.strftime("%Y%m%d%H%M", time.localtime()) + "-" + args["dataset"].strip("/").replace("/", "_") + \
        "-" + args["split_way"].strip("/") + "-" + str(args["foldnum"])
    os.makedirs(args["modelpath"], exist_ok=True)
    path = os.path.join(args["modelpath"], "model.ckpt-" + suf)
    model.sync_updates()
    model.sync_item_table()                  # catalog-sharded training: collect every owner's rows (and moments) first
    model.sync_optimizer_state()             # data-parallel sharded update: collect every rank's moment slices
    if getattr(model, "rank", 0) == 0:       # now every rank holds the same state; one writer
        torch.save(model.ps.state_dict(), path)
    return path


def restore_model(model, path):
    import torch
    model.sync_updates()
    # the state dict holds tensors, ints and a dict of tensors only: no pickled code is ever executed
    model.ps.load_state_dict(torch.load(path, map_location="cpu", weights_only=True))
