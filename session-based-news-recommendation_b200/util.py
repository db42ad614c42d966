"""Host utilities mirroring the reference's util.py: data_partition (pickle loader, util.py:20-57), cau_metrics
(util.py:8-18), save_model (util.py:102-106; the reference version is broken -- stray `self`, wrong key)."""
import os
import pickle
import time

import numpy as np


def cau_metrics(preds, labels, cutoff=20):
    """util.py:8-18 on a materialised score matrix (used by tests / debugging; the hot path gets the rank from
    tcar_eval_topk's n_greater instead)."""
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
