"""Host-side batch production -- mirrors the reference's sampler.Sampler (sampler.py:23-140) API and RNG use.

`Sampler(len_dict, session_dict, session_time_dict, neighbor_dict, item_dict, neg_num, batch_size)` with
`has_next()` / `next_batch()` returning the reference's 6-tuple of Python lists, plus `next_packed()`, which emits
the same indices as ONE contiguous int32 array (the layout `model_combine.Batch` consumes) so that a batch costs a
single pinned host->device copy.

Differences from the reference, all documented in DESIGN.md:
  * per-click time features are extracted once per session and cached (the reference re-reads datetime attributes
    for every click of every epoch); the values are identical;
  * the dwell-time bucket is clamped to 10: `bucketized` returns 11 for active_t >= 1024 s, which is out of range
    for the 11-row duration table (sampler.py:18-21; TF-CPU would raise, TF-GPU returns zeros);
  * negatives of a batch come from one vectorised `np.random.randint` call per session -- the legacy global NumPy
    stream yields the same values as the reference's scalar calls (tests/test_host_logic.py).
"""
import math
import random

import numpy as np

_FEATURE_CACHE = {}
_COLUMNAR_CACHE = {}


class _Columnar:
    """Packed columnar view of one dataset split (SURVEY 8f-1: "replace pickled-dict iteration with a packed columnar
    cache"): per session length L, the item sequences [n, L+1], the six per-click features [6, n, L] (publish month,
    day, isoweekday, hour+1, minute+1, clamped dwell bucket) and the click context [2, n] (isoweekday-1, hour), plus
    key -> row.  Built once per (session_dict, session_time_dict) pair and reused by every epoch's Sampler."""

    def __init__(self, session_dict, session_time_dict):
        by_len = {}
        for key, seq in session_dict.items():
            by_len.setdefault(len(seq) - 1, []).append(key)
        self.row, self.seq, self.feats, self.ctx = {}, {}, {}, {}
        for L, keys in by_len.items():
            n = len(keys)
            seq = np.empty((n, L + 1), dtype=np.int32)
            feats = np.empty((6, n, L), dtype=np.int32)
            ctx = np.empty((2, n), dtype=np.int32)
            for r, key in enumerate(keys):
                self.row[key] = r
                seq[r] = session_dict[key]
                f, c = _session_features(session_time_dict[key])
                feats[:, r, :] = f
                ctx[0, r], ctx[1, r] = c[2], c[3]
            np.minimum(feats[5], 10, out=feats[5])
            self.seq[L], self.feats[L], self.ctx[L] = seq, feats, ctx


def _columnar(session_dict, session_time_dict):
    key = (id(session_dict), id(session_time_dict))
    ent = _COLUMNAR_CACHE.get(key)
    if ent is None or ent[0] is not session_dict or ent[1] is not session_time_dict:
        ent = _COLUMNAR_CACHE[key] = (session_dict, session_time_dict, _Columnar(session_dict, session_time_dict))
    return ent[2]


def bucketized(seconds):
    """sampler.py:18-21 -- index of the first boundary in [0..10] that is >= log2(seconds + 1)."""
    return int(np.searchsorted(np.arange(0, 11), np.log2(seconds + 1)))


def _session_features(times):
    """[(month, day, isoweekday, hour+1, minute+1, gap)] per input click and the click context of the last input
    click (sampler.py:79-87,105-109)."""
    n = len(times) - 1
    feats = np.empty((6, n), dtype=np.int32)
    for j in range(n):
        t = times[j]
        p = t["publish_t"]
        feats[0, j], feats[1, j], feats[2, j] = p.month, p.day, p.isoweekday()
        feats[3, j], feats[4, j] = p.hour + 1, p.minute + 1
        feats[5, j] = bucketized(t["active_t"])
    c = times[n - 1]["click_t"]
    ctx = (c.month - 1, c.day - 1, c.isoweekday() - 1, c.hour, c.minute)
    return feats, ctx


class Sampler(object):
    def __init__(self, len_dict, session_dict, session_time_dict=None, neighbor_dict=None, item_dict=None,
                 neg_num=None, batch_size=1024, negative_mode="uniform", verbose=True):
        if verbose:
            print("Sampler init begin...")
        self.session_num = len(session_dict)
        self.batch_size = batch_size
        self.batch_i = 0
        self.neighbor_dict = neighbor_dict
        self.item_dict = item_dict
        if item_dict is not None:
            self.item_num = len(item_dict)
        self.neg_num = neg_num
        self.negative_mode = negative_mode          # "uniform" (shipped, sampler.py:98-99) | "impression" (:96,118-131)
        self.len_dict = len_dict
        self.session_dict = session_dict
        self.session_time_dict = session_time_dict
        self.session_id_batches = []
        for _slen, session_ids in self.len_dict.items():
            random.shuffle(session_ids)             # in place, like the reference (affects later epochs)
            while len(session_ids) > batch_size:
                self.session_id_batches.append(session_ids[:batch_size])
                session_ids = session_ids[batch_size:]
            if len(session_ids):
                self.session_id_batches.append(session_ids)
        self.batch_num = len(self.session_id_batches)
        random.shuffle(self.session_id_batches)
        # cache keyed by the dict object (kept alive by the cache entry so the id cannot be recycled)
        self._cache = _FEATURE_CACHE.setdefault(id(session_time_dict), (session_time_dict, {}))[1] \
            if session_time_dict else None
        self.last_in = self.last_out = self.last_neg = None
        if verbose:
            print("Sampler init finished, batch size : {}, # batch: {}.".format(self.batch_size, self.batch_num))

    def has_next(self):
        return self.batch_i < self.batch_num

    def restrict_to_rank(self, rank, world):
        """Multi-GPU training with one batch PER RANK (global batch = world x batch_size): this sampler was built with
        batch_size = world x the per-GPU batch, identically on every rank (same `random` seed, main.py:9-10); keep only
        this rank's contiguous share of every global batch (parallel.shard_sessions), so that each rank's host thread
        gathers features / draws negatives for its own <= batch_size sessions only.  `global_sizes[i]` keeps the size
        of global batch i (all ranks derive the same per-rank counts from it), `batch_T[i]` its session length (a
        rank's share of a small tail batch may be empty).  Impression negatives switch to a per-rank `random.Random`
        so that the global `random` stream -- which shuffles the next epoch's batches -- stays identical on all ranks;
        the NumPy stream of the uniform negatives is per process anyway (reseed it per rank for distinct draws)."""
        from .parallel import shard_sessions
        self._record_global_batches()
        out = []
        for b in self.session_id_batches:
            lo, hi = shard_sessions(len(b), rank, world)
            out.append(b[lo:hi])
        self.session_id_batches = out
        self._choice = random.Random(2020 + 7919 * rank).choice
        return self

    def keep_rank_batches(self, rank, world):
        """Evaluation under torchrun: batch i of the split goes to rank i mod world, so keep this rank's whole batches
        rank, rank + world, ...  `global_sizes` / `batch_T` keep the size and session length of every batch of the
        split (as restrict_to_rank does), from which all ranks derive the same rounds."""
        self._record_global_batches()
        self.session_id_batches = self.session_id_batches[rank::world]
        self.batch_num = len(self.session_id_batches)
        return self

    def _record_global_batches(self):
        self.global_sizes = [len(b) for b in self.session_id_batches]
        self.batch_T = [len(self.session_dict[b[0]]) - 1 for b in self.session_id_batches]

    def _features(self, sid):
        f = self._cache.get(sid)
        if f is None:
            f = self._cache[sid] = _session_features(self.session_time_dict[sid])
        return f

    def _negatives(self, sid):
        if not self.neighbor_dict:
            return []
        if self.negative_mode == "impression":
            return self.neg_neighbor_from_impre(int(str(sid).split("_")[0]))
        return np.random.randint(0, self.item_num, size=self.neg_num).tolist()

    def next_batch(self):
        """The reference's return value: (batch_in, batch_out, 5 publish lists, 5 click lists, neg, gap)."""
        ids = self.session_id_batches[self.batch_i]
        batch_in, batch_out, neg_all, gap_all = [], [], [], []
        pt = ([], [], [], [], [])
        ct = ([], [], [], [], [])
        for sid in ids:
            seq = self.session_dict[sid]
            batch_in.append(seq[:-1])
            batch_out.append(seq[-1] - 1)
            neg, gap = [], []
            if self.session_time_dict:
                feats, ctx = self._features(sid)
                for k in range(5):
                    pt[k].append(feats[k].tolist())
                    ct[k].append(ctx[k])
                gap = feats[5].tolist()
                neg = self._negatives(sid)
            neg_all.append(neg)
            gap_all.append(gap)
        self.batch_i += 1
        self.last_in, self.last_out, self.last_neg = batch_in, batch_out, neg_all
        return batch_in, batch_out, pt, ct, neg_all, gap_all

    def next_packed(self):
        """Same batch as next_batch() as one int32 array [7*B*T | 2*B | B | B*Nn] (see model_combine.Batch), assembled
        with array gathers from the columnar cache instead of a Python loop over clicks (~0.2 ms vs ~10 ms for 512
        sessions).  Uniform negatives come from ONE np.random.randint call of shape [B, Nn]: the legacy global stream
        yields exactly the values of the reference's B consecutive calls of size Nn (sampler.py:98-99)."""
        ids = self.session_id_batches[self.batch_i]
        B = len(ids)
        # an empty share of restrict_to_rank takes its global batch's length (batch_T is indexed by global batch)
        T = len(self.session_dict[ids[0]]) - 1 if B else self.batch_T[self.batch_i]
        Nn = self.neg_num if (self.neighbor_dict and self.neg_num) else 0
        M = B * T
        col = _columnar(self.session_dict, self.session_time_dict)
        rows = np.fromiter(map(col.row.__getitem__, ids), dtype=np.int64, count=B)
        seq = col.seq[T][rows]                                    # [B, T+1]
        out = np.empty(7 * M + 3 * B + B * Nn, dtype=np.int32)
        idx = out[: 7 * M].reshape(7, B, T)
        idx[0] = seq[:, :T]
        idx[1:] = col.feats[T][:, rows, :]
        out[7 * M: 7 * M + 2 * B].reshape(2, B)[:] = col.ctx[T][:, rows]
        label = out[7 * M + 2 * B: 7 * M + 3 * B]
        label[:] = seq[:, T] - 1
        negs = None
        if Nn:
            negs = out[7 * M + 3 * B:].reshape(B, Nn)
            if self.negative_mode == "impression":
                for b, sid in enumerate(ids):
                    negs[b] = self._negatives(sid)
            else:
                negs[:] = np.random.randint(0, self.item_num, size=(B, Nn))
        self.batch_i += 1
        self._last = (idx[0], label, negs)
        self.last_in = self.last_out = self.last_neg = None       # materialised lazily (last_lists())
        return out, B, T, Nn

    def last_lists(self):
        """(batch_in, batch_out, neg) of the most recent next_packed() as Python lists (what next_batch() returns)."""
        if self.last_in is None and getattr(self, "_last", None) is not None:
            seq, label, negs = self._last
            self.last_in, self.last_out = seq.tolist(), label.tolist()
            self.last_neg = negs.tolist() if negs is not None else [[] for _ in range(len(label))]
        return self.last_in, self.last_out, self.last_neg

    def neg_neighbor_from_impre(self, sessionid):
        """sampler.py:118-131."""
        neighor_set = self.neighbor_dict[sessionid]
        neg, cnt = [], 0
        choice = getattr(self, "_choice", None) or random.choice
        while len(neg) < self.neg_num:
            cnt += 1
            randomid = choice(neighor_set)
            if randomid in self.item_dict:
                neg.append(self.item_dict[randomid] - 1)
            if cnt > 20:
                break
        while len(neg) < self.neg_num:
            neg.append(int(np.random.randint(0, self.item_num)))
        return neg

    def neg_neighbor(self, itemid):
        """sampler.py:133-140 (publish-time neighbours; needs data_process/generate_neighbor.py output)."""
        neighor_set = self.neighbor_dict[itemid]
        neg = []
        while len(neg) < self.neg_num:
            randomid = random.choice(neighor_set)
            if randomid != itemid:
                neg.append(randomid)
        return neg


def impression_candidates(keys, labels, impressions, item_dict):
    """Candidate lists of a batch for ranking each session's impression list (the MIND protocol): session key k's list
    is impressions[int(str(k).split("_")[0])] (the key rule of the impression negatives), its article ids mapped
    through item_dict to 0-based ids.  Articles outside item_dict are dropped (the impression logs name more articles
    than the clicked-item dictionary, mind_preprocess.py:275-280), repeats keep their first occurrence, and the label
    is appended when absent, so every list holds it exactly once; a session without a list gets [label].
    Returns (off int32 [B+1], ids int32 [nnz]) in CSR form."""
    off = np.zeros(len(keys) + 1, dtype=np.int32)
    ids = []
    for b, (key, lab) in enumerate(zip(keys, labels)):
        seen = {}
        for art in impressions.get(int(str(key).split("_")[0]), ()):
            i = item_dict.get(art)
            if i is not None:
                seen.setdefault(i - 1, None)
        seen.setdefault(int(lab), None)
        ids.extend(seen)
        off[b + 1] = len(ids)
    return off, np.asarray(ids, dtype=np.int32)


def pack_batch(batch_in, batch_out, batch_pt, batch_ct, neg, gap):
    """Reference 6-tuple of lists -> (int32 array, B, T, Nn) in the model_combine.Batch layout."""
    B, T = len(batch_in), len(batch_in[0])
    Nn = len(neg[0]) if neg and len(neg[0]) else 0
    M = B * T
    out = np.empty(7 * M + 3 * B + B * Nn, dtype=np.int32)
    idx = out[: 7 * M].reshape(7, B, T)
    idx[0] = np.asarray(batch_in, dtype=np.int32)
    for k in range(5):
        idx[1 + k] = np.asarray(batch_pt[k], dtype=np.int32)
    idx[6] = np.minimum(np.asarray(gap, dtype=np.int32), 10)
    out[7 * M: 7 * M + B] = np.asarray(batch_ct[2], dtype=np.int32)
    out[7 * M + B: 7 * M + 2 * B] = np.asarray(batch_ct[3], dtype=np.int32)
    out[7 * M + 2 * B: 7 * M + 3 * B] = np.asarray(batch_out, dtype=np.int32)
    if Nn:
        out[7 * M + 3 * B:] = np.asarray(neg, dtype=np.int32).reshape(-1)
    return out, B, T, Nn
