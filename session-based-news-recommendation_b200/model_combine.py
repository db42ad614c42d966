"""TCAR model -- drop-in for the reference's model_combine.Seq2SeqAttNN (model_combine.py:10-315).

Same constructor (`Seq2SeqAttNN(args: dict)`), same `train(sess, item_dict, train_data, neighbor_dict, args,
test_data, saver, threshold_acc)` / `test(sess, test_data, args)` methods and the same feed-dict vocabulary; the
TensorFlow graph underneath is replaced by hand-written sm_100a kernels called through the C ABI in
include/tcar_b200.h (the dense projections too: tcar_gemm_tf32, tcgen05 kind::tf32).  `sess` / `saver` are accepted
and ignored.  PyTorch is used for device memory, streams and torch.distributed only.

There is no CPU path: constructing the model without CUDA + libtcar_b200.so raises.
"""
import math
import os
import time

import numpy as np
import torch

from . import _native as nv
from . import parallel
from .catalog_parallel import CatalogShardedTraining
from .params import ParamStore, SMALL
from .sampler import Sampler, pack_batch
from .util import (category_layout, check_decay, check_id_lists, check_item_categories, check_item_times,
                   check_windows, pad_sources)

H, TH, XW, PW, NB, KEXT, QROWS, TOPK = nv.H, nv.TH, nv.XW, nv.PW, nv.NBINS, nv.KEXT, nv.QROWS, nv.TOPK


class Batch:
    """One length-bucketed batch on the device: the reference's 11-entry feed dict (model_combine.py:214-227)
    packed into a single int32 buffer  [7*B*T idx | 2*B ctx | B label | B*Nn neg]."""

    def __init__(self, buf, B, T, Nn):
        self.buf, self.B, self.T, self.Nn = buf, B, T, Nn
        self.counts = None       # sessions per rank of the global batch this slice was cut from (catalog_parallel.py)
        M = B * T
        self.idx = buf[: 7 * M]
        self.ctx = buf[7 * M: 7 * M + 2 * B]
        self.label = buf[7 * M + 2 * B: 7 * M + 3 * B]
        self.neg = buf[7 * M + 3 * B: 7 * M + 3 * B + B * Nn] if Nn > 0 else None
        self.seq = buf[:M]


def prefetch_packed(sampler, depth=4):
    """Iterate `sampler.next_packed()` from a producer thread (NumPy gathers release the GIL), `depth` batches ahead
    of the GPU.  One producer, FIFO queue: the RNG streams are consumed in exactly the order of a plain loop."""
    import queue
    import threading
    q = queue.Queue(maxsize=depth)
    done = object()

    def work():
        try:
            while sampler.has_next():
                q.put(sampler.next_packed())
            q.put(done)
        except BaseException as exc:          # surface producer errors in the consumer
            q.put(exc)

    # The producer and the launching thread share the GIL; with CPython's default 5 ms switch interval the thread that
    # wants it back (35 short library calls per step on this side, a few NumPy gathers per batch on the other) can wait
    # milliseconds for a hand-over.  100 us keeps both fed (measured on the producer/consumer pair: 1.17 -> 0.89 ms per
    # batch); restored when the epoch's iterator ends.
    import sys
    old_interval = sys.getswitchinterval()
    sys.setswitchinterval(min(old_interval, 1e-4))
    threading.Thread(target=work, daemon=True).start()
    try:
        while True:
            item = q.get()
            if item is done:
                return
            if isinstance(item, BaseException):
                raise item
            yield item
    finally:
        sys.setswitchinterval(old_interval)


def pipelined(items, launch, consume):
    """One item of look-ahead, the loop of test() / test_impressions() / recommend_split(): launch(cur, nxt) enqueues
    item i (nxt = item i + 1, None for the last; items are never None) and returns the handles of its results, or
    None when there is nothing to read back; consume(*handles) of item i runs after item i + 1 has been launched, so
    the host reads item i's results from pinned memory while item i + 1 runs on the device."""
    it = iter(items)
    cur, pending = next(it, None), None
    while cur is not None:
        nxt = next(it, None)
        handles = launch(cur, nxt)
        if pending is not None:
            consume(*pending)
        pending, cur = handles, nxt
    if pending is not None:
        consume(*pending)


class PinnedRing:
    """A few reusable pinned staging buffers: pin_memory() per batch costs a cudaHostAlloc; a slot is reused only
    after the H2D copy that read it has completed (event per slot)."""

    def __init__(self, slots=4):
        self.slots, self.bufs, self.events, self.i = slots, [None] * slots, [None] * slots, 0

    def stage(self, packed):
        i = self.i
        self.i = (i + 1) % self.slots
        if self.events[i] is not None:
            self.events[i].synchronize()
        n = packed.size
        if self.bufs[i] is None or self.bufs[i].numel() < n:
            self.bufs[i] = torch.empty(max(n, 1 << 16), dtype=torch.int32).pin_memory()
        view = self.bufs[i][:n]
        view.numpy()[:] = packed
        self.events[i] = torch.cuda.Event()
        return view, self.events[i]


class HostFetch:
    """Device -> host hand-off of a small per-step result (the [B] loss, the top-20 block) WITHOUT stalling the launch
    queue: the copy goes into a slot of a pinned ring on the producing stream and an event is recorded behind it;
    `get()` waits for that one event only.  Reading step i's loss while step i+1 is being enqueued keeps the GPU fed
    (a blocking `.cpu()` per step leaves it idle for the host's whole enqueue time of the next step)."""

    SLOT_BYTES = 1 << 16           # a [512, 20] int32 block is 40 KB

    def __init__(self, slots=16):
        # ONE pinned allocation up front (cudaHostAlloc synchronises the device: never inside the step loop)
        self.slots, self.i = slots, 0
        self._pool = torch.empty(slots * self.SLOT_BYTES, dtype=torch.uint8).pin_memory()
        self.bufs = [self._pool[k * self.SLOT_BYTES: (k + 1) * self.SLOT_BYTES] for k in range(slots)]

    class Handle:
        def __init__(self, view, event):
            self.view, self.event = view, event

        def get(self):
            self.event.synchronize()
            return self.view

    def fetch(self, t):
        i = self.i
        self.i = (i + 1) % self.slots
        nbytes = t.numel() * t.element_size()
        buf = self.bufs[i]
        if buf.numel() < nbytes:           # unusually large result: give this slot its own (one-off) allocation
            buf = self.bufs[i] = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        view = buf[:nbytes].view(t.dtype).view(t.shape)
        view.copy_(t, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        return HostFetch.Handle(view, ev)


class Seq2SeqAttNN(CatalogShardedTraining):
    def __init__(self, args):
        if not torch.cuda.is_available():
            raise RuntimeError("tcar_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        nv.lib()
        torch.backends.cuda.matmul.allow_tf32 = False
        self.args = args
        self.itemnum = args["itemnum"]
        self.category_id = args.get("category_id")
        self.item_freq_dict_norm = args.get("item_freq_dict_norm")
        self.reverse_item = args.get("reverse_item")
        content = np.asarray(args["content_emb"], dtype=np.float32)
        self.candidate_n = content.shape[0]
        self.N = self.candidate_n - 1                       # model_combine.py:42,135
        self.emb_stddev, self.stddev = args["emb_stddev"], args["stddev"]
        self.hidden_size, self.time_hidden_size = args["hidden_size"], args["time_hidden_size"]
        if self.hidden_size != H or content.shape[1] != H or self.time_hidden_size != TH:
            raise ValueError("this build is specialised for hidden_size=250 (== content width), time_hidden_size=64")
        self.batch_size, self.epoch, self.neg_num = args["batch_size"], args["epoch"], args["neg_num"]
        if self.batch_size > QROWS:
            raise ValueError(f"batch_size <= {QROWS} (one scoring call holds at most {QROWS} sessions)")
        self.lr = float(args["lr"])
        self.max_grad = args.get("max_grad")
        self.max_grad_f = float(self.max_grad) if self.max_grad is not None else 3.0e38
        # catalog sharding for evaluation / data-parallel training (torch.distributed, NCCL)
        self.rank = int(args.get("rank", 0))
        self.world = int(args.get("world_size", 1))
        self.cluster = int(args.get("cluster", nv.CLUSTER_PAIR))
        dev = torch.device("cuda", torch.cuda.current_device())
        self.dev = dev
        self.ps = ParamStore(self.N, content, args["publish_time_MWDHM"], dev)
        self.ps.init_reference(self.emb_stddev, self.stddev)
        self.variables_names = ["item"] + [n for n, _ in SMALL]
        self._alloc()
        self._cat_array = None
        self.curEpoch = 0
        self.error_during_train = False
        self.global_step = 0
        # software pipelining of the train loop (train_step(bt, next_bt)): the table-wide item Adam of step s runs on a
        # side stream while the session forward of step s+1 runs on the caller's stream
        # `_side`: the table-wide Adam; `_ahead` (high priority, so that its CTAs are dispatched as soon as Adam CTAs
        # retire): the next batch's session forward
        self._side = torch.cuda.Stream(device=dev)
        self._ahead = torch.cuda.Stream(device=dev, priority=-1)
        # `_aux`: independent branches of the backward / update (query-path gradients, small-tensor Adam) that run
        # beside the main chain; joined by events, results do not depend on the interleaving (disjoint buffers)
        self._aux = torch.cuda.Stream(device=dev)
        self._la_events = None
        self._update_done = None           # event recorded on `_side` after the pending item update
        self._ahead_done = None            # event recorded on `_ahead` after the prefetched session forward
        self._prefetched = None            # the Batch whose session forward has already been launched
        self.adam_overlap_ctas = 64
        # multi-GPU training layout: "dp" = data parallel + gradient all-reduce (north_star), "catalog" = the softmax
        # sharded over the item catalog (catalog_parallel.py; SURVEY 8e row 2)
        # overflow guard of the full-catalog softmax (TCAR_EXP_LIMIT2 in include/tcar_b200.h): TF subtracts the row
        # maximum (model_combine.py:145), the scoring kernel shifts by the label score; rows whose best candidate
        # outscores the label by more than 55 nats are re-run shifted by their maximum (two empty launches otherwise)
        self.softmax_guard = bool(args.get("softmax_guard", os.environ.get("TCAR_SOFTMAX_GUARD", "1") != "0"))
        self.eval_group_launch = True
        # single item range, <= 512 queries: the fused CTA-per-query kernel (121 us) beats warp-per-query selection +
        # re-scoring (63 + 72 us: 512 warps cannot fill the GPU); the sharded rounds select for world x 512 queries per
        # launch, where the warp kernel's time stays flat (tcar_eval_select_groups)
        self.eval_warp_select = False
        self.train_parallel = "dp"
        self._item_table_synced = True
        mode = args.get("train_parallel") or "dp"
        if mode not in ("dp", "catalog"):
            raise ValueError("train_parallel must be 'dp' or 'catalog'")
        if mode == "catalog":
            self.enable_catalog_training(int(args.get("catalog_virtual_shards") or 1))

    # ------------------------------------------------------------------------------------------- workspaces
    def _alloc(self):
        dev, Bm, Tm = self.dev, QROWS, nv.MAXT
        Mm = Bm * Tm
        f = lambda *s: torch.zeros(*s, device=dev)
        self.X, self.P, self.D, self.CT = f(Mm, XW), f(Mm, PW), f(Mm, TH), f(Bm, 2 * TH)
        HP = nv.HP
        self.U1, self.U2, self.dU1, self.dU2 = f(Mm, HP), f(Mm, HP), f(Mm, HP), f(Mm, HP)   # 256-float pitch (TMA)
        self.dXi, self.dP, self.dD = f(Mm, HP), f(Mm, PW), f(Mm, TH)
        self.alpha, self.de = f(3, Mm), f(3, Mm)
        self.h1, self.dh1, self.q, self.dq = f(Bm, HP), f(Bm, HP), f(Bm, XW), f(Bm, XW)
        self.dpooled, self.dpooled_t = f(Bm, XW), f(Bm, PW)
        self.gW_tmp = f(XW, H)
        self.col_scratch = f(2, 32 * H + 8)         # TCAR_COL_SCRATCH(250) floats per long column job
        self.gemm_part = f(int(nv.lib().tcar_gemm_tf32_part_elems(XW, H, 16)) * 4)     # split-reduction scratch
        self._part_off = 0
        self.pooled, self.pooled_t = f(Bm, XW), f(Bm, PW)
        self.a_ic, self.a_pt = f(Bm, XW), f(Bm, PW)
        self.d_a_ic, self.d_a_pt, self.dA_neg = f(Bm, XW), f(Bm, PW), f(Bm, XW)
        self.Tq, self.dTq = f(Bm, NB), f(Bm, NB)
        self.a_ic_eval, self.Tq_eval = f(Bm, XW), f(Bm, NB)      # eval look-ahead: parked copies for the re-scoring
        self.c_ref, self.ce = f(Bm), f(Bm)
        # one shard's evaluation results as ONE block (TCAR_EVAL_OFF_* in include/tcar_b200.h): the kernels write its
        # planes, the catalog-sharded evaluation exchanges the whole block in a single collective
        self._evblock = f(nv.EVAL_BLOCK_WORDS)
        ev_i = self._evblock.view(torch.int32)
        self.top_scores = self._evblock[nv.EVAL_OFF_SCORES: nv.EVAL_OFF_SCORES + Bm * TOPK].view(Bm, TOPK)
        self.top_ids = ev_i[nv.EVAL_OFF_IDS: nv.EVAL_OFF_IDS + Bm * TOPK].view(Bm, TOPK)
        self.n_greater = ev_i[nv.EVAL_OFF_NGT: nv.EVAL_OFF_NGT + Bm]
        self.sumexp = self._evblock[nv.EVAL_OFF_SUMEXP: nv.EVAL_OFF_SUMEXP + Bm]
        self.rowmax = self._evblock[nv.EVAL_OFF_ROWMAX: nv.EVAL_OFF_ROWMAX + Bm]
        # merged (global) results of a sharded evaluation
        self.m_ids = torch.zeros(Bm, TOPK, device=dev, dtype=torch.int32)
        self.m_scores, self.m_ce = f(Bm, TOPK), f(Bm)
        self.m_ngt = torch.zeros(Bm, device=dev, dtype=torch.int32)
        # certification of the top-20 candidate selection (tcar_eval_topk_certified / tcar_eval_topk_widen)
        self.uncertain = torch.zeros(Bm, device=dev, dtype=torch.int32)
        self.tau, self.cat_stats = f(Bm), f(2)
        self._sel1 = f(2 * Bm * nv.EVAL_NSEL)            # candidate list of the single-range evaluation (vals | ids)
        self.widen_ws = torch.zeros(int(nv.lib().tcar_eval_topk_widen_ws_bytes(1)), device=dev, dtype=torch.uint8)
        self._cat_stats_version = -1
        self.negloss, self.loss, self.coef = f(Bm), f(Bm), f(Bm)
        self.Q = torch.zeros(QROWS, KEXT, device=dev, dtype=torch.bfloat16)
        self.Qs = torch.zeros(QROWS, nv.HP, device=dev, dtype=torch.bfloat16)
        self.dq_raw = f(QROWS, KEXT)
        self.dCT = f(Bm, 2 * TH)
        self._score_ws = {}
        self.hash_size = 0
        self._alloc_scatter(Bm * 20 + Bm + Bm * max(int(self.neg_num or 0), 20))   # reference defaults: T<=20, Nn=20
        self.sq_partial = f(256)
        self.table_part = f(148 * 19600)            # TCAR_TABLE_GRAD_CHUNKS x TCAR_TABLE_GRAD_PART

    def _alloc_scatter(self, entries):
        """Scratch of the deterministic scatter-add, sized for `entries` sparse rows (clicks + labels + negatives):
        a power-of-two hash with load factor <= 1/2.  Grows on demand (MIND-shaped runs use up to 100 negatives)."""
        need = 1 << max(16, (2 * entries - 1).bit_length())
        if need <= self.hash_size:
            return
        dev = self.dev
        self.hash_size = need
        self.hash_keys = torch.full((need,), -1, device=dev, dtype=torch.int32)
        self.hash_acc = torch.zeros(need, nv.HP, device=dev, dtype=torch.int64)
        self.hash_cnt = torch.zeros(need, device=dev, dtype=torch.int32)
        self.entry_slot = torch.zeros(need // 2, device=dev, dtype=torch.int32)
        self.slot_sq = torch.zeros(need, device=dev)

    def _part(self, M, N, splits):
        """Carve a disjoint split-reduction scratch for one problem of a GEMM group (None when not split)."""
        if splits <= 1:
            return None
        n = int(nv.lib().tcar_gemm_tf32_part_elems(M, N, splits))
        if self._part_off + n > self.gemm_part.numel():
            raise ValueError("GEMM split scratch exhausted")
        out = self.gemm_part[self._part_off:]
        self._part_off += n
        return out

    def _score_buffers(self, n_pad, train):
        """E / partial-sum / chunk-max buffers sized for a catalog (shard) of n_pad items; allocated once."""
        key = (n_pad, train)
        if key not in self._score_ws:
            dev = self.dev
            tiles = nv.lib().tcar_score_fwd_tiles(n_pad)
            ws = {"part": torch.zeros(tiles, QROWS, device=dev), "pmax": torch.zeros(tiles, QROWS, device=dev),
                  "tiles": tiles}
            if train:
                ws["E"] = torch.zeros(QROWS, n_pad, device=dev, dtype=torch.bfloat16)
                splits = max(nv.lib().tcar_score_bwd_q_splits(b, n_pad) for b in (1, 129, 257, 385))
                ws["qpart"] = torch.zeros(splits, QROWS, KEXT, device=dev)
            else:
                ws["cmax"] = torch.zeros(QROWS, n_pad // nv.CHUNK, device=dev)
                ws["tmax"] = torch.zeros(QROWS, n_pad // 128, device=dev)
            self._score_ws[key] = ws
        return self._score_ws[key]

    # ------------------------------------------------------------------------------------------- batches
    def to_device(self, packed, B, T, Nn):
        """H2D copy of one packed int32 batch (pinned host buffer -> device)."""
        buf = torch.empty(packed.numel(), device=self.dev, dtype=torch.int32)
        buf.copy_(packed, non_blocking=True)
        return Batch(buf, B, T, Nn)

    def stage_to_device(self, packed_np, B, T, Nn):
        """NumPy packed batch -> pinned ring slot -> device (the path of the train / test loops)."""
        return Batch(self._stage_ints(packed_np), B, T, Nn)

    def _stage_ints(self, arr_np):
        """int32 NumPy array -> pinned ring slot -> new device tensor, without blocking the host."""
        if getattr(self, "_ring", None) is None:
            self._ring = PinnedRing()
        view, ev = self._ring.stage(arr_np)
        buf = torch.empty(view.numel(), device=self.dev, dtype=torch.int32)
        buf.copy_(view, non_blocking=True)
        ev.record()
        return buf

    def fetch_async(self, t):
        """Start the device -> host copy of a result tensor into pinned memory; returns a handle whose .get() blocks
        only until THAT copy is done (see HostFetch).  A slot is reused after 16 further fetches."""
        if getattr(self, "_fetch", None) is None:
            self._fetch = HostFetch()
        return self._fetch.fetch(t)

    def make_batch(self, batch_in, batch_out, batch_pt, batch_ct, neg, gap):
        """From the reference sampler's 6-tuple of Python lists (sampler.py:113) to a device Batch."""
        packed, B, T, Nn = pack_batch(batch_in, batch_out, batch_pt, batch_ct, neg, gap)
        return self.to_device(torch.from_numpy(packed).pin_memory(), B, T, Nn)

    # ------------------------------------------------------------------------------------------- forward
    def sync_updates(self):
        """Make the caller's stream wait for an item-table update still running on the side stream (only pending after
        train_step(bt, next_bt)).  Every entry point that reads parameters calls this first."""
        cur = torch.cuda.current_stream()
        if self._update_done is not None:
            cur.wait_event(self._update_done)
            self._update_done = None
        if self._ahead_done is not None:
            cur.wait_event(self._ahead_done)
            self._ahead_done = None

    def _session_forward(self, bt, prefetch=False):
        """Everything up to a_ic / a_pt / Q: model_combine.py:52-127.  With prefetch=True the caller guarantees that
        the rows of the item table this batch reads (clicks, labels) are already up to date, so the pending table-wide
        update is NOT waited for."""
        if not prefetch:
            self.sync_updates()
            self._prefetched = None
        ps, w, B, T = self.ps, self.ps.w, bt.B, bt.T
        M = B * T
        p = nv.ptr
        nv.counted_call("tcar_gather_fwd", 1, p(bt.idx), p(bt.ctx), p(ps.item), p(ps.content), p(w["pos"]),
                        p(w["month"]), p(w["day"]), p(w["week"]), p(w["hour"]), p(w["minute"]), p(w["dur"]),
                        p(self.X), p(self.P), p(self.D), p(self.CT), B, T)
        # linear_3d / linear_2d projections (modules.py:126-131, :94-96, :138-139; model_combine.py:119,127) on the
        # tensor cores in 3xTF32 (fp32-class accuracy); bias + activation fused into the GEMM epilogue
        wh, wl, pr = ps.wh, ps.wl, nv.problem
        nv.gemm_group([
            pr([(self.X, XW, 0, wh["W_in1"], wl["W_in1"], 256, 1, XW), (self.D, TH, 0, wh["W_i"], wl["W_i"], 256, 1, TH)],
               M, H, self.U1, nv.HP, precise=True),
            pr([(self.P, PW, 0, wh["W1"], wl["W1"], 256, 1, PW), (self.X, XW, 0, wh["W2x"], wl["W2x"], 256, 1, XW)],
               M, H, self.U2, nv.HP, precise=True),
            pr([(self.CT, 2 * TH, 0, wh["Wq1"], wl["Wq1"], 256, 1, 2 * TH)], B, H, self.h1, nv.HP, bias=w["bq1"], act=1,
               precise=True)])
        nv.gemm([(self.h1, nv.HP, 0, wh["Wq2"], wl["Wq2"], 512, 1, H)], B, XW, self.q, XW, bias=w["bq2"], act=2,
                precise=True)
        nv.counted_call("tcar_pool_fwd", 1, p(self.X), p(self.P), p(self.U1), p(self.U2), p(self.q), p(w["w_r"]),
                        p(w["w_t"]), p(self.alpha), p(self.pooled), p(self.pooled_t), B, T)
        nv.gemm_group([
            pr([(self.pooled, XW, 0, wh["W_a"], wl["W_a"], 512, 1, XW)], B, XW, self.a_ic, XW, bias=w["b_a"], act=2,
               precise=True),
            pr([(self.pooled_t, PW, 0, wh["W_p"], wl["W_p"], 320, 1, PW)], B, PW, self.a_pt, PW, bias=w["b_p"], act=2,
               precise=True)])
        self._session_query(bt)

    def _session_query(self, bt):
        """Second half of the session forward: Tq, the bf16 session operand Q and the exact label scores c_ref (the
        buffers the scoring GEMM and its overflow-guard pass read)."""
        ps, w, p, B = self.ps, self.ps.w, nv.ptr, bt.B
        nv.counted_call("tcar_clip_time_tables", 1, p(w["month"]), p(w["day"]), p(w["week"]), p(w["hour"]),
                        p(w["minute"]), p(ps.ct_tab), p(ps.ct_scale))
        nv.counted_call("tcar_build_query", 1, p(self.a_ic), p(self.a_pt), p(ps.ct_tab), p(ps.item), p(ps.content),
                        p(ps.mwdhm), p(bt.label), p(self.Tq), p(self.Q), p(self.c_ref), B)

    @staticmethod
    def _splits_for(k):
        return max(1, min(16, (k // 32) // 24))

    def _cluster_for(self, B):
        if self.cluster == nv.CLUSTER_PAIR:
            return nv.CLUSTER_PAIR
        mt = (B + 127) // 128
        c = min(self.cluster, 4)
        while c > 1 and c > mt:
            c //= 2
        return max(c, 1)

    def forward_train(self, bt):
        """loss [B], cross_loss [B] (model_combine.py:145-147) and everything the backward needs."""
        ps, p, B = self.ps, nv.ptr, bt.B
        if self._prefetched is bt:
            self._prefetched = None        # session forward already launched by the previous train_step
            self.sync_updates()            # the scoring operand / negative rows need the whole table
        else:
            self._session_forward(bt)
        ws = self._score_buffers(ps.n_pad, True)
        if self.world == 1:
            # the negative-feedback term needs a_ic and item rows only: beside the scoring GEMM on the auxiliary stream
            # (its CTAs use no shared memory to speak of, so they fit next to the GEMM's), off the critical path
            main = torch.cuda.current_stream()
            ev = torch.cuda.Event()
            ev.record(main)

            def neg_side():
                self._aux.wait_event(ev)
                with torch.cuda.stream(self._aux):
                    nv.counted_call("tcar_neg_loss", 1, p(self.a_ic), p(ps.item), p(ps.content), p(bt.neg), None,
                                    p(self.negloss), p(self.loss), p(self.coef), p(self.dA_neg), B, bt.Nn)
                    self._neg_done = torch.cuda.Event()
                    self._neg_done.record(self._aux)

            self._score_and_sum(ws, ps.iext, p(ws["E"]), None, None, B, ps.N, ps.n_pad, 0, after_gemm=neg_side)
            main.wait_event(self._neg_done)
            nv.counted_call("tcar_loss_combine", 1, p(self.ce), p(self.negloss), p(self.loss), B)
        else:
            self._score_and_sum(ws, ps.iext, p(ws["E"]), None, None, B, ps.N, ps.n_pad, 0)
            nv.counted_call("tcar_neg_loss", 1, p(self.a_ic), p(ps.item), p(ps.content), p(bt.neg), p(self.ce),
                            p(self.negloss), p(self.loss), p(self.coef), p(self.dA_neg), B, bt.Nn)
        return self.loss[:B], self.ce[:B]

    def _score_and_sum(self, ws, iext, e_ptr, cmax_ptr, tmax_ptr, B, n_items, n_pad, mode, q=None, c=None, sumexp=None,
                       ce=None, rowmax=None, after_gemm=None):
        """Scoring GEMM + softmax sums: E / chunk maxima, sumexp, ce = logsumexp(S) - S[label], with the overflow
        guard (pass 2 is two empty launches unless a row's best score beats the label by > 55 nats).  q / c / sumexp /
        ce / rowmax default to this model's own buffers (another rank's queries in the sharded evaluation)."""
        p, cl = nv.ptr, self._cluster_for(B)
        q, c, part = p(self.Q if q is None else q), p(self.c_ref if c is None else c), p(ws["part"])
        sumexp, ce = p(self.sumexp if sumexp is None else sumexp), p(self.ce if ce is None else ce)
        rowmax_t = self.rowmax if rowmax is None else rowmax
        if not self.softmax_guard:
            nv.counted_call("tcar_score_fwd", 1, q, p(iext), c, e_ptr, part, cmax_ptr, tmax_ptr, B, n_items, n_pad,
                            mode, cl)
            if after_gemm is not None:
                after_gemm()
            nv.counted_call("tcar_ce_finish", 1, part, sumexp, ce, ws["tiles"], B)
            if mode == 1:
                rowmax_t[:B].zero_()       # result blocks carry the shift: none here
            return
        pmax, rowmax = p(ws["pmax"]), p(rowmax_t)
        nv.counted_call("tcar_score_fwd_guarded", 1, q, p(iext), c, e_ptr, part, cmax_ptr, tmax_ptr, pmax, None, B,
                        n_items, n_pad, mode, cl)
        if after_gemm is not None:
            after_gemm()           # pass 2 below still reads q / c: the hook must not let anything overwrite them
        nv.counted_call("tcar_ce_finish_guarded", 1, part, pmax, sumexp, ce, rowmax, ws["tiles"], B, 1)
        nv.counted_call("tcar_score_fwd_guarded", 1, q, p(iext), c, e_ptr, part, cmax_ptr, tmax_ptr, None, rowmax, B,
                        n_items, n_pad, mode, cl)
        nv.counted_call("tcar_ce_finish_guarded", 1, part, None, sumexp, ce, rowmax, ws["tiles"], B, 2)

    def backward(self, bt, scatter=True):
        """Gradients of sum_b loss_b wrt all 23 tensors (model_combine.py:156) into ps.item_g / ps.theta_g.
        scatter=False leaves the sparse item rows (clicks, labels, negatives) to a later _scatter_item_grads(bt)."""
        ps, p, B = self.ps, nv.ptr, bt.B
        ws = self._score_buffers(ps.n_pad, True)
        nv.counted_call("tcar_score_bwd_q", 2, p(ws["E"]), p(ps.iext), p(ws["qpart"]), p(self.dq_raw), B, ps.n_pad)
        nv.counted_call("tcar_score_bwd_finish", 1, p(self.dq_raw), p(self.sumexp), p(self.dA_neg), p(self.a_ic),
                        p(ps.ct_tab), p(ps.item), p(ps.content), p(ps.mwdhm), p(bt.label), p(self.d_a_ic),
                        p(self.d_a_pt), p(self.dTq), p(self.Qs), B)
        if self.world == 1:
            # the dense item gradient GEMM (HBM-bound, persistent CTAs) on the side stream, the session-side backward
            # (a chain of short latency-bound kernels that only needs d a_ic / d a_pt / dTq) beside it on this stream
            main = torch.cuda.current_stream()
            fork = torch.cuda.Event()
            fork.record(main)
            self._side.wait_event(fork)
            with torch.cuda.stream(self._side):
                nv.counted_call("tcar_score_bwd_i", 1, p(ws["E"]), p(self.Qs), p(ps.item_g), p(self.sq_partial), B,
                                ps.N, ps.n_pad)
                join = torch.cuda.Event()
                join.record(self._side)
            self._session_backward(bt)
            main.wait_event(join)
        else:
            nv.counted_call("tcar_score_bwd_i", 1, p(ws["E"]), p(self.Qs), p(ps.item_g), p(self.sq_partial), B, ps.N,
                            ps.n_pad)
            self._session_backward(bt)
        if scatter:
            self._scatter_item_grads(bt)

    def _session_backward(self, bt):
        """Everything below the scoring layer: from d a_ic / d a_pt / dTq (tcar_score_bwd_finish) to the gradients of
        the 22 small tensors (ps.theta_g) and dXi, the gradient wrt the gathered item rows."""
        ps, w, g, p, B, T = self.ps, self.ps.w, self.ps.g, nv.ptr, bt.B, bt.T
        M = B * T
        # ---- session-side backward: weight / data gradients on the tensor cores in single-pass TF32 (gradients carry
        # a 2e-2 norm-wise tolerance, dominated by the bf16 scoring GEMMs); operands are consumed in place, K-major or
        # MN-major as they lie, so no transposes are materialised.
        wh, pr, HPp = ps.wh, nv.problem, nv.HP
        self._part_off = 0
        dz_a, dz_p = self.d_a_ic, self.d_a_pt
        nv.col_jobs([(dz_a, self.a_ic, dz_a, g["b_a"], B, XW, XW, 0), (dz_p, self.a_pt, dz_p, g["b_p"], B, PW, PW, 0)])
        # split the reduction dimension across CTAs only when one CTA would walk more than ~48 K blocks of 32: a split
        # costs a second (reduction) launch, which is worth it for long reductions only
        ksp = self._splits_for(B)
        nv.gemm_group([
            pr([(self.pooled, XW, 1, dz_a, None, XW, 1, B)], XW, XW, g["W_a"], XW, splits=ksp, part=self._part(XW, XW, ksp)),
            pr([(self.pooled_t, PW, 1, dz_p, None, PW, 1, B)], PW, PW, g["W_p"], PW, splits=ksp, part=self._part(PW, PW, ksp)),
            pr([(dz_a, XW, 0, wh["W_a"], None, 512, 0, XW)], B, XW, self.dpooled, XW),
            pr([(dz_p, PW, 0, wh["W_p"], None, 320, 0, PW)], B, PW, self.dpooled_t, PW)])
        nv.counted_call("tcar_pool_bwd", 1, p(self.X), p(self.P), p(self.U1), p(self.U2), p(self.q), p(w["w_r"]),
                        p(w["w_t"]), p(self.alpha), p(self.dpooled), p(self.dpooled_t), p(self.dU1), p(self.dU2),
                        p(self.dXi), p(self.dP), p(self.dq), p(self.de), B, T)
        de = self.de.view(-1)                      # kernel layout: [3][B*T] with the ACTUAL B*T as stride
        dzq = self.dq
        main = torch.cuda.current_stream()
        branch = self._aux if self.world == 1 else main
        if branch is not main:
            ev = torch.cuda.Event()
            ev.record(main)
            branch.wait_event(ev)
        with torch.cuda.stream(branch):
            # ---- branch B (independent of dU1 / dU2's consumers): w_r / w_t gradients (S1^T de1, S2^T de_t), the query
            # path backward (modules.py:138-139) down to dCT.  ksp == 1 here, so no split scratch is shared with branch A
            nv.col_jobs([(de[:M], self.U1, None, g["w_r"], M, H, HPp, 2, self.col_scratch[0]),
                         (de[2 * M: 3 * M], self.U2, None, g["w_t"], M, H, HPp, 2, self.col_scratch[1]),
                         (dzq, self.q, dzq, g["bq2"], B, XW, XW, 0)])
            nv.gemm_group([
                pr([(self.h1, HPp, 1, dzq, None, XW, 1, B)], H, XW, g["Wq2"], XW),
                pr([(dzq, XW, 0, wh["Wq2"], None, 512, 0, XW)], B, H, self.dh1, HPp)])
            nv.counted_call("tcar_act_bwd_colsum", 1, p(self.dh1), p(self.h1), p(self.dh1), p(g["bq1"]), B, H, HPp, 1)
            nv.gemm_group([
                pr([(self.CT, 2 * TH, 1, self.dh1, None, HPp, 1, B)], 2 * TH, H, g["Wq1"], H),
                pr([(self.dh1, HPp, 0, wh["Wq1"], None, 256, 0, H)], B, 2 * TH, self.dCT, 2 * TH)])
            if branch is not main:
                ev_b = torch.cuda.Event()
                ev_b.record(branch)
        # every gradient that consumes dU1 / dU2, one launch: four weight gradients (reduction over the B*T clicks
        # split across CTAs) and three data gradients
        msp = self._splits_for(M)
        self._part_off = 0
        nv.gemm_group([
            # rows 250..499 of X^T dU1 / X^T dU2 (the content half of X) are W_c's and W2's gradients: second
            # destination of the same problem, no copy kernels
            pr([(self.X, XW, 1, self.dU1, None, HPp, 1, M)], XW, H, g["W_in"], H, splits=msp, part=self._part(XW, H, msp),
               out2=g["W_c"], out2_row0=H),
            pr([(self.D, TH, 1, self.dU1, None, HPp, 1, M)], TH, H, g["W_i"], H, splits=msp, part=self._part(TH, H, msp)),
            pr([(self.P, PW, 1, self.dU2, None, HPp, 1, M)], PW, H, g["W1"], H, splits=msp, part=self._part(PW, H, msp)),
            pr([(self.X, XW, 1, self.dU2, None, HPp, 1, M)], XW, H, self.gW_tmp, H, splits=msp,
               part=self._part(XW, H, msp), out2=g["W2"], out2_row0=H),
            pr([(self.dU1, HPp, 0, wh["W_in1"], None, 256, 0, H)], M, H, self.dXi, HPp, accumulate=True),
            pr([(self.dU1, HPp, 0, wh["W_i"], None, 256, 0, H)], M, TH, self.dD, TH),
            pr([(self.dU2, HPp, 0, wh["W1"], None, 256, 0, H)], M, PW, self.dP, PW, accumulate=True)])
        if branch is not main:
            main.wait_event(ev_b)              # the table gradients consume dCT
        nv.counted_call("tcar_small_table_grads", 1, p(bt.idx), p(bt.ctx), p(self.dXi), p(self.dP), p(self.dD),
                        p(self.dCT), p(self.dTq), p(self.a_pt), p(w["pos"]), p(w["month"]), p(w["day"]),
                        p(w["week"]), p(w["hour"]), p(w["minute"]), p(w["dur"]), p(g["pos"]), p(g["month"]),
                        p(g["day"]), p(g["week"]), p(g["hour"]), p(g["minute"]), p(g["dur"]), p(self.table_part), B, T)

    def _scatter_item_grads(self, bt):
        """Deterministic scatter-add of the sparse item-row gradients into the dense ps.item_g."""
        ps, p, B, T = self.ps, nv.ptr, bt.B, bt.T
        entries = B * T + B + B * bt.Nn
        self._alloc_scatter(entries)
        nv.counted_call("tcar_scatter_add_rows", 3, p(bt.seq), p(bt.label), p(bt.neg), p(self.dXi), p(self.a_ic),
                        p(self.coef), p(ps.item), p(ps.item_g), p(self.hash_keys), p(self.hash_cnt), p(self.hash_acc),
                        p(self.entry_slot), p(self.slot_sq), self.hash_size, B, T, bt.Nn)
        self._fused_norm = True

    def _sharded_update(self):
        """True when the data-parallel step uses reduce-scatter -> per-rank Adam slice -> all-gather (the two halves of
        an all-reduce with the optimiser in between) instead of all-reduce + replicated Adam."""
        return parallel.is_distributed(self.world) and self.ps.rows_alloc % self.world == 0

    def allreduce_grads(self):
        """Data-parallel training: SUM (not mean -- the loss is a batch sum, model_combine.py:156) over ranks."""
        if self._sharded_update():
            parallel.allreduce_sum((self.ps.theta_g,), self.world)      # the item gradient is reduce-scattered later
        else:
            parallel.allreduce_sum((self.ps.item_g, self.ps.theta_g), self.world)

    def _apply_item_sharded(self):
        """Item table update of the data-parallel step: every rank reduces and owns one contiguous slice of rows."""
        import torch.distributed as dist
        ps, p = self.ps, nv.ptr
        per = ps.rows_alloc // self.world
        lo = self.rank * per
        if getattr(self, "_g_slice", None) is None or self._g_slice.shape[0] != per:
            self._g_slice = torch.empty(per, nv.HP, device=self.dev)
        dist.reduce_scatter_tensor(self._g_slice, ps.item_g_full, op=dist.ReduceOp.SUM)
        # clip norm of the WHOLE reduced gradient: per-slice sums of squares, summed over ranks
        nv.counted_call("tcar_sqnorm_big", 2, p(self._g_slice), p(ps.norm_partial), p(ps.sqnorm_item),
                        self._g_slice.numel())
        dist.all_reduce(ps.sqnorm_item, op=dist.ReduceOp.SUM)
        # no bf16 refresh here (iext = NULL): the slice of the LAST rank runs over the alignment rows N+1 .. rows_alloc-1,
        # which have no row in the scoring operand, and tcar_refresh_iext_items rebuilds it after the all-gather anyway
        nv.counted_call("tcar_adam_item", 1, p(ps.item_full[lo:]), p(ps.item_m_full[lo:]), p(ps.item_v_full[lo:]),
                        p(self._g_slice), p(ps.sqnorm_item), p(ps.step), self.lr, self.max_grad_f, None, lo, per,
                        None, 0)
        dist.all_gather_into_tensor(ps.item_full, ps.item_full[lo: lo + per])
        nv.counted_call("tcar_refresh_iext_items", 1, p(ps.item), p(ps.iext), ps.N)
        self._moments_synced = False       # every rank holds the Adam moments of its own row slice only

    def sync_optimizer_state(self):
        """Data-parallel training with the sharded update keeps the item table's Adam moments distributed (rank r owns
        the rows of its slice).  A checkpoint is 'parameters + moments + step': gather the slices first, so that the
        writer holds the moments of EVERY row (a resumed run would otherwise restart Adam for (world-1)/world of them)."""
        if getattr(self, "_moments_synced", True) or not self._sharded_update():
            return
        import torch.distributed as dist
        ps = self.ps
        per = ps.rows_alloc // self.world
        lo = self.rank * per
        self.sync_updates()
        for t in (ps.item_m_full, ps.item_v_full):
            dist.all_gather_into_tensor(t, t[lo: lo + per])
        self._moments_synced = True

    def apply_gradients(self, next_bt=None):
        """per-tensor clip_by_norm + TF Adam (model_combine.py:155-163); also refreshes the bf16 scoring operand.
        With next_bt (single GPU): the item rows next_bt gathers are updated first, then the table-wide item update is
        forked onto the side stream and next_bt's session forward is launched behind it on the caller's stream."""
        ps, p = self.ps, nv.ptr
        ps.version += 1                    # the item table changes: statistics derived from it are stale
        small_done, self._small_done = getattr(self, "_small_done", None), None
        if self._sharded_update():
            nv.counted_call("tcar_sqnorm_segments", 1, p(ps.theta_g), p(ps.seg_off), p(ps.sqnorm_small), len(SMALL))
            ps.step.add_(1)
            self.global_step += 1
            nv.counted_call("tcar_adam_small", 1, p(ps.theta), p(ps.theta_m), p(ps.theta_v), p(ps.theta_g),
                            p(ps.seg_off), p(ps.sqnorm_small), len(SMALL), p(ps.step), self.lr, self.max_grad_f)
            self._apply_item_sharded()
            ps.prep_weights()
            self._fused_norm = False
            return
        if small_done is not None:
            # the small tensors were updated on the auxiliary stream beside the scatter (train_step): only the item
            # norm is left -- per-CTA sums of the dense gradient GEMM + per-row corrections of the scatter
            nv.counted_call("tcar_update_norms", 1, None, None, None, 0, p(self.sq_partial),
                            nv.lib().tcar_score_bwd_i_ctas(ps.n_pad), p(self.slot_sq), self.hash_size,
                            p(ps.sqnorm_item), p(ps.norm_partial), p(ps.norm_ticket), None)
            torch.cuda.current_stream().wait_event(small_done)
            self._fused_norm = False
            self.global_step += 1
        elif self.world == 1 and getattr(self, "_fused_norm", False):
            # every clip norm of the step + the step counter in one launch.  ||g_item||^2 comes from the per-CTA sums
            # of the dense gradient GEMM + the per-row corrections of the scatter: no pass over the 364 MB gradient
            nv.counted_call("tcar_update_norms", 1, p(ps.theta_g), p(ps.seg_off), p(ps.sqnorm_small), len(SMALL),
                            p(self.sq_partial), nv.lib().tcar_score_bwd_i_ctas(ps.n_pad), p(self.slot_sq),
                            self.hash_size, p(ps.sqnorm_item), p(ps.norm_partial), p(ps.norm_ticket), p(ps.step))
        else:
            # data parallel: the clip norm is the norm of the all-reduced gradient
            nv.counted_call("tcar_sqnorm_segments", 1, p(ps.theta_g), p(ps.seg_off), p(ps.sqnorm_small), len(SMALL))
            nv.counted_call("tcar_sqnorm_big", 2, p(ps.item_g), p(ps.norm_partial), p(ps.sqnorm_item),
                            ps.item_g.numel())
            ps.step.add_(1)
        if small_done is None:
            self._fused_norm = False
            self.global_step += 1
            self._update_small()
        item_args = (p(ps.item), p(ps.item_m), p(ps.item_v), p(ps.item_g), p(ps.sqnorm_item), p(ps.step), self.lr,
                     self.max_grad_f, p(ps.iext))
        if next_bt is None or next_bt.B == 0 or self.world != 1 or self.adam_overlap_ctas <= 0:
            nv.counted_call("tcar_adam_item", 1, *item_args, 0, ps.N + 1, None, 0)
            return
        nv.counted_call("tcar_adam_item_rows", 1, *item_args, p(next_bt.seq), next_bt.B * next_bt.T, p(next_bt.label),
                        next_bt.B, p(ps.row_flags), ps.N + 1)
        timed = self._la_events is not None         # tools/lookahead_times.py: how long both branches really take
        main = torch.cuda.current_stream()
        fork = torch.cuda.Event(enable_timing=timed)
        fork.record(main)
        self._side.wait_event(fork)
        with torch.cuda.stream(self._side):
            nv.counted_call("tcar_adam_item", 1, *item_args, 0, ps.N + 1, p(ps.row_flags), self.adam_overlap_ctas)
            done = torch.cuda.Event(enable_timing=timed)
            done.record(self._side)
        self._update_done = done
        self._ahead.wait_event(fork)
        with torch.cuda.stream(self._ahead):
            self._session_forward(next_bt, prefetch=True)
            adone = torch.cuda.Event(enable_timing=timed)
            adone.record(self._ahead)
        self._ahead_done = adone
        if timed:
            self._la_events.append((fork, done, adone))
        self._prefetched = next_bt

    def _update_small(self):
        """clip + TF-Adam of the 22 small tensors (their norms and the step counter are ready) + tf32 hi/lo refresh."""
        ps, p = self.ps, nv.ptr
        nv.counted_call("tcar_adam_small", 1, p(ps.theta), p(ps.theta_m), p(ps.theta_v), p(ps.theta_g), p(ps.seg_off),
                        p(ps.sqnorm_small), len(SMALL), p(ps.step), self.lr, self.max_grad_f)
        ps.prep_weights()

    def train_step(self, bt, next_bt=None, counts=None):
        """One `sess.run([loss, global_step, train_op])` (model_combine.py:231-234). Returns loss [B] (device).
        next_bt (optional) is the batch of the following call: its session forward is overlapped with this step's
        table-wide Adam pass.  Results are bit-identical with and without it; after a call with next_bt, parameters
        must be read through this object's methods (or after sync_updates()).
        counts (catalog-sharded training only): sessions of every rank in this step, see train_step_catalog."""
        if self.train_parallel == "catalog":
            return self.train_step_catalog(bt, counts if counts is not None else getattr(bt, "counts", None), next_bt,
                                           getattr(next_bt, "counts", None) if next_bt is not None else None)
        if bt.B == 0:
            # data-parallel tail batch with fewer sessions than ranks: contribute a zero gradient to the all-reduce
            self.sync_updates()
            self._prefetched = None
            self.ps.item_g_full.zero_()
            self.ps.theta_g.zero_()
            loss = self.loss[:0]
        else:
            loss, _ = self.forward_train(bt)
            if self.world == 1:
                # the small-tensor update (norms, step counter, Adam, weight split) needs theta_g only: it runs on the
                # auxiliary stream beside the scatter-add of the sparse item rows
                self.backward(bt, scatter=False)
                ps, p = self.ps, nv.ptr
                main = torch.cuda.current_stream()
                ev = torch.cuda.Event()
                ev.record(main)
                self._aux.wait_event(ev)
                with torch.cuda.stream(self._aux):
                    nv.counted_call("tcar_update_norms", 1, p(ps.theta_g), p(ps.seg_off), p(ps.sqnorm_small), len(SMALL),
                                    None, 0, None, 0, None, None, None, p(ps.step))
                    self._update_small()
                    self._small_done = torch.cuda.Event()
                    self._small_done.record(self._aux)
                self._scatter_item_grads(bt)
            else:
                self.backward(bt)
        self.allreduce_grads()
        self.apply_gradients(next_bt)
        return loss

    # ------------------------------------------------------------------------------------------- evaluation
    def _etrace(self, name, stream=None):
        """Timing mark for tools/eval_probe.py (self._eval_trace = [] switches it on)."""
        tr = getattr(self, "_eval_trace", None)
        if tr is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record(stream if stream is not None else torch.cuda.current_stream())
            tr.append((name, ev))

    def _prefetch_forward(self, next_bt):
        """Launch next_bt's session forward on the high-priority stream behind everything queued so far."""
        main = torch.cuda.current_stream()
        fork = torch.cuda.Event()
        fork.record(main)
        self._ahead.wait_event(fork)
        with torch.cuda.stream(self._ahead):
            self._session_forward(next_bt, prefetch=True)
            adone = torch.cuda.Event()
            adone.record(self._ahead)
            self._etrace("ahead: session forward")
        self._ahead_done = adone
        self._prefetched = next_bt

    def eval_step(self, bt, shard=None, next_bt=None):
        """Scores every candidate, returns (top20 ids [B,20], n_greater [B], cross_loss [B]) on the device.
        shard = (item_lo, item_hi, iext_shard) restricts the scoring to a catalog shard (multi-GPU eval).
        next_bt (optional) = the batch of the following call: its session forward (latency-bound) is launched beside
        this batch's top-20 selection (latency-bound too); identical results."""
        ps, p, B = self.ps, nv.ptr, bt.B
        if not self._item_table_synced:
            self.sync_item_table()         # after catalog-sharded training every rank holds only its own rows
        self._etrace("begin")
        if self._prefetched is bt:
            self._prefetched = None
            self.sync_updates()
        else:
            self._session_forward(bt)
        ahead = next_bt is not None and next_bt.B > 0
        if shard is None:
            lo, n_loc, n_pad, iext = 0, ps.N, ps.n_pad, ps.iext
        else:
            lo, hi, iext = shard
            n_loc, n_pad = hi - lo, iext.shape[0]
        if n_loc <= 0:
            # this rank's slice of a small catalog is empty: contribute empty lists to the merge
            self.top_ids[:B].fill_(-1)
            self.top_scores[:B].fill_(float("-inf"))
            self.n_greater[:B].zero_()
            self.sumexp[:B].zero_()
            self.rowmax[:B].zero_()
        else:
            self._ensure_cat_stats()
            ws = self._score_buffers(n_pad, False)
            a_ic, Tq = self.a_ic, self.Tq
            self._etrace("session forward (or wait for the prefetched one)")
            self._score_and_sum(ws, iext, None, p(ws["cmax"]), p(ws["tmax"]), B, n_loc, n_pad, 1)
            self._etrace("scoring GEMM + softmax sums + guard")
            if ahead:
                # the exact re-scoring below reads this batch's session vectors: park them before next_bt's forward
                # overwrites the live buffers.  (Starting that forward right behind the GEMM, beside the softmax sums,
                # was measured and bought nothing: the window between two GEMMs is set by the top-20 selection +
                # widening, 180 us in situ, not by the 130 us session forward -- tools/eval_probe.py.)
                self.a_ic_eval[:B].copy_(self.a_ic[:B])
                self.Tq_eval[:B].copy_(self.Tq[:B])
                a_ic, Tq = self.a_ic_eval, self.Tq_eval
                self._prefetch_forward(next_bt)
                ahead = False
            self._topk(ws, a_ic, Tq, bt.label, self._evblock, B, n_loc, n_pad, lo)
            self._etrace("top-20")
        if ahead:
            self._prefetch_forward(next_bt)
        if shard is not None and parallel.is_distributed(self.world):
            # ONE collective: every rank's result block (top-20 pairs, rank counts, softmax partial sums and their
            # exponent shifts), then one merge kernel
            if getattr(self, "_evblocks", None) is None or self._evblocks.shape[0] != self.world:
                self._evblocks = torch.zeros(self.world, nv.EVAL_BLOCK_WORDS, device=self.dev)
            parallel.gather_eval_blocks(self._evblock, self.world, out=self._evblocks)
            return self._merge_blocks(self._evblocks, self.world, B)
        return self.top_ids[:B], self.n_greater[:B], self.ce[:B]

    def _ensure_cat_stats(self):
        """Largest row norm / bf16 rounding-error norm of the candidate rows (the error bound behind the certified
        top-20): recomputed only after the item table changed."""
        ps = self.ps
        if self._cat_stats_version != ps.version:
            nv.counted_call("tcar_catalog_stats", 1, nv.ptr(ps.item), nv.ptr(ps.content), 1, ps.N + 1,
                            nv.ptr(self.cat_stats))
            self._cat_stats_version = ps.version

    def _topk(self, ws, a_ic, Tq, label, block, B, n_loc, n_pad, lo):
        """Certified top-20 + rank counts of B queries over the n_loc items behind ws's chunk / tile maxima, written
        into the result block `block` (TCAR_EVAL_OFF_* planes)."""
        ps, p = self.ps, nv.ptr
        bi = block.view(torch.int32)
        ids, sc, ngt = p(bi[nv.EVAL_OFF_IDS:]), p(block[nv.EVAL_OFF_SCORES:]), p(bi[nv.EVAL_OFF_NGT:])
        if self.eval_warp_select:
            # selection by one warp per query (tcar_eval_select), exact re-scoring + certification by one CTA per query
            sel = self._sel1
            nv.counted_call("tcar_eval_select", 1, p(ws["cmax"]), p(ws["tmax"]), p(sel), p(sel.view(torch.int32)[QROWS * nv.EVAL_NSEL:]),
                            B, n_loc, n_pad, lo)
            nv.counted_call("tcar_eval_rescore", 1, p(sel), p(sel.view(torch.int32)[QROWS * nv.EVAL_NSEL:]), 1,
                            QROWS * nv.EVAL_NSEL, p(a_ic), p(Tq), p(ps.item), p(ps.content), p(ps.mwdhm), p(label), ids, sc,
                            ngt, B, ps.N, p(self.cat_stats), p(self.uncertain), p(self.tau))
        else:
            nv.counted_call("tcar_eval_topk_certified", 1, p(ws["cmax"]), p(ws["tmax"]), p(a_ic), p(Tq), p(ps.item),
                            p(ps.content), p(ps.mwdhm), p(label), ids, sc, ngt, B, n_loc, n_pad, lo, p(self.cat_stats),
                            p(self.uncertain), p(self.tau))
        self._etrace("top-20: certified selection")
        nv.counted_call("tcar_eval_topk_widen", 1, p(ws["cmax"]), p(ws["tmax"]), p(a_ic), p(Tq), p(ps.item),
                        p(ps.content), p(ps.mwdhm), p(label), p(self.uncertain), p(self.tau), ids, sc, ngt, B, n_loc,
                        n_pad, lo, p(self.widen_ws))

    def _merge_blocks(self, blocks, G, B):
        """G shard result blocks -> global top-20 ids, rank counts, cross_loss (one launch)."""
        p = nv.ptr
        nv.counted_call("tcar_eval_merge", 1, p(blocks), blocks.stride(0), p(self.m_ids), p(self.m_scores),
                        p(self.m_ngt), p(self.m_ce), G, B)
        return self.m_ids[:B], self.m_ngt[:B], self.m_ce[:B]

    # ------------------------------------------------------------- catalog-sharded evaluation, one batch per rank
    EQ_Q, EQ_C = QROWS * KEXT * 2, QROWS * 4
    EQ_A, EQ_T = QROWS * XW * 4, QROWS * NB * 4
    EQ_BYTES = EQ_Q + EQ_C + EQ_A + EQ_T + QROWS * 4

    def _alloc_eval_round(self, R):
        if getattr(self, "_eq", None) is not None and self._eq_all.shape[0] == R:
            return
        dev = self.dev
        self._eq = torch.zeros(self.EQ_BYTES, device=dev, dtype=torch.uint8)
        self._eq_all = torch.zeros(R, self.EQ_BYTES, device=dev, dtype=torch.uint8) if R > 1 else self._eq.view(1, -1)
        self._ev_send = torch.zeros(R, nv.EVAL_BLOCK_WORDS, device=dev)
        self._ev_recv = torch.zeros(R, nv.EVAL_BLOCK_WORDS, device=dev) if R > 1 else self._ev_send
        self._ce_scratch = torch.zeros(QROWS, device=dev)

    def _eq_views(self, blk):
        """(Q bf16 [512,640], c_ref [512], a_ic [512,500], Tq [512,139], label int32 [512]) inside one exchange block."""
        o1 = self.EQ_Q
        o2 = o1 + self.EQ_C
        o3 = o2 + self.EQ_A
        o4 = o3 + self.EQ_T
        return (blk[:o1].view(torch.bfloat16).view(QROWS, KEXT), blk[o1:o2].view(torch.float32),
                blk[o2:o3].view(torch.float32).view(QROWS, XW), blk[o3:o4].view(torch.float32).view(QROWS, NB),
                blk[o4:].view(torch.int32))

    def _round_forward(self, bt, block):
        """Step 1 of eval_round: session forward of the local queries, written straight into an exchange block."""
        if bt.B == 0:
            return
        if self._prefetched is bt:
            raise RuntimeError("eval_round does not take prefetched batches")
        mine = self._eq_views(block)
        keep = (self.Q, self.c_ref, self.a_ic, self.Tq)
        self.Q, self.c_ref, self.a_ic, self.Tq = mine[:4]
        try:
            self._session_forward(bt)
        finally:
            self.Q, self.c_ref, self.a_ic, self.Tq = keep
        mine[4][:bt.B].copy_(bt.label)

    # Two-stage round (the default): an item range only SELECTS its 32 best chunks per query (bf16 chunk
    # maxima, no re-scoring); the query's owner merges the ranges' lists and re-scores the 32 best chunks overall from
    # the replicated fp32 tables -- the exact re-scoring (256 candidate rows per query, the bandwidth-heavy part) is done
    # once per query instead of once per (query, item range).  Queries the owner cannot certify are widened by every
    # range (tcar_eval_topk_widen with the owner's bound) and merged: still the exact top-20.
    def _group_ws(self, n_pad, g):
        key = (n_pad, "eval-group", g)
        if key not in self._score_ws:
            tiles = nv.lib().tcar_score_fwd_tiles(n_pad)
            f = lambda *s_: torch.zeros(*s_, device=self.dev)
            self._score_ws[key] = {"part": f(tiles, QROWS), "pmax": f(tiles, QROWS), "tiles": tiles,
                                   "cmax": f(QROWS, n_pad // nv.CHUNK), "tmax": f(QROWS, n_pad // 128)}
        return self._score_ws[key]

    def _groups_ws(self, n_pad, R):
        """Chunk / tile maxima and softmax partials of R session groups against one item range, group-major."""
        key = (n_pad, "eval-groups", R)
        if key not in self._score_ws:
            tiles = nv.lib().tcar_score_fwd_tiles(n_pad)
            f = lambda *s_: torch.zeros(*s_, device=self.dev)
            self._score_ws[key] = {"part": f(R, tiles * QROWS), "pmax": f(R, tiles * QROWS), "tiles": tiles,
                                   "cmax": f(R, QROWS * (n_pad // nv.CHUNK)), "tmax": f(R, QROWS * (n_pad // 128)),
                                   "widen": torch.zeros(int(nv.lib().tcar_eval_topk_widen_ws_bytes(R)), device=self.dev,
                                                        dtype=torch.uint8)}
        return self._score_ws[key]

    def _round_select(self, eq_all, counts, shard, sel_send):
        """Stage 1 on an item range: every rank's queries -> chunk / tile maxima (kept per group for a later widening),
        guarded softmax partial sums and the candidate lists, written into sel_send[g] (layout nv.SEL_OFF_*).  With
        CTA pairs (the production configuration) the groups share ONE launch per phase: scoring GEMM (both guard
        passes), partial-sum reduction, selection."""
        p = nv.ptr
        lo, hi, iext = shard
        n_loc, n_pad = hi - lo, iext.shape[0]
        R = len(counts)
        if n_loc > 0 and self.cluster == nv.CLUSTER_PAIR and self.eval_group_launch and eq_all.is_contiguous():
            ws = self._groups_ws(n_pad, R)
            cnt = (nv.C.c_int * R)(*counts)
            qs, cs = self.EQ_BYTES // 2, self.EQ_BYTES // 4
            q0 = nv.C.c_void_p(eq_all.data_ptr())
            c0 = nv.C.c_void_p(eq_all.data_ptr() + self.EQ_Q)
            cm_s, tm_s, pt_s = ws["cmax"].stride(0), ws["tmax"].stride(0), ws["part"].stride(0)
            sumexp, rowmax = p(sel_send[0, nv.SEL_OFF_SUMEXP:]), p(sel_send[0, nv.SEL_OFF_ROWMAX:])
            guard = self.softmax_guard
            nv.counted_call("tcar_score_fwd_multi_eval", 1, q0, qs, c0, cs, p(iext), p(ws["cmax"]), cm_s, p(ws["tmax"]),
                            tm_s, p(ws["part"]), pt_s, p(ws["pmax"]), None, sel_send.stride(0), cnt, R, n_loc, n_pad)
            nv.counted_call("tcar_ce_finish_groups", 1, p(ws["part"]), p(ws["pmax"]), pt_s, sumexp, rowmax,
                            sel_send.stride(0), ws["tiles"], cnt, R, 1)
            if guard:
                nv.counted_call("tcar_score_fwd_multi_eval", 1, q0, qs, c0, cs, p(iext), p(ws["cmax"]), cm_s,
                                p(ws["tmax"]), tm_s, p(ws["part"]), pt_s, None, rowmax, sel_send.stride(0), cnt, R, n_loc,
                                n_pad)
                nv.counted_call("tcar_ce_finish_groups", 1, p(ws["part"]), None, pt_s, sumexp, rowmax,
                                sel_send.stride(0), ws["tiles"], cnt, R, 2)
            else:
                sel_send[:, nv.SEL_OFF_ROWMAX:].zero_()
            nv.counted_call("tcar_eval_select_groups", 1, p(ws["cmax"]), cm_s, p(ws["tmax"]), tm_s, p(sel_send),
                            p(sel_send.view(torch.int32)[0, nv.SEL_OFF_IDS:]), sel_send.stride(0), cnt, R, n_loc, n_pad, lo)
            return
        for g, Bg in enumerate(counts):
            if Bg == 0:
                continue
            blk = sel_send[g]
            bi = blk.view(torch.int32)
            if n_loc <= 0:                                   # empty item range: no candidates, no softmax mass
                bi[nv.SEL_OFF_IDS: nv.SEL_OFF_IDS + Bg * nv.EVAL_NSEL].fill_(-1)
                blk[: Bg * nv.EVAL_NSEL].fill_(float("-inf"))
                blk[nv.SEL_OFF_SUMEXP:].zero_()
                continue
            ws = self._group_ws(n_pad, g)
            Qg, cg, _, _, _ = self._eq_views(eq_all[g])
            self._score_and_sum(ws, iext, None, p(ws["cmax"]), p(ws["tmax"]), Bg, n_loc, n_pad, 1, q=Qg, c=cg,
                                sumexp=blk[nv.SEL_OFF_SUMEXP:], ce=self._ce_scratch, rowmax=blk[nv.SEL_OFF_ROWMAX:])
            nv.counted_call("tcar_eval_select", 1, p(ws["cmax"]), p(ws["tmax"]), p(blk), p(bi[nv.SEL_OFF_IDS:]), Bg,
                            n_loc, n_pad, lo)

    def _round_rescore(self, sel_recv, R, eq_block, B, flags):
        """Stage 2 at the queries' owner: merge the R candidate lists, exact re-scoring, top-20 / rank counts into
        m_ids / m_scores / m_ngt, cross loss into m_ce, uncertified queries flagged in `flags` (uncertain | tau)."""
        p = nv.ptr
        ps = self.ps
        self._ensure_cat_stats()
        _, _, a_ic, Tq, lab = self._eq_views(eq_block)
        si = sel_recv.view(torch.int32)
        fi = flags.view(torch.int32)
        nv.counted_call("tcar_eval_rescore", 1, p(sel_recv), p(si[:, nv.SEL_OFF_IDS:]), R, sel_recv.stride(0), p(a_ic),
                        p(Tq), p(ps.item), p(ps.content), p(ps.mwdhm), p(lab), p(self.m_ids), p(self.m_scores),
                        p(self.m_ngt), B, ps.N, p(self.cat_stats), p(fi[:QROWS]), p(flags[QROWS:]))
        nv.counted_call("tcar_eval_ce_combine", 1, p(sel_recv[:, nv.SEL_OFF_SUMEXP:]), p(sel_recv[:, nv.SEL_OFF_ROWMAX:]),
                        sel_recv.stride(0), p(self.m_ce), R, B)

    def _round_widen(self, eq_all, counts, shard, flag_all, send):
        """Stage 3 on an item range: for the flagged queries of every rank, ALL local chunks at or above the owner's
        bound re-scored exactly -> partial top-20 lists and rank counts in send[g] (result-block planes)."""
        p = nv.ptr
        ps = self.ps
        lo, hi, iext = shard
        n_loc, n_pad = hi - lo, iext.shape[0]
        R = len(counts)
        if (n_loc > 0 and self.cluster == nv.CLUSTER_PAIR and self.eval_group_launch and eq_all.is_contiguous()
                and flag_all.is_contiguous()):
            ws = self._groups_ws(n_pad, R)
            cnt = (nv.C.c_int * R)(*counts)
            base = eq_all.data_ptr()
            o_a = self.EQ_Q + self.EQ_C
            o_t, o_l = o_a + self.EQ_A, o_a + self.EQ_A + self.EQ_T
            si = send.view(torch.int32)
            nv.counted_call("tcar_eval_topk_widen_groups", 1, p(ws["cmax"]), ws["cmax"].stride(0), p(ws["tmax"]),
                            ws["tmax"].stride(0), nv.C.c_void_p(base + o_a), nv.C.c_void_p(base + o_t),
                            nv.C.c_void_p(base + o_l), self.EQ_BYTES // 4, p(ps.item), p(ps.content), p(ps.mwdhm),
                            p(flag_all.view(torch.int32)), p(flag_all[0, QROWS:]), flag_all.stride(0),
                            p(si[0, nv.EVAL_OFF_IDS:]), p(send[0, nv.EVAL_OFF_SCORES:]), p(si[0, nv.EVAL_OFF_NGT:]),
                            send.stride(0), cnt, R, n_loc, n_pad, lo, p(ws["widen"]))
            return
        for g, Bg in enumerate(counts):
            if Bg == 0:
                continue
            blk = send[g]
            bi = blk.view(torch.int32)
            if n_loc <= 0:
                bi[nv.EVAL_OFF_IDS: nv.EVAL_OFF_IDS + Bg * TOPK].fill_(-1)
                blk[nv.EVAL_OFF_SCORES: nv.EVAL_OFF_SCORES + Bg * TOPK].fill_(float("-inf"))
                blk[nv.EVAL_OFF_NGT: nv.EVAL_OFF_NGT + QROWS].zero_()
                continue
            ws = self._group_ws(n_pad, g)
            _, _, ag, Tg, lg = self._eq_views(eq_all[g])
            fl = flag_all[g]
            nv.counted_call("tcar_eval_topk_widen", 1, p(ws["cmax"]), p(ws["tmax"]), p(ag), p(Tg), p(ps.item),
                            p(ps.content), p(ps.mwdhm), p(lg), p(fl.view(torch.int32)[:QROWS]), p(fl[QROWS:]),
                            p(bi[nv.EVAL_OFF_IDS:]), p(blk[nv.EVAL_OFF_SCORES:]), p(bi[nv.EVAL_OFF_NGT:]), Bg, n_loc,
                            n_pad, lo, p(self.widen_ws))

    def _round_finish(self, recv, R, B, flags):
        nv.counted_call("tcar_eval_merge_flagged", 1, nv.ptr(recv), recv.stride(0),
                        nv.ptr(flags.view(torch.int32)[:QROWS]), nv.ptr(self.m_ids), nv.ptr(self.m_scores),
                        nv.ptr(self.m_ngt), R, B)
        return self.m_ids[:B], self.m_ngt[:B], self.m_ce[:B]

    def _alloc_two_stage(self, R):
        if getattr(self, "_sel_send", None) is not None and self._sel_send.shape[0] == R:
            return
        f = lambda *s_: torch.zeros(*s_, device=self.dev)
        self._sel_send, self._flag = f(R, nv.SEL_BLOCK_WORDS), f(2 * QROWS)
        self._sel_recv = f(R, nv.SEL_BLOCK_WORDS) if R > 1 else self._sel_send
        self._flag_all = f(R, 2 * QROWS) if R > 1 else self._flag.view(1, -1)

    def _round_score(self, eq_all, counts, shard, send):
        """Step 3 of the one-stage eval_round: every rank's queries (exchange blocks eq_all [R, EQ_BYTES]) against the
        item range `shard` = (lo, hi, iext rows): scoring GEMM + guarded softmax sums + certified top-20 -> send[g]."""
        p = nv.ptr
        lo, hi, iext = shard
        n_loc, n_pad = hi - lo, iext.shape[0]
        if n_loc > 0:
            ws = self._score_buffers(n_pad, False)
            self._ensure_cat_stats()
        for g, Bg in enumerate(counts):
            if Bg == 0:
                continue
            blk = send[g]
            if n_loc <= 0:                                   # empty item range of a small catalog: empty lists
                bi = blk.view(torch.int32)
                bi[nv.EVAL_OFF_IDS: nv.EVAL_OFF_IDS + Bg * TOPK].fill_(-1)
                blk[nv.EVAL_OFF_SCORES: nv.EVAL_OFF_SCORES + Bg * TOPK].fill_(float("-inf"))
                blk[nv.EVAL_OFF_NGT: nv.EVAL_OFF_NGT + 3 * QROWS].zero_()
                continue
            Qg, cg, ag, Tg, lg = self._eq_views(eq_all[g])
            self._score_and_sum(ws, iext, None, p(ws["cmax"]), p(ws["tmax"]), Bg, n_loc, n_pad, 1, q=Qg, c=cg,
                                sumexp=blk[nv.EVAL_OFF_SUMEXP:], ce=self._ce_scratch, rowmax=blk[nv.EVAL_OFF_ROWMAX:])
            self._topk(ws, ag, Tg, lg, blk, Bg, n_loc, n_pad, lo)

    def eval_round(self, bt, counts, shard=None, two_stage=True, next_bt=None):
        """Catalog-sharded evaluation that SCALES: every rank brings its OWN batch of <= 512 queries (bt; B may be 0 in
        the last round), so one round evaluates sum(counts) queries.  counts[g] = queries of rank g (the same list on
        every rank).  Per round (two-stage form, the default):
          1. session forward of the local queries -> [Q | label scores | a_ic | Tq | labels] (1.97 MB, written in place)
          2. all-gather of those blocks: every rank now holds every rank's queries
          3. for every rank g: scoring GEMM of g's queries against the LOCAL item range, guarded softmax partial sums,
             and the range's 32 best chunks per query (tcar_eval_select: no re-scoring) -> candidate block g
          4. all-to-all: rank g receives the candidate blocks about ITS queries from every item range
          5. the owner merges the lists and re-scores the 32 best chunks overall exactly (tcar_eval_rescore) -> top-20,
             rank counts, cross loss; queries it cannot certify are flagged with their bound
          6. all-gather of the flags; every range widens the flagged queries (tcar_eval_topk_widen); all-to-all of the
             partial lists; the owner merges them (tcar_eval_merge_flagged)
        two_stage=False: the one-stage form (every range computes its certified local top-20; one all-gather + one
        all-to-all).  Same results as eval_step(bt) on one GPU either way, bit for bit on the ids
        (model_combine.py:283-306, util.py:8-18).
        next_bt (two-stage form): this rank's batch of the FOLLOWING round; its session forward (a latency-bound chain
        of small kernels) is launched on the high-priority stream beside this round's owner-side phases (re-scoring,
        widening, merge) into the second exchange block.  Identical results."""
        import torch.distributed as dist
        if not self._item_table_synced:
            self.sync_item_table()
        on = parallel.is_distributed(self.world)
        R, me = (self.world, self.rank) if on else (1, 0)
        two_stage = two_stage and R * nv.EVAL_NSEL <= 512
        counts = [int(c) for c in counts]
        B = bt.B
        if len(counts) != R or counts[me] != B:
            raise ValueError("counts must list the queries of every rank (and counts[rank] == bt.B)")
        self._alloc_eval_round(R)
        if shard is None:
            lo, hi = self.shard_bounds(R)[me]
            shard = (lo, hi, self.iext_shard(lo, hi))
        trace = getattr(self, "_round_trace", None)       # tools/eval_round_probe.py: (phase, CUDA event) pairs

        def mark(name):
            if trace is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                trace.append((name, ev))

        mark("start")
        pre, self._round_pre = getattr(self, "_round_pre", None), None
        if pre is not None and pre[0] is bt:
            torch.cuda.current_stream().wait_event(pre[1])       # forward already launched by the previous round
            self._eq, self._eq_next = self._eq_next, self._eq
            self._prefetched = None
        else:
            self._round_forward(bt, self._eq)
        mark("forward")
        if on:
            dist.all_gather_into_tensor(self._eq_all.view(-1), self._eq)
        mark("gather_queries")
        if not two_stage:
            self._round_score(self._eq_all, counts, shard, self._ev_send)
            if on:
                dist.all_to_all_single(self._ev_recv.view(-1), self._ev_send.view(-1))
            if B == 0:
                return self.m_ids[:0], self.m_ngt[:0], self.m_ce[:0]
            return self._merge_blocks(self._ev_recv, R, B)
        self._alloc_two_stage(R)
        self._round_select(self._eq_all, counts, shard, self._sel_send)
        mark("score+select")
        if on:
            dist.all_to_all_single(self._sel_recv.view(-1), self._sel_send.view(-1))
        mark("exchange_lists")
        if next_bt is not None and next_bt.B > 0:
            if getattr(self, "_eq_next", None) is None:
                self._eq_next = torch.zeros_like(self._eq)
            main = torch.cuda.current_stream()
            fork = torch.cuda.Event()
            fork.record(main)
            self._ahead.wait_event(fork)
            with torch.cuda.stream(self._ahead):
                self._round_forward(next_bt, self._eq_next)
                done = torch.cuda.Event()
                done.record(self._ahead)
            self._round_pre = (next_bt, done)
            self._ahead_done = done            # any other entry point waits for it too (sync_updates)
        if B > 0:
            self._round_rescore(self._sel_recv, R, self._eq, B, self._flag)
        else:
            self._flag.zero_()
        mark("rescore")
        if on:
            dist.all_gather_into_tensor(self._flag_all.view(-1), self._flag)
        mark("gather_flags")
        self._round_widen(self._eq_all, counts, shard, self._flag_all, self._ev_send)
        mark("widen")
        if on:
            dist.all_to_all_single(self._ev_recv.view(-1), self._ev_send.view(-1))
        mark("exchange_widened")
        if B == 0:
            return self.m_ids[:0], self.m_ngt[:0], self.m_ce[:0]
        out = self._round_finish(self._ev_recv, R, B, self._flag)
        mark("merge")
        return out

    def eval_round_virtual(self, bts, two_stage=True):
        """Single-GPU emulation of eval_round over V = len(bts) ranks (tests): the same kernels with the same shard
        offsets and block layouts, the collectives replaced by copies.  Returns the per-rank results."""
        V = len(bts)
        counts = [b.B for b in bts]
        two_stage = two_stage and V * nv.EVAL_NSEL <= 512
        self._alloc_eval_round(1)
        eq_all = torch.zeros(V, self.EQ_BYTES, device=self.dev, dtype=torch.uint8)
        for v, bt in enumerate(bts):                      # step 1 of every rank + "all-gather"
            self._round_forward(bt, eq_all[v])
        shards = [(lo, hi, self.iext_shard(lo, hi)) for lo, hi in self.shard_bounds(V)]
        f = lambda *s_: torch.zeros(*s_, device=self.dev)
        outs = []
        if not two_stage:
            sends = []
            for v in range(V):                            # step 3 of every rank
                send = f(V, nv.EVAL_BLOCK_WORDS)
                self._round_score(eq_all, counts, shards[v], send)
                sends.append(send)
            for v in range(V):                            # "all-to-all" + merge of every rank
                if counts[v] == 0:
                    outs.append(None)
                    continue
                recv = torch.stack([sends[src][v] for src in range(V)])
                outs.append(tuple(x.clone() for x in self._merge_blocks(recv, V, counts[v])))
            return outs
        # two-stage: the chunk / tile maxima of (range v, group g) must survive until the widening -> one workspace
        # set per virtual range
        saved_ws = self._score_ws
        ws_of = [dict() for _ in range(V)]
        sel = []
        for v in range(V):
            self._score_ws = ws_of[v]
            blk = f(V, nv.SEL_BLOCK_WORDS)
            self._round_select(eq_all, counts, shards[v], blk)
            sel.append(blk)
        flags, firsts = f(V, 2 * QROWS), []
        for v in range(V):
            if counts[v] == 0:
                firsts.append(None)
                continue
            recv = torch.stack([sel[src][v] for src in range(V)])
            self._round_rescore(recv, V, eq_all[v], counts[v], flags[v])
            firsts.append((self.m_ids.clone(), self.m_scores.clone(), self.m_ngt.clone(), self.m_ce.clone()))
        wid = []
        for v in range(V):
            self._score_ws = ws_of[v]
            send = f(V, nv.EVAL_BLOCK_WORDS)
            self._round_widen(eq_all, counts, shards[v], flags, send)
            wid.append(send)
        self._score_ws = saved_ws
        for v in range(V):
            if counts[v] == 0:
                outs.append(None)
                continue
            ids, sc, ngt, ce = firsts[v]
            self.m_ids.copy_(ids); self.m_scores.copy_(sc); self.m_ngt.copy_(ngt); self.m_ce.copy_(ce)
            recv = torch.stack([wid[src][v] for src in range(V)])
            outs.append(tuple(x.clone() for x in self._round_finish(recv, V, counts[v], flags[v])))
        self.last_round_flagged = int(flags.view(torch.int32)[:, :QROWS].sum().item())
        return outs

    def shard_bounds(self, G):
        """Contiguous item-id ranges [lo, hi) per shard, aligned to 256 rows so that a shard of the bf16 scoring
        operand is a plain row-slice of ps.iext."""
        return parallel.shard_bounds(self.ps.N, self.ps.n_pad, G)

    def iext_shard(self, lo, hi):
        n_pad = max((hi - lo + 255) // 256 * 256, 256)
        return self.ps.iext[lo: lo + n_pad]

    def eval_step_virtual_shards(self, bt, G):
        """Single-GPU emulation of the catalog-sharded evaluation: every shard is scored in turn and the per-shard
        top-20 lists are merged with the same kernel the NCCL path uses (tests the merge logic without G GPUs)."""
        B = bt.B
        blocks = torch.zeros(G, nv.EVAL_BLOCK_WORDS, device=self.dev)
        world, self.world = self.world, 1
        try:
            for g, (lo, hi) in enumerate(self.shard_bounds(G)):
                self.eval_step(bt, shard=(lo, hi, self.iext_shard(lo, hi)))
                blocks[g].copy_(self._evblock)
        finally:
            self.world = world
        return self._merge_blocks(blocks, G, B)

    def softmax_input(self, bt):
        """Debug aid mirroring the reference's `softmax_input` fetch (model_combine.py:138): materialises the
        [B,N] fp32 scores from the same bf16 operands with a library GEMM.  Not used on the hot path."""
        self._session_forward(bt)
        return self.Q[:bt.B].float() @ self.ps.iext[: self.ps.N].float().t()

    # ------------------------------------------------------------------------------------------- candidate re-ranking
    def rerank(self, bt, cand_off, cand_ids, metrics=True):
        """Rank a given candidate list per session (tcar_rerank).  Session b's candidates are
        cand_ids[cand_off[b]:cand_off[b + 1]]: 0-based item ids in host arrays (NumPy, lists or CPU tensors), duplicates
        allowed, at most nv.RERANK_MAXL per session; cand_off has B + 1 entries from 0 to len(cand_ids).  The scores are
        the exact fp32 scores of the full-catalog evaluation (bit for bit what eval_step reports for the same item), not
        the bf16 products of softmax_input().

        Returns device tensors (scores [nnz] in input order, ranked [nnz] = every list's ids ordered by (score desc,
        id asc), label_rank [B], auc [B]).  bt.label is read for the metrics only: it is the positive of its session's
        list and every other entry a negative; label_rank = 1 + #negatives scoring above it (the label wins ties),
        auc counts a tied negative as 1/2 and is NaN for a list without negatives.  metrics=False returns None for
        the last two, so a serving caller may fill bt.label with any valid item id."""
        B, N = bt.B, self.N
        host, max_len = check_id_lists(cand_off, cand_ids, B, N, names=("cand_off", "cand_ids"),
                                       nouns=("candidate id", "candidates"), limit=nv.RERANK_MAXL,
                                       limit_name="TCAR_RERANK_MAXL")
        nnz = host.shape[0] - (B + 1)
        dev, p, ps = self.dev, nv.ptr, self.ps
        scores = torch.empty(nnz, device=dev)
        ranked = torch.empty(nnz, device=dev, dtype=torch.int32)
        label_rank = torch.empty(B, device=dev, dtype=torch.int32) if metrics else None
        auc = torch.empty(B, device=dev) if metrics else None
        if B == 0:
            return scores, ranked, label_rank, auc
        if not self._item_table_synced:
            self.sync_item_table()         # after catalog-sharded training every rank holds only its own rows
        self._session_forward(bt)
        csr = self._stage_ints(host)
        nv.counted_call("tcar_rerank", 1, p(self.a_ic), p(self.Tq), p(ps.item), p(ps.content), p(ps.mwdhm), p(csr),
                        p(csr[B + 1:]), p(bt.label) if metrics else None, B, N, max_len, p(scores), p(ranked),
                        p(label_rank), p(auc))
        return scores, ranked, label_rank, auc

    def _eval_sampler(self, test_data):
        """The batches of a split as test() walks them; under torchrun only this rank's (Sampler.keep_rank_batches)."""
        sampler = Sampler(*test_data, batch_size=self.batch_size)
        if parallel.is_distributed(self.world):
            sampler.keep_rank_batches(self.rank, self.world)
        return sampler

    def _sum_over_ranks(self, sums):
        """This rank's float64 metric sums -> their sum over all ranks (unchanged on one GPU)."""
        if not parallel.is_distributed(self.world):
            return sums
        t = torch.as_tensor(sums, device=self.dev)
        parallel.allreduce_sum((t,), self.world)
        return t.cpu().numpy()

    def test_impressions(self, sess, test_data, impressions, item_dict, args):
        """Rank every session's impression list (the MIND protocol): the clicked article (the label) is the positive,
        the listed articles known to item_dict the negatives (sampler.impression_candidates).  Prints and returns
        {"auc", "mrr", "ndcg5", "ndcg10", "sessions", "skipped"}: averages over the sessions with at least one
        negative (util.impression_sums); `skipped` counts the others.  Walks the split in the batches test() uses.
        Under torchrun batch i goes to rank i mod world and the sums are all-reduced, so every rank returns the
        metrics of the whole split."""
        from .sampler import impression_candidates
        from .util import impression_metrics, impression_sums
        print("Ranking impression lists...")
        self.sync_item_table()
        session_dict_test = test_data[1]
        sampler = self._eval_sampler(test_data)
        # this rank's lists up front, so that the producer thread does no dictionary work per batch
        cands = [impression_candidates(keys, [session_dict_test[k][-1] - 1 for k in keys], impressions, item_dict)
                 for keys in sampler.session_id_batches]
        sums = np.zeros(6)

        def launch(cur, nxt):
            bt, (off, ids) = cur
            _, _, rank, auc = self.rerank(bt, off, ids)
            return np.diff(off) - 1, self.fetch_async(rank), self.fetch_async(auc)

        def consume(n_neg, rank, auc):
            sums[:] += impression_sums(rank.get().numpy(), auc.get().numpy(), n_neg)

        pipelined(zip((self.stage_to_device(packed, B, T, Nn) for packed, B, T, Nn in prefetch_packed(sampler)), cands),
                  launch, consume)
        m = impression_metrics(self._sum_over_ranks(sums))
        self.last_impression_metrics = m
        print("Impressions: AUC: {}, MRR: {}, nDCG@5: {}, nDCG@10: {} ({} sessions, {} without a negative skipped)".format(
            m["auc"], m["mrr"], m["ndcg5"], m["ndcg10"], m["sessions"], m["skipped"]))
        return m

    # ------------------------------------------------------------------------------------------- top-K recommendation
    def set_item_times(self, times):
        """One time per item for recommend(window=..., decay=...): N integers of any integer type, each within int32, in whatever
        clock unit the windows use (recommend_split: minutes since the epoch).  Checked on the host (ValueError, nothing
        uploaded), then copied once to an int32 [n_pad] device buffer; may be called again at any time, e.g. to
        withdraw an article by giving it a time no window reaches."""
        t = check_item_times(times, self.N)
        if getattr(self, "_item_time", None) is None:
            self._item_time = torch.zeros(self.ps.n_pad, device=self.dev, dtype=torch.int32)
        self._item_time[:self.N].copy_(torch.from_numpy(t))
        self._item_time_min = int(t.min()) if self.N else 0     # the oldest item: check_decay's largest penalty

    def set_item_categories(self, codes, n_categories=None):
        """One category code per item for recommend(max_per_category=..., categories=...): N integers in [0, G),
        G = n_categories (default max(codes) + 1) <= nv.RECOMMEND_MAXG.  Checked on the host (ValueError, nothing
        uploaded).  Builds the catalog in category order (util.category_layout: N' <= N + 7 G positions) and iext_cat,
        a second copy of the bf16 scoring operand whose row p is the ps.iext row of the item at position p, about
        N' x 1280 bytes; recommend() rebuilds it whenever the item table has changed.  May be called again."""
        codes, G = check_item_categories(codes, self.N, n_categories)
        perm, off, n2 = category_layout(codes, G)
        n_pad = (n2 + 255) // 256 * 256
        dev = self.dev
        if getattr(self, "_iext_cat", None) is None or self._iext_cat.shape[0] != n_pad:
            old = getattr(self, "_cat_n_pad", None)
            if old is not None and old != self.ps.n_pad:
                self._score_ws.pop((old, False), None)       # the previous layout's score buffers
            self._iext_cat = torch.zeros(n_pad, nv.KEXT, device=dev, dtype=torch.bfloat16)
        else:
            self._iext_cat[n2:].zero_()                      # rows >= N' are zero
        self._cat_perm = torch.from_numpy(perm).to(dev)
        self._cat_src = torch.from_numpy(pad_sources(perm)).to(dev)
        self._cat_off = torch.from_numpy(off).to(dev)
        self._item_cat = torch.from_numpy(codes).to(dev)
        self._cat_G, self._cat_n, self._cat_n_pad = G, n2, n_pad
        self._iext_cat_version = -1

    def _ensure_iext_cat(self):
        """Gather iext_cat from ps.iext again when the item table has changed since the last build (the rule of
        _ensure_cat_stats): a plain row gather, off the per-batch path."""
        if self._iext_cat_version != self.ps.version:
            torch.index_select(self.ps.iext, 0, self._cat_src, out=self._iext_cat[:self._cat_n])
            self._iext_cat_version = self.ps.version

    def recommend(self, bt, k=20, exclude_off=None, exclude_ids=None, exclude_clicked=False, window=None,
                  max_per_category=None, categories=None, decay=None):
        """The exact top-k of the whole catalog for every session of bt (tcar_recommend), 1 <= k <= nv.RECOMMEND_MAXK,
        ordered by (score desc, id asc).  Scores are the exact fp32 scores of the full-catalog evaluation: with k <= 20
        and no exclusions the result is the prefix of eval_step's top-20, and an item scores bit for bit what eval_step
        and rerank report for it.

        Exclusions: session b never gets exclude_ids[exclude_off[b]:exclude_off[b + 1]] (0-based item ids in host
        arrays, duplicates allowed; exclude_off has B + 1 entries from 0 to len(exclude_ids)) nor, with
        exclude_clicked=True, the articles of its own clicks (read on the device from bt.seq).  A session's list
        length plus T (with exclude_clicked) is at most nv.RECOMMEND_MAXX.

        Returns device tensors (ids [B, k] int32, scores [B, k] fp32); a catalog of fewer than k eligible items pads
        with -1 / -inf.  The number of items each session re-scored exactly is left in self.rec_rescored[:B].
        bt.label plays no part in the result (the session forward reads it, so a serving caller fills it with any
        valid item id).

        Publish-time window: window = (lo, hi), host arrays of B integers within int32, lo[b] <= hi[b], restricts
        session b to the items with lo[b] <= t[n] <= hi[b], t = the times of set_item_times (same clock unit).  The
        result is the exact top-k of the in-window, non-excluded items, with the same exact scores; a window with fewer
        than k of them pads with -1 / -inf.  The mask sits in the scoring GEMM's epilogue (tcar_score_fwd_window,
        tcar_recommend_window), so the selection stays exact however few items a window holds.

        Freshness decay: decay = (t_ref, rate), t_ref a host array of B integers within int32 (the request times, in
        the clock unit of set_item_times) and rate one number or B numbers, finite and >= 0 (score units per clock
        unit), ranks session b by r = s - p, p = rate[b] * age, age = min(max(t_ref[b] - t[n], 0), DECAY_MAX_AGE)
        (util.decay_penalty: age exact in float32, one float32 multiply and one float32 subtract; items published
        after t_ref get age 0).  The result is the exact top-k by (r desc, id asc) and scores holds r.  A rate whose
        penalty for the oldest item is not finite in float32 is refused.  The penalty sits in the scoring GEMM's
        epilogue (tcar_score_fwd_decay, tcar_recommend_decay), so an article just outside the undecayed top-k is still
        found.  Composes with the exclusions and window.

        Categories (after set_item_categories): max_per_category = C >= 1 leaves out an item that has C better items of
        its category in the list (C >= k: no cap); categories = (off, codes) restricts session b to the categories
        codes[off[b]:off[b + 1]] (CSR as the exclusion lists, codes in [0, G), duplicates allowed; an empty list gives
        -1 / -inf throughout).  Exclusions compose with both; window and decay do not (ValueError).  The result is the exact
        capped, filtered top-k in the same format, by the scoring GEMM over iext_cat and tcar_recommend_category."""
        if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)) or not 1 <= k <= nv.RECOMMEND_MAXK:
            raise ValueError(f"k must be an integer in [1, TCAR_RECOMMEND_MAXK = {nv.RECOMMEND_MAXK}], got {k!r}")
        if (exclude_off is None) != (exclude_ids is None):
            raise ValueError("exclude_off and exclude_ids are given together")
        k, B, N = int(k), bt.B, self.N
        extra = bt.T if exclude_clicked else 0
        host = None
        if exclude_off is not None:
            host, _ = check_id_lists(exclude_off, exclude_ids, B, N, names=("exclude_off", "exclude_ids"),
                                     nouns=("excluded id", "exclusions"), limit=nv.RECOMMEND_MAXX,
                                     limit_name="TCAR_RECOMMEND_MAXX", extra=extra)
        elif extra > nv.RECOMMEND_MAXX:
            raise ValueError(f"session 0: more than TCAR_RECOMMEND_MAXX = {nv.RECOMMEND_MAXX} clicks")
        win = None
        if window is not None:
            if getattr(self, "_item_time", None) is None:
                raise ValueError("window needs item times: call set_item_times first")
            win = check_windows(window, B)
        dec = None
        if decay is not None:
            if getattr(self, "_item_time", None) is None:
                raise ValueError("decay needs item times: call set_item_times first")
            dec = check_decay(decay, B, [self._item_time_min])
        by_cat = max_per_category is not None or categories is not None
        if by_cat:
            if getattr(self, "_iext_cat", None) is None:
                raise ValueError("max_per_category / categories need item categories: call set_item_categories first")
            if window is not None:
                raise ValueError("window cannot be combined with max_per_category / categories")
            if decay is not None:
                raise ValueError("decay cannot be combined with max_per_category / categories")
            C = k
            if max_per_category is not None:
                if isinstance(max_per_category, (bool, np.bool_)) or not isinstance(max_per_category, (int, np.integer)) \
                        or max_per_category < 1:
                    raise ValueError(f"max_per_category must be an integer >= 1, got {max_per_category!r}")
                C = int(min(max_per_category, k))
            allowed = None
            if categories is not None:
                if not isinstance(categories, (tuple, list)) or len(categories) != 2:
                    raise ValueError("categories must be a pair (off, codes) of integer arrays")
                allowed, _ = check_id_lists(categories[0], categories[1], B, self._cat_G,
                                            names=("categories off", "categories codes"),
                                            nouns=("category", "categories"), limit=float("inf"), limit_name="")
        dev, p, ps = self.dev, nv.ptr, self.ps
        out_ids = torch.empty(B, k, device=dev, dtype=torch.int32)
        out_sc = torch.empty(B, k, device=dev)
        if B == 0:
            return out_ids, out_sc
        if getattr(self, "_rec_ws", None) is None:
            # one workspace for the three selections, sized for the category one (tcar_recommend's layout plus the
            # per-category thresholds: QROWS x TCAR_RECOMMEND_MAXG x 4 B = 2 MiB more); its ticket counters come first:
            # zero once, every call leaves them at zero
            self._rec_ws = torch.zeros(int(nv.lib().tcar_recommend_category_ws_bytes(QROWS)), device=dev,
                                       dtype=torch.uint8)
            self.rec_rescored = torch.zeros(QROWS, device=dev, dtype=torch.int32)
        if not self._item_table_synced:
            self.sync_item_table()         # after catalog-sharded training every rank holds only its own rows
        self._session_forward(bt)
        self._ensure_cat_stats()
        # the chunk / tile maxima of one unguarded eval-mode GEMM (its softmax partial sums, which may overflow without
        # the guard, are not read): over ps.iext, with the windows applied in the epilogue, or over iext_cat (N' items
        # in category order); the windows and the decay go up through the pinned ring like the exclusion lists.  With a
        # decay the GEMM writes the maxima of the decayed scores, with its window if there is one.
        if dec is not None:
            ws = self._score_buffers(ps.n_pad, False)
            wv = self._stage_ints(win) if win is not None else None
            dv = self._stage_ints(dec)
            wargs = (p(wv), p(wv[B:])) if wv is not None else (None, None)
            nv.counted_call("tcar_score_fwd_decay", 1, p(self.Q), p(ps.iext), p(ws["cmax"]), p(ws["tmax"]),
                            p(self._item_time), p(dv), p(dv[B:]), *wargs, B, N, ps.n_pad)
        elif win is not None:
            ws = self._score_buffers(ps.n_pad, False)
            wv = self._stage_ints(win)
            nv.counted_call("tcar_score_fwd_window", 1, p(self.Q), p(ps.iext), p(self.c_ref), p(ws["part"]),
                            p(ws["cmax"]), p(ws["tmax"]), p(self._item_time), p(wv), p(wv[B:]), B, N, ps.n_pad)
        else:
            if by_cat:
                self._ensure_iext_cat()
            iext, n, n_pad = (self._iext_cat, self._cat_n, self._cat_n_pad) if by_cat else (ps.iext, N, ps.n_pad)
            ws = self._score_buffers(n_pad, False)
            nv.counted_call("tcar_score_fwd", 1, p(self.Q), p(iext), p(self.c_ref), None, p(ws["part"]), p(ws["cmax"]),
                            p(ws["tmax"]), B, n, n_pad, 1, self._cluster_for(B))
        csr = self._stage_ints(host) if host is not None else None
        query = (p(self.a_ic), p(self.Tq), p(ps.item), p(ps.content), p(ps.mwdhm), p(self.cat_stats), p(csr),
                 p(csr[B + 1:]) if csr is not None else None, p(bt.seq) if exclude_clicked else None, bt.T, B)
        out = (p(self._rec_ws), p(out_ids), p(out_sc), p(self.rec_rescored))
        if by_cat:
            acsr = self._stage_ints(allowed) if allowed is not None else None
            nv.counted_call("tcar_recommend_category", 2, p(ws["cmax"]), *query, self._cat_n_pad, k,
                            p(self._cat_perm), p(self._item_cat), p(self._cat_off), self._cat_G, p(acsr),
                            p(acsr[B + 1:]) if acsr is not None else None, C, *out)
        elif dec is not None:
            nv.counted_call("tcar_recommend_decay", 2, p(ws["cmax"]), p(ws["tmax"]), *query, N, ps.n_pad, k, *out,
                            p(self._item_time), p(dv), p(dv[B:]), *wargs)
        elif win is not None:
            nv.counted_call("tcar_recommend_window", 2, p(ws["cmax"]), p(ws["tmax"]), *query, N, ps.n_pad, k, *out,
                            p(self._item_time), p(wv), p(wv[B:]))
        else:
            nv.counted_call("tcar_recommend", 2, p(ws["cmax"]), p(ws["tmax"]), *query, N, ps.n_pad, k, *out)
        return out_ids, out_sc

    def recommend_split(self, sess, test_data, item_dict, args):
        """Recommend the top-K articles (args["recommend_k"], default 20) for every session of a split, optionally
        without the session's own clicks (args["recommend_exclude_clicked"]), in the batches test() uses.  Writes one
        line per session to saved/recommend_<foldnum>[_rank<r>].txt (util.recommend_line: the session key, then K
        `article:score` pairs with the original article ids) and prints and returns {"hr", "mrr", "ndcg", "sessions"}
        @K, where a session's rank is its label's 1-based position in the returned list (ties go to the lower id).
        Under torchrun batch i goes to rank i mod world (each rank writes its own file) and the sums are all-reduced,
        so every rank returns the metrics of the whole split.

        args["recommend_max_age_h"] = H > 0 (hours) restricts every session to the articles published in
        [t_req - round(60 H) min, t_req], t_req = the click time of its last input click (util.session_windows): the
        time-aware protocol, which never recommends an article published after the request.  Article times are
        args["publish_time"] (one datetime per item, main.load_datas) in minutes since the epoch.  Then the result
        also holds "label_outside": the sessions whose label was published outside their window (never a hit).

        args["recommend_max_per_category"] = C returns at most C articles of one category per list (exact: the capped
        top-K, recommend(max_per_category=C)), with the categories of args["category_id"]; it cannot be combined with
        recommend_max_age_h.  The articles without a category share one extra code here, unlike _categories(), which
        gives each its own: every category is padded to whole 8-item chunks in the category-ordered catalog, and one
        padded category per unknown article would blow up its size.  Then the result also holds "ild" and "unexp",
        the reference's intra-list diversity and unexpectedness (getILD / getUnexp, padding dropped) averaged as test()
        averages them: over the returned lists of at least two items.

        args["recommend_half_life_h"] = H > 0 (hours) ranks every session by the decayed score of recommend(decay=...)
        with t_ref = t_req (util.session_request_times) and rate = ln 2 / (60 H) per minute, so that an article's
        recommendation probability halves every H hours of age; it composes with recommend_max_age_h and cannot be
        combined with recommend_max_per_category.  Then the result also holds "mean_age_h": the mean age
        max(t_req - publish time, 0) of the returned articles in hours (padding dropped)."""
        from .util import (count_outside, diversity_sums, epoch_minutes, label_positions, recommend_line,
                           session_request_times, session_windows, topk_metrics, topk_sums)
        k = int(args.get("recommend_k") or 20)
        clicked = bool(args.get("recommend_exclude_clicked"))
        max_age = args.get("recommend_max_age_h")
        windowed = max_age is not None
        half_life = args.get("recommend_half_life_h")
        decayed = half_life is not None
        cap = args.get("recommend_max_per_category")
        capped = cap is not None
        if capped:
            if windowed:
                raise ValueError("recommend_max_per_category cannot be combined with recommend_max_age_h")
            if decayed:
                raise ValueError("recommend_max_per_category cannot be combined with recommend_half_life_h")
            self.set_item_categories(self._split_category_codes())
        if windowed and not float(max_age) > 0:
            raise ValueError(f"recommend_max_age_h must be > 0 hours, got {max_age!r}")
        if decayed and not (0 < float(half_life) < float("inf")):
            raise ValueError(f"recommend_half_life_h must be a finite number of hours > 0, got {half_life!r}")
        if windowed or decayed:
            if args.get("publish_time") is None:
                raise ValueError("{} needs every article's publish time in args['publish_time']".format(
                    "recommend_max_age_h" if windowed else "recommend_half_life_h"))
            item_time = epoch_minutes(args["publish_time"])
            self.set_item_times(item_time)
        if windowed:
            max_age_min = int(round(60 * float(max_age)))
        if decayed:
            rate = float(np.log(2.0) / (60.0 * float(half_life)))
        print("Recommending the top-{} articles{}{}{}{}...".format(
            k, " without the clicked ones" if clicked else "",
            " published at most {} h before the request".format(max_age) if windowed else "",
            ", at most {} per category".format(cap) if capped else "",
            ", ranked with a freshness half-life of {} h".format(half_life) if decayed else ""))
        self.sync_item_table()
        session_dict_test = test_data[1]
        reverse = self.reverse_item if self.reverse_item is not None else \
            {cnt - 1: art for art, cnt in item_dict.items()}
        sampler = self._eval_sampler(test_data)
        keys = list(sampler.session_id_batches)
        # this rank's windows up front, so that the producer thread does no dictionary work per batch
        wins = [session_windows(kb, test_data[2], max_age_min) for kb in keys] if windowed else [None] * len(keys)
        t_reqs = [session_request_times(kb, test_data[2]) for kb in keys] if decayed else [None] * len(keys)
        os.makedirs("saved", exist_ok=True)
        dist_on = parallel.is_distributed(self.world)
        path = "saved/recommend_{}{}.txt".format(args.get("foldnum", 0), "_rank{}".format(self.rank) if dist_on else "")
        # HR / MRR / nDCG / sessions, then label_outside (window), ILD / unexpectedness / lists (cap), and the summed
        # age in minutes / number of returned articles (decay)
        sums = np.zeros((5 if windowed else 7 if capped else 4) + (2 if decayed else 0))

        def launch(cur, nxt):
            bt, (kb, win, t_req) = cur
            ids, sc = self.recommend(bt, k, exclude_clicked=clicked, window=win,
                                     **({"max_per_category": int(cap)} if capped else {}),
                                     **({"decay": (t_req, rate)} if decayed else {}))
            return kb, win, t_req, self.fetch_async(ids), self.fetch_async(sc)

        def consume(kb, win, t_req, ids_h, sc_h):
            ids, sc = ids_h.get().numpy(), sc_h.get().numpy()
            labels = [session_dict_test[key][-1] - 1 for key in kb]
            sums[:4] += topk_sums(label_positions(ids, labels))
            if windowed:
                sums[4] += count_outside(item_time[labels], *win)
            if capped:
                sums[4:7] += diversity_sums(ids, [np.asarray(session_dict_test[key][:-1]) - 1 for key in kb],
                                            self._categories())
            if decayed:
                got = ids >= 0
                age = np.maximum(t_req[:, None] - item_time[np.maximum(ids, 0)], 0)
                sums[-2:] += (age[got].sum(), got.sum())
            f.writelines(recommend_line(key, ids[b], sc[b], reverse) for b, key in enumerate(kb))

        with open(path, "w") as f:
            pipelined(zip((self.stage_to_device(packed, B, T, Nn) for packed, B, T, Nn in prefetch_packed(sampler)),
                          zip(keys, wins, t_reqs)), launch, consume)
        total = self._sum_over_ranks(sums)
        m = topk_metrics(total[:4])
        if windowed:
            m["label_outside"] = int(total[4])
        if capped:
            n = total[6]
            m["ild"], m["unexp"] = (float(total[4] / n), float(total[5] / n)) if n > 0 else (float("nan"),) * 2
        if decayed:
            m["mean_age_h"] = float(total[-2] / total[-1] / 60) if total[-1] > 0 else float("nan")
        self.last_recommend_metrics = m
        self.last_recommend_path = path
        print("Recommend: HR@{k}: {}, MRR@{k}: {}, nDCG@{k}: {} ({} sessions{}, written to {})".format(
            m["hr"], m["mrr"], m["ndcg"], m["sessions"],
            ", {} labels published outside their window".format(m["label_outside"]) if windowed else "", path, k=k))
        if capped:
            print("Recommend: ILD: {}, unexpectedness: {}".format(m["ild"], m["unexp"]))
        if decayed:
            print("Recommend: mean age of the returned articles: {} h (half-life {} h)".format(m["mean_age_h"],
                                                                                              half_life))
        return m

    def _split_category_codes(self):
        """Category code of every item for recommend_split: args["category_id"] through reverse_item, codes in order
        of first appearance; every item without a category gets one shared extra code (see recommend_split)."""
        codes, index, none = np.empty(self.N, dtype=np.int64), {}, object()
        getter = self.category_id.get if hasattr(self.category_id, "get") else None
        for i in range(self.N):
            art = self.reverse_item.get(i, none) if hasattr(self.reverse_item, "get") else self.reverse_item[i]
            c = getter(art, none) if getter is not None else self.category_id[art]
            codes[i] = index.setdefault(c, len(index))
        return codes

    # ------------------------------------------------------------------------------------------- metrics
    def _categories(self):
        if self._cat_array is None:
            cat = np.zeros(self.N, dtype=np.int64)
            codes = {}
            for i in range(self.N):
                # items without a category (MIND's extra candidates, mind_preprocess.py:275-280) get their own code
                c = self.category_id.get(self.reverse_item.get(i, ("?", i)), ("?", i)) \
                    if hasattr(self.category_id, "get") else self.category_id[self.reverse_item[i]]
                cat[i] = codes.setdefault(c, len(codes))
            self._cat_array = cat
        return self._cat_array

    def getILD(self, recList):
        """model_combine.py:174-182, vectorised over the category codes."""
        c = self._categories()[np.asarray(recList)]
        n = len(c)
        return float((c[:, None] != c[None, :]).sum()) / (n * (n - 1))

    def getUnexp(self, inSeq, recList):
        """model_combine.py:184-194."""
        if len(recList) == 0:
            return 0
        cat = self._categories()
        c, ci = cat[np.asarray(recList)], cat[np.asarray(inSeq) - 1]
        return float((c[:, None] != ci[None, :]).sum()) / (len(c) * len(ci))

    def printData(self, filename, batch_in, batch_out, batch_pred):
        os.makedirs("saved", exist_ok=True)
        with open("saved/CAR+P_Normal_predict_exa_" + filename + ".txt", "a+") as f:
            for index in range(len(batch_in)):
                f.write("# batch in: {} # batch out: {} # batch pred: {} \n".format(
                    str(batch_in[index]), str(batch_out[index]), str(batch_pred[index])))

    # ------------------------------------------------------------------------------------------- loops
    def train(self, sess, item_dict, train_data, neighbor_dict, args, test_data=None, saver=None, threshold_acc=0.99):
        """model_combine.py:196-252."""
        (len_dict_train, session_dict_train, session_time_dict_train) = train_data
        # Multi-GPU (torchrun): "per_rank" (default) = every rank trains on its OWN batch of <= batch_size sessions of
        # the same length bucket, i.e. the global batch is world x batch_size -- this changes the optimisation
        # trajectory against the single-GPU loop (model_combine.py:196-252 sees batch_size sessions per step), which is
        # what weak scaling means; "split" = ONE batch of batch_size sessions split over the ranks: the single-GPU
        # trajectory, no throughput gain from more GPUs.
        dist_batch = (args.get("dist_batch") or "per_rank") if self.world > 1 else "single"
        if dist_batch not in ("per_rank", "split", "single"):
            raise ValueError("dist_batch must be 'per_rank' or 'split'")
        gbatch = self.batch_size * (self.world if dist_batch == "per_rank" else 1)
        neg_mode = args.get("negative_mode") or "uniform"
        if dist_batch == "per_rank":
            print("rank {}: global batch = {} x {} sessions".format(self.rank, self.world, self.batch_size))
            np.random.seed(2020 + 7919 * self.rank)       # distinct uniform negatives per rank (main.py:11-12 seeds 2020)
        for epoch in range(self.epoch):
            self.curEpoch = epoch
            print("Epoch {}".format(epoch))
            c = []
            mode = args.get("device_sampler") or "off"
            if mode != "off":
                # GPU-resident sampler (SURVEY 8f-2): "host" = negatives from the reference's NumPy stream (batches
                # identical to the host sampler's), "device" = Philox negatives drawn on the device
                from .device_sampler import DeviceSampler
                sampler = DeviceSampler(self, len_dict_train, session_dict_train, session_time_dict_train,
                                        neighbor_dict, item_dict, args["neg_num"], batch_size=gbatch,
                                        negative_mode=neg_mode, negatives=mode, seed=2020 + epoch, rank=self.rank,
                                        world=self.world)
            else:
                sampler = Sampler(len_dict_train, session_dict_train, session_time_dict_train, neighbor_dict,
                                  item_dict, args["neg_num"], batch_size=gbatch, negative_mode=neg_mode)
                if self.world > 1:
                    sampler.restrict_to_rank(self.rank, self.world)
            batch = 0

            def staged():
                nonlocal batch
                if mode != "off":
                    while sampler.has_next():
                        batch += 1
                        yield sampler.next_device()
                    return
                sizes = getattr(sampler, "global_sizes", None)
                for packed, B, T, Nn in prefetch_packed(sampler):
                    if batch < 2 and Nn and B:
                        print(packed[7 * B * T + 3 * B: 7 * B * T + 3 * B + min(Nn, 10)].tolist())
                    # every rank walks the same global batches (same `random` seed, main.py:9-10) and has gathered
                    # only its own share of the sessions (Sampler.restrict_to_rank)
                    bt_ = self.stage_to_device(packed, B, T, Nn)
                    bt_.counts = parallel.catalog_counts(sizes[batch], self.world) if sizes is not None else None
                    batch += 1
                    yield bt_

            # one batch of look-ahead: batch i+1 is on the device before step i is launched, so that its session
            # forward can overlap step i's table-wide Adam pass (train_step(bt, next_bt))
            it = staged()
            bt = next(it, None)
            while bt is not None:
                nxt = next(it, None)
                c.append(self.train_step(bt, nxt).clone())
                bt = nxt
            self.sync_updates()
            tot = torch.stack([torch.cat(c).sum(), torch.tensor(float(sum(len(x) for x in c)), device=self.dev)]) \
                if c else torch.zeros(2, device=self.dev)
            parallel.allreduce_sum((tot,), self.world)
            avgc = float((tot[0] / tot[1]).item()) if float(tot[1].item()) > 0 else float("nan")
            if math.isnan(avgc):
                print("Epoch {}: NaN error!".format(str(epoch)))
                self.error_during_train = True
                return
            print("\tloss: {:.6f}".format(avgc))
            if test_data is not None:
                recall = self.test(sess, test_data, args)
                if recall > threshold_acc and args.get("save"):
                    from .util import save_model
                    print("Model saved - {}".format(save_model(self, args)))

    def test(self, sess, test_data, args):
        """model_combine.py:254-315.  Under torchrun the catalog is sharded across the ranks AND every rank evaluates
        its own batches (eval_round: batch i goes to rank i mod world); the metric sums are then reduced over the
        ranks, so every rank prints / returns the metrics of the whole test set."""
        print("Measuring...")
        self.sync_item_table()
        acc = {"mrr": [], "recall": [], "ndcg": [], "ild": [], "unexp": [], "loss": [], "items": {}}
        sampler = self._eval_sampler(test_data)         # the producer thread packs only this rank's batches
        dist_on = parallel.is_distributed(self.world)
        batch = 0

        def consume(packed, B, T, top, ngt, ce):
            nonlocal batch
            batch += 1
            batch_in = packed[: B * T].reshape(B, T).tolist()
            batch_out = packed[7 * B * T + 2 * B: 7 * B * T + 3 * B].tolist()
            top, ngt, ce = top.get().numpy(), ngt.get().numpy(), ce.get().numpy()
            if batch < 3:
                print("batch_in:", batch_in[0])
                print("batch_out:", batch_out[0])
                print("batch pred:", top[0][:10].tolist())
            ranks = ngt.astype(np.int64) + 1                                    # util.py:14
            hit = ranks <= 20
            acc["recall"] += hit.tolist()
            acc["mrr"] += np.where(hit, 1.0 / ranks, 0.0).tolist()
            acc["ndcg"] += np.where(hit, 1.0 / np.log2(ranks + 1.0), 0.0).tolist()
            acc["loss"] += ce.tolist()
            batch_pred = [[int(x) for x in row if x >= 0] for row in top]
            for idx, pred in enumerate(batch_pred):
                if self.category_id is not None and len(pred) > 1:
                    acc["ild"].append(self.getILD(pred))
                    acc["unexp"].append(self.getUnexp(batch_in[idx], pred))
                for pi in pred:
                    acc["items"][pi] = acc["items"].get(pi, 0) + 1
            if args.get("is_print"):
                self.printData(str(args["foldnum"]) + "_" + str(self.curEpoch), batch_in, batch_out, batch_pred)

        staged = ((packed, B, T, self.stage_to_device(packed, B, T, Nn)) for packed, B, T, Nn in prefetch_packed(sampler))
        if dist_on:
            # round r evaluates batches r * R ... r * R + R - 1, one per rank; a rank without a batch in the last round
            # still takes part in its collectives with B = 0
            R, me, sizes = self.world, self.rank, sampler.global_sizes

            def rounds():
                for r in range(0, len(sizes), R):
                    counts = [sizes[r + g] if r + g < len(sizes) else 0 for g in range(R)]
                    if counts[me]:
                        yield counts, next(staged)
                    else:
                        T = sampler.batch_T[0]
                        yield counts, (None, 0, T, Batch(torch.zeros(0, device=self.dev, dtype=torch.int32), 0, T, 0))

            def launch(cur, nxt):
                counts, (packed, B, T, bt) = cur
                top, ngt, ce = self.eval_round(bt, counts)
                return (packed, B, T, *[self.fetch_async(x) for x in (top, ngt, ce)]) if B else None

            pipelined(rounds(), launch, consume)
        else:
            def launch(cur, nxt):
                packed, B, T, bt = cur
                top, ngt, ce = self.eval_step(bt, next_bt=nxt[3] if nxt is not None else None)
                return (packed, B, T, *[self.fetch_async(x) for x in (top, ngt, ce)])

            pipelined(staged, launch, consume)
        sums = np.array([np.sum(acc["loss"]), len(acc["loss"]), np.sum(acc["ild"]), len(acc["ild"]), np.sum(acc["unexp"]),
                         np.sum(acc["mrr"]), np.sum(acc["recall"]), np.sum(acc["ndcg"])], dtype=np.float64)
        sums = self._sum_over_ranks(sums)
        coverage = len(acc["items"])
        if dist_on:
            import torch.distributed as dist
            seen = torch.zeros(self.N, device=self.dev, dtype=torch.int32)
            if acc["items"]:
                seen[torch.tensor(list(acc["items"].keys()), device=self.dev, dtype=torch.long)] = 1
            dist.all_reduce(seen, op=dist.ReduceOp.MAX)
            coverage = int(seen.sum().item())
        n = max(sums[1], 1.0)
        self.last_metrics = {"loss": float(sums[0] / n), "ild": float(sums[2] / sums[3]) if sums[3] else 0.0,
                             "unexp": float(sums[4] / sums[3]) if sums[3] else 0.0, "coverage": coverage,
                             "mrr": float(sums[5] / n), "recall": float(sums[6] / n), "ndcg": float(sums[7] / n)}
        print("avg loss...", self.last_metrics["loss"])
        print("avg ILD...", self.last_metrics["ild"])
        print("avg unexp...", self.last_metrics["unexp"])
        print("len of result dict: ", coverage)
        print("MRR@20: {}, Recall@20: {}, nDCG@20: {}".format(self.last_metrics["mrr"], self.last_metrics["recall"],
                                                                self.last_metrics["ndcg"]))
        return self.last_metrics["recall"]
