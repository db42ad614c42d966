"""Catalog-sharded TCAR train step (SURVEY 8e row 2, 8f-3): the softmax over the N candidates is split across ranks.

The data-parallel step of model_combine.Seq2SeqAttNN.train_step all-reduces the dense item gradient (364 MB at the
Globo shape) and repeats the table-wide Adam pass (2.7 GB of HBM traffic) on every rank.  Here every rank OWNS a
contiguous range of items -- the rows of the bf16 scoring operand, the fp32 master rows, their Adam moments and their
gradient -- and the step exchanges only session-sized tensors:

    all-gather   packed batch ids                 (orders the owners' previous update before the row fetch below)
    peer loads   item rows of the rank's own sessions, straight from the owners' HBM      (tcar_peer_fetch_rows)
    all-gather   Q [512,640] bf16 + label scores c [512]          -> every rank scores ALL sessions against its range
    all-reduce   softmax partial sums [R,512]                     (model_combine.py:145: CE = log sum exp(S - c))
    reduce-scat. dQ partials [R,512,640] fp32                     -> each rank keeps its own sessions' dQ
    all-gather   Qs = a_ic / sumexp [512,256] bf16                -> dense item gradient of the owned rows, complete
    all-gather   a_ic, coef, dXi of every rank's sessions         -> each owner applies the sparse rows it owns
    all-reduce   gradients of the 22 small tensors + the squared norm of the item gradient (per-tensor clip_by_norm,
                 model_combine.py:158-160, needs the norm of the WHOLE item gradient)

and then runs clip + Adam on its own rows only.  Same function as the single-GPU step (the sums over sessions and over
items are merely regrouped); verified against it by tools/dist_check.py and tests/test_gpu_parity.py.

`Seq2SeqAttNN(args)` with args["train_parallel"] == "catalog" enables it; `train_step_catalog(bt, counts)` is the
step, `sync_item_table()` re-assembles the full fp32 table + scoring operand on every rank (before evaluation, export
or a checkpoint).  With world_size == 1, args["catalog_virtual_shards"] = V makes the single process own V shards and
walk them one after the other -- the same kernels with the same shard offsets, used by the single-GPU parity test.
"""
import ctypes as C

import torch

from . import _native as nv
from . import parallel
from .params import SMALL

H, XW, KEXT, QROWS, HP = nv.H, nv.XW, nv.KEXT, nv.QROWS, nv.HP
Q_BYTES = QROWS * KEXT * 2                 # bf16 query operand
QC_BYTES = Q_BYTES + QROWS * 4             # + fp32 label scores
PAY_HEAD = QROWS * XW + QROWS              # a_ic [512,500] + coef [512] floats in front of dXi


class CatalogShardedTraining:
    """Mixin of Seq2SeqAttNN (needs its workspaces and kernels wrappers)."""

    # ------------------------------------------------------------------------------------------- set-up
    def enable_catalog_training(self, virtual_shards=1):
        dev, ps = self.dev, self.ps
        self._cat_dist = parallel.is_distributed(self.world)
        if self.world > 1 and not self._cat_dist:
            raise RuntimeError("catalog-sharded training needs an initialised torch.distributed process group")
        R = self.world if self._cat_dist else 1
        if R > nv.MAX_PEERS:
            raise ValueError(f"at most {nv.MAX_PEERS} ranks")
        self._cat_R = R
        nshards = R if self._cat_dist else max(1, int(virtual_shards))
        bounds = parallel.shard_bounds(ps.N, ps.n_pad, nshards)
        self._cat_row_bounds = parallel.catalog_row_bounds(bounds, ps.N)        # table rows, [nshards + 1]
        mine = [self.rank] if self._cat_dist else list(range(nshards))
        self._cat_shards = []
        for s in mine:
            lo, hi = bounds[s]
            n_pad = max((hi - lo + 255) // 256 * 256, 256)
            self._cat_shards.append({"lo": lo, "hi": hi, "n_pad": n_pad, "iext": ps.iext[lo: lo + n_pad],
                                     "row_lo": self._cat_row_bounds[s], "row_hi": self._cat_row_bounds[s + 1]})
        # exchange buffers; the kernels keep writing self.Q / self.c_ref / self.a_ic / self.coef / self.dXi, which now
        # alias the send buffers of the collectives (no packing kernels)
        self._qc = torch.zeros(QC_BYTES, device=dev, dtype=torch.uint8)
        self.Q = self._qc[:Q_BYTES].view(torch.bfloat16).view(QROWS, KEXT)
        self.c_ref = self._qc[Q_BYTES:].view(torch.float32)
        self._qc_all = torch.zeros(R, QC_BYTES, device=dev, dtype=torch.uint8) if R > 1 else self._qc.view(1, -1)
        self._pay = torch.zeros(PAY_HEAD + QROWS * nv.MAXT * HP, device=dev)
        self.a_ic = self._pay[: QROWS * XW].view(QROWS, XW)
        self.coef = self._pay[QROWS * XW: PAY_HEAD]
        self.dXi = self._pay[PAY_HEAD:].view(QROWS * nv.MAXT, HP)
        self._pay_all = None
        self._ids = torch.zeros(1, device=dev, dtype=torch.int32)
        self._ids_all = torch.zeros(1, device=dev, dtype=torch.int32)
        # look-ahead across ranks (opt-in, TCAR_CATALOG_LOOKAHEAD=1; see train_step_catalog): the NEXT batch's ids are
        # gathered one step early into the second buffer pair
        import os
        self.cat_lookahead = os.environ.get("TCAR_CATALOG_LOOKAHEAD", "0") == "1"
        self._ids_n = torch.zeros(1, device=dev, dtype=torch.int32)
        self._ids_all_n = torch.zeros(1, device=dev, dtype=torch.int32)
        self._cat_pre = None               # {"bt", "counts", "L"} of the batch whose ids / rows / forward are ahead
        self._bar = torch.zeros(1, device=dev)
        self._sumexp_all = torch.zeros(R, QROWS, device=dev)
        self._rowmax_all = torch.zeros(R, QROWS, device=dev)          # largest exponent argument of every session row
        self._rowmax_tmp = torch.zeros(R, QROWS, device=dev) if len(self._cat_shards) > 1 else None
        self._dq_all = torch.zeros(R, QROWS, KEXT, device=dev)
        self._qs_all = torch.zeros(R, QROWS, HP, device=dev, dtype=torch.bfloat16) if R > 1 else self.Qs.view(1, QROWS, HP)
        self._dq_tmp = torch.zeros(R, QROWS, KEXT, device=dev) if len(self._cat_shards) > 1 else None
        self._sq_tmp = torch.zeros(1, device=dev)
        # one all-reduce carries [theta_g | squared norm of the owned item-gradient rows]: the small-tensor gradients
        # now live at the front of that buffer (the kernels write them through ps.g / ps.theta_g as before)
        self._red = torch.zeros(ps.flat_size + 4, device=dev)
        ps.theta_g = self._red[: ps.flat_size]
        ps.g = {n: ps._view(ps.theta_g, i) for i, (n, _) in enumerate(SMALL)}
        self._sq_slot = self._red[ps.flat_size: ps.flat_size + 1]
        self._cat_trace = None          # tools/catalog_probe.py: list collecting (phase name, CUDA event)
        for sh in self._cat_shards:
            tiles = nv.lib().tcar_score_fwd_tiles(sh["n_pad"])
            sh["tiles"] = tiles
            # one E / partial-sum block per session group, a fixed stride apart (tcar_score_*_groups)
            sh["E"] = torch.zeros(R, QROWS * sh["n_pad"], device=dev, dtype=torch.bfloat16)
            sh["part"] = torch.zeros(R, tiles * QROWS, device=dev)
            sh["pmax"] = torch.zeros(R, tiles * QROWS, device=dev)          # softmax overflow guard, pass 1
            splits = max(nv.lib().tcar_score_bwd_q_splits(b, sh["n_pad"]) for b in (1, 129, 257, 385))
            qelems = splits * QROWS * KEXT
            if R > 1:
                qelems = max(qelems, int(nv.lib().tcar_score_bwd_q_multi_part_elems(R)))
            sh["qpart"] = torch.zeros(qelems, device=dev)
            sh["ctas"] = nv.lib().tcar_score_bwd_i_ctas(sh["n_pad"])
            sh["sqp"] = torch.zeros(sh["ctas"], device=dev)
        self._slot_sq_g = None
        # peer pointers of the fp32 item table (single node, CUDA IPC): exported once, opened once
        self._peer_ptrs = (C.c_void_p * nv.MAX_PEERS)()
        self._peer_ptrs[self.rank if self._cat_dist else 0] = ps.item_full.data_ptr()
        self._peer_bounds = (C.c_int32 * (nv.MAX_PEERS + 1))(*self._cat_row_bounds) if self._cat_dist else None
        self._peer_opened = []
        if self._cat_dist:
            self._open_peers()
        self._item_table_synced = True
        self.train_parallel = "catalog"

    def _open_peers(self):
        """Export the own fp32 item table and open every other rank's (CUDA IPC).  All ranks agree on the outcome before
        anyone raises, so that a node without peer access fails cleanly instead of hanging in a later collective."""
        import torch.distributed as dist
        err = None
        handle = (C.c_ubyte * nv.PEER_HANDLE_BYTES)()
        off = C.c_longlong(0)
        rc = nv.lib().tcar_peer_export(C.c_void_p(self.ps.item_full.data_ptr()), handle, C.byref(off))
        if rc != 0:
            err = (f"tcar_peer_export failed with code {rc} (cudaIpcGetMemHandle; the item table must live in a plain "
                   "cudaMalloc block -- PYTORCH_CUDA_ALLOC_CONF=expandable_segments is not supported)")
        everyone = [None] * self.world
        dist.all_gather_object(everyone, (bytes(handle), int(off.value), rc))
        for g, (hb, o, rc_g) in enumerate(everyone):
            if g == self.rank or rc_g != 0 or err is not None:
                continue
            out = C.c_void_p()
            rc = nv.lib().tcar_peer_open((C.c_ubyte * nv.PEER_HANDLE_BYTES).from_buffer_copy(hb), o, C.byref(out))
            if rc != 0 or not out.value:
                err = (f"tcar_peer_open(rank {g}) failed with code {rc}: catalog-sharded training needs CUDA IPC peer "
                       "access between the GPUs of the node")
                break
            self._peer_ptrs[g] = out.value
            self._peer_opened.append((out.value, o))
        bad = torch.tensor([0 if err is None else 1], device=self.dev, dtype=torch.int32)
        dist.all_reduce(bad, op=dist.ReduceOp.MAX)
        if int(bad.item()):
            self.close_peers()
            raise nv.TcarNativeError(err or "another rank could not export / open the peer item tables")

    def close_peers(self):
        for ptr, off in getattr(self, "_peer_opened", ()):     # data-parallel models never opened any
            nv.lib().tcar_peer_close(C.c_void_p(ptr), off)
        self._peer_opened = []

    # ------------------------------------------------------------------------------------------- the step
    def _fetch_rows(self, bt):
        """Item rows this rank's sessions read (clicks, labels, negatives) from their owners' HBM."""
        p = nv.ptr
        nv.LAUNCHES["count"] += 1
        rc = nv.lib().tcar_peer_fetch_rows(p(bt.seq), p(bt.label), p(bt.neg), bt.B, bt.T, bt.Nn, self._peer_ptrs,
                                           self._peer_bounds, self._cat_R, self.rank, p(self.ps.item_full),
                                           nv.stream_ptr())
        if rc != 0:
            raise nv.TcarNativeError(f"tcar_peer_fetch_rows failed with code {rc}")

    def _gather(self, out_flat, inp_flat):
        """all_gather_into_tensor on flat views: out = [rank 0 | rank 1 | ...]."""
        import torch.distributed as dist
        dist.all_gather_into_tensor(out_flat, inp_flat)

    def train_step_catalog(self, bt, counts=None, next_bt=None, next_counts=None):
        """One train step with the catalog sharded across ranks.  bt = this rank's sessions (B may be 0 for a tail
        batch); counts[g] = sessions of rank g in this step (default: bt.B on every rank) -- all ranks must pass the
        same list, and the same T / Nn.  Returns this rank's loss [B].

        next_bt / next_counts (used when self.cat_lookahead): the batch of the FOLLOWING call.  Its packed ids are
        all-gathered at the end of this step, every owner first updates the rows those ids name (tcar_adam_item_rows_
        groups on its own range), one barrier later the rest of the owned rows is updated on the side stream while the
        peer loads and the session forward of next_bt run on the high-priority stream -- the look-ahead of
        Seq2SeqAttNN.train_step, across ranks.  Same arithmetic per row whichever kernel applies it."""
        import torch.distributed as dist
        ps, p = self.ps, nv.ptr
        R, me, on = self._cat_R, (self.rank if self._cat_dist else 0), self._cat_dist
        B, T, Nn = bt.B, bt.T, bt.Nn
        counts = [B] * R if counts is None else [int(c) for c in counts]
        if len(counts) != R or counts[me] != B:
            raise ValueError("counts must list the sessions of every rank (and counts[rank] == bt.B)")
        Bmax = max(counts)
        if Bmax == 0:
            return self.loss[:0]
        pre, self._cat_pre = self._cat_pre, None
        ahead = pre is not None and pre["bt"] is bt and pre["counts"] == counts
        self.sync_updates()                # pending table-wide Adam (side stream) / prefetched forward (ahead stream)
        self._prefetched = None
        self._item_table_synced = False
        ps.version += 1
        groups = [g for g in range(R) if counts[g] > 0]
        trace = self._cat_trace

        def mark(name):
            if trace is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                trace.append((name, ev))

        mark("start")
        L = 7 * Bmax * T + 3 * Bmax + Bmax * Nn
        # ---- packed ids of every rank (sparse-row scatter below); as the first collective of the step it also orders
        # every owner's previous Adam pass before the peer loads
        if ahead:
            # ids gathered, rows fetched and session forward launched by the previous call: take over its ids buffers
            self._ids, self._ids_n = self._ids_n, self._ids
            self._ids_all, self._ids_all_n = self._ids_all_n, self._ids_all
        else:
            if on:
                self._gather_ids(bt, L, False)
                if B > 0:
                    self._fetch_rows(bt)
        mark("ids+fetch")
        # ---- session forward of the local sessions -> Q, c_ref (views of the send buffer)
        if B > 0 and not ahead:
            self._session_forward(bt)
        mark("session_fwd")
        if B > 0:
            nv.counted_call("tcar_neg_loss", 1, p(self.a_ic), p(ps.item), p(ps.content), p(bt.neg), None,
                            p(self.negloss), p(self.loss), p(self.coef), p(self.dA_neg), B, Nn)
        if on:
            self._gather(self._qc_all.view(-1), self._qc)
        mark("gather_q")
        # ---- every session group against every owned item range (one call per phase and shard: the loops over the
        # groups are in the library)
        cnt = (C.c_int * R)(*counts)
        ng = len(groups)
        qc_ptr = self._qc_all.data_ptr()
        shards = [sh for sh in self._cat_shards if sh["hi"] > sh["lo"]]
        multi = len(self._cat_shards) > 1
        guard = self.softmax_guard

        def score_fwd(sh, pmax, rowmax):
            nv.counted_call("tcar_score_fwd_groups_guarded", ng, C.c_void_p(qc_ptr), QC_BYTES // 2,
                            C.c_void_p(qc_ptr + Q_BYTES), QC_BYTES // 4, p(sh["iext"]), p(sh["E"]), QROWS * sh["n_pad"],
                            p(sh["part"]), sh["tiles"] * QROWS, pmax, rowmax, cnt, R, sh["hi"] - sh["lo"], sh["n_pad"],
                            self._cluster_for(Bmax))

        for k, sh in enumerate(shards):
            score_fwd(sh, p(sh["pmax"]) if guard else None, None)
            if guard:
                dst = self._rowmax_all if k == 0 else self._rowmax_tmp
                nv.counted_call("tcar_rowmax_groups", 1, p(sh["pmax"]), sh["tiles"] * QROWS, p(dst), sh["tiles"], cnt, R)
                if k > 0:
                    torch.maximum(self._rowmax_all, self._rowmax_tmp, out=self._rowmax_all)
        if guard:
            # overflow guard of the softmax (TCAR_EXP_LIMIT2): every owner must shift a session row by the same amount,
            # so the row maxima are reduced over the ranks; pass 2 is `ng` empty launches unless a row is above the limit
            if on:
                dist.all_reduce(self._rowmax_all, op=dist.ReduceOp.MAX)
            for sh in shards:
                score_fwd(sh, None, p(self._rowmax_all))
        mark("score_fwd")
        # ---- dQ partial sums over the owned items for every group; the softmax partial sums travel in the zero pad
        # column of dQ, so ONE reduce-scatter hands both to the sessions' ranks (model_combine.py:145: CE = log sum)
        for k, sh in enumerate(shards):
            dst = self._dq_all if k == 0 else self._dq_tmp
            # launches: one GEMM + one split reduction over all groups (per group when only one is present) + one
            # partial-sum kernel per group
            nv.counted_call("tcar_score_bwd_q_groups", 2 + ng if ng > 1 else 3, p(sh["E"]), QROWS * sh["n_pad"], p(sh["iext"]),
                            p(sh["qpart"]), p(dst), QROWS * KEXT, p(sh["part"]), sh["tiles"] * QROWS, sh["tiles"], cnt, R,
                            sh["n_pad"])
            if k > 0:
                self._dq_all += self._dq_tmp
        mark("score_bwd_q")
        if on:
            dist.reduce_scatter_tensor(self.dq_raw, self._dq_all, op=dist.ReduceOp.SUM)
            dq_raw = self.dq_raw
        else:
            dq_raw = self._dq_all[0]
        if B > 0:
            # CE = log(sum) (+ shift ln 2 for rows the guard shifted) from the strided sums column
            nv.counted_call("tcar_ce_from_sums", 1, p(dq_raw[:, KEXT - 1:]), KEXT,
                            p(self._rowmax_all[me]) if guard else None, p(self.sumexp), p(self.ce), B)
            nv.counted_call("tcar_loss_combine", 1, p(self.ce), p(self.negloss), p(self.loss), B)
            nv.counted_call("tcar_score_bwd_finish", 1, p(dq_raw), p(self.sumexp), p(self.dA_neg), p(self.a_ic),
                            p(ps.ct_tab), p(ps.item), p(ps.content), p(ps.mwdhm), p(bt.label), p(self.d_a_ic),
                            p(self.d_a_pt), p(self.dTq), p(self.Qs), B)
        mark("loss+finish")
        # Collectives are overlapped with chains of short kernels only, never with the persistent GEMMs: an NCCL kernel
        # that gets a few SMs first delays the GEMM CTAs bound to them by its whole duration (static tile schedule)
        w_qs = dist.all_gather_into_tensor(self._qs_all.view(-1), self.Qs.view(-1), async_op=True) if on else None
        # ---- session-side backward of the local sessions (beside the all-gather of Qs)
        if B > 0:
            self._session_backward(bt)
        else:
            ps.theta_g.zero_()
        mark("session_bwd")
        n_pay = PAY_HEAD + Bmax * T * HP
        if on:
            if self._pay_all is None or self._pay_all.numel() < R * n_pay:
                self._pay_all = torch.zeros(R * n_pay, device=self.dev)
            w_qs.wait()
            self._gather(self._pay_all[: R * n_pay], self._pay[:n_pay])
            ids_ptr, ids_stride, pay_ptr, pay_stride = self._ids_all.data_ptr(), L, self._pay_all.data_ptr(), n_pay
        else:
            ids_ptr, ids_stride, pay_ptr, pay_stride = bt.buf.data_ptr(), 0, self._pay.data_ptr(), 0
        mark("gather_payload")
        # ---- dense gradient of the owned item rows: complete after the last group (sum over ALL sessions)
        for sh in shards:
            # the kernel writes table row n + 1 for local item n
            nv.counted_call("tcar_score_bwd_i_groups", ng, p(sh["E"]), QROWS * sh["n_pad"], p(self._qs_all), QROWS * HP,
                            p(ps.item_g_full[sh["lo"]:]), p(sh["sqp"]), cnt, R, sh["hi"] - sh["lo"], sh["n_pad"])
        mark("score_bwd_i")
        # ---- the sparse rows (clicks, labels, negatives) of every rank's sessions that fall into the owned ranges
        # all source ranks against ONE hash table (tcar_scatter_add_rows_multi: three launches per step instead of
        # three per source rank)
        merged = ng > 1
        ent = Bmax * T + Bmax + Bmax * Nn
        self._alloc_scatter(R * ent if merged else ent)
        nsq = self.hash_size if merged else R * self.hash_size
        if self._slot_sq_g is None or self._slot_sq_g.numel() != nsq:
            self._slot_sq_g = torch.zeros(nsq, device=self.dev)
        if multi:
            self._sq_slot.zero_()
        for sh in self._cat_shards:
            if sh["row_hi"] <= sh["row_lo"]:
                continue
            nv.counted_call("tcar_scatter_add_rows_multi" if merged else "tcar_scatter_add_rows_groups",
                            3 if merged else 3 * ng, C.c_void_p(ids_ptr), ids_stride, C.c_void_p(pay_ptr),
                            pay_stride, p(ps.item), p(ps.item_g), p(self.hash_keys), p(self.hash_cnt), p(self.hash_acc),
                            p(self.entry_slot), p(self._slot_sq_g), self.hash_size, cnt, R, T, Nn, sh["row_lo"],
                            sh["row_hi"])
            # squared norm of the owned gradient rows without re-reading them: per-CTA sums of the dense GEMM (last
            # group = accumulated values) + the per-slot corrections of the scatter passes
            dense = sh["hi"] > sh["lo"]
            nv.counted_call("tcar_update_norms", 1, None, None, None, 0, p(sh["sqp"]) if dense else None,
                            sh["ctas"] if dense else 0, p(self._slot_sq_g), nsq,
                            p(self._sq_tmp if multi else self._sq_slot), p(ps.norm_partial), p(ps.norm_ticket), None)
            if multi:
                self._sq_slot += self._sq_tmp
        mark("scatter+norm")
        # ---- [small-tensor gradients | item-gradient norm] summed over ranks; per-tensor clip + Adam (model_combine.py:
        # 155-163) on the replicated small tensors and on the owned item rows
        if on:
            dist.all_reduce(self._red, op=dist.ReduceOp.SUM)
        mark("allreduce")
        nv.counted_call("tcar_sqnorm_segments", 1, p(ps.theta_g), p(ps.seg_off), p(ps.sqnorm_small), len(SMALL))
        ps.step.add_(1)
        self.global_step += 1
        self._update_small()
        look = (self.cat_lookahead and next_bt is not None and self.adam_overlap_ctas > 0 and next_bt.T >= 1)
        if look:
            ncounts = [next_bt.B] * R if next_counts is None else [int(c) for c in next_counts]
            look = len(ncounts) == R and ncounts[me] == next_bt.B and max(ncounts) > 0
        flags = None
        if look:
            # (a) the next step's ids, one step early; (b) the rows they name inside the owned ranges first
            nBmax, nT, nNn = max(ncounts), next_bt.T, next_bt.Nn
            nL = 7 * nBmax * nT + 3 * nBmax + nBmax * nNn
            if on:
                self._gather_ids(next_bt, nL, True)
                nids_ptr, nids_stride = self._ids_all_n.data_ptr(), nL
            else:
                nids_ptr, nids_stride = next_bt.buf.data_ptr(), 0
            ncnt = (C.c_int * R)(*ncounts)
            flags = ps.row_flags
            for sh in self._cat_shards:
                if sh["row_hi"] <= sh["row_lo"]:
                    continue
                nv.counted_call("tcar_adam_item_rows_groups", 2 * sum(1 for c in ncounts if c > 0), p(ps.item_full),
                                p(ps.item_m_full), p(ps.item_v_full), p(ps.item_g_full), p(self._sq_slot), p(ps.step),
                                self.lr, self.max_grad_f, p(ps.iext), C.c_void_p(nids_ptr), nids_stride, ncnt, R, nT,
                                nNn, p(flags), sh["row_lo"], sh["row_hi"])
            # (c) every owner has updated the rows anyone is about to load
            if on:
                dist.all_reduce(self._bar, op=dist.ReduceOp.SUM)
            main = torch.cuda.current_stream()
            fork = torch.cuda.Event()
            fork.record(main)
            self._side.wait_event(fork)
            self._ahead.wait_event(fork)
        # ---- the owned rows (all of them, or those not yet updated: on the side stream, beside the next forward)
        with torch.cuda.stream(self._side if look else torch.cuda.current_stream()):
            for sh in self._cat_shards:
                lo, n = sh["row_lo"], sh["row_hi"] - sh["row_lo"]
                if n <= 0:
                    continue
                nv.counted_call("tcar_adam_item", 1, p(ps.item_full[lo:]), p(ps.item_m_full[lo:]),
                                p(ps.item_v_full[lo:]), p(ps.item_g_full[lo:]), p(self._sq_slot), p(ps.step), self.lr,
                                self.max_grad_f, p(ps.iext), lo, n, p(flags) if look else None,
                                self.adam_overlap_ctas if look else 0)
            if look:
                done = torch.cuda.Event()
                done.record(self._side)
                self._update_done = done
        if look:
            # (d) peer loads + session forward of the next batch on the high-priority stream
            with torch.cuda.stream(self._ahead):
                if next_bt.B > 0:
                    if on:
                        self._fetch_rows(next_bt)
                    self._session_forward(next_bt, prefetch=True)
                adone = torch.cuda.Event()
                adone.record(self._ahead)
            self._ahead_done = adone
            self._cat_pre = {"bt": next_bt, "counts": ncounts, "L": nL}
        mark("adam")
        self._fused_norm = False
        return self.loss[:B]

    def _gather_ids(self, bt, L, nxt):
        """All-gather one packed batch (L int32 per rank, zero padded) into the current / the look-ahead ids buffers."""
        R = self._cat_R
        loc, allb = (self._ids_n, self._ids_all_n) if nxt else (self._ids, self._ids_all)
        if loc.numel() < L:
            loc = torch.zeros(L, device=self.dev, dtype=torch.int32)
            allb = torch.zeros(R * L, device=self.dev, dtype=torch.int32)
            if nxt:
                self._ids_n, self._ids_all_n = loc, allb
            else:
                self._ids, self._ids_all = loc, allb
        if bt.B > 0:
            loc[: bt.buf.numel()].copy_(bt.buf)
        self._gather(allb[: R * L], loc[:L])

    # ------------------------------------------------------------------------------------------- re-assembly
    def sync_item_table(self):
        """Every rank receives every owner's fp32 rows and rebuilds the whole bf16 scoring operand: evaluation, export
        and checkpoints read the full table.  A no-op when nothing was trained since the last call."""
        if getattr(self, "train_parallel", "dp") != "catalog" or self._item_table_synced:
            return
        self.sync_updates()
        if self._cat_dist:
            import torch.distributed as dist
            rb = self._cat_row_bounds
            for g in range(self._cat_R):
                if rb[g + 1] > rb[g]:
                    for t in (self.ps.item_full, self.ps.item_m_full, self.ps.item_v_full):
                        dist.broadcast(t[rb[g]: rb[g + 1]], src=g)
        self.ps.rebuild_iext()
        self._item_table_synced = True
