#!/usr/bin/env python
"""bench.py -- TCAR train sessions/s (+ full-catalog top-20 eval queries/s) on synthetic Globo-shaped data.

    python bench.py [--gpus N] [--steps K] [--warmup W]                  this repo's B200 path
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]  the reference's CPU arithmetic (oracle port)
    python bench.py ... --dump-outputs DIR                               also write the last timed step's results to DIR

One "step" = one `sess.run([loss, global_step, train_op])` of the reference (model_combine.py:231-234): forward,
losses, gradients, per-tensor clip and Adam over one length-bucketed batch of 512 sessions against the full
364 047-article catalog.  N>1 (torchrun, one rank per GPU): data-parallel, every rank owns a batch of 512 sessions
(weak scaling) and the gradients are summed with one NCCL all-reduce per step.  Rank 0 prints ONE JSON line.

Nothing here reads /root/reference.  oracle/ is executed only by the `cpu_baseline` leg and by `--impl reference`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GLOBO_N = 364047           # SURVEY 8d: Globo articles_metadata.csv row count
MIND_N = 103630            # SURVEY 8d cfg 4: articles_timeDict_103630.pkl (data_process/mind_preprocess.py:358)
ADRESSA_N = 20000          # SURVEY 8d cfg 5 (our choice; the reference does not ship Adressa statistics)
SHAPE = {"globo": ("Globo", GLOBO_N), "mind": ("MIND", MIND_N), "adressa": ("Adressa", ADRESSA_N)}
K_REF = 820                # scoring K of the reference graph (2H + 5Th, model_combine.py:132-136)
K_DITEM = 570              # columns of the candidate matrix that carry trainable parameters (250 item + 320 time)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--items", type=int, default=0, help="catalog size; 0 = the workload's (364 047 / 103 630 / 20 000)")
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--session_len", type=int, default=0,
                    help="clicks per session; 0 = SURVEY 8d mix: one length per batch drawn from P(T) ~ 0.55^T, "
                         "T in [1,20] (Globo-like, prefix-augmented sessions are short); 20 = the reference --maxlen")
    ap.add_argument("--neg_num", type=int, default=20)
    ap.add_argument("--negative_mode", default="uniform", choices=["uniform", "impression"],
                    help="negatives of the sampler-inclusive train_loop lines: uniform (what the reference ships, "
                         "sampler.py:98-99) or drawn from the sessions' impression lists (sampler.py:118-131, MIND)")
    ap.add_argument("--workload", default="globo", choices=["globo", "mind", "adressa"],
                    help="globo = BASELINE config 2/3 (default; what the driver measures); mind = config 4: MIND shape "
                         "(103 630 articles, impression-list negatives, neg_num sweep 20/50/100); adressa = config 5: "
                         "Adressa shape (20 000 articles), sweep over the session length T = 1..40")
    ap.add_argument("--train_parallel", default=os.environ.get("TCAR_TRAIN_PARALLEL", "catalog"),
                    choices=["dp", "catalog"],
                    help="multi-GPU training layout: catalog (default) = softmax sharded over the item catalog, only "
                         "session-sized exchanges (catalog_parallel.py); dp = data parallel + all-reduce of the dense "
                         "364 MB item gradient.  Ignored at --gpus 1")
    ap.add_argument("--no_cpu_baseline", action="store_true")
    ap.add_argument("--no_kernels", action="store_true", help="skip the per-kernel roofline pass")
    ap.add_argument("--no_lookahead", action="store_true",
                    help="call train_step(bt) without the next batch (no overlap of Adam with the next session forward)")
    ap.add_argument("--cpu_sample_sessions", type=int, default=512)
    ap.add_argument("--loop_sessions", type=int, default=32768,
                    help="sessions of the in-memory synthetic split used for the sampler-inclusive `train_loop` line")
    ap.add_argument("--profile_region", action="store_true",
                    help="for `ncu --profile-from-start off`: warm up, then ONE train step (T=20) and ONE eval step "
                         "between cudaProfilerStart/Stop; prints nothing")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed loops, write DIR/<name>.npy (float32 / float64): the loss and the updated "
                         "parameters (dense tensors, a fixed sample of item rows) of the last timed train step, the "
                         "top-20 ids, ranks and cross loss of the last timed eval step.  The inputs depend only on the "
                         "arguments, so two builds can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the results of the B200 path")
    if a.items <= 0:
        a.items = SHAPE[a.workload][1]
    if a.workload == "mind":
        a.negative_mode = "impression"
    return a


# ----------------------------------------------------------------------------------------------------- helpers
def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm": float(d["hbm_gbs"]), "tensor_burst": float(d["bf16_tflops"]),
                "tensor_sustained": float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "source": "measured"}
    return {"hbm": 6650.0, "tensor_burst": 1590.0, "tensor_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def wait_first(self, timeout=15.0):
        """Block until the first sample has arrived: nvidia-smi takes about a second to attach to every GPU of the box
        and holds driver locks meanwhile -- a timed loop whose HOST is on the critical path (the e2e loops) must not
        overlap that start-up (it cost 0.7 ms per step on a 20-step loop, measured: tools/e2e_probe.py is clean)."""
        t0 = time.perf_counter()
        while self.proc is not None and not self.lines and time.perf_counter() - t0 < timeout:
            time.sleep(0.05)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # "under load" = samples in the upper half of the observed power range
        thr = (max(pw) + min(pw)) / 2
        load = [s for s, p in zip(sm, pw) if p >= thr] or sm
        load.sort()
        return {"sm_mhz": load[len(load) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw),
                "samples": len(sm), "reasons": sorted(reasons)}


NBATCH = 16


def session_lengths(a, n=NBATCH):
    """One session length per length-bucketed batch (sampler.py:40-49 buckets by exact length)."""
    import numpy as np
    if a.session_len > 0:
        return [a.session_len] * n
    rs = np.random.RandomState(2020)
    pr = 0.55 ** np.arange(1, 21)
    return [int(t) for t in rs.choice(np.arange(1, 21), size=n, p=pr / pr.sum())]


def make_batches(synth, N, B, Ts, Nn, mwdhm, seed0):
    import torch
    out = []
    for i, T in enumerate(Ts):
        packed = synth.make_index_batch(N, B, T, Nn, mwdhm, seed=seed0 + i)
        out.append(torch.from_numpy(packed).pin_memory() if torch.cuda.is_available() else torch.from_numpy(packed))
    return out


# ----------------------------------------------------------------------------------------------------- CPU arms
def oracle_train_rate(N, B, Ts, Nn, steps, warmup, content, mwdhm, seed=11):
    """Times the CPU oracle's train step (fwd + bwd + clip + TF-Adam, fp32, all host threads) on batches of B
    sessions against the full N-item catalog.  Returns (sessions/s, ms/step, threads)."""
    import numpy as np
    import torch
    from oracle import tcar_oracle as O
    from tcar_b200 import synth
    torch.set_num_threads(os.cpu_count() or 1)
    p = O.init_params(N)
    adam = O.TFAdam(p, 0.001)
    c = torch.from_numpy(content)
    mw = torch.from_numpy(mwdhm.astype(np.int64))
    batches = []
    for i in range(min(steps, len(Ts))):
        packed = synth.make_index_batch(N, B, Ts[i], Nn, mwdhm, seed=seed + i)
        batches.append({k: torch.from_numpy(v) for k, v in synth.unpack(packed, B, Ts[i], Nn).items()})
    for i in range(warmup):
        O.train_step(p, adam, c, mw, batches[-1 - i % len(batches)])
    t0 = time.perf_counter()
    for i in range(steps):
        O.train_step(p, adam, c, mw, batches[i % len(batches)])
    dt = time.perf_counter() - t0
    return B * steps / dt, dt / steps * 1e3, torch.get_num_threads()


def oracle_eval_rate(N, B, T, steps, content, mwdhm, seed=17):
    """The reference's eval iteration (model_combine.py:283-301): scores, cau_metrics, argsort top-20."""
    import numpy as np
    import torch
    from oracle import tcar_oracle as O
    from tcar_b200 import synth
    p = O.init_params(N)
    c = torch.from_numpy(content)
    mw = torch.from_numpy(mwdhm.astype(np.int64))
    packed = synth.make_index_batch(N, B, T, 0, mwdhm, seed=seed)
    batch = {k: torch.from_numpy(v) for k, v in synth.unpack(packed, B, T, 0).items()}
    t0 = time.perf_counter()
    for _ in range(steps):
        with torch.no_grad():
            S = O.forward(p, c, mw, batch)["softmax_input"].numpy()
        O.cau_metrics(S, batch["label"].numpy(), 20)
        [np.argsort(r)[::-1][:20] for r in S]
    dt = time.perf_counter() - t0
    return B * steps / dt


def run_reference(a):
    """`--impl reference`: the reference's own implementation is a TensorFlow-1 graph that cannot run here (no
    TensorFlow, and model_combine.py:113/115 is a SyntaxError), so this arm times the oracle port of its arithmetic on
    the host cores, on the same workload config; each step is a bounded sample of `cpu_sample_sessions` sessions."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import __graft_entry__ as ge
    ge.load_package()
    from tcar_b200 import synth
    content, mwdhm, _ = synth.make_catalog(a.items)
    Bs = a.cpu_sample_sessions
    Ts = session_lengths(a)
    rate, ms, threads = oracle_train_rate(a.items, Bs, Ts, a.neg_num, a.steps, a.warmup, content, mwdhm)
    sample = (f"{a.steps} train steps of {Bs} sessions (session lengths {Ts[:min(a.steps, len(Ts))]}, Nn={a.neg_num}) "
              f"against the full {a.items}-item catalog, torch CPU fp32")
    line = {"impl": "reference", "metric": f"TCAR train sessions/sec ({SHAPE[a.workload][0]} shape)", "value": rate,
            "unit": "sessions/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(a, 1),
            "cpu_baseline": {"value": rate, "unit": "sessions/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": "sessions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def workload_config(a, world):
    Ts = session_lengths(a)
    tdesc = (f"session length {a.session_len} for every batch" if a.session_len > 0 else
             f"one session length per batch drawn from P(T)~0.55^T on [1,20] (SURVEY 8d; cycle {Ts})")
    extra = {"mind": "; sampler-inclusive lines draw impression-list negatives (sampler.py:118-131), neg_sweep = "
                     "neg_num 20 / 50 / 100",
             "adressa": "; len_sweep = every batch at T = 1, 2, 4, 8, 16, 20, 30, 40 (position table limit, "
                        "model_combine.py:57)"}.get(a.workload, "")
    return {"workload": f"TCAR train step, {SHAPE[a.workload][0]} shape: {a.items} articles x 250-d content, batch "
                        f"{a.batch} sessions/GPU, {tdesc}, {a.neg_num} negatives{extra}",
            "name": a.workload,
            "items": a.items, "batch_per_gpu": a.batch, "global_batch": a.batch * world,
            "session_len": a.session_len if a.session_len > 0 else "mix", "mean_session_len": sum(Ts) / len(Ts),
            "neg_num": a.neg_num,
            "parallelism": (f"catalog{world} (softmax sharded over the item catalog, sessions of all ranks scored by every "
                            f"rank; catalog_parallel.py)" if getattr(a, "train_parallel", "dp") == "catalog" else
                            f"dp{world}") if world > 1 else "single",
            "l2": "inputs larger than L2: bf16 candidate matrix %d MB, E %d MB, item table + grad + Adam moments "
                  "4 x %d MB streamed every step (L2 = 126 MB)" % (a.items * 640 * 2 >> 20, a.items * 1024 >> 20,
                                                                  a.items * 1024 >> 20)}


# ----------------------------------------------------------------------------------------------------- B200 arm
DUMP_ITEM_ROWS = 4096      # item-table rows in the dump: a fixed sample keeps it at 4 MB instead of the 364 MB table
DUMP_MAX_BYTES = 64 << 20


def train_outputs(model, loss):
    """What a caller of train_step holds after its last call, on the host: the returned per-session loss and the
    updated parameters (every dense tensor, and the item-table rows of a fixed seeded sample with their ids)."""
    import numpy as np
    import torch
    from tcar_b200.params import H
    ps = model.ps
    rows = np.sort(np.random.RandomState(7).choice(ps.N + 1, min(DUMP_ITEM_ROWS, ps.N + 1), replace=False))
    out = {"train_loss": loss.float().cpu().numpy(), "item_row_ids": rows.astype(np.float64),
           "item_rows": ps.item.index_select(0, torch.from_numpy(rows).to(ps.item.device))[:, :H].cpu().numpy()}
    for name, t in ps.w.items():
        out["param_" + name] = t.cpu().numpy()
    return out


def eval_outputs(top, ngt, ce):
    """What eval_step / eval_round returned, on the host; the integer results as float64 (exact)."""
    import numpy as np
    return {"eval_top20_ids": top.cpu().numpy().astype(np.float64),
            "eval_n_greater": ngt.cpu().numpy().astype(np.float64), "eval_cross_loss": ce.float().cpu().numpy()}


def dump_outputs(path, arrays):
    """DIR/<name>.npy per array, float32 or float64 only, at most DUMP_MAX_BYTES in all."""
    import numpy as np
    assert all(v.dtype in (np.float32, np.float64) for v in arrays.values())
    assert sum(v.nbytes for v in arrays.values()) <= DUMP_MAX_BYTES
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(path, name + ".npy"), v)


def time_kernel(torch, fn, iters, flush):
    """Average CUDA-event duration (ms) of fn() over `iters` launches on the current stream; `flush` (a >L2 buffer)
    is rewritten before every launch, outside the event pair."""
    fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        if flush is not None:
            flush.add_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / iters


def kernel_rooflines(torch, nv, model, bt, peaks, traffic):
    """Per-kernel achieved throughput against the measured roofline (kernels timed alone -> burst peaks)."""
    ps, p, B, T, Nn = model.ps, nv.ptr, bt.B, bt.T, bt.Nn
    N = ps.N
    M = B * T
    model.forward_train(bt)
    model.backward(bt)
    torch.cuda.synchronize()
    ws = model._score_buffers(ps.n_pad, True)
    wse = model._score_buffers(ps.n_pad, False)
    flush = torch.zeros(64 * 1024 * 1024, device=model.dev, dtype=torch.int32)        # 256 MB > 126 MB L2
    cl = model._cluster_for(B)
    w = ps.w
    specs = [
        ("score_fwd_train", "tensor", 2.0 * B * N * K_REF,
         lambda: nv.call("tcar_score_fwd", p(model.Q), p(ps.iext), p(model.c_ref), p(ws["E"]), p(ws["part"]), None, None,
                         B, N, ps.n_pad, 0, cl)),
        ("score_fwd_eval", "tensor", 2.0 * B * N * K_REF,
         lambda: nv.call("tcar_score_fwd", p(model.Q), p(ps.iext), p(model.c_ref), None, p(wse["part"]),
                         p(wse["cmax"]), p(wse["tmax"]), B, N, ps.n_pad, 1, cl)),
        ("score_bwd_q", "tensor", 2.0 * B * N * K_REF,
         lambda: nv.call("tcar_score_bwd_q", p(ws["E"]), p(ps.iext), p(ws["qpart"]), p(model.dq_raw), B, ps.n_pad)),
        ("score_bwd_i", "tensor", 2.0 * B * N * K_DITEM,
         lambda: nv.call("tcar_score_bwd_i", p(ws["E"]), p(model.Qs), p(ps.item_g), p(model.sq_partial), B, N,
                         ps.n_pad)),
        # SURVEY 8d unit: reads p, m, v, g and writes p, m, v = 7 x (N+1) x 250 x 4 bytes.  The kernel also rewrites the
        # bf16 item columns of the scoring operand in the same pass (+ (N+1) x 250 x 2 bytes, reported separately as
        # frac_with_operand_refresh)
        ("adam_item", "hbm", (N + 1) * 7.0 * 250 * 4,
         lambda: nv.call("tcar_adam_item", p(ps.item), p(ps.item_m), p(ps.item_v), p(ps.item_g), p(ps.sqnorm_item),
                         p(ps.step), 0.0, model.max_grad_f, p(ps.iext), 0, N + 1, None, 0)),
        ("sqnorm_item_grad", "hbm", (N + 1) * 250 * 4.0,
         lambda: nv.call("tcar_sqnorm_big", p(ps.item_g), p(ps.norm_partial), p(ps.sqnorm_item), ps.item_g.numel())),
        # table rows read + X/P/D/CT written + the index words
        ("gather_fwd", "hbm", M * (2 * 250 + 250 + 6 * 64) * 4.0 + M * (500 + 320 + 64) * 4.0 + B * 4 * 128 * 4.0
         + (7 * M + 2 * B) * 4.0,
         lambda: nv.call("tcar_gather_fwd", p(bt.idx), p(bt.ctx), p(ps.item), p(ps.content), p(w["pos"]),
                         p(w["month"]), p(w["day"]), p(w["week"]), p(w["hour"]), p(w["minute"]), p(w["dur"]),
                         p(model.X), p(model.P), p(model.D), p(model.CT), B, T)),
        # reads X, P, U1, U2 and rewrites U1, U2 (sigmoid) + alpha + pooled
        ("pool_fwd", "hbm", M * (500 + 320 + 4 * 250 + 3) * 4.0 + B * (500 + 500 + 320) * 4.0,
         lambda: nv.call("tcar_pool_fwd", p(model.X), p(model.P), p(model.U1), p(model.U2), p(model.q), p(w["w_r"]),
                         p(w["w_t"]), p(model.alpha), p(model.pooled), p(model.pooled_t), B, T)),
        # sparse rows: read dXi / a_ic rows + item rows, RMW of the touched g_item rows
        ("scatter_add_rows", "hbm", (M * 3 + (B + B * Nn) * 3) * 250 * 4.0,
         lambda: nv.call("tcar_scatter_add_rows", p(bt.seq), p(bt.label), p(bt.neg), p(model.dXi), p(model.a_ic),
                         p(model.coef), p(ps.item), p(ps.item_g), p(model.hash_keys), p(model.hash_cnt),
                         p(model.hash_acc), p(model.entry_slot), p(model.slot_sq), model.hash_size, B, T, Nn)),
    ]
    # eval top-k (certified selection + widening of the queries it could not certify): reads tilemax [B, n_pad/128]
    # + 512 chunk maxima and re-scores 256 candidates x 2 KB of fp32 rows
    model._ensure_cat_stats()
    specs.append(("eval_topk", "hbm", B * (ps.n_pad / 128 + 512) * 4.0 + B * 256 * 2 * 250 * 4.0,
                  lambda: model._topk(wse, model.a_ic, model.Tq, bt.label, model._evblock, B, N, ps.n_pad, 0)))
    out = {}
    for name, bound, work, fn in specs:
        ms = time_kernel(torch, fn, 10, flush)
        if bound == "tensor":
            ach, peak, unit = work / (ms * 1e-3) / 1e12, peaks["tensor_burst"], "TFLOP/s"
        else:
            ach, peak, unit = work / (ms * 1e-3) / 1e9, peaks["hbm"], "GB/s"
        out[name] = {"bound": bound, "ms": ms, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                     "peak_source": peaks["source"], "work_per_launch": work, "traffic": traffic.get(name)}
        if name == "adam_item":
            out[name]["frac_with_operand_refresh"] = (work + (N + 1) * 250 * 2.0) / (ms * 1e-3) / 1e9 / peak
        if bound == "tensor":
            out[name]["note"] = ("credited with the REFERENCE's FLOPs (K = 820 scoring / dA, 570 dItems, SURVEY 8d); the "
                                 "kernel multiplies K = 640 / 256 columns (time-term factorisation)")
            k_exec = {"score_bwd_i": 256.0 / K_DITEM}.get(name, 640.0 / K_REF)
            out[name]["frac_executed_flops"] = ach * k_exec / peak
    del flush
    return out


def multi_gpu_parity(torch, dist, synth, Model, margs, model, mwdhm, rank, world):
    """N-GPU step == 1-GPU step, checked inside the bench run (so the driver's SCALE record carries it): ONE train step
    on a global batch of <= 512 sessions split over the ranks (the layout being benchmarked) against the same batch on a
    single-GPU model built here with the same initial values, then one eval batch.  Returns the "parity" object."""
    import numpy as np
    from tcar_b200 import parallel
    N, Nn = margs["itemnum"], margs["neg_num"]
    Bg, T = 64 * world if 64 * world <= 512 else 512, 5
    packed = synth.make_index_batch(N, Bg, T, Nn, mwdhm, seed=424242)
    pl, Bl, _, _ = parallel.shard_packed(packed, Bg, T, Nn, rank, world)
    # fresh models: the benchmarked one has trained already
    np.random.seed(2020)
    multi = Model(dict(margs))
    np.random.seed(2020)
    single = Model(dict(margs, rank=0, world_size=1, train_parallel="dp"))
    bt = multi.to_device(torch.from_numpy(pl).pin_memory(), Bl, T, Nn)
    bt.counts = parallel.catalog_counts(Bg, world)
    loss_m = multi.train_step(bt).clone()
    multi.sync_updates()
    multi.sync_item_table()
    if getattr(multi, "sync_optimizer_state", None):
        multi.sync_optimizer_state()      # data-parallel sharded update: every rank holds the moments of its own rows only
    btf = single.to_device(torch.from_numpy(packed).pin_memory(), Bg, T, Nn)
    loss_s = single.train_step(btf).clone()
    single.sync_updates()
    lo, hi = parallel.shard_sessions(Bg, rank, world)
    rel = lambda x, y: float((x - y).double().norm() / (y.double().norm() + 1e-30))
    res = {"loss_maxabs": float((loss_m - loss_s[lo:hi]).abs().max()) if hi > lo else 0.0,
           "theta_rel": rel(multi.ps.theta, single.ps.theta), "item_rel": rel(multi.ps.item, single.ps.item),
           "item_moment_rel": rel(multi.ps.item_m, single.ps.item_m)}
    # evaluation: catalog sharded across the ranks vs the single-GPU result on the SAME parameters
    single.ps.load_state_dict(multi.ps.state_dict())
    ep = synth.make_index_batch(N, 256, 3, 0, mwdhm, seed=434343)
    eb_m = multi.to_device(torch.from_numpy(ep).pin_memory(), 256, 3, 0)
    eb_s = single.to_device(torch.from_numpy(ep).pin_memory(), 256, 3, 0)
    s_lo, s_hi = multi.shard_bounds(world)[rank]
    top_m, ngt_m, ce_m = [x.clone() for x in multi.eval_step(eb_m, shard=(s_lo, s_hi, multi.iext_shard(s_lo, s_hi)))]
    top_s, ngt_s, ce_s = single.eval_step(eb_s)
    hit = ngt_s < 20
    res["eval_top20_equal"] = bool(torch.equal(top_m, top_s))
    res["eval_rank_equal"] = bool(torch.equal(hit, ngt_m < 20) and torch.equal(ngt_m[hit], ngt_s[hit]))
    res["eval_ce_maxabs"] = float((ce_m - ce_s).abs().max())
    # the layout the bench times (eval_round): every rank its OWN batch, two collectives per round
    Br = 200 + 7 * rank
    er = synth.make_index_batch(N, Br, 2 + rank % 3, 0, mwdhm, seed=444444 + rank)
    er_m = multi.to_device(torch.from_numpy(er).pin_memory(), Br, 2 + rank % 3, 0)
    er_s = single.to_device(torch.from_numpy(er).pin_memory(), Br, 2 + rank % 3, 0)
    top_r, ngt_r, ce_r = [x.clone() for x in multi.eval_round(er_m, [200 + 7 * g for g in range(world)])]
    top_s, ngt_s, ce_s = single.eval_step(er_s)
    hit = ngt_s < 20
    res["round_top20_equal"] = bool(torch.equal(top_r, top_s))
    res["round_rank_equal"] = bool(torch.equal(hit, ngt_r < 20) and torch.equal(ngt_r[hit], ngt_s[hit]))
    res["eval_ce_maxabs"] = max(res["eval_ce_maxabs"], float((ce_r - ce_s).abs().max()))
    ok = (res["loss_maxabs"] < 1e-4 and res["theta_rel"] < 1e-4 and res["item_rel"] < 1e-4
          and res["item_moment_rel"] < 1e-3 and res["eval_top20_equal"]
          and res["eval_rank_equal"] and res["round_top20_equal"] and res["round_rank_equal"]
          and res["eval_ce_maxabs"] < 1e-3)
    flag = torch.tensor([1 if ok else 0], device=model.dev, dtype=torch.int32)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    worst = torch.tensor([res["loss_maxabs"], res["theta_rel"], res["item_rel"], res["item_moment_rel"],
                          res["eval_ce_maxabs"]], device=model.dev, dtype=torch.float64)
    dist.all_reduce(worst, op=dist.ReduceOp.MAX)
    for k, v in zip(("loss_maxabs", "theta_rel", "item_rel", "item_moment_rel", "eval_ce_maxabs"), worst.tolist()):
        res[k] = v
    res["ok"] = bool(int(flag.item()))
    for k in ("eval_top20_equal", "eval_rank_equal", "round_top20_equal", "round_rank_equal"):
        f2 = torch.tensor([1 if res[k] else 0], device=model.dev, dtype=torch.int32)
        dist.all_reduce(f2, op=dist.ReduceOp.MIN)
        res[k] = bool(int(f2.item()))
    res["what"] = (f"one {margs['train_parallel']} train step on a global batch of {Bg} sessions over {world} GPUs vs the same "
                   f"batch on one GPU (loss, parameters after Adam), then one catalog-sharded eval batch of 256 queries vs "
                   f"one GPU (top-20 ids bit-equal, ranks, cross loss); worst value over the ranks")
    if getattr(multi, "close_peers", None):
        multi.close_peers()
    del multi, single
    torch.cuda.empty_cache()
    return res


def run_b200(a):
    import numpy as np
    import torch
    import __graft_entry__ as ge
    ge.load_package()
    from tcar_b200 import _native as nv, synth
    from tcar_b200.model_combine import Seq2SeqAttNN

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local),
                                timeout=datetime.timedelta(seconds=180))
    N, B, Nn, K, W = a.items, a.batch, a.neg_num, a.steps, a.warmup
    clocks = ClockSampler(local)
    if rank == 0 and not a.profile_region:
        clocks.start()           # started before the model is built: its start-up is over when the timed loops begin
    Ts = session_lengths(a)
    T = 20                     # worst-case length, used for the per-kernel pass and the `t20` line
    content, mwdhm, category = synth.make_catalog(N)
    np.random.seed(2020)
    margs = dict(publish_time_MWDHM=mwdhm, itemnum=N, category_id=None, item_freq_dict_norm={}, reverse_item=None,
                 content_emb=content, emb_stddev=0.002, stddev=0.05, hidden_size=250, time_hidden_size=64, l2_emb=0.0,
                 batch_size=B, epoch=1, neg_num=Nn, lr=0.001, max_grad=150, rank=rank, world_size=world,
                 train_parallel=a.train_parallel if world > 1 else "dp")
    layout_note = None
    try:
        model = Seq2SeqAttNN(margs)
    except nv.TcarNativeError as exc:
        if margs["train_parallel"] != "catalog":
            raise
        # no CUDA IPC peer access on this node (every rank raises together, catalog_parallel._open_peers): measure the
        # data-parallel layout instead and say so in the JSON line
        layout_note = f"catalog layout unavailable ({exc}); data parallel measured instead"
        a.train_parallel = margs["train_parallel"] = "dp"
        np.random.seed(2020)
        model = Seq2SeqAttNN(margs)
    peaks = load_peaks()
    nbatch = len(Ts)
    host = make_batches(synth, N, B, Ts, Nn, mwdhm, seed0=1000 * (rank + 1))
    dev = [model.to_device(h, B, t, Nn) for h, t in zip(host, Ts)]
    host20 = make_batches(synth, N, B, [T] * 4, Nn, mwdhm, seed0=5000 * (rank + 1))
    dev20 = [model.to_device(h, B, T, Nn) for h in host20]
    torch.cuda.synchronize()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    if a.profile_region:
        pb = model.to_device(make_batches(synth, N, B, [T], Nn, mwdhm, seed0=3)[0], B, T, Nn)
        eb = model.to_device(make_batches(synth, N, B, [T], 0, mwdhm, seed0=4)[0], B, T, 0)
        pb2 = model.to_device(make_batches(synth, N, B, [T], Nn, mwdhm, seed0=5)[0], B, T, Nn)
        for _ in range(2):
            model.train_step(pb)
            model.eval_step(eb)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        model.train_step(pb, pb2)      # with the look-ahead: rows of pb2 updated first, its session forward prefetched
        model.sync_updates()
        model.eval_step(eb)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], device=model.dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- kernel-resident train throughput: inputs already in HBM --------------------------------------------
    clocks.wait_first()          # samples cover warm-up + every timed loop below (a timed loop alone is ~60 ms)
    # train_step(bt, next_bt): the train loop's one-batch look-ahead (Seq2SeqAttNN.train) -- the session forward of the
    # next batch overlaps this step's table-wide Adam pass.  Every timed step therefore contains exactly one session
    # forward (its successor's) and the step after the last timed one is launched the same way.
    # (catalog layout: only with the opt-in look-ahead across ranks, TCAR_CATALOG_LOOKAHEAD=1)
    pipe = (world == 1 or bool(getattr(model, "cat_lookahead", False))) and not a.no_lookahead
    nxt = (lambda lst, i: lst[(i + 1) % len(lst)]) if pipe else (lambda lst, i: None)
    for i in range(W):
        model.train_step(dev[i % nbatch], nxt(dev, i))
    model.sync_updates()
    barrier()
    nv.LAUNCHES["count"] = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    marks = []
    for i in range(W, W + K):
        loss_dev = model.train_step(dev[i % nbatch], nxt(dev, i))
        ev = torch.cuda.Event(enable_timing=True)      # per-step marks on the launching stream: spread of the K steps
        ev.record()
        marks.append(ev)
    model.sync_updates()
    e1.record()
    barrier()
    train_ms = max_over_ranks(e0.elapsed_time(e1))
    launches = nv.LAUNCHES["count"]
    seq_ms = [a_.elapsed_time(b_) for a_, b_ in zip([e0] + marks[:-1], marks)]
    per_step = sorted(seq_ms)
    step_spread = {"min_ms": per_step[0], "median_ms": per_step[len(per_step) // 2], "max_ms": per_step[-1],
                   "first_ms": [round(x, 3) for x in seq_ms[:12]], "last_ms": [round(x, 3) for x in seq_ms[-6:]],
                   "note": "rank 0, time between consecutive steps' last launches on the main stream"}
    loss_last = float(model.loss[:B].mean().item())
    outputs = {}
    if a.dump_outputs:
        model.sync_item_table()    # catalog layout: rank 0 holds only its own item rows until this collective
        if rank == 0:
            outputs.update(train_outputs(model, loss_dev))

    # ---- end to end through the public API: pinned host batch -> H2D -> train_step -> D2H of the loss -------
    def e2e_loop(hosts, lens, n):
        """n steps through the public API, each: H2D of the NEXT batch (pinned -> device), train_step, D2H of this
        step's [B] loss into pinned memory (Seq2SeqAttNN.fetch_async); the host READS a step's loss one step later, so
        that it never stalls the launch queue.  Every loss is read inside the timed region."""
        bt = model.to_device(hosts[0], B, lens[0], Nn)
        pending, total = None, 0.0
        e2e_wall.clear()
        for i in range(n):
            e2e_wall.append(time.perf_counter())
            j = (i + 1) % len(hosts)
            nb = model.to_device(hosts[j], B, lens[j], Nn)
            h = model.fetch_async(model.train_step(bt, nb if pipe else None))
            if pending is not None:
                total += float(pending.get().sum())
            pending = h
            bt = nb
        model.sync_updates()
        total += float(pending.get().sum())
        return total

    e2e_wall = []
    e2e_loop(host, Ts, max(W, 2))
    barrier()
    e0.record()
    e2e_loop(host, Ts, K)
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    # host wall time per step of that loop: a step far above the median is interference on the host side (another
    # process holding driver locks), not the path's cost -- reported, not removed
    dts = sorted(b_ - a_ for a_, b_ in zip(e2e_wall, e2e_wall[1:]))
    e2e_host = {"median_ms": dts[len(dts) // 2] * 1e3, "max_ms": dts[-1] * 1e3} if dts else None
    h2d = sum(host[i % nbatch].numel() for i in range(K)) * 4 / K
    d2h = B * 4
    # ---- the same two measurements at the reference's --maxlen (every batch T = 20): the heaviest session side
    for i in range(2):
        model.train_step(dev20[i % 4], nxt(dev20, i))
    model.sync_updates()
    barrier()
    e0.record()
    for i in range(2, 2 + K):
        model.train_step(dev20[i % 4], nxt(dev20, i))
    model.sync_updates()
    e1.record()
    barrier()
    t20_ms = max_over_ranks(e0.elapsed_time(e1))
    e0.record()
    e2e_loop(host20, [T] * 4, K)
    e1.record()
    barrier()
    t20_e2e_ms = max_over_ranks(e0.elapsed_time(e1))

    def time_train(batches, steps, warm=3):
        n = len(batches)
        for i in range(warm):
            model.train_step(batches[i % n], nxt(batches, i))
        model.sync_updates()
        barrier()
        e0.record()
        for i in range(warm, warm + steps):
            model.train_step(batches[i % n], nxt(batches, i))
        model.sync_updates()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps

    def time_eval(batches, steps, shard_, warm=3):
        n = len(batches)
        nx = (lambda i: batches[(i + 1) % n]) if not a.no_lookahead else (lambda i: None)
        ev = (lambda b, nb: model.eval_round(b, [B] * world, shard=shard_)) if world > 1 else \
            (lambda b, nb: model.eval_step(b, next_bt=nb))
        for i in range(warm):
            ev(batches[i % n], nx(i))
        model.sync_updates()
        barrier()
        e0.record()
        for i in range(warm, warm + steps):
            ev(batches[i % n], nx(i))
        model.sync_updates()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps

    sweeps = {}
    if a.workload == "mind":
        # BASELINE config 4: heavier negative-feedback sampling -- the same step at neg_num 20 / 50 / 100
        sweeps["neg_sweep"] = {}
        for nn in (20, 50, 100):
            hb = make_batches(synth, N, B, Ts, nn, mwdhm, seed0=7000 * (rank + 1) + nn)
            db = [model.to_device(h, B, t, nn) for h, t in zip(hb, Ts)]
            ms = time_train(db, K)
            sweeps["neg_sweep"][str(nn)] = {"ms_per_step": ms, "value": world * B / (ms * 1e-3), "unit": "sessions/s"}
            del db
    if a.workload == "adressa":
        # BASELINE config 5: throughput over the session length (every batch at one T)
        sweeps["len_sweep"] = {}
        sh = None
        if world > 1:
            s_lo, s_hi = model.shard_bounds(world)[rank]
            sh = (s_lo, s_hi, model.iext_shard(s_lo, s_hi))
        for tt in (1, 2, 4, 8, 16, 20, 30, 40):
            hb = make_batches(synth, N, B, [tt] * 4, Nn, mwdhm, seed0=9000 * (rank + 1) + tt)
            db = [model.to_device(h, B, tt, Nn) for h in hb]
            ms = time_train(db, K)
            he = make_batches(synth, N, B, [tt] * 4, 0, mwdhm, seed0=9100 + tt + 100 * rank)
            de = [model.to_device(h, B, tt, 0) for h in he]
            model.sync_item_table()
            ems = time_eval(de, K, sh)
            sweeps["len_sweep"][str(tt)] = {"train_ms_per_step": ms, "train_sessions_per_s": world * B / (ms * 1e-3),
                                            "eval_ms_per_step": ems, "eval_queries_per_s": world * B / (ems * 1e-3)}
            del db, de

    # ---- evaluation: full-catalog top-20, catalog sharded across ranks when N > 1 ----------------------------
    # one batch of 512 queries per rank and step (Seq2SeqAttNN.test: batch i goes to rank i mod world; eval_round)
    ehost = make_batches(synth, N, B, Ts, 0, mwdhm, seed0=77 + 1000 * rank)
    edev = [model.to_device(h, B, t, 0) for h, t in zip(ehost, Ts)]
    shard = None
    if world > 1:
        lo, hi = model.shard_bounds(world)[rank]
        shard = (lo, hi, model.iext_shard(lo, hi))
    ecounts = [B] * world
    # eval_step(bt, next_bt=...): the test loop's one-batch look-ahead (Seq2SeqAttNN.test)
    look = not a.no_lookahead
    enxt = (lambda i: edev[(i + 1) % nbatch]) if look else (lambda i: None)

    def estep(bt_, nxt_):
        if world > 1:
            return model.eval_round(bt_, ecounts, shard=shard)
        return model.eval_step(bt_, next_bt=nxt_)

    for i in range(W):
        estep(edev[i % nbatch], enxt(i))
    model.sync_updates()
    barrier()
    e0.record()
    for i in range(W, W + K):
        eres = estep(edev[i % nbatch], enxt(i))
    model.sync_updates()
    e1.record()
    barrier()
    eval_ms = max_over_ranks(e0.elapsed_time(e1))
    if a.dump_outputs and rank == 0:
        outputs.update(eval_outputs(*eres))
    # share of the queries the certified selection handed to the widening pass, averaged over the batches
    unc = []
    for b_ in edev:
        estep(b_, None)
        unc.append(float(model.uncertain[:B].float().mean().item()))
    model.sync_updates()
    eval_uncertified = sum(unc) / len(unc)
    e0.record()
    bt = model.to_device(ehost[0], B, Ts[0], 0)
    pend = None
    for i in range(K):
        j = (i + 1) % nbatch
        nb = model.to_device(ehost[j], B, Ts[j], 0)              # H2D of the next batch, then this batch's step + D2H
        top, ngt, ce = estep(bt, nb if look else None)
        hs = [model.fetch_async(top), model.fetch_async(ngt), model.fetch_async(ce)]
        if pend is not None:
            [h.get() for h in pend]                              # read one step late: the launch queue never drains
        pend = hs
        bt = nb
    model.sync_updates()
    [h.get() for h in pend]
    e1.record()
    barrier()
    eval_e2e_ms = max_over_ranks(e0.elapsed_time(e1))
    eval_qp_ms = None
    if world > 1:
        # for comparison: query-parallel evaluation (every rank scores its own queries against the whole catalog)
        for i in range(2):
            model.eval_step(edev[(i + rank) % nbatch])
        barrier()
        e0.record()
        for i in range(K):
            model.eval_step(edev[(i + rank) % nbatch])
        e1.record()
        barrier()
        eval_qp_ms = max_over_ranks(e0.elapsed_time(e1))
    clk = clocks.stop() if rank == 0 else None
    eval_queries = world * B * K
    eval_layout = ("item catalog sharded across the ranks; per step every rank brings its own batch of %d queries: one "
                   "all-gather of the query blocks, every rank scores all %d queries against its item range (certified "
                   "local top-20), one all-to-all of the result blocks, merge (Seq2SeqAttNN.eval_round)" % (B, world * B)
                   if world > 1 else "single GPU")
    parity = multi_gpu_parity(torch, dist, synth, Seq2SeqAttNN, margs, model, mwdhm, rank, world) if world > 1 else None

    # ---- the loop a user runs (Seq2SeqAttNN.train): reference-API Sampler on a host thread -> pinned ring -> H2D ->
    # train_step, on an in-memory synthetic split with Globo-like session lengths
    train_loop = None
    if a.loop_sessions > 0:
        import random as pyrandom
        from tcar_b200.model_combine import prefetch_packed
        from tcar_b200.sampler import Sampler
        # multi-GPU: the loop of Seq2SeqAttNN.train with dist_batch="per_rank" -- every rank walks the same GLOBAL
        # batches of world x B sessions (same `random` seed, as main.py does) and its host thread gathers only its own
        # share of <= B sessions (Sampler.restrict_to_rank): all ranks run the same number of steps / collectives
        from tcar_b200 import parallel
        ld, sd, td, idict, impr = synth.make_sessions(N, a.loop_sessions * world, seed=2020,
                                                      impressions="mind" if a.negative_mode == "impression" else "few")
        pyrandom.seed(2020)
        np.random.seed(2020 + 7919 * rank)
        t_h0 = time.perf_counter()
        smp = Sampler(ld, sd, td, impr, idict, Nn, batch_size=B * world, negative_mode=a.negative_mode, verbose=False)
        smp.next_packed()                                    # builds the columnar cache (once per split)
        t_cache = time.perf_counter() - t_h0
        pyrandom.seed(2020)
        smp = Sampler(ld, sd, td, impr, idict, Nn, batch_size=B * world, negative_mode=a.negative_mode, verbose=False)
        if world > 1:
            smp.restrict_to_rank(rank, world)
        gsizes = getattr(smp, "global_sizes", None)
        nsess, nb = 0, 0
        barrier()
        t_w0 = time.perf_counter()
        e0.record()
        def staged_batches():
            for i, (packed, Bl, Tb, Nb) in enumerate(prefetch_packed(smp)):
                Bb = gsizes[i] if gsizes is not None else Bl
                sbt = model.stage_to_device(packed, Bl, Tb, Nb)
                sbt.counts = parallel.catalog_counts(Bb, world)
                yield Bb, sbt

        staged = staged_batches()
        cur = next(staged, None)
        while cur is not None:
            nx = next(staged, None)
            loss_dev = model.train_step(cur[1], nx[1] if (pipe and nx is not None) else None)
            nsess += cur[0]                              # sessions of the GLOBAL batch
            nb += 1
            cur = nx
        model.sync_updates()
        loss_dev.cpu()
        e1.record()
        barrier()
        loop_ms = max_over_ranks(e0.elapsed_time(e1))
        train_loop = {"note": "Sampler.next_packed (host thread) -> pinned ring -> H2D -> train_step over one epoch of "
                              "an in-memory synthetic split; length-bucketed batches, tail batches included; "
                              "multi-GPU: one batch of <= %d sessions per rank and step (global batch = GPUs x %d), "
                              "each rank's host thread samples only its own sessions" % (B, B),
                      "negative_mode": a.negative_mode,
                      "value": nsess / (loop_ms * 1e-3), "unit": "sessions/s", "batches": nb,
                      "sessions": nsess, "ms_per_batch": loop_ms / nb,
                      "wall_s": time.perf_counter() - t_w0, "columnar_cache_build_s": t_cache}

        # the same loop with the GPU-resident sampler (SURVEY 8f-2): bucket rows uploaded, batch assembled and
        # negatives drawn (Philox) on the device
        from tcar_b200.device_sampler import DeviceSampler
        pyrandom.seed(2020)
        dsm = DeviceSampler(model, ld, sd, td, impr, idict, Nn, batch_size=B * world, negative_mode=a.negative_mode,
                            negatives="device", seed=2020, rank=rank, world=world, verbose=False)
        nsess2, nb2 = 0, 0
        barrier()
        e0.record()
        cur = dsm.next_device() if dsm.has_next() else None
        while cur is not None:
            nx = dsm.next_device() if dsm.has_next() else None
            loss_dev = model.train_step(cur, nx if pipe else None)
            nsess2 += sum(cur.counts) if cur.counts is not None else cur.B
            nb2 += 1
            cur = nx
        model.sync_updates()
        loss_dev.cpu()
        e1.record()
        barrier()
        dloop_ms = max_over_ranks(e0.elapsed_time(e1))
        train_loop["device_sampler"] = {"note": "DeviceSampler(negatives='device'): host sends B bucket rows per batch; "
                                                "gather of the 7 index planes + Philox negatives (uniform, or the "
                                                "impression-list algorithm of sampler.py:118-131) on the device",
                                        "value": nsess2 / (dloop_ms * 1e-3), "unit": "sessions/s", "batches": nb2,
                                        "ms_per_batch": dloop_ms / nb2}

    kernels = {}
    traffic = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f)
    model.sync_item_table()        # catalog-sharded training: every rank holds the whole table again (collective)
    if rank == 0 and not a.no_kernels:
        kernels = kernel_rooflines(torch, nv, model, dev20[0], peaks, traffic)
    cpu_baseline = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        del model
        torch.cuda.empty_cache()
        Bs = a.cpu_sample_sessions
        rate, ms, threads = oracle_train_rate(N, Bs, Ts, Nn, 3, 1, content, mwdhm)
        erate = oracle_eval_rate(N, Bs, Ts[0], 1, content, mwdhm)
        cpu_baseline = {"value": rate, "unit": "sessions/s", "cores": threads, "kind": "port",
                        "sample": f"3 train steps of {Bs} sessions (session lengths {Ts[:3]}, Nn={Nn}) against the full "
                                  f"{N}-item catalog after 1 warm-up, torch CPU fp32 oracle ({ms:.0f} ms/step)",
                        "eval_queries_per_s": erate}
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, outputs)
    sessions = world * B * K
    value = sessions / (train_ms * 1e-3)
    # dominant kernel of the step = largest share of the isolated kernel times
    roof = None
    if kernels:
        step_k = ["score_fwd_train", "score_bwd_q", "score_bwd_i", "adam_item", "sqnorm_item_grad", "gather_fwd",
                  "pool_fwd", "scatter_add_rows"]
        top = max(step_k, key=lambda k: kernels[k]["ms"])
        kk = kernels[top]
        roof = {"kernel": top, "bound": kk["bound"], "achieved": kk["achieved"], "peak": kk["peak"],
                "unit": kk["unit"], "frac": kk["frac"], "traffic": kk["traffic"], "peak_source": kk["peak_source"],
                "ms_per_launch": kk["ms"]}
    line = {"metric": f"TCAR train sessions/sec ({SHAPE[a.workload][0]} shape)", "value": value, "unit": "sessions/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": train_ms / K, "ms_per_step_spread": step_spread,
            "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 tensor-core scoring GEMMs (fp32 accumulate), fp32 elsewhere",
            "data": "synthetic", "config": dict(workload_config(a, world), lookahead=bool(pipe),
                                                **({"layout_note": layout_note} if layout_note else {})),
            "e2e": {"value": sessions / (e2e_ms * 1e-3), "unit": "sessions/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / K, "host_step_wall": e2e_host},
            "t20": {"note": "same measurement with every batch at the reference --maxlen (T = 20)",
                    "value": sessions / (t20_ms * 1e-3), "ms_per_step": t20_ms / K,
                    "e2e_value": sessions / (t20_e2e_ms * 1e-3), "unit": "sessions/s"},
            "train_loop": train_loop, **sweeps,
            "gpu_launches": launches, "launches_per_step": launches / K, "loss_last_step": loss_last,
            "clocks": clk, "kernels": kernels, "roofline": roof, "cpu_baseline": cpu_baseline,
            "parity": parity,
            "eval_query_parallel": None if eval_qp_ms is None else {
                "note": "queries sharded across ranks instead of the catalog (no collective); not the north_star layout",
                "value": world * B * K / (eval_qp_ms * 1e-3), "unit": "queries/s", "ms_per_step": eval_qp_ms / K},
            # last, so that a consumer keeping only the tail of the line keeps the second half of BASELINE's metric
            "eval": {"metric": "full-catalog top-20 eval queries/sec", "value": eval_queries / (eval_ms * 1e-3),
                     "unit": "queries/s", "ms_per_step": eval_ms / K, "queries_per_step": eval_queries / K,
                     "layout": eval_layout, "uncertified_share": eval_uncertified,
                     "e2e": {"value": eval_queries / (eval_e2e_ms * 1e-3), "unit": "queries/s",
                             "h2d_bytes_per_step": sum(ehost[i % nbatch].numel() for i in range(K)) * 4 / K,
                             "d2h_bytes_per_step": B * (20 + 1 + 1) * 4},
                     "scaling": "weak (512 queries per GPU and step)" if world > 1 else "single"}}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
