"""Top-K recommendation on the GPU (tcar_recommend, Seq2SeqAttNN.recommend): one JSON line per workload at the Globo
shape (364 047 items) and the MIND shape (103 630 items), 512 sessions per batch, T in {1, 20}, K in {20, 100, 256},
with and without the session's own clicks excluded.

    python tools/recommend_probe.py [--shapes globo,mind]
    python tools/recommend_probe.py --window [--shapes globo,mind]
    python tools/recommend_probe.py --category [--shapes globo,mind]
    python tools/recommend_probe.py --decay [--shapes globo,mind]

recommend_split across ranks is checked by tools/split_check.py.

Per workload:
  select_us_cold / scan_us_cold   recommend_select_kernel / recommend_scan_kernel alone (torch.profiler, CUDA
                                  activities), the L2 overwritten (256 MB memset) before each tcar_recommend call
  select_us_warm / scan_us_warm   the same, back-to-back calls on the same batch
  recommend_us                    Seq2SeqAttNN.recommend per batch (session forward, scoring GEMM, both kernels),
                                  CUDA events over 32 batches
  eval_step_us                    Seq2SeqAttNN.eval_step per batch on the same batches (the certified top-20)
  ratio                           recommend_us / eval_step_us
  rescored_mean / rescored_max    items re-scored exactly per query (the width of the error band)

--window: publish-time windows (tcar_score_fwd_window / tcar_recommend_window) instead, one JSON line per shape,
window width (100 %, 10 %, 1 %, 0.05 % of the catalog: item times are a random permutation of 0 .. N-1, every session
its own window of that many consecutive times) and K in {20, 100}, T = 1, no exclusions:
  gemm_mode1_us_cold / gemm_window_us_cold   score_fwd_pair_kernel<1> / <2> alone (torch.profiler), the L2
                                             overwritten before each call; gemm_ratio = window / mode 1
  recommend_us / recommend_window_us         Seq2SeqAttNN.recommend without / with the window per batch (CUDA events
                                             over 32 batches); ratio = window / none
  rescored_mean / rescored_max               items re-scored exactly per query with the window (rescored_nowin_mean:
                                             without)

--category: at most C items per category and allowed categories (set_item_categories / recommend(max_per_category,
categories) / tcar_recommend_category), item codes drawn uniformly from G categories: Globo (G = 461) and MIND
(G = 17, 264) shapes, B = 512, T in {1, 20}, K in {20, 100}, C in {1, 2, K}, allowed = all / one category per session /
10 % of the categories per session, no exclusions.  One JSON line per workload:
  gemm_us_cold / gemm_cat_us_cold            the mode-1 scoring GEMM over ps.iext / over iext_cat alone
                                             (torch.profiler, L2 overwritten before each call); gemm_ratio
  select_us_cold / scan_us_cold (_warm)      recommend_category_select_kernel / _scan_kernel alone, as above
  recommend_us / recommend_cat_us            Seq2SeqAttNN.recommend per batch without / with the categories (CUDA
                                             events over 32 batches); ratio = with / without
  rescored_mean / rescored_max               items re-scored exactly per query
  rebuild_us                                 one rebuild of iext_cat from ps.iext (CUDA events, mean of 10)

--decay: the freshness decay (recommend(decay=...) / tcar_score_fwd_decay / tcar_recommend_decay), item times uniform
over ten days in minutes and every session's t_ref at their end, half-lives of 6, 24 and 48 h, K in {20, 100}, B = 512,
T = 1, no exclusions.  One JSON line per shape, half-life and K:
  gemm_mode1_us_cold / gemm_decay_us_cold    score_fwd_pair_kernel<1> / <3> alone (torch.profiler), the L2
                                             overwritten before each call; gemm_ratio = decay / mode 1
  recommend_us / recommend_decay_us          Seq2SeqAttNN.recommend without / with the decay per batch (CUDA events
                                             over 32 batches); ratio = decay / none
  rescored_mean / rescored_max               items re-scored exactly per query with the decay (rescored_plain_mean:
                                             without; rescored_ratio = with / without)
"""
import argparse
import json

import numpy as np
import torch

from probe_common import B, gpu_info, make_model
from tcar_b200 import _native as nv, synth, util as nv_util

SHAPES = {"globo": 364047, "mind": 103630}


def kernel_times(model, bt, K, clicked, flush):
    """Mean device time of the two kernels over 20 tcar_recommend calls on bt's chunk maxima (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    model.recommend(bt, K, exclude_clicked=clicked)         # leaves bt's maxima and session vectors in place
    ps, p = model.ps, nv.ptr
    ws = model._score_buffers(ps.n_pad, False)
    ids = torch.empty(B, K, device=model.dev, dtype=torch.int32)
    sc = torch.empty(B, K, device=model.dev)
    args = (p(ws["cmax"]), p(ws["tmax"]), p(model.a_ic), p(model.Tq), p(ps.item), p(ps.content), p(ps.mwdhm),
            p(model.cat_stats), None, None, p(bt.seq) if clicked else None, bt.T, B, ps.N, ps.n_pad, K,
            p(model._rec_ws), p(ids), p(sc), p(model.rec_rescored))
    for _ in range(3):
        nv.call("tcar_recommend", *args)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            if flush is not None:
                flush.zero_()
            nv.call("tcar_recommend", *args)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for name in ("select", "scan"):
            if f"recommend_{name}_kernel" in e.key:
                out[name] = e.device_time_total / e.count
    return out["select"], out["scan"]


def workload(model, mwdhm, shape, T, K, clicked, info, flush):
    N = model.N
    bts = []
    for i in range(4):
        packed = synth.make_index_batch(N, B, T, 0, mwdhm, seed=100 * T + i)
        bts.append(model.to_device(torch.from_numpy(packed).pin_memory(), B, T, 0))
    sel_c, scan_c = kernel_times(model, bts[0], K, clicked, flush)
    sel_w, scan_w = kernel_times(model, bts[0], K, clicked, None)
    resc = []
    for bt in bts:
        model.recommend(bt, K, exclude_clicked=clicked)
        resc.append(model.rec_rescored[:B].cpu().numpy())
        model.eval_step(bt)
    resc = np.concatenate(resc)
    torch.cuda.synchronize()
    KB = 32
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {}
    for name, fn in (("recommend", lambda bt: model.recommend(bt, K, exclude_clicked=clicked)),
                     ("eval_step", lambda bt: model.eval_step(bt))):
        t0.record()
        for i in range(KB):
            fn(bts[i % 4])
        t1.record()
        torch.cuda.synchronize()
        times[name] = t0.elapsed_time(t1) / KB * 1e3
    res = dict(info, workload=f"{shape} N={N} B={B} T={T} K={K}" + (" exclude_clicked" if clicked else ""), N=N, B=B,
               T=T, K=K, exclude_clicked=clicked, select_us_cold=round(sel_c, 2), scan_us_cold=round(scan_c, 2),
               select_us_warm=round(sel_w, 2), scan_us_warm=round(scan_w, 2),
               recommend_us=round(times["recommend"], 1), eval_step_us=round(times["eval_step"], 1),
               ratio=round(times["recommend"] / times["eval_step"], 3), rescored_mean=round(float(resc.mean()), 1),
               rescored_max=int(resc.max()))
    print("recommend_probe " + json.dumps(res), flush=True)


def gemm_times(model, bt, wins, flush):
    """Mean device time of score_fwd_pair_kernel<1> and <2> over 20 calls each on bt's queries, cold L2."""
    from torch.profiler import ProfilerActivity, profile
    model.recommend(bt, 20)                                 # leaves bt's session vectors in place
    ps, p = model.ps, nv.ptr
    ws = model._score_buffers(ps.n_pad, False)
    wv = torch.from_numpy(np.concatenate(wins).astype(np.int32)).cuda()
    calls = (("tcar_score_fwd", p(model.Q), p(ps.iext), p(model.c_ref), None, p(ws["part"]), p(ws["cmax"]),
              p(ws["tmax"]), B, ps.N, ps.n_pad, 1, nv.CLUSTER_PAIR),
             ("tcar_score_fwd_window", p(model.Q), p(ps.iext), p(model.c_ref), p(ws["part"]), p(ws["cmax"]),
              p(ws["tmax"]), p(model._item_time), p(wv), p(wv[B:]), B, ps.N, ps.n_pad))
    for c in calls:
        nv.call(*c)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            for c in calls:
                flush.zero_()
                nv.call(*c)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for mode in (1, 2):
            if f"score_fwd_pair_kernel<{mode}>" in e.key:
                out[mode] = e.device_time_total / e.count
    return out[1], out[2]


def window_workloads(model, mwdhm, shape, info, flush):
    N = model.N
    rs = np.random.RandomState(5)
    model.set_item_times(rs.permutation(N))
    bts = []
    for i in range(4):
        packed = synth.make_index_batch(N, B, 1, 0, mwdhm, seed=100 + i)
        bts.append(model.to_device(torch.from_numpy(packed).pin_memory(), B, 1, 0))
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    KB = 32
    for frac in (1.0, 0.1, 0.01, 0.0005):
        width = max(1, int(round(frac * N)))
        wins = []
        for _ in range(4):
            lo = rs.randint(0, N - width + 1, B)
            wins.append((lo, lo + width - 1))
        g1, g2 = gemm_times(model, bts[0], wins[0], flush)
        for K in (20, 100):
            resc, resc0 = [], []
            for bt, w in zip(bts, wins):
                model.recommend(bt, K)
                resc0.append(model.rec_rescored[:B].cpu().numpy())
                model.recommend(bt, K, window=w)
                resc.append(model.rec_rescored[:B].cpu().numpy())
            resc, resc0 = np.concatenate(resc), np.concatenate(resc0)
            times = {}
            for name, kw in (("none", lambda i: {}), ("window", lambda i: {"window": wins[i % 4]})):
                t0.record()
                for i in range(KB):
                    model.recommend(bts[i % 4], K, **kw(i))
                t1.record()
                torch.cuda.synchronize()
                times[name] = t0.elapsed_time(t1) / KB * 1e3
            res = dict(info, workload=f"{shape} N={N} B={B} T=1 K={K} window={frac:g}", N=N, B=B, T=1, K=K,
                       window_frac=frac, window_items=width, gemm_mode1_us_cold=round(g1, 2),
                       gemm_window_us_cold=round(g2, 2), gemm_ratio=round(g2 / g1, 3),
                       recommend_us=round(times["none"], 1), recommend_window_us=round(times["window"], 1),
                       ratio=round(times["window"] / times["none"], 3), rescored_mean=round(float(resc.mean()), 1),
                       rescored_max=int(resc.max()), rescored_nowin_mean=round(float(resc0.mean()), 1))
            print("recommend_probe_window " + json.dumps(res), flush=True)


def profiled(calls, names, flush, reps=20):
    """Mean device time per launch of the kernels whose names contain names[i], over reps rounds of calls."""
    from torch.profiler import ProfilerActivity, profile
    for c in calls:
        nv.call(*c)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            for c in calls:
                if flush is not None:
                    flush.zero_()
                nv.call(*c)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for n in names:
            if n in e.key:
                out[n] = e.device_time_total / e.count
    return [out[n] for n in names]


def events_us(fn, n):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(n):
        fn(i)
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / n * 1e3


def decay_workloads(model, mwdhm, shape, info, flush):
    """--decay: item times uniform over ten days in minutes, every session's t_ref at their end, half-lives of 6, 24
    and 48 h (rate = ln 2 / (60 H) per minute)."""
    N, ps, p = model.N, model.ps, nv.ptr
    rs = np.random.RandomState(5)
    model.set_item_times(rs.randint(0, 14400, N))
    bts = []
    for i in range(4):
        packed = synth.make_index_batch(N, B, 1, 0, mwdhm, seed=100 + i)
        bts.append(model.to_device(torch.from_numpy(packed).pin_memory(), B, 1, 0))
    t_ref = np.full(B, 14400)
    for hl in (6, 24, 48):
        rate = np.log(2) / (60 * hl)
        model.recommend(bts[0], 20)                         # leaves bts[0]'s session vectors in place
        ws = model._score_buffers(ps.n_pad, False)
        dv = torch.from_numpy(nv_util.check_decay((t_ref, rate), B, [0])).cuda()
        calls = (("tcar_score_fwd", p(model.Q), p(ps.iext), p(model.c_ref), None, p(ws["part"]), p(ws["cmax"]),
                  p(ws["tmax"]), B, N, ps.n_pad, 1, nv.CLUSTER_PAIR),
                 ("tcar_score_fwd_decay", p(model.Q), p(ps.iext), p(ws["cmax"]), p(ws["tmax"]), p(model._item_time),
                  p(dv), p(dv[B:]), None, None, B, N, ps.n_pad))
        g1, g3 = profiled(calls, ("score_fwd_pair_kernel<1>", "score_fwd_pair_kernel<3>"), flush)
        for K in (20, 100):
            resc, resc0 = [], []
            for bt in bts:
                model.recommend(bt, K)
                resc0.append(model.rec_rescored[:B].cpu().numpy())
                model.recommend(bt, K, decay=(t_ref, rate))
                resc.append(model.rec_rescored[:B].cpu().numpy())
            resc, resc0 = np.concatenate(resc), np.concatenate(resc0)
            t_plain = events_us(lambda i: model.recommend(bts[i % 4], K), 32)
            t_decay = events_us(lambda i: model.recommend(bts[i % 4], K, decay=(t_ref, rate)), 32)
            res = dict(info, workload=f"{shape} N={N} B={B} T=1 K={K} half_life={hl}h", N=N, B=B, T=1, K=K,
                       half_life_h=hl, gemm_mode1_us_cold=round(g1, 2), gemm_decay_us_cold=round(g3, 2),
                       gemm_ratio=round(g3 / g1, 3), recommend_us=round(t_plain, 1),
                       recommend_decay_us=round(t_decay, 1), ratio=round(t_decay / t_plain, 3),
                       rescored_mean=round(float(resc.mean()), 1), rescored_max=int(resc.max()),
                       rescored_plain_mean=round(float(resc0.mean()), 1),
                       rescored_ratio=round(float(resc.mean() / resc0.mean()), 3))
            print("recommend_probe_decay " + json.dumps(res), flush=True)


def category_workloads(model, mwdhm, shape, G, info, flush):
    N, ps, p = model.N, model.ps, nv.ptr
    rs = np.random.RandomState(G)
    model.set_item_categories(rs.randint(0, G, N), G)
    model._ensure_iext_cat()

    def rebuild(i):
        model._iext_cat_version = -1
        model._ensure_iext_cat()
    rebuild_us = events_us(rebuild, 10)
    KB = 32
    for T in (1, 20):
        bts = []
        for i in range(4):
            packed = synth.make_index_batch(N, B, T, 0, mwdhm, seed=300 * T + i)
            bts.append(model.to_device(torch.from_numpy(packed).pin_memory(), B, T, 0))
        model.recommend(bts[0], 20, max_per_category=2)                # bts[0]'s session vectors stay in place
        ws, wc = model._score_buffers(ps.n_pad, False), model._score_buffers(model._cat_n_pad, False)
        g_plain = profiled([("tcar_score_fwd", p(model.Q), p(ps.iext), p(model.c_ref), None, p(ws["part"]),
                             p(ws["cmax"]), p(ws["tmax"]), B, ps.N, ps.n_pad, 1, nv.CLUSTER_PAIR)],
                           ["score_fwd_pair_kernel<1>"], flush)[0]
        g_cat = profiled([("tcar_score_fwd", p(model.Q), p(model._iext_cat), p(model.c_ref), None, p(wc["part"]),
                           p(wc["cmax"]), p(wc["tmax"]), B, model._cat_n, model._cat_n_pad, 1, nv.CLUSTER_PAIR)],
                         ["score_fwd_pair_kernel<1>"], flush)[0]
        allowed = {"all": None}
        one = rs.randint(0, G, B).astype(np.int32)
        allowed["one"] = (np.arange(B + 1, dtype=np.int32), one)
        m = max(1, G // 10)
        allowed["10%"] = (np.arange(B + 1, dtype=np.int32) * m,
                          np.concatenate([rs.choice(G, m, replace=False) for _ in range(B)]).astype(np.int32))
        for K in (20, 100):
            plain = events_us(lambda i: model.recommend(bts[i % 4], K), KB)
            for C in (1, 2, K):
                for name, cats in allowed.items():
                    kw = dict(max_per_category=C, categories=cats)
                    resc = []
                    for bt in bts:
                        model.recommend(bt, K, **kw)
                        resc.append(model.rec_rescored[:B].cpu().numpy())
                    resc = np.concatenate(resc)
                    model.recommend(bts[0], K, **kw)
                    acsr = torch.from_numpy(np.concatenate(cats).astype(np.int32)).cuda() if cats else None
                    ids = torch.empty(B, K, device=model.dev, dtype=torch.int32)
                    sc = torch.empty(B, K, device=model.dev)
                    call = [("tcar_recommend_category", p(wc["cmax"]), p(model.a_ic), p(model.Tq), p(ps.item),
                             p(ps.content), p(ps.mwdhm), p(model.cat_stats), None, None, None, T, B,
                             model._cat_n_pad, K, p(model._cat_perm), p(model._item_cat), p(model._cat_off), G,
                             p(acsr), p(acsr[B + 1:]) if acsr is not None else None, C, p(model._rec_ws), p(ids),
                             p(sc), p(model.rec_rescored))]
                    names = ["recommend_category_select_kernel", "recommend_category_scan_kernel"]
                    sel_c, scan_c = profiled(call, names, flush)
                    sel_w, scan_w = profiled(call, names, None)
                    cat_us = events_us(lambda i: model.recommend(bts[i % 4], K, **kw), KB)
                    res = dict(info, workload=f"{shape} N={N} G={G} B={B} T={T} K={K} C={C} allowed={name}", N=N,
                               N_cat=model._cat_n, G=G, B=B, T=T, K=K, C=C, allowed=name,
                               gemm_us_cold=round(g_plain, 2), gemm_cat_us_cold=round(g_cat, 2),
                               gemm_ratio=round(g_cat / g_plain, 3), select_us_cold=round(sel_c, 2),
                               scan_us_cold=round(scan_c, 2), select_us_warm=round(sel_w, 2),
                               scan_us_warm=round(scan_w, 2), recommend_us=round(plain, 1),
                               recommend_cat_us=round(cat_us, 1), ratio=round(cat_us / plain, 3),
                               rescored_mean=round(float(resc.mean()), 1), rescored_max=int(resc.max()),
                               rebuild_us=round(rebuild_us, 1))
                    print("recommend_probe_category " + json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="globo,mind")
    ap.add_argument("--window", action="store_true", help="publish-time windows (see the module docstring)")
    ap.add_argument("--category", action="store_true", help="caps and allowed categories (see the module docstring)")
    ap.add_argument("--decay", action="store_true", help="freshness decay (see the module docstring)")
    a = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    flush = torch.empty(256 << 20, device="cuda", dtype=torch.uint8)
    for shape in a.shapes.split(","):
        model, mwdhm = make_model(SHAPES[shape])
        if a.category:
            for G in ((461,) if shape == "globo" else (17, 264)):
                category_workloads(model, mwdhm, shape, G, info, flush)
            del model
            torch.cuda.empty_cache()
            continue
        if a.decay:
            decay_workloads(model, mwdhm, shape, info, flush)
            del model
            torch.cuda.empty_cache()
            continue
        if a.window:
            window_workloads(model, mwdhm, shape, info, flush)
            del model
            torch.cuda.empty_cache()
            continue
        for T in (1, 20):
            for K in (20, 100, 256):
                for clicked in (False, True):
                    workload(model, mwdhm, shape, T, K, clicked, info, flush)
        del model
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
