"""Top-K recommendation on the GPU (tcar_recommend, Seq2SeqAttNN.recommend): one JSON line per workload at the Globo
shape (364 047 items) and the MIND shape (103 630 items), 512 sessions per batch, T in {1, 20}, K in {20, 100, 256},
with and without the session's own clicks excluded.

    python tools/recommend_probe.py [--shapes globo,mind]

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
"""
import argparse
import json

import numpy as np
import torch

from probe_common import B, gpu_info, make_model
from tcar_b200 import _native as nv, synth

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="globo,mind")
    a = ap.parse_args()
    torch.cuda.set_device(0)
    info = gpu_info()
    flush = torch.empty(256 << 20, device="cuda", dtype=torch.uint8)
    for shape in a.shapes.split(","):
        model, mwdhm = make_model(SHAPES[shape])
        for T in (1, 20):
            for K in (20, 100, 256):
                for clicked in (False, True):
                    workload(model, mwdhm, shape, T, K, clicked, info, flush)
        del model
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
