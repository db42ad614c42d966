"""Top-K recommendation on the GPU (tcar_recommend, Seq2SeqAttNN.recommend): one JSON line per workload at the Globo
shape (364 047 items) and the MIND shape (103 630 items), 512 sessions per batch, T in {1, 20}, K in {20, 100, 256},
with and without the session's own clicks excluded.

    python tools/recommend_probe.py          every workload
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29514 \\
        tools/recommend_probe.py --check     recommend_split at world 2 == world 1 on a synthetic split, file for file
                                             and metric for metric (NCCL with a GPU per rank; ranks sharing a GPU use
                                             gloo)

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
import copy
import json
import os
import random
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

ge.load_package()
from tcar_b200 import _native as nv, synth  # noqa: E402
from tcar_b200.model_combine import Seq2SeqAttNN  # noqa: E402

SHAPES = {"globo": 364047, "mind": 103630}
B = 512


def make_model(N, rank=0, world=1, seed=2020):
    content, mwdhm, _ = synth.make_catalog(N, seed=seed)
    np.random.seed(2020)
    return Seq2SeqAttNN(dict(publish_time_MWDHM=mwdhm, itemnum=N, category_id=None, item_freq_dict_norm={},
                             reverse_item=None, content_emb=content, emb_stddev=0.04, stddev=0.05, hidden_size=250,
                             time_hidden_size=64, l2_emb=0.0, batch_size=B, epoch=1, neg_num=20, lr=0.001,
                             max_grad=150, rank=rank, world_size=world, train_parallel="dp")), mwdhm


def gpu_info():
    idx = torch.cuda.current_device()
    out = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True).stdout.strip()
    return {"gpu": torch.cuda.get_device_name(idx), "power_limit_w": float(out) if out else None}


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


def check():
    """recommend_split under torchrun (batch i on rank i mod world, sums all-reduced) == the same split on one GPU: the
    ranks' files together hold exactly the lines of the single-GPU file, and the metrics agree."""
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    gpus = torch.cuda.device_count()
    torch.cuda.set_device(local % gpus)
    if gpus >= world:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:                                                # ranks share a GPU: NCCL needs one GPU per rank, gloo does not
        dist.init_process_group("gloo")
    N = 20000
    len_dict, sdict, tdict, item_dict, _ = synth.make_sessions(N, 3000, train=False)
    base = os.path.join(tempfile.gettempdir(), "recommend_check")
    out, files = {}, {}
    for w in (world, 1):
        d = os.path.join(base, f"world{w}" + (f"_rank{rank}" if w == 1 else ""))
        os.makedirs(d, exist_ok=True)
        os.chdir(d)
        model, _ = make_model(N, rank if w > 1 else 0, w, seed=3)
        random.seed(7)                                   # same batches for both runs
        args = {"recommend_k": 100, "recommend_exclude_clicked": True, "foldnum": 0}
        out[w] = model.recommend_split(None, (copy.deepcopy(len_dict), sdict, tdict), item_dict, args)
        files[w] = model.last_recommend_path if w == 1 else None
        dist.barrier()
    a, b = out[world], out[1]
    lines_n = []
    for r in range(world):
        lines_n += open(os.path.join(base, f"world{world}", f"saved/recommend_0_rank{r}.txt")).read().splitlines()
    lines_1 = open(os.path.join(base, f"world1_rank{rank}", files[1])).read().splitlines()
    same_files = sorted(lines_n) == sorted(lines_1) and len(lines_1) == b["sessions"]
    same = same_files and a["sessions"] == b["sessions"] and all(abs(a[k] - b[k]) <= 1e-12 for k in ("hr", "mrr", "ndcg"))
    print(f"rank {rank} recommend_check " + json.dumps(dict(gpu_info(), world=world, gpus=min(gpus, world),
                                                            backend=dist.get_backend(), K=100, exclude_clicked=True,
                                                            world_n=a, world_1=b, lines=len(lines_1),
                                                            files_equal=same_files, equal=same)), flush=True)
    dist.destroy_process_group()
    if not same:
        sys.exit(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--shapes", default="globo,mind")
    a = ap.parse_args()
    if a.check:
        return check()
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
