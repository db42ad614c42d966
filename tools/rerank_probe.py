"""Candidate re-ranking on the GPU (tcar_rerank, Seq2SeqAttNN.rerank): one JSON line per workload at the MIND shape
(catalog of 103 630 items, 512 sessions per batch).

    python tools/rerank_probe.py             T in {1, 20} x MIND-like list lengths (LogNormal, mean 37); T = 20 x 300
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 \
        tools/rerank_probe.py --check        test_impressions at world 2 == world 1 on a synthetic split
                                             (NCCL with a GPU per rank; ranks sharing a GPU use gloo)

Per workload:
  kernel_us_cold  tcar_rerank alone, CUDA events around every launch, L2 overwritten (256 MB memset) before each one:
                  the candidate rows come from HBM, as they do when a batch's lists are new
  kernel_us_warm  back-to-back launches on the same lists (their rows stay in the 126 MB L2)
  batch_us        Seq2SeqAttNN.rerank per batch: host validation, list upload, session forward, kernel
  forward_us      the session forward alone; sessions_per_s = B / batch_us
  bytes           what the kernel must read: L x (item row 1 KB + content row 1 KB + 20 B of publish-time bins) per
                  session plus the session vectors (500 + 139 floats) and the list itself
  hbm_share       bytes / 7.7 TB/s (B200 data sheet HBM3e bandwidth) over kernel_us_cold
"""
import argparse
import copy
import json
import os
import random
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

ge.load_package()
from tcar_b200 import _native as nv, synth  # noqa: E402
from tcar_b200.model_combine import Seq2SeqAttNN  # noqa: E402

N_MIND, B = 103630, 512
HBM_BPS = 7.7e12


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


def lists_for(rs, labels, lens):
    off = np.zeros(len(lens) + 1, dtype=np.int32)
    off[1:] = np.cumsum(lens)
    ids = rs.randint(0, N_MIND, int(off[-1])).astype(np.int32)
    for b, L in enumerate(lens):
        ids[off[b] + rs.randint(L)] = labels[b]          # the clicked article is on its impression list
    return off, ids


def workload(model, mwdhm, T, fixed_len, info):
    rs = np.random.RandomState(T * 1000 + fixed_len)
    bts, lists = [], []
    for i in range(4):
        packed = synth.make_index_batch(N_MIND, B, T, 0, mwdhm, seed=100 * T + i)
        bt = model.to_device(torch.from_numpy(packed).pin_memory(), B, T, 0)
        lens = [fixed_len] * B if fixed_len else \
            [len(v) for v in synth.make_impressions(N_MIND, B, seed=10 * T + i).values()]
        bts.append(bt)
        lists.append(lists_for(rs, packed[7 * B * T + 2 * B: 7 * B * T + 3 * B], lens))
    # ---- the kernel alone, on batch 0's session vectors
    model.rerank(bts[0], *lists[0])
    off, ids = lists[0]
    nnz, max_len = len(ids), int(np.diff(off).max())
    csr = torch.from_numpy(np.concatenate([off, ids]).astype(np.int32)).to(model.dev)
    sc, rk = torch.empty(nnz, device=model.dev), torch.empty(nnz, device=model.dev, dtype=torch.int32)
    lr, au = torch.empty(B, device=model.dev, dtype=torch.int32), torch.empty(B, device=model.dev)
    ps, p = model.ps, nv.ptr
    args = (p(model.a_ic), p(model.Tq), p(ps.item), p(ps.content), p(ps.mwdhm), p(csr), p(csr[B + 1:]),
            p(bts[0].label), B, ps.N, max_len, p(sc), p(rk), p(lr), p(au))
    for _ in range(20):
        nv.call("tcar_rerank", *args)
    flush = torch.empty(256 << 20, device=model.dev, dtype=torch.uint8)
    K = 200
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    for e0, e1 in evs:
        flush.zero_()
        e0.record()
        nv.call("tcar_rerank", *args)
        e1.record()
    torch.cuda.synchronize()
    cold = sum(e0.elapsed_time(e1) for e0, e1 in evs) / K * 1e3
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0.record()
    for _ in range(K):
        nv.call("tcar_rerank", *args)
    w1.record()
    torch.cuda.synchronize()
    warm = w0.elapsed_time(w1) / K * 1e3
    # ---- per batch: session forward + rerank, and the forward alone
    for i in range(8):
        model.rerank(bts[i % 4], *lists[i % 4])
    torch.cuda.synchronize()
    KB = 64
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(KB):
        model.rerank(bts[i % 4], *lists[i % 4])
    t1.record()
    torch.cuda.synchronize()
    batch_us = t0.elapsed_time(t1) / KB * 1e3
    t0.record()
    for i in range(KB):
        model._session_forward(bts[i % 4])
    t1.record()
    torch.cuda.synchronize()
    fwd_us = t0.elapsed_time(t1) / KB * 1e3
    nbytes = nnz * (2 * 1024 + 5 * 4) + B * (nv.XW + nv.NBINS) * 4 + (B + 1 + nnz) * 4 + B * 4
    res = dict(info, workload=f"T={T}, " + (f"L={fixed_len}" if fixed_len else "L~LogNormal(mean 37)"),
               N=N_MIND, B=B, T=T, mean_len=round(nnz / B, 2), max_len=max_len, kernel_us_cold=round(cold, 2),
               kernel_us_warm=round(warm, 2), batch_us=round(batch_us, 1), forward_us=round(fwd_us, 1),
               sessions_per_s=round(B / batch_us * 1e6), bytes=nbytes,
               gbps_cold=round(nbytes / cold / 1e3, 1), hbm_share=round(nbytes / HBM_BPS / (cold * 1e-6), 4),
               hbm_bound="7.7 TB/s HBM3e (B200 data sheet)")
    print("rerank_probe " + json.dumps(res), flush=True)


def check():
    """test_impressions under torchrun (batch i on rank i mod world, sums all-reduced) == the same split on one GPU."""
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    gpus = torch.cuda.device_count()
    torch.cuda.set_device(local % gpus)
    if gpus >= world:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:                                                # ranks share a GPU: NCCL needs one GPU per rank, gloo does not
        dist.init_process_group("gloo")
    N = 20000
    len_dict, sdict, tdict, item_dict, impr = synth.make_sessions(N, 3000, train=False, impressions="mind")
    impr[0] = ["x1"]                                     # one session without a known negative: skipped
    out = {}
    for w in (world, 1):
        model, _ = make_model(N, rank if w > 1 else 0, w, seed=3)
        random.seed(7)                                   # same batches for both runs
        out[w] = model.test_impressions(None, (copy.deepcopy(len_dict), sdict, tdict), impr, item_dict, {})
    a, b = out[world], out[1]
    same = a["sessions"] == b["sessions"] and a["skipped"] == b["skipped"] and \
        all(abs(a[k] - b[k]) <= 1e-12 for k in ("auc", "mrr", "ndcg5", "ndcg10"))
    print(f"rank {rank} rerank_check " + json.dumps(dict(gpu_info(), world=world, gpus=min(gpus, world),
                                                         backend=dist.get_backend(), world_n=a, world_1=b, equal=same)),
          flush=True)
    dist.destroy_process_group()
    if not same:
        sys.exit(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    if ap.parse_args().check:
        return check()
    torch.cuda.set_device(0)
    info = gpu_info()
    model, mwdhm = make_model(N_MIND)
    for T, L in ((1, 0), (20, 0), (20, 300)):
        workload(model, mwdhm, T, L, info)


if __name__ == "__main__":
    main()
