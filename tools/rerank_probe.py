"""Candidate re-ranking on the GPU (tcar_rerank, Seq2SeqAttNN.rerank): one JSON line per workload at the MIND shape
(catalog of 103 630 items, 512 sessions per batch).

    python tools/rerank_probe.py             T in {1, 20} x MIND-like list lengths (LogNormal, mean 37); T = 20 x 300

test_impressions across ranks is checked by tools/split_check.py.

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
import json

import numpy as np
import torch

from probe_common import B, gpu_info, make_model
from tcar_b200 import _native as nv, synth

N_MIND = 103630
HBM_BPS = 7.7e12


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


def main():
    torch.cuda.set_device(0)
    info = gpu_info()
    model, mwdhm = make_model(N_MIND)
    for T, L in ((1, 0), (20, 0), (20, 300)):
        workload(model, mwdhm, T, L, info)


if __name__ == "__main__":
    main()
