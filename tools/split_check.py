"""Run under torchrun: the split walkers of Seq2SeqAttNN -- test() (catalog-sharded eval_round, one round per `world`
batches), test_impressions() and recommend_split() (batch i on rank i mod world; once more with 24 h publish-time
windows, once more with at most 2 articles per category, once more with a 6 h freshness half-life inside 48 h
windows) -- on one synthetic split at world N equal the same walkers at world 1.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 \\
        tools/split_check.py

NCCL with a GPU per rank; ranks sharing a GPU use gloo.  Equal means: metrics within 1e-12 absolute (test()'s loss
within 1e-5 relative: the sharded softmax sums in another order), session counts, `skipped` and test()'s coverage
equal, and the ranks' recommend_split files together hold line for line the single-process file.  Prints one JSON line
per rank and exits with status 1 on a mismatch.
"""
import copy
import datetime
import json
import os
import random
import sys
import tempfile

import numpy as np
import torch.distributed as dist

from probe_common import gpu_info, init_torchrun, make_model
from tcar_b200 import synth

N, SESSIONS, K = 20000, 3000, 100


def publish_times(n):
    """Article publish times over the sessions' two weeks (synth.make_sessions: clicks from day 31 to 45 after
    2017-10-01), so that a 24 h window holds a few percent of the catalog."""
    rs = np.random.RandomState(11)
    t0 = datetime.datetime(2017, 10, 1) + datetime.timedelta(days=30)
    return [t0 + datetime.timedelta(minutes=int(m)) for m in rs.randint(0, 60 * 24 * 16, n)]


def categories(item_dict):
    """Article -> category over G = 461 codes, every 50th article without one."""
    rs = np.random.RandomState(12)
    return {art: int(rs.randint(0, 461)) for art, cnt in item_dict.items() if cnt % 50}


def run_walkers(model, split, impressions, item_dict):
    """The walkers on the same batches (Sampler shuffles len_dict in place and draws from `random`); recommend_split
    also with 24 h publish-time windows (written to recommend_1*.txt), with at most 2 articles per category
    (recommend_2*.txt) and with a 6 h half-life inside 48 h windows (recommend_3*.txt)."""
    def fresh():
        random.seed(7)
        return (copy.deepcopy(split[0]), *split[1:])
    out = {"impressions": model.test_impressions(None, fresh(), impressions, item_dict, {}),
           "recommend": model.recommend_split(None, fresh(), item_dict,
                                              {"recommend_k": K, "recommend_exclude_clicked": True, "foldnum": 0}),
           "recommend_window": model.recommend_split(None, fresh(), item_dict,
                                                     {"recommend_k": K, "recommend_exclude_clicked": True,
                                                      "recommend_max_age_h": 24.0, "publish_time": publish_times(N),
                                                      "foldnum": 1}),
           "recommend_decay": model.recommend_split(None, fresh(), item_dict,
                                                    {"recommend_k": K, "recommend_exclude_clicked": True,
                                                     "recommend_half_life_h": 6.0, "recommend_max_age_h": 48.0,
                                                     "publish_time": publish_times(N), "foldnum": 3})}
    model.reverse_item = {cnt - 1: art for art, cnt in item_dict.items()}
    model.category_id = categories(item_dict)
    out["recommend_capped"] = model.recommend_split(None, fresh(), item_dict,
                                                    {"recommend_k": K, "recommend_exclude_clicked": True,
                                                     "recommend_max_per_category": 2, "foldnum": 2})
    model.reverse_item = model.category_id = model._cat_array = None
    model.test(None, fresh(), {})
    out["test"] = model.last_metrics
    return out


def close(a, b, exact=(), rel=()):
    return all(a[k] == b[k] if k in exact else
               abs(a[k] - b[k]) <= (1e-5 * abs(b[k]) if k in rel else 1e-12) for k in b)


def main():
    rank, world, gpus = init_torchrun()
    len_dict, sdict, tdict, item_dict, impr = synth.make_sessions(N, SESSIONS, train=False, impressions="mind")
    impr[0] = ["x1"]                                     # one session without a known negative: skipped
    base = [tempfile.mkdtemp(prefix="split_check_") if rank == 0 else None]
    dist.broadcast_object_list(base)
    base = base[0]
    res = {}
    for w in (world, 1):
        d = os.path.join(base, f"world{w}" + (f"_rank{rank}" if w == 1 else ""))
        os.makedirs(d, exist_ok=True)
        os.chdir(d)
        model, _ = make_model(N, rank if w > 1 else 0, w, seed=3)
        res[w] = run_walkers(model, (len_dict, sdict, tdict), impr, item_dict)
        dist.barrier()
    a, b = res[world], res[1]

    def lines(fold):
        n = []
        for r in range(world):
            with open(os.path.join(base, f"world{world}", f"saved/recommend_{fold}_rank{r}.txt")) as f:
                n += f.read().splitlines()
        with open(os.path.join(base, f"world1_rank{rank}", f"saved/recommend_{fold}.txt")) as f:
            return n, f.read().splitlines()
    lines_n, lines_1 = lines(0)
    win_n, win_1 = lines(1)
    cap_n, cap_1 = lines(2)
    dec_n, dec_1 = lines(3)
    equal = {"test": close(a["test"], b["test"], exact=("coverage",), rel=("loss",)),
             "impressions": close(a["impressions"], b["impressions"], exact=("sessions", "skipped")),
             "recommend": close(a["recommend"], b["recommend"], exact=("sessions",)),
             "recommend_files": sorted(lines_n) == sorted(lines_1) and len(lines_1) == b["recommend"]["sessions"],
             "recommend_window": close(a["recommend_window"], b["recommend_window"],
                                       exact=("sessions", "label_outside")),
             "recommend_window_files": sorted(win_n) == sorted(win_1) and
             len(win_1) == b["recommend_window"]["sessions"],
             "recommend_capped": close(a["recommend_capped"], b["recommend_capped"], exact=("sessions",)),
             "recommend_capped_files": sorted(cap_n) == sorted(cap_1) and
             len(cap_1) == b["recommend_capped"]["sessions"],
             "recommend_decay": close(a["recommend_decay"], b["recommend_decay"],
                                      exact=("sessions", "label_outside")),
             "recommend_decay_files": sorted(dec_n) == sorted(dec_1) and
             len(dec_1) == b["recommend_decay"]["sessions"]}
    ok = all(equal.values())
    print(f"rank {rank} split_check " + json.dumps(dict(gpu_info(), world=world, gpus=gpus, backend=dist.get_backend(),
                                                        sessions=SESSIONS, K=K, exclude_clicked=True, world_n=a,
                                                        world_1=b, lines=len(lines_1), equal=equal, ok=ok)), flush=True)
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
