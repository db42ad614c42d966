"""Run under torchrun: the split walkers of Seq2SeqAttNN -- test() (catalog-sharded eval_round, one round per `world`
batches), test_impressions() and recommend_split() (batch i on rank i mod world) -- on one synthetic split at world N
equal the same walkers at world 1.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29513 \\
        tools/split_check.py

NCCL with a GPU per rank; ranks sharing a GPU use gloo.  Equal means: metrics within 1e-12 absolute (test()'s loss
within 1e-5 relative: the sharded softmax sums in another order), session counts, `skipped` and test()'s coverage
equal, and the ranks' recommend_split files together hold line for line the single-process file.  Prints one JSON line
per rank and exits with status 1 on a mismatch.
"""
import copy
import json
import os
import random
import sys
import tempfile

import torch.distributed as dist

from probe_common import gpu_info, init_torchrun, make_model
from tcar_b200 import synth

N, SESSIONS, K = 20000, 3000, 100


def run_walkers(model, split, impressions, item_dict):
    """The three walkers on the same batches (Sampler shuffles len_dict in place and draws from `random`)."""
    def fresh():
        random.seed(7)
        return (copy.deepcopy(split[0]), *split[1:])
    out = {"impressions": model.test_impressions(None, fresh(), impressions, item_dict, {}),
           "recommend": model.recommend_split(None, fresh(), item_dict,
                                              {"recommend_k": K, "recommend_exclude_clicked": True, "foldnum": 0})}
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
    lines_n = []
    for r in range(world):
        with open(os.path.join(base, f"world{world}", f"saved/recommend_0_rank{r}.txt")) as f:
            lines_n += f.read().splitlines()
    with open(os.path.join(base, f"world1_rank{rank}", "saved/recommend_0.txt")) as f:
        lines_1 = f.read().splitlines()
    equal = {"test": close(a["test"], b["test"], exact=("coverage",), rel=("loss",)),
             "impressions": close(a["impressions"], b["impressions"], exact=("sessions", "skipped")),
             "recommend": close(a["recommend"], b["recommend"], exact=("sessions",)),
             "recommend_files": sorted(lines_n) == sorted(lines_1) and len(lines_1) == b["recommend"]["sessions"]}
    ok = all(equal.values())
    print(f"rank {rank} split_check " + json.dumps(dict(gpu_info(), world=world, gpus=gpus, backend=dist.get_backend(),
                                                        sessions=SESSIONS, K=K, exclude_clicked=True, world_n=a,
                                                        world_1=b, lines=len(lines_1), equal=equal, ok=ok)), flush=True)
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
