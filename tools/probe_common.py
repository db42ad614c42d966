"""What the GPU probes and tools/split_check.py share: the package import from the repository tree, a model on a
synthetic catalog, the card's name and power limit (which belong beside every number), and the torchrun set-up."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

ge.load_package()
from tcar_b200 import synth  # noqa: E402
from tcar_b200.model_combine import Seq2SeqAttNN  # noqa: E402

B = 512


def make_model(N, rank=0, world=1, seed=2020, emb_stddev=0.04):
    """A freshly initialised model (batch size B) on synth.make_catalog(N, seed); returns (model, publish-time bins)."""
    content, mwdhm, _ = synth.make_catalog(N, seed=seed)
    np.random.seed(2020)
    return Seq2SeqAttNN(dict(publish_time_MWDHM=mwdhm, itemnum=N, category_id=None, item_freq_dict_norm={},
                             reverse_item=None, content_emb=content, emb_stddev=emb_stddev, stddev=0.05, hidden_size=250,
                             time_hidden_size=64, l2_emb=0.0, batch_size=B, epoch=1, neg_num=20, lr=0.001,
                             max_grad=150, rank=rank, world_size=world, train_parallel="dp")), mwdhm


def gpu_info():
    idx = torch.cuda.current_device()
    out = subprocess.run(["nvidia-smi", "-i", str(idx), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True).stdout.strip()
    return {"gpu": torch.cuda.get_device_name(idx), "power_limit_w": float(out) if out else None}


def init_torchrun():
    """Join the torchrun process group: NCCL with a GPU per rank; ranks sharing a GPU use gloo (NCCL needs one GPU per
    rank).  Returns (rank, world, GPUs in use)."""
    import torch.distributed as dist
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    gpus = torch.cuda.device_count()
    torch.cuda.set_device(local % gpus)
    if gpus >= world:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        dist.init_process_group("gloo")
    return rank, world, min(gpus, world)
