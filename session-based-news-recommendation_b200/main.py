# coding=utf-8
"""CLI with the reference's 23 flags (main.py:91-125).  Additions: --impression_path / --category_path replace the
two hard-coded /home/sansa/... paths of the reference (util.py:47, main.py:36)."""
import argparse
import importlib
import os
import pickle
import random

import numpy as np

random.seed(2020)
np.random.seed(2020)


def load_datas(args):
    """main.py:14-47."""
    from .util import data_partition
    print("load the datasets.")
    base = args.datapath + args.dataset + args.split_way
    dataset = data_partition(base, args.foldnum, args.impression_path)
    train_data, test_data, item_dict, neighbor, content_emb, publish_time, _ = dataset
    item_freq_dict_norm = pickle.load(open(base + "item_freq_dict_norm_" + str(args.foldnum) + ".txt", "rb"))
    args = vars(args)
    args["itemnum"] = len(item_dict)
    args["reverse_item"] = {cnt - 1: idx for idx, cnt in item_dict.items()}
    cat_path = args.get("category_path") or base + "articles_category.pkl"
    args["category_id"] = pickle.load(open(cat_path, "rb"))
    args["item_freq_dict_norm"] = item_freq_dict_norm
    args["publish_time"] = publish_time[0]
    args["publish_time_MWDHM"] = publish_time[1]
    args["content_emb"] = content_emb
    print("------", len(item_dict), len(publish_time[1]))
    return train_data, test_data, neighbor, args, item_dict


def main(args):
    is_train, model_path, input_data, modelname = args.train, args.modelpath, args.inputdata, args.model
    train_data, test_data, neighbor, args, item_dict = load_datas(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        # launched with torchrun: one process per GPU (NCCL over NVLink); every rank loads the same data and draws the
        # same batches (same seeds above), see parallel.py
        import torch
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        args["rank"], args["world_size"] = int(os.environ["RANK"]), world
    pkg = __package__ or "tcar_b200"
    module = importlib.import_module(pkg + "." + modelname)            # main.py:65-66 `__import__(args.model)`
    model = getattr(module, "Seq2SeqAttNN")(args)
    if is_train:
        print("Begin Training")
        model.train(None, item_dict, train_data, neighbor, args, test_data, None)
    else:
        from .util import restore_model
        sent_data = train_data if input_data == "train" else test_data
        print("Begin Testing. Test data is %s data" % ("train" if input_data == "train" else "test"))
        restore_model(model, model_path)
        model.test(None, sent_data, args)
    if args.get("impression_eval"):
        model.test_impressions(None, test_data if is_train else sent_data, neighbor, item_dict, args)
    if args.get("recommend_k") is not None or args.get("recommend_exclude_clicked"):
        model.recommend_split(None, test_data if is_train else sent_data, item_dict, args)
    return model


def recommend_k(text):
    """--recommend_k: an integer in [1, TCAR_RECOMMEND_MAXK], checked before any data is loaded."""
    from ._native import RECOMMEND_MAXK
    k = int(text)
    if not 1 <= k <= RECOMMEND_MAXK:
        raise argparse.ArgumentTypeError(f"must be in [1, {RECOMMEND_MAXK}]")
    return k


def max_age_hours(text):
    """--recommend_max_age_h: a float number of hours > 0."""
    h = float(text)
    if not h > 0:
        raise argparse.ArgumentTypeError("must be > 0 hours")
    return h


def half_life_hours(text):
    """--recommend_half_life_h: a finite float number of hours > 0."""
    h = float(text)
    if not 0 < h < float("inf"):
        raise argparse.ArgumentTypeError("must be a finite number of hours > 0")
    return h


def max_per_category(text):
    """--recommend_max_per_category: an integer >= 1."""
    c = int(text)
    if c < 1:
        raise argparse.ArgumentTypeError("must be >= 1")
    return c


class _Parser(argparse.ArgumentParser):
    """Checks the flags that depend on one another right after parsing, before any data is loaded."""

    def parse_args(self, args=None, namespace=None):
        ns = super().parse_args(args, namespace)
        if getattr(ns, "recommend_max_age_h", None) is not None and ns.recommend_k is None:
            self.error("--recommend_max_age_h requires --recommend_k")
        if getattr(ns, "recommend_max_per_category", None) is not None:
            if ns.recommend_k is None:
                self.error("--recommend_max_per_category requires --recommend_k")
            if ns.recommend_max_age_h is not None:
                self.error("--recommend_max_per_category cannot be combined with --recommend_max_age_h")
        if getattr(ns, "recommend_half_life_h", None) is not None:
            if ns.recommend_k is None:
                self.error("--recommend_half_life_h requires --recommend_k")
            if ns.recommend_max_per_category is not None:
                self.error("--recommend_half_life_h cannot be combined with --recommend_max_per_category")
        return ns


def build_parser():
    parser = _Parser()
    # DATASET PARAMETERS
    parser.add_argument("--datapath", default="./data/", type=str, help="Location of pre-processed dataset")
    parser.add_argument("--dataset", default="mind/TCAR-mid/", type=str, help="Dataset")
    parser.add_argument("--split_way", default="Normal/", type=str, choices=["Normal/", "TrainLen/", "TestLen/"])
    parser.add_argument("--foldnum", default=1, type=int)
    # TRAIN PARAMETERS
    parser.add_argument("--batch_size", default=512, type=int)
    parser.add_argument("--lr", default=0.001, type=float)
    parser.add_argument("--epoch", default=10, type=int)
    parser.add_argument("--maxlen", default=20, type=int)
    parser.add_argument("--neg_num", default=20, type=int)
    # MODEL PARAMETERS
    parser.add_argument("--model", default="model_combine", type=str)
    parser.add_argument("--hidden_size", default=250, type=int)
    parser.add_argument("--time_hidden_size", default=64, type=int)
    parser.add_argument("--max_grad", default=150, type=int)
    parser.add_argument("--stddev", default=0.05, type=float)
    parser.add_argument("--emb_stddev", default=0.002, type=float)
    parser.add_argument("--dropout_rate", default=0.5, type=float)
    parser.add_argument("--l2_emb", default=0.0, type=float)
    # OTHER SETTING (type=bool kept: any non-empty string is True, like the reference)
    parser.add_argument("--save", default=False, type=bool)
    parser.add_argument("--is_print", default=False, type=bool)
    parser.add_argument("--train", default=True, type=bool)
    parser.add_argument("--modelpath", default="./ckpt/", type=str)
    # not a reference flag: GPU-resident sampler (SURVEY 8f-2).  off = host Sampler; host = batches assembled on the
    # device with the reference's NumPy negatives (identical batches); device = Philox negatives drawn on the device
    parser.add_argument("--device_sampler", default="off", choices=["off", "host", "device"], type=str)
    # not a reference flag: multi-GPU training layout under torchrun.  dp = data parallel + gradient all-reduce,
    # catalog = softmax sharded over the item catalog (catalog_parallel.py, SURVEY 8e row 2 / 8f-3)
    parser.add_argument("--train_parallel", default="dp", choices=["dp", "catalog"], type=str)
    # not a reference flag: what a step is under torchrun.  per_rank = every GPU its own batch of --batch_size sessions
    # (global batch = GPUs x batch_size: weak scaling, a different optimisation trajectory than one GPU); split = ONE
    # batch of --batch_size sessions split over the GPUs (the single-GPU trajectory)
    parser.add_argument("--dist_batch", default="per_rank", choices=["per_rank", "split"], type=str)
    # not a reference flag: the reference ships uniform negatives (sampler.py:98-99) and keeps the impression-list
    # sampler of the MIND experiments commented out (sampler.py:96,118-131); this switch selects it
    parser.add_argument("--negative_mode", default="uniform", choices=["uniform", "impression"], type=str)
    # not a reference flag: after training / testing, also rank every session's impression list (the MIND protocol:
    # AUC, MRR, nDCG@5, nDCG@10; Seq2SeqAttNN.test_impressions) with the impression file as the neighbour dict
    parser.add_argument("--impression_eval", action="store_true")
    # not a reference flag: after training / testing, also write every session's exact top-K of the whole catalog
    # (Seq2SeqAttNN.recommend_split: saved/recommend_<foldnum>.txt, HR / MRR / nDCG@K); K defaults to 20, at most 256
    parser.add_argument("--recommend_k", default=None, type=recommend_k)
    # not a reference flag: leave a session's own clicked articles out of its recommendations
    parser.add_argument("--recommend_exclude_clicked", action="store_true")
    # not a reference flag: recommend only articles published at most H hours before the session's last input click
    # (the time-aware protocol: publish-time windows applied exactly on the device, Seq2SeqAttNN.recommend_split)
    parser.add_argument("--recommend_max_age_h", default=None, type=max_age_hours)
    # not a reference flag: at most C articles of one category per recommended list (exact capped top-K on the device,
    # Seq2SeqAttNN.recommend_split); also prints the lists' ILD and unexpectedness
    parser.add_argument("--recommend_max_per_category", default=None, type=max_per_category)
    # not a reference flag: rank by the score minus a freshness penalty that halves an article's recommendation
    # probability every H hours of age at the session's last input click (exact on the device, recommend(decay=...));
    # also prints the mean age of the returned articles
    parser.add_argument("--recommend_half_life_h", default=None, type=half_life_hours)
    parser.add_argument("--inputdata", default="test", type=str)
    parser.add_argument("--threshold_acc", default=0.27, type=float)
    # additions
    parser.add_argument("--impression_path", default=None, type=str)
    parser.add_argument("--category_path", default=None, type=str)
    return parser


if __name__ == "__main__":
    main(build_parser().parse_args())
