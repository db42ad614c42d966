"""Host-side mirror of the reference interface (no GPU): the product Sampler / util / main against the golden vectors
that tests/golden/make_golden.py produced by running the reference's own sampler.py / util.py, and the on-disk
pickle layout round trip."""
import datetime
import json
import os
import random
import tempfile

import numpy as np
import pytest

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _datasets():
    d = json.load(open(os.path.join(G, "sampler_ref.json")))
    len_dict = {int(k): list(v) for k, v in d["len_dict"].items()}
    time_dict = {k: [{"click_t": datetime.datetime.fromisoformat(t["click_t"]),
                      "publish_t": datetime.datetime.fromisoformat(t["publish_t"]), "active_t": t["active_t"]}
                     for t in v] for k, v in d["time_dict"].items()}
    item_dict = {"orig%d" % i: i + 1 for i in range(d["N"])}
    impressions = {int(k): v for k, v in d["impressions"].items()}
    return d, len_dict, d["session_dict"], time_dict, item_dict, impressions


def test_product_sampler_reproduces_reference_batches():
    """Same RNG streams, same shuffles, same negatives, same time features as sampler.py (bit-exact lists)."""
    from tcar_b200.sampler import Sampler
    d, len_dict, session_dict, time_dict, item_dict, impressions = _datasets()
    for run in d["runs"]:
        random.seed(2020)
        np.random.seed(2020)
        ld = {k: list(v) for k, v in len_dict.items()}
        s = Sampler(ld, session_dict, time_dict, impressions, item_dict, run["neg_num"], batch_size=run["batch_size"],
                    verbose=False)
        got = []
        while s.has_next():
            b_in, b_out, pt, ct, neg, gap = s.next_batch()
            got.append({"in": b_in, "out": b_out, "pt": [list(x) for x in pt], "ct": [list(x) for x in ct],
                        "neg": neg, "gap": gap})
        assert got == run["batches"]
        assert [s.neg_neighbor_from_impre(i) for i in range(5)] == run["impre"]
        assert {str(k): v for k, v in ld.items()} == run["shuffled_len_dict"]


def test_vectorised_next_packed_reproduces_reference_batches():
    """The columnar / single-randint path yields the reference's batches (same shuffles, same negatives)."""
    from tcar_b200.sampler import Sampler, pack_batch
    d, len_dict, session_dict, time_dict, item_dict, impressions = _datasets()
    for run in d["runs"]:
        random.seed(2020)
        np.random.seed(2020)
        s = Sampler({k: list(v) for k, v in len_dict.items()}, session_dict, time_dict, impressions, item_dict,
                    run["neg_num"], batch_size=run["batch_size"], verbose=False)
        for ref in run["batches"]:
            packed, B, T, Nn = s.next_packed()
            want, *_ = pack_batch(ref["in"], ref["out"], ref["pt"], ref["ct"], ref["neg"], ref["gap"])
            np.testing.assert_array_equal(packed, want)
            b_in, b_out, neg = s.last_lists()
            assert b_in == ref["in"] and b_out == ref["out"] and neg == ref["neg"]
        assert not s.has_next()


def test_prefetcher_preserves_order_and_content():
    from tcar_b200.model_combine import prefetch_packed
    from tcar_b200.sampler import Sampler
    d, len_dict, session_dict, time_dict, item_dict, impressions = _datasets()
    run = d["runs"][0]
    outs = []
    for use_thread in (False, True):
        random.seed(5)
        np.random.seed(5)
        s = Sampler({k: list(v) for k, v in len_dict.items()}, session_dict, time_dict, impressions, item_dict,
                    run["neg_num"], batch_size=run["batch_size"], verbose=False)
        if use_thread:
            outs.append([p.copy() for p, *_ in prefetch_packed(s, depth=2)])
        else:
            got = []
            while s.has_next():
                got.append(s.next_packed()[0].copy())
            outs.append(got)
    assert len(outs[0]) == len(outs[1]) > 0
    for a, b in zip(*outs):
        np.testing.assert_array_equal(a, b)


def test_prefetcher_lowers_the_gil_switch_interval_only_while_it_runs():
    """The producer thread and the launching thread share the GIL: prefetch_packed shortens CPython's switch interval
    for the lifetime of the iterator (also when the consumer abandons it early) and restores the caller's value."""
    import sys
    from tcar_b200.model_combine import prefetch_packed
    from tcar_b200.sampler import Sampler
    d, len_dict, session_dict, time_dict, item_dict, impressions = _datasets()
    run = d["runs"][0]
    before = sys.getswitchinterval()
    for abandon in (False, True):
        random.seed(5)
        np.random.seed(5)
        s = Sampler({k: list(v) for k, v in len_dict.items()}, session_dict, time_dict, impressions, item_dict,
                    run["neg_num"], batch_size=run["batch_size"], verbose=False)
        it = prefetch_packed(s, depth=2)
        next(it)
        assert sys.getswitchinterval() <= 1e-4 + 1e-12
        if abandon:
            it.close()
        else:
            for _ in it:
                pass
        assert sys.getswitchinterval() == before


def test_next_packed_is_the_same_batch_in_one_buffer():
    from tcar_b200.sampler import Sampler, pack_batch
    d, len_dict, session_dict, time_dict, item_dict, impressions = _datasets()
    run = d["runs"][0]
    twins = []
    for _ in range(2):
        random.seed(7)
        np.random.seed(7)
        twins.append(Sampler({k: list(v) for k, v in len_dict.items()}, session_dict, time_dict, impressions, item_dict,
                             run["neg_num"], batch_size=run["batch_size"], verbose=False))
    a, b = twins
    n = 0
    while a.has_next():
        # the two samplers share the global NumPy stream: draw them one after the other from the same state
        state = np.random.get_state()
        ref = a.next_batch()
        np.random.set_state(state)
        packed, B, T, Nn = b.next_packed()
        want, B2, T2, Nn2 = pack_batch(*ref)
        assert (B, T, Nn) == (B2, T2, Nn2)
        np.testing.assert_array_equal(packed, want)
        assert packed.dtype == np.int32 and packed.size == 7 * B * T + 3 * B + B * Nn
        n += 1
    assert n == len(run["batches"]) and not b.has_next()


def test_dwell_bucket_is_clamped_to_the_table():
    """bucketized(active_t >= 1024 s) = 11 is out of range for the 11-row duration table (sampler.py:18-21):
    next_packed / pack_batch clamp it to 10 (documented deviation)."""
    from tcar_b200.sampler import bucketized, pack_batch
    assert bucketized(1023) == 10 and bucketized(1024) == 11
    packed, B, T, Nn = pack_batch([[1, 2]], [0], ([[1, 1]], [[1, 1]], [[1, 1]], [[1, 1]], [[1, 1]]),
                                  ([0], [0], [3], [5], [0]), [[]], [[11, 4]])
    assert (B, T, Nn) == (1, 2, 0)
    assert packed[6 * 2: 7 * 2].tolist() == [10, 4]
    assert packed[7 * 2: 7 * 2 + 2].tolist() == [3, 5]          # click week, click hour


def test_cau_metrics_match_reference():
    from tcar_b200.util import cau_metrics
    m = json.load(open(os.path.join(G, "metrics_ref.json")))
    recall, mrr, ndcg = cau_metrics(np.array(m["preds"], dtype=np.float32), m["labels"], 20)
    assert [bool(x) for x in recall] == m["recall"]
    np.testing.assert_allclose(mrr, m["mrr"])
    np.testing.assert_allclose(ndcg, m["ndcg"])


def test_cli_keeps_the_reference_flags_and_defaults():
    """main.py:94-123 -- 23 flags, names and defaults."""
    from tcar_b200.main import build_parser
    ref = {"datapath": "./data/", "dataset": "mind/TCAR-mid/", "split_way": "Normal/", "foldnum": 1,
           "batch_size": 512, "lr": 0.001, "epoch": 10, "maxlen": 20, "neg_num": 20, "model": "model_combine",
           "hidden_size": 250, "time_hidden_size": 64, "max_grad": 150, "stddev": 0.05, "emb_stddev": 0.002,
           "dropout_rate": 0.5, "l2_emb": 0.0, "save": False, "is_print": False, "train": True,
           "modelpath": "./ckpt/", "inputdata": "test", "threshold_acc": 0.27}
    got = vars(build_parser().parse_args([]))
    for k, v in ref.items():
        assert got[k] == v, k
    assert len(ref) == 23
    # type=bool flags keep the reference quirk: any non-empty string is True (main.py:118-120)
    assert build_parser().parse_args(["--train", "False"]).train is True


def test_pickle_layout_round_trip():
    """synth.write_dataset emits the reference's on-disk layout (SURVEY 8f-1); util.data_partition / main.load_datas
    read it back with the reference's 7-tuple / args keys."""
    from tcar_b200 import main as tmain, synth
    from tcar_b200.util import data_partition
    with tempfile.TemporaryDirectory() as d:
        root = d + "/synth/TCAR-mid/Normal/"
        synth.write_dataset(root, N=300, n_train=120, n_test=40, fold=0)
        train, test, item_dict, neighbor, content, publish, _ = data_partition(root, 0)
        len_dict, session_dict, time_dict = train
        assert len(item_dict) == 300 and content.shape == (301, 250) and np.all(content[0] == 0)
        assert publish[1].shape == (300, 5) and len(publish[0]) == 300
        for L, keys in len_dict.items():
            for k in keys:
                assert len(session_dict[k]) == L + 1 and len(time_dict[k]) == L + 1      # inputs + target
                assert str(k).endswith("_%d" % L)                                        # train key "<sid>_<len>"
        assert all(isinstance(k, int) for k in test[1])                                  # test key = sid
        args = tmain.build_parser().parse_args(["--datapath", d + "/", "--dataset", "synth/TCAR-mid/", "--foldnum", "0"])
        _, _, _, a, _ = tmain.load_datas(args)
        for key in ("itemnum", "reverse_item", "category_id", "item_freq_dict_norm", "publish_time_MWDHM",
                    "content_emb"):
            assert key in a
        assert a["reverse_item"][0] == "a0" and a["itemnum"] == 300


def test_model_refuses_to_run_without_cuda(monkeypatch):
    """No CPU fallback: constructing the product model on a GPU-less host fails loudly (a host with a GPU is made to
    look GPU-less)."""
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    from tcar_b200.model_combine import Seq2SeqAttNN
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Seq2SeqAttNN({"itemnum": 1})


def test_cfg1_plumbing_epoch_on_cpu():
    """BASELINE.json configs[0] (`main.py --foldnum=0 --epoch=1` on small synthetic Globo-shaped sessions, CPU): the
    host side of the product (pickle loader, CLI args, Sampler / next_packed) drives the ORACLE's train step and eval
    for one epoch -- the plumbing the reference runs around sess.run (model_combine.py:196-315), minus the device."""
    import torch
    from oracle import tcar_oracle as O
    from tcar_b200 import main as tmain, synth
    from tcar_b200.sampler import Sampler
    with tempfile.TemporaryDirectory() as d:
        synth.write_dataset(d + "/synth/TCAR-mid/Normal/", N=150, n_train=90, n_test=30, fold=0)
        cli = tmain.build_parser().parse_args(["--datapath", d + "/", "--dataset", "synth/TCAR-mid/", "--foldnum", "0",
                                               "--epoch", "1", "--batch_size", "32"])
        train, test, neighbor, a, item_dict = tmain.load_datas(cli)
    N = a["itemnum"]
    content = torch.from_numpy(np.asarray(a["content_emb"], dtype=np.float64))
    mwdhm = torch.from_numpy(np.asarray(a["publish_time_MWDHM"]).astype(np.int64))
    np.random.seed(2020)
    params = {k: v.double() for k, v in O.init_params(N, a["emb_stddev"], a["stddev"]).items()}
    adam = O.TFAdam(params, a["lr"])
    sampler = Sampler(*train, neighbor, item_dict, a["neg_num"], batch_size=a["batch_size"], verbose=False)
    losses, sessions = [], 0
    while sampler.has_next():
        packed, B, T, Nn = sampler.next_packed()
        batch = {k: torch.from_numpy(v) for k, v in synth.unpack(packed, B, T, Nn).items()}
        assert B <= a["batch_size"] and Nn == a["neg_num"] and int(batch["seq"].min()) >= 1
        out, _ = O.train_step(params, adam, content, mwdhm, batch, max_grad=float(a["max_grad"]))
        losses.append(float(out["loss"].mean()))
        sessions += B
    assert sessions == sum(len(v) for v in train[0].values()) and np.isfinite(losses).all()
    # cross-entropy of an untrained softmax over N items ~ log N; negative feedback adds 0.01 * ~log 2
    assert abs(losses[0] - np.log(N)) < 0.5
    # evaluation loop (model_combine.py:254-315): metrics of every test session, Recall/MRR in [0, 1]
    ev = Sampler(*test, batch_size=a["batch_size"], verbose=False)
    recall, mrr, n = [], [], 0
    while ev.has_next():
        packed, B, T, Nn = ev.next_packed()
        assert Nn == 0
        batch = {k: torch.from_numpy(v) for k, v in synth.unpack(packed, B, T, 0).items()}
        with torch.no_grad():
            res = O.eval_batch(params, content, mwdhm, batch, a["category_id"], a["reverse_item"])
        recall += list(res["recall"])
        mrr += list(res["mrr"])
        n += B
    assert n == sum(len(v) for v in test[0].values())
    assert 0.0 <= float(np.mean(recall)) <= 1.0 and 0.0 <= float(np.mean(mrr)) <= 1.0


def test_print_data_dump_parses_with_the_reference_evaluation_script(tmp_path, monkeypatch):
    """--is_print dump (model_combine.py:165-169): every line must split the way data_process/evaluation_predict.py:16-26
    splits it (restated below: the script itself reads a hard-coded path and cannot be imported as a function of text)."""
    from tcar_b200.model_combine import Seq2SeqAttNN
    monkeypatch.chdir(tmp_path)
    batch_in = [[5, 17, 3], [9, 9, 1]]
    batch_out = [41, 0]
    batch_pred = [[7, 41, 2, 300000], []]                 # an empty recommendation list is legal (pred_split[0] == '')
    Seq2SeqAttNN.printData(None, "0_3", batch_in, batch_out, batch_pred)
    Seq2SeqAttNN.printData(None, "0_3", batch_in[:1], batch_out[:1], batch_pred[:1])      # appended ('a+')
    lines = open(tmp_path / "saved" / "CAR+P_Normal_predict_exa_0_3.txt").readlines()
    assert len(lines) == 3
    got = []
    for line in lines:
        in_ = [int(x) for x in line.split("# batch in: [")[1].split("]")[0].split(", ")]       # evaluation_predict.py:16
        out_ = int(line.split("# batch out: ")[1].split(" #")[0])                              # :18
        pred_split = line.split("# batch pred: [")[1].split("]")[0].split(", ")                # :19
        pred_ = [] if pred_split[0] == "" else [int(x) for x in pred_split]                    # :20-23
        got.append((in_, out_, pred_))
    assert got == [(batch_in[0], 41, batch_pred[0]), (batch_in[1], 0, []), (batch_in[0], 41, batch_pred[0])]


def test_restrict_to_rank_partitions_every_global_batch():
    """Per-rank batches of the multi-GPU train loop (Seq2SeqAttNN.train, dist_batch='per_rank'): samplers built alike
    on every rank (same `random` seed) and restricted to their rank must partition every global batch -- same order,
    same session length, shares of at most batch_size sessions -- and the shares' packed planes must be the rows of
    the global batch's."""
    import random
    from tcar_b200 import parallel, synth
    from tcar_b200.sampler import Sampler
    N, world, B = 400, 4, 16
    ld, sd, td, idict, impr = synth.make_sessions(N, 700, seed=8)
    random.seed(5)
    np.random.seed(5)
    ref = Sampler({k: list(v) for k, v in ld.items()}, sd, td, impr, idict, 3, batch_size=B * world, verbose=False)
    global_ids = [list(b) for b in ref.session_id_batches]
    parts = []
    for r in range(world):
        random.seed(5)
        s = Sampler({k: list(v) for k, v in ld.items()}, sd, td, impr, idict, 3, batch_size=B * world, verbose=False)
        s.restrict_to_rank(r, world)
        assert s.global_sizes == [len(b) for b in global_ids]
        parts.append(s)
    for i, ids in enumerate(global_ids):
        got = []
        for r, s in enumerate(parts):
            share = s.session_id_batches[i]
            assert len(share) <= B
            assert len(share) == parallel.catalog_counts(len(ids), world)[r]
            got += share
        assert got == ids
    # packed shares: sequence plane and labels are slices of the global batch's
    full = [ref.next_packed() for _ in range(3)]
    for r, s in enumerate(parts):
        for i in range(3):
            packed, Bl, T, Nn = s.next_packed()
            gp, Bg, Tg, _ = full[i]
            lo, hi = parallel.shard_sessions(Bg, r, world)
            assert (Bl, T) == (hi - lo, Tg)
            np.testing.assert_array_equal(packed[: Bl * T].reshape(Bl, T), gp[: Bg * Tg].reshape(Bg, Tg)[lo:hi])
            np.testing.assert_array_equal(packed[7 * Bl * T + 2 * Bl: 7 * Bl * T + 3 * Bl],
                                          gp[7 * Bg * Tg + 2 * Bg: 7 * Bg * Tg + 3 * Bg][lo:hi])


def test_restrict_to_rank_keeps_the_global_random_stream_in_lockstep():
    """Impression negatives of a restricted sampler use a private random.Random: the global `random` stream -- which
    shuffles the next epoch's batches and must stay identical on all ranks -- is not consumed by sampling."""
    import random
    from tcar_b200 import synth
    from tcar_b200.sampler import Sampler
    N = 300
    ld, sd, td, idict, _ = synth.make_sessions(N, 200, seed=9)
    impr = synth.make_impressions(N, 200, seed=9, mean_len=5.0, miss=0.3)
    states = []
    for r in range(2):
        random.seed(11)
        s = Sampler({k: list(v) for k, v in ld.items()}, sd, td, impr, idict, 4, batch_size=32,
                    negative_mode="impression", verbose=False)
        s.restrict_to_rank(r, 2)
        while s.has_next():
            s.next_packed()
        states.append(random.getstate())
    assert states[0] == states[1]
