"""Host side of the split walkers (no GPU): the look-ahead loop, the per-rank batches of evaluation under torchrun and
the checks of per-session id lists."""
import random

import numpy as np
import pytest


# ------------------------------------------------------------------------------------------------- pipelined
def run_pipelined(items, empty=()):
    from tcar_b200.model_combine import pipelined
    log = []

    def launch(cur, nxt):
        log.append(("launch", cur, nxt))
        return None if cur in empty else (cur, "h" + cur)

    def consume(item, handle):
        assert handle == "h" + item
        log.append(("consume", item))

    pipelined(items, launch, consume)
    return log


def test_pipelined_consumes_each_item_after_the_next_launch():
    assert run_pipelined(iter(["a", "b", "c"])) == [
        ("launch", "a", "b"), ("launch", "b", "c"), ("consume", "a"), ("launch", "c", None), ("consume", "b"),
        ("consume", "c")]


def test_pipelined_zero_and_one_item():
    assert run_pipelined([]) == []
    assert run_pipelined(["a"]) == [("launch", "a", None), ("consume", "a")]


def test_pipelined_skips_an_item_without_handles():
    """An empty torchrun round is launched (its collectives must run) but has nothing to read back."""
    assert run_pipelined(["a", "b", "c"], empty={"b"}) == [
        ("launch", "a", "b"), ("launch", "b", "c"), ("consume", "a"), ("launch", "c", None), ("consume", "c")]
    assert run_pipelined(["a", "b"], empty={"b"}) == [("launch", "a", "b"), ("launch", "b", None), ("consume", "a")]


# ------------------------------------------------------------------------------------------------- keep_rank_batches
@pytest.mark.parametrize("world", [1, 2, 3, 5])
def test_keep_rank_batches_partitions_the_split(world):
    """Ranks built alike (same `random` seed) keep batches rank, rank + world, ...: together, in order, the whole
    split; global_sizes / batch_T describe the whole split on every rank, and a rank packs exactly the batches the
    single-process sampler packs for them."""
    from tcar_b200 import synth
    from tcar_b200.sampler import Sampler
    ld, sd, td, _, _ = synth.make_sessions(500, 600, train=False, seed=4)
    random.seed(3)
    ref = Sampler({k: list(v) for k, v in ld.items()}, sd, td, batch_size=32, verbose=False)
    global_ids = [list(b) for b in ref.session_id_batches]
    full = [ref.next_packed() for _ in range(ref.batch_num)]
    assert len(global_ids) > world
    kept = []
    for r in range(world):
        random.seed(3)
        s = Sampler({k: list(v) for k, v in ld.items()}, sd, td, batch_size=32, verbose=False).keep_rank_batches(r, world)
        assert s.global_sizes == [len(b) for b in global_ids]
        assert s.batch_T == [len(sd[b[0]]) - 1 for b in global_ids]
        assert s.batch_num == len(s.session_id_batches) == len(range(r, len(global_ids), world))
        for j, ids in enumerate(s.session_id_batches):
            kept.append((r + j * world, ids))
            packed, B, T, Nn = s.next_packed()
            gp, Bg, Tg, Ng = full[r + j * world]
            assert (B, T, Nn) == (Bg, Tg, Ng)
            np.testing.assert_array_equal(packed, gp)
        assert not s.has_next()
    assert [ids for _, ids in sorted(kept, key=lambda x: x[0])] == global_ids


# ------------------------------------------------------------------------------------------------- check_id_lists
RERANK = dict(names=("cand_off", "cand_ids"), nouns=("candidate id", "candidates"), limit=6, limit_name="TCAR_RERANK_MAXL")
RECOMMEND = dict(names=("exclude_off", "exclude_ids"), nouns=("excluded id", "exclusions"), limit=6,
                 limit_name="TCAR_RECOMMEND_MAXX")
N, B = 500, 4
GOOD_OFF, GOOD_IDS = np.array([0, 2, 3, 3, 5]), np.array([1, 2, 3, 4, 5])


def check(off, ids, words=RERANK, n_items=N, sessions=B, extra=0):
    from tcar_b200.util import check_id_lists
    return check_id_lists(off, ids, sessions, n_items, extra=extra, **words)


@pytest.mark.parametrize("words", [RERANK, RECOMMEND], ids=["rerank", "recommend"])
@pytest.mark.parametrize("off, ids, extra, what", [
    (GOOD_OFF, np.array([1, 2, 3, N, 5]), 0, "session 3: {id} 500 outside [0, 500)"),
    (GOOD_OFF, np.array([1, -1, 3, 4, 5]), 0, "session 0: {id} -1 outside [0, 500)"),
    (np.array([0, 2, 1, 3, 5]), GOOD_IDS, 0, "session 1: {off} decreases"),
    (np.array([0, 1, 1, 1, 8]), np.zeros(8, np.int32), 0, "session 3: more than {limit} = 6 {entries}"),
    (np.array([0, 0, 5, 5, 5]), np.zeros(5, np.int32), 2, "session 1: more than {limit} = 6 {entries} with its 2 clicks"),
    (GOOD_OFF[:-1], GOOD_IDS[:3], 0, "{off} must hold B + 1 = 5 offsets from 0 to len({ids}) = 3"),
    (np.array([1, 2, 3, 3, 5]), GOOD_IDS, 0, "{off} must hold B + 1 = 5 offsets from 0 to len({ids}) = 5"),
    (GOOD_OFF, GOOD_IDS[:4], 0, "{off} must hold B + 1 = 5 offsets from 0 to len({ids}) = 4"),
    (GOOD_OFF.astype(np.float64), GOOD_IDS, 0, "{off} and {ids} must hold integers"),
    (GOOD_OFF, GOOD_IDS.astype(np.float32), 0, "{off} and {ids} must hold integers"),
])
def test_check_id_lists_rejects(words, off, ids, extra, what):
    msg = what.format(off=words["names"][0], ids=words["names"][1], id=words["nouns"][0], entries=words["nouns"][1],
                      limit=words["limit_name"])
    with pytest.raises(ValueError) as e:
        check(off, ids, words, extra=extra)
    assert str(e.value) == msg


@pytest.mark.parametrize("dtype", [np.int32, np.int64, np.uint16, np.uint32, np.uint64])
def test_check_id_lists_packs_any_integer_type(dtype):
    host, longest = check(GOOD_OFF.astype(dtype), GOOD_IDS.astype(dtype))
    assert host.dtype == np.int32 and host.tolist() == GOOD_OFF.tolist() + GOOD_IDS.tolist() and longest == 2
    with pytest.raises(ValueError, match="session 3: candidate id 500 outside"):
        check(GOOD_OFF.astype(dtype), np.array([1, 2, 3, N, 5], dtype))
    with pytest.raises(ValueError, match="session 1: cand_off decreases"):
        check(np.array([0, 2, 1, 3, 5], dtype), GOOD_IDS.astype(dtype))


def test_check_id_lists_limit_counts_the_extra_entries():
    assert check(np.array([0, 0, 6, 6, 6]), np.zeros(6, np.int32), RECOMMEND)[1] == 6
    assert check(np.array([0, 0, 4, 4, 4]), np.zeros(4, np.int32), RECOMMEND, extra=2)[1] == 4
    with pytest.raises(ValueError, match="session 1: more than TCAR_RECOMMEND_MAXX = 6 exclusions with its 3 clicks"):
        check(np.array([0, 0, 4, 4, 4]), np.zeros(4, np.int32), RECOMMEND, extra=3)


def test_check_id_lists_empty_lists_and_no_sessions():
    for ids in ([], np.zeros(0, np.int64), np.zeros(0, np.float64)):    # an empty list of any type holds no id
        host, longest = check([0, 0, 0, 0, 0], ids)
        assert host.tolist() == [0] * 5 and longest == 0
        host, longest = check([0], ids, sessions=0)
        assert host.tolist() == [0] and longest == 0
    with pytest.raises(ValueError, match="offsets from 0"):
        check([0], [1], sessions=0)
    with pytest.raises(ValueError, match="outside"):
        check([0, 1], [0], n_items=0, sessions=1)
