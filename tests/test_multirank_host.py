"""world_size-2 check of the multi-GPU host logic on CPU (gloo): pairs shard in contiguous
blocks, each rank computes its own block (here with the CPU oracle standing in for the GPU),
and one all_gather of 64-byte records reproduces the single-rank result on every rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import free_port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _records(first, count):
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    rec = np.zeros(count, tracking.PAIR_RESULT_DTYPE)
    for i in range(count):
        p = first + i
        rec[i]["q"] = [1, 0, 0, p]
        rec[i]["t"] = [p, 2 * p, 3 * p]
        rec[i]["num_matches"] = 1000 + p
        rec[i]["best_hypothesis"] = p % 7
    return rec


def _worker(rank, world, port, n_pairs, out_dir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    first, count, per = tracking.shard_pairs(n_pairs, world, rank)
    local = torch.from_numpy(_records(first, count).view(np.uint8).reshape(-1, 64).copy())
    full = tracking.gather_results(local, n_pairs, world)
    # ... and the persistent form bench.py uses: records written in place into the send buffer, two steps
    gat = tracking.ResultGather(n_pairs, world, rank, torch.device("cpu"))
    assert (gat.first, gat.count, gat.per) == (first, count, per)
    for step in range(2):
        gat.send.copy_(local)
        again = gat.gather()
        assert again.shape == full.shape and bool((again == full).all()), step
    # ... and unequal blocks (the host-buffer path on a box with unequal host links): padding rows of the
    # short block must not show up between the blocks
    for weights in ([1.0, 2.0], [3.0, 1.0], [1.0, 0.0]):
        blocks = tracking.shard_pairs_weighted(n_pairs, weights)
        counts = [c for _, c in blocks]
        gw = tracking.ResultGather(n_pairs, world, rank, torch.device("cpu"), counts=counts)
        assert (gw.first, gw.count) == blocks[rank]
        mine = torch.from_numpy(_records(gw.first, gw.count).view(np.uint8).reshape(-1, 64).copy())
        for step in range(2):
            gw.send.copy_(mine)
            again = gw.gather()
            assert again.shape == full.shape and bool((again == full).all()), (weights, step)
    np.save(os.path.join(out_dir, f"rank{rank}.npy"), full.numpy())
    dist.destroy_process_group()


def test_shard_bounds():
    sys.path.insert(0, ROOT)
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    for n, w in [(4540, 8), (4540, 1), (5, 8), (17, 4), (0, 2)]:
        seen = []
        for r in range(w):
            first, count, per = tracking.shard_pairs(n, w, r)
            seen += list(range(first, first + count))
            assert count <= per
        assert seen == list(range(n))
    assert tracking.shard_pairs(4540, 8, 7) == (3976, 564, 568)     # SURVEY §8e


def test_weighted_blocks_and_balancing():
    sys.path.insert(0, ROOT)
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    for n, weights in [(4540, [23.1] * 4 + [35.2] * 4), (7, [1, 1, 1]), (5, [0, 1]), (100, [1e-9, 1.0]), (0, [1, 2])]:
        blocks = tracking.shard_pairs_weighted(n, weights)
        assert [f for f, _ in blocks] == [sum(c for _, c in blocks[:r]) for r in range(len(weights))]
        assert sum(c for _, c in blocks) == n and min(c for _, c in blocks) >= 0
        tot = float(sum(weights))
        assert all(abs(c - n * w / tot) < 1.0 for (_, c), w in zip(blocks, weights))
    # the pool's 8-GPU box: 568 pairs take 22.0 ms on ranks 0-3 and 15.2 ms on ranks 4-7
    counts = [568] * 7 + [564]
    secs = [22.0e-3] * 4 + [15.2e-3] * 3 + [15.1e-3]
    new = tracking.balance_shards(counts, secs)
    assert sum(new) == 4540 and max(new[:4]) < 568 < min(new[4:])
    finish = [c / (k / s) for c, k, s in zip(new, counts, secs)]      # at the measured rates
    assert max(finish) < 1.02 * min(finish) and max(finish) < 0.85 * max(secs)
    # within the tolerance nothing moves; ranks without work are left alone
    assert tracking.balance_shards([568] * 8, [20.0e-3 + 1e-4 * r for r in range(8)]) == [568] * 8
    assert tracking.balance_shards([5, 0], [1.0, 0.0]) == [5, 0]


def test_two_rank_gather_equals_single_rank(tmp_path):
    n_pairs, world = 37, 2
    port = free_port()
    mp.spawn(_worker, args=(world, port, n_pairs, str(tmp_path)), nprocs=world, join=True)
    want = _records(0, n_pairs).view(np.uint8).reshape(-1, 64)
    for r in range(world):
        got = np.load(os.path.join(str(tmp_path), f"rank{r}.npy"))
        assert got.shape == want.shape and (got == want).all()
