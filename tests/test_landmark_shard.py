"""The landmark path split at the table: speculate / resolve (mv_landmarks_speculate, mv_landmarks_resolve), the
frame-level block (mv_track_landmarks_prepare / step_table / solve) and the table relay over ranks
(tracking.track_sequence_landmarks_sharded).

References: mv_landmarks_sequence and mv_track_sequence_landmarks on the same inputs (themselves pinned to the
per-frame kernels and the oracle in tests/test_landmark_sequence.py), and the oracle's table loop.
The device one-call is itself held to a CPU reference of the whole path, tests/landmark_reference.py
(tests/test_landmark_reference.py).
"""
import os
import sys

import numpy as np
import pytest

from helpers import (N_FRAMES, WARMS, StandIn, cycled_blocks, dev, drive_host_pool, free_port, landmark_sequence,
                     ref_vocab, table_bytes, upload_table)
from landmark_reference import orc_landmarks_sequence

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cases():
    """The streams of tests/test_landmark_sequence.py, plus streams built for the resolve step's branches.  Each
    case: a stream of frames, split at `k` into a prefix (which gives the true entry table) and the block."""
    rng = np.random.default_rng(11)
    cases = {}
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib
    snaps = drive_host_pool(lib.load())
    word = np.stack([s[0] for s in snaps]).astype(np.int32)
    cases["churn"] = dict(n_words=10000, first=0, word=word, qc=np.full(len(snaps), 200, np.int32),
                          coords=np.stack([s[1] for s in snaps]).astype(np.float32), init=None, k=(0, 23, 40))
    n, top_n = 40, 300
    word = rng.integers(-3, 520, (n, top_n)).astype(np.int32)
    word[5, 10:30] = 77
    word[:, :4] = 3
    word[word == 42] = 43
    word[np.arange(n) % 13 < 2, 4] = 42
    qc = np.full(n, top_n, np.int32)
    qc[7], qc[9], qc[21] = 0, 150, 1000
    cases["churn_dups"] = dict(n_words=500, first=0, word=word, qc=qc,
                               coords=rng.normal(size=(n, top_n, 3)).astype(np.float32), init=None, k=(6, 20))
    from oracle import orc
    o = orc.Oracle()
    init = o.pool_new(500)
    w0 = rng.integers(0, 500, (25, 200)).astype(np.int32)
    orc_landmarks_sequence(o, init, 975, w0, np.full(25, 200, np.int32), rng.normal(size=(25, 200, 3)).astype(np.float32))
    word = rng.integers(0, 520, (30, 200)).astype(np.int32)
    cases["resume"] = dict(n_words=500, first=1000, word=word, qc=np.full(30, 200, np.int32),
                           coords=rng.normal(size=(30, 200, 3)).astype(np.float32), init=init, k=(0, 12))
    cases["one_word"] = dict(n_words=10000, first=3, word=np.full((24, 1000), 9999, np.int32),
                             qc=np.full(24, 1000, np.int32), coords=rng.normal(size=(24, 1000, 3)).astype(np.float32),
                             init=None, k=(0, 10))
    # the patch branches, around a block that starts at frame k = 30
    n, top_n, k = 70, 64, 30
    word = np.full((n, top_n), -1, np.int32)
    word[:, 40:] = rng.integers(100, 160, (n, top_n - 40))      # background churn
    word[:, 0] = 1                                                 # alive throughout: frame_ptr moves, coords old
    word[k - 1, 1:10] = 2; word[k + 3, 1:12] = 2; word[k + 4, 1] = 2   # full ring in one frame (rotation)
    for f in range(0, n, 7): word[f, 12] = 3                       # gaps of 7
    for f in range(0, n, 8): word[f, 13] = 4                       # gaps of 8
    for f in range(0, n, 9): word[f, 14] = 5                       # gaps of 9
    word[k - 8, 15] = 6                                            # deleted exactly at the block's first step
    word[k - 3, 16] = 7; word[k + 7, 16] = 7                       # deleted inside the block, then re-inserted
    word[k - 20, 17:25] = 8; word[k - 1, 17] = 8                   # live entries older than a short warm-up
    word[k - 40 if k >= 40 else 0, 25] = 9; word[k - 2, 25] = 9; word[k + 1, 25] = 9
    word[k - 5:k, 26] = 10                                         # guess alive, truth depends on the warm-up
    word[2:5, 27] = 11; word[k + 2, 27] = 11                       # truth empty at the block, guess from old frames
    cases["branches"] = dict(n_words=200, first=500, word=word, qc=np.full(n, top_n, np.int32),
                             coords=rng.normal(size=(n, top_n, 3)).astype(np.float32), init=None, k=(k, 1, 55))
    # a random initial table: records of every shape, stale slots and foreign word ids included
    rt = o.pool_new(200)
    rt["word_id"] = np.where(rng.random(200) < 0.3, -1, np.where(rng.random(200) < 0.1, 7, np.arange(200)))
    rt["frame_ptr"] = rng.integers(0, 8, 200)
    rt["num_frames"] = rng.integers(1, 9, 200)
    rt["frames"] = rng.integers(480, 500, (200, 8))
    rt["coords"] = rng.normal(size=(200, 3))
    cases["random_table"] = dict(n_words=200, first=500, word=cases["branches"]["word"], qc=np.full(n, top_n, np.int32),
                                 coords=cases["branches"]["coords"], init=rt, k=(0, 5))
    return cases


@pytest.fixture(scope="module")
def cases():
    return _cases()


def _split(tracker, oracle, c, k, n_warm, rng):
    """-> (entry table on the device, warm-up + block words / counts, block coordinates)."""
    word, qc, coords, n_words, first = c["word"], c["qc"], c["coords"], c["n_words"], c["first"]
    init = c["init"] if c["init"] is not None else oracle.pool_new(n_words)
    entry = upload_table(tracker, init)
    if k > 0:
        tracker.landmarks_sequence(entry, first, dev(tracker, word[:k]), dev(tracker, qc[:k]), dev(tracker, coords[:k]))
    # warm-up frames: the stream's, and where it has too few, made-up frames (a guess that is simply wrong)
    pad = max(0, n_warm - k)
    ww = np.concatenate([rng.integers(-1, n_words, (pad, word.shape[1])).astype(np.int32), word[k - n_warm + pad:k]])
    wq = np.concatenate([np.full(pad, word.shape[1], np.int32), qc[k - n_warm + pad:k]])
    return entry, np.concatenate([ww, word[k:]]), np.concatenate([wq, qc[k:]]), coords[k:]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["churn", "churn_dups", "resume", "one_word", "branches", "random_table"])
def test_speculate_resolve_equals_sequence(tracker, oracle, cases, case):
    import torch
    c = cases[case]
    rng = np.random.default_rng(5)
    rewalked = []
    for k in c["k"]:
        for n_warm in WARMS:
            entry, word, qc, coords = _split(tracker, oracle, c, k, n_warm, rng)
            first = c["first"] + k
            want_t = entry.clone()
            want = tracker.landmarks_sequence(want_t, first, dev(tracker, word[n_warm:]), dev(tracker, qc[n_warm:]),
                                              dev(tracker, coords)).cpu().numpy()
            spec = tracker.landmarks_speculate(c["n_words"], first, n_warm, dev(tracker, word), dev(tracker, qc),
                                               dev(tracker, coords))
            got_t = entry.clone()
            n_rw = torch.full((1,), -1, dtype=torch.int32, device=tracker.device)
            got = tracker.landmarks_resolve(spec, got_t, n_rewalked=n_rw).cpu().numpy()
            tracker.landmarks_release(spec)
            assert table_bytes(got_t) == table_bytes(want_t), (k, n_warm)
            assert got.tobytes() == want.tobytes(), (k, n_warm)
            rewalked.append(int(n_rw.item()))
            if case != "random_table" and n_warm in (0, 16):
                o_table = entry.cpu().numpy().view(oracle.pool_new(1).dtype).reshape(-1).copy()
                o_out = orc_landmarks_sequence(oracle, o_table, first, word[n_warm:], qc[n_warm:], coords)
                assert table_bytes(got_t) == o_table.tobytes() and got.tobytes() == o_out.tobytes(), (k, n_warm)
    assert min(rewalked) >= 0
    if case in ("branches", "churn"):   # both paths of the resolve step run
        assert min(rewalked) == 0 and max(rewalked) > 0, rewalked


@pytest.mark.gpu
def test_speculate_resolve_refusals(tracker, cases):
    import torch
    from maveric_slam_b200 import lib
    c = cases["churn_dups"]
    word, qc, coords = (dev(tracker, c[x]) for x in ("word", "qc", "coords"))
    with pytest.raises(lib.MvError, match="bad argument"):
        tracker.landmarks_speculate(c["n_words"], 0, 40, word, qc, coords)   # no block step left
    from maveric_slam_b200 import tracking
    other = tracking.Tracker(0)
    spec = tracker.landmarks_speculate(c["n_words"], 5, 5, word, qc, coords[5:])
    table = tracker.landmarks_new(c["n_words"])
    with pytest.raises(lib.MvError, match="another context"):
        other.landmarks_resolve(spec, table)
    with pytest.raises(lib.MvError, match="NULL landmark table"):
        tracker.ctx.check(tracker.lib.mv_landmarks_resolve(tracker.ctx.h, spec["h"], None, tracker._d(coords), None))
    tracker.landmarks_resolve(spec, table)
    with pytest.raises(lib.MvError, match="already resolved"):
        tracker.landmarks_resolve(spec, table)
    tracker.landmarks_release(spec)
    torch.cuda.synchronize()


# ------------------------------------------------------------------ frame level
@pytest.fixture(scope="module")
def seq(tracker, synth):
    s = landmark_sequence(tracker, synth)
    return dict(s, frames=tuple(s["d"].values()))


def _prepare(tr, seq, lo, count, n_warm):
    from maveric_slam_b200 import tracking
    w = min(n_warm, lo)
    p = tracking.kitti_track_params(hypotheses=256, first_pair=lo)
    f = [x[lo - w:lo + count + 1] for x in seq["frames"]]
    return tr.track_landmarks_prepare(p, w, seq["first"] + lo, *f, seq["n_words"])


@pytest.mark.gpu
def test_prepare_step_solve_whole_sequence(tracker, seq):
    from maveric_slam_b200 import tracking
    block = _prepare(tracker, seq, 0, N_FRAMES - 1, 0)
    table = tracker.landmarks_new(seq["n_words"])
    tracker.track_landmarks_step_table(block, table)
    res, nl = tracker.track_landmarks_solve(block)
    tracker.track_landmarks_release(block)
    assert tracking.results_to_numpy(res).tobytes() == seq["res"].tobytes()
    assert (nl.cpu().numpy() == seq["nl"]).all() and table_bytes(table) == seq["table"]


@pytest.mark.gpu
@pytest.mark.parametrize("two_contexts", [False, True])
def test_blocks_prepared_first_then_stepped_in_order(tracker, seq, two_contexts):
    import torch
    from maveric_slam_b200 import tracking
    other = tracker
    if two_contexts:
        other = tracking.Tracker(0)
        other.bow_set_vocabulary(*ref_vocab())
    for n_warm in WARMS:
        blocks = cycled_blocks([1, 2, 3, 7], N_FRAMES - 1)
        trs = [(tracker, other)[i % 2] for i in range(len(blocks))]
        # prepared in reverse order, all before the first table step
        prepared = {i: _prepare(trs[i], seq, lo, c, n_warm) for i, (lo, c) in reversed(list(enumerate(blocks)))}
        # another sequence call on the same contexts between prepare and solve changes nothing
        scratch_table = tracker.landmarks_new(seq["n_words"])
        tracker.track_sequence_landmarks(seq["p"], *[x[:9] for x in seq["frames"]], scratch_table)
        table = tracker.landmarks_new(seq["n_words"])
        res, nls = [], []
        n_rw = torch.zeros((1,), dtype=torch.int32, device=tracker.device)
        for i, (lo, c) in enumerate(blocks):
            trs[i].track_landmarks_step_table(prepared[i], table, n_rw)
            r, nl = trs[i].track_landmarks_solve(prepared[i])
            res.append(tracking.results_to_numpy(r)); nls.append(nl.cpu().numpy())
            trs[i].track_landmarks_release(prepared[i])
        assert np.concatenate(res).tobytes() == seq["res"].tobytes(), n_warm
        assert (np.concatenate(nls) == seq["nl"]).all(), n_warm
        assert table_bytes(table) == seq["table"], n_warm


@pytest.mark.gpu
def test_block_refusals(tracker, seq):
    import torch
    from maveric_slam_b200 import lib, tracking
    semi, sscale, desc, dscale, depth = seq["frames"]
    table = tracker.landmarks_new(seq["n_words"])
    before = table_bytes(table)
    for part, field, val in (("pnp", "lanes_per_hypothesis", 4), ("pnp", "hypotheses", 0), ("pnp", "sample_size", 0),
                             ("match", "radius", -1)):
        bad = tracking.kitti_track_params(hypotheses=256)
        setattr(getattr(bad, part), field, val)
        launches = tracker.ctx.launches
        with pytest.raises(lib.MvError, match="bad argument"):
            tracker.track_landmarks_prepare(bad, 2, seq["first"] + 2, semi[:8], sscale[:8], desc[:8], dscale[:8],
                                            depth[:8], seq["n_words"])
        assert tracker.ctx.launches == launches, field
    launches = tracker.ctx.launches
    for n_warm, n in ((-1, 4), (3, 4), (0, 1)):   # n_warm < 0; n_warm leaves one block frame; one frame
        with pytest.raises(lib.MvError, match="bad argument"):
            tracker.track_landmarks_prepare(seq["p"], n_warm, 0, semi[:n], sscale[:n], desc[:n], dscale[:n], depth[:n],
                                            seq["n_words"])
    with pytest.raises(lib.MvError, match="n_words must be positive"):
        tracker.track_landmarks_prepare(seq["p"], 0, 0, semi[:4], sscale[:4], desc[:4], dscale[:4], depth[:4], 0)
    assert tracker.ctx.launches == launches
    assert table_bytes(table) == before
    # phases
    block = _prepare(tracker, seq, 0, 5, 0)
    launches = tracker.ctx.launches
    with pytest.raises(lib.MvError, match="out of phase"):
        tracker.track_landmarks_solve(block)
    with pytest.raises(lib.MvError, match="NULL landmark table"):
        tracker.ctx.check(tracker.lib.mv_track_landmarks_step_table(tracker.ctx.h, block["h"], None, None))
    other = tracking.Tracker(0)
    with pytest.raises(lib.MvError, match="another context"):
        other.track_landmarks_step_table(block, table)
    assert tracker.ctx.launches == launches and table_bytes(table) == before
    tracker.track_landmarks_step_table(block, table)
    with pytest.raises(lib.MvError, match="out of phase"):
        tracker.track_landmarks_step_table(block, table)
    tracker.track_landmarks_solve(block)
    with pytest.raises(lib.MvError, match="out of phase"):
        tracker.track_landmarks_solve(block)
    tracker.track_landmarks_release(block)
    # released without solve (and without a table step): the context still gives the stored answers
    for steps in (0, 1):
        block = _prepare(tracker, seq, 10, 20, 8)
        if steps:
            tracker.track_landmarks_step_table(block, tracker.landmarks_new(seq["n_words"]))
        tracker.track_landmarks_release(block)
    table = tracker.landmarks_new(seq["n_words"])
    res, nl = tracker.track_sequence_landmarks(seq["p"], *seq["frames"], table, first_frame=seq["first"])
    assert tracking.results_to_numpy(res).tobytes() == seq["res"].tobytes() and (nl.cpu().numpy() == seq["nl"]).all()
    assert table_bytes(table) == seq["table"]
    torch.cuda.synchronize()


# ------------------------------------------------------------------ ranks
def _gpu_worker(rank, world, port, out_dir, n_warm):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import synth, tracking
    tr = tracking.Tracker(rank)
    s = landmark_sequence(tr, synth)
    table = tr.landmarks_new(s["n_words"])
    rec, nl, _ = tracking.track_sequence_landmarks_sharded(tr, s["p"], tuple(s["d"].values()), table,
                                                           first_frame=s["first"], n_warm=n_warm)
    ok = (rec.cpu().numpy().tobytes() == s["res"].tobytes() and bool((nl.cpu().numpy() == s["nl"]).all())
          and table_bytes(table) == s["table"])
    open(os.path.join(out_dir, f"rank{rank}_{n_warm}.txt"), "w").write("ok" if ok else "differs")
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_sharded_equals_one_gpu(tmp_path, world):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    for n_warm in (0, 16):
        mp.spawn(_gpu_worker, args=(world, free_port(), str(tmp_path), n_warm), nprocs=world, join=True)
        for r in range(world):
            assert open(tmp_path / f"rank{r}_{n_warm}.txt").read() == "ok", (r, n_warm)


def _relay_worker(rank, world, port, n_pairs, out_dir):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    p = tracking.kitti_track_params(hypotheses=16)
    frames = tuple(torch.zeros((n_pairs + 1, 1)) for _ in range(5))
    table = torch.arange(128, dtype=torch.uint8).reshape(2, 64).clone() if rank == 0 else \
        torch.full((2, 64), 99, dtype=torch.uint8)
    rec, nl, rw = tracking.track_sequence_landmarks_sharded(StandIn(), p, frames, table, first_frame=10, n_warm=4)
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), rec=rec.numpy(), nl=nl.numpy(), table=table.numpy(),
             rw=rw.numpy())
    dist.destroy_process_group()


def test_relay_order_cpu(tmp_path):
    """Rank r steps the table rank r - 1 sent, in rank order; records and counts land in pair order on every rank;
    the last rank's table is broadcast."""
    import torch
    import torch.multiprocessing as mp
    sys.path.insert(0, ROOT)
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    n_pairs = 11
    for world in (1, 3):
        mp.spawn(_relay_worker, args=(world, free_port(), n_pairs, str(tmp_path)), nprocs=world, join=True)
        st = StandIn()
        table = torch.arange(128, dtype=torch.uint8).reshape(2, 64).clone()
        block = {"first": 0, "n_pairs": n_pairs, "n_warm": 0, "frame": 10}
        st.track_landmarks_step_table(block, table)
        want_t = table.numpy()
        # records of the sequential chain: pair q's record is the table after its block's last step, plus its index
        chain = torch.arange(128, dtype=torch.uint8).reshape(2, 64).clone()
        want_rec = np.zeros((n_pairs, 64), np.uint8)
        for r in range(world):
            first, count, _ = tracking.shard_pairs(n_pairs, world, r)
            b = {"first": first, "n_pairs": count, "n_warm": 0, "frame": 10 + first}
            st.track_landmarks_step_table(b, chain)
            for i in range(count):
                want_rec[first + i] = (chain.reshape(-1)[:64] + i).numpy()
        for r in range(world):
            got = np.load(tmp_path / f"rank{r}.npz")
            assert (got["table"] == want_t).all(), (world, r)
            assert (got["rec"] == want_rec).all(), (world, r)
            assert (got["nl"] == 10 + np.arange(n_pairs)).all(), (world, r)
            first = tracking.shard_pairs(n_pairs, world, r)[0]
            assert int(got["rw"][0]) == min(4, first), (world, r)
