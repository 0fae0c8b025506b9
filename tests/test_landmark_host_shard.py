"""The landmark block prepared from host buffers (mv_track_landmarks_prepare_host) and the host-buffer relay over ranks
(tracking.track_sequence_landmarks_host_sharded).

References: the device landmark path on the same 66-frame fixture (mv_track_sequence_landmarks, which
tests/test_landmark_host.py equates with mv_track_sequence_landmarks_host) and the device-prepared block
(tests/test_landmark_shard.py).  Staged bytes are checked against a formula computed from the public detector
outputs, as tests/test_landmark_host.py does for the one host call.
The device one-call is itself held to a CPU reference of the whole path, tests/landmark_reference.py
(tests/test_landmark_reference.py)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from helpers import (FIRST, KEYS, N_FRAMES, WARMS, HostStandIn, StandIn, cycled_blocks, free_port, landmark_sequence,
                     landmarks_host, pinned, ref_vocab, table_bytes)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lmseq(tracker, synth):
    """The 66-frame sequence of tests/test_landmark_host.py, its pinned host copies and the device path's answer."""
    s = landmark_sequence(tracker, synth, host=True)
    return dict(s, res=s["res"].tobytes())


def _params(lo):
    from maveric_slam_b200 import tracking
    return tracking.kitti_track_params(hypotheses=256, first_pair=lo)


def _prep_host(tr, s, lo, count, n_warm, h=None):
    w = min(n_warm, lo)
    h = h or s["h"]
    return tr.track_landmarks_prepare_host(_params(lo), w, FIRST + lo, *[h[k][lo - w:lo + count + 1] for k in KEYS],
                                           s["n_words"])


def _prep_device(tr, s, lo, count, n_warm):
    w = min(n_warm, lo)
    return tr.track_landmarks_prepare(_params(lo), w, FIRST + lo, *[s["d"][k][lo - w:lo + count + 1] for k in KEYS],
                                      s["n_words"])


def _chain(s, prepared, trs):
    """Steps prepared blocks in order from an empty table -> (records bytes, counts, table bytes)."""
    table = trs[0].landmarks_new(s["n_words"])
    res, nls = [], []
    for tr, b in zip(trs, prepared):
        tr.track_landmarks_step_table(b, table)
        r, nl = tr.track_landmarks_solve(b)
        res.append(r.cpu().numpy()); nls.append(nl.cpu().numpy())
        tr.track_landmarks_release(b)
    return np.concatenate(res).tobytes(), np.concatenate(nls), table_bytes(table)


def _assert_one_call(s, got, what=""):
    res, nl, table = got
    assert res == s["res"], what
    assert nl.tobytes() == s["nl"].tobytes(), what
    assert table == s["table"], what


def _second(tracker, s):
    from maveric_slam_b200 import tracking
    other = tracking.Tracker(0)
    other.bow_set_vocabulary(*ref_vocab())
    return other


@pytest.mark.gpu
def test_whole_sequence(tracker, lmseq):
    b = _prep_host(tracker, lmseq, 0, N_FRAMES - 1, 0)
    _assert_one_call(lmseq, _chain(lmseq, [b], [tracker]))
    res, nl, table, _, _ = landmarks_host(tracker, lmseq)
    assert (res.tobytes(), nl.tobytes(), table_bytes(table)) == (lmseq["res"], lmseq["nl"].tobytes(), lmseq["table"])


@pytest.mark.gpu
@pytest.mark.parametrize("two_contexts", [False, True])
def test_blocks_in_reverse_with_a_device_block(tracker, lmseq, two_contexts):
    s = lmseq
    other = _second(tracker, s) if two_contexts else tracker
    blocks = cycled_blocks([1, 2, 3, 7, 40], N_FRAMES - 1)
    for n_warm in WARMS:
        trs = [(tracker, other)[i % 2] for i in range(len(blocks))]
        prepared = {}
        for i, (lo, c) in reversed(list(enumerate(blocks))):
            # block 3 (7 pairs) is prepared on the device: blocks of either prepare chain with each other
            prep = _prep_device if i == 3 else _prep_host
            prepared[i] = prep(trs[i], s, lo, c, n_warm)
        _assert_one_call(s, _chain(s, [prepared[i] for i in range(len(blocks))], trs), n_warm)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["chunk1", "chunk7", "chunk40", "pageable"])
def test_chunking_and_staging_change_nothing(tracker, lmseq, monkeypatch, mode):
    s = lmseq
    h = s["h"]
    if mode.startswith("chunk"):
        monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", mode[5:])
    else:
        h = {k: v.numpy().copy() for k, v in h.items()}
    blocks = [(0, 10), (10, 40), (50, 15)]
    prepared = [_prep_host(tracker, s, lo, c, 8, h=h) for lo, c in blocks]
    _assert_one_call(s, _chain(s, prepared, [tracker] * 3), mode)


def _rows_per_frame(tracker, s):
    """-> (candidate-or-query rows, query rows) per frame, from the public detector outputs."""
    p = s["p"]
    idx, prob, _ = tracker.softmax(s["d"]["semi"], s["d"]["sscale"])
    qp, _, _, qc, _ = tracker.top_n(idx, prob, p.top_n, p.max_valid)
    idx, prob, qp, qc = (t.cpu().numpy() for t in (idx, prob, qp, qc))
    need = (idx != 64) & ~(prob.astype(np.float64) < p.match.min_prob0)
    query = np.zeros_like(need)
    for f in range(idx.shape[0]):
        query[f, qp[f, :min(int(qc[f]), p.top_n)]] = True
    return (need | query).sum(1), query.sum(1), idx.shape[1]


@pytest.mark.gpu
def test_byte_accounting(tracker, lmseq, monkeypatch):
    """Block frames: per chunk of pairs (one halo frame), the logits, depth, both scales and 256 B per candidate-or-query
    row, as the one host call; warm-up frames, in chunks without a halo: logits, both scales and query rows only."""
    s, chunk = lmseq, 9
    monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", str(chunk))
    rows, qrows, cells = _rows_per_frame(tracker, s)
    lo, count = 20, 30
    for n_warm in (0, 16):
        b = _prep_host(tracker, s, lo, count, n_warm)
        want = 0
        for f in range(lo - n_warm, lo):
            want += cells * 65 + 4 + 4 + 256 * int(qrows[f])
        for p0 in range(0, count, chunk):
            f0, nf = lo + p0, min(chunk, count - p0) + 1
            want += nf * (cells * (65 + 4) + 4 + 4) + 256 * int(rows[f0:f0 + nf].sum())
        assert b["h2d_bytes"] == want, n_warm
        whole = (n_warm + count + 1) * (cells * (65 + 256 + 4) + 4 + 4)
        assert b["h2d_bytes"] < whole
        tracker.track_landmarks_release(b)
        if n_warm == 0:   # the same frames through the one host call move the same bytes
            _, _, _, up, _ = landmarks_host(tracker, s, first=FIRST + lo, lo=lo, hi=lo + count + 1, p=_params(lo))
            assert up == want


@pytest.mark.gpu
def test_host_buffers_free_at_return(tracker, lmseq):
    import torch
    s = lmseq
    prepared = []
    for lo, c in ((0, 30), (30, 35)):
        w = min(8, lo)
        h = {k: pinned(s["h"][k][lo - w:lo + c + 1]) for k in KEYS}
        prepared.append(tracker.track_landmarks_prepare_host(_params(lo), w, FIRST + lo, *[h[k] for k in KEYS],
                                                             s["n_words"]))
        for k in KEYS:   # overwritten as soon as the call returns, before any later stream work
            h[k].fill_(-7 if h[k].dtype == torch.int8 else 3.0)
    _assert_one_call(s, _chain(s, prepared, [tracker] * 2))


@pytest.mark.gpu
def test_refusals(tracker, lmseq):
    from maveric_slam_b200 import lib, tracking
    s, h = lmseq, lmseq["h"]

    def call(tr=tracker, p=None, n_warm=2, n=8, n_words=None, **over):
        hb = dict(h, **over)
        ptr = [None if hb[k] is None else C.c_void_p(hb[k].data_ptr()) for k in KEYS]
        out = C.c_void_p(1234)
        tr.ctx.check(tr.lib.mv_track_landmarks_prepare_host(
            tr.ctx.h, C.byref(p or _params(2)), n_warm, n - n_warm, FIRST + 2, *ptr,
            s["n_words"] if n_words is None else n_words, C.byref(out), None))
        raise AssertionError("accepted")

    launches = tracker.ctx.launches
    for part, field, val in (("pnp", "lanes_per_hypothesis", 4), ("pnp", "hypotheses", 0), ("pnp", "sample_size", 0),
                             ("match", "radius", -1)):
        bad = tracking.kitti_track_params(hypotheses=256)
        setattr(getattr(bad, part), field, val)
        with pytest.raises(lib.MvError, match="bad argument"):
            call(p=bad)
    for n_warm, n in ((-1, 4), (3, 4), (0, 1)):   # n_warm < 0; n_warm leaves one block frame; one frame
        with pytest.raises(lib.MvError, match="bad argument"):
            call(n_warm=n_warm, n=n)
    with pytest.raises(lib.MvError, match="65535 frames in all"):
        call(n_warm=65534, n=65538)            # refused before any host read: the buffers hold 66 frames
    for nw in (0, -5):
        with pytest.raises(lib.MvError, match="n_words must be positive"):
            call(n_words=nw)
    for k in KEYS:
        with pytest.raises(lib.MvError, match="bad argument"):
            call(**{k: None})
    with pytest.raises(lib.MvError, match="bad argument"):
        tracker.ctx.check(tracker.lib.mv_track_landmarks_prepare_host(
            tracker.ctx.h, C.byref(s["p"]), 0, 4, FIRST, *[C.c_void_p(h[k].data_ptr()) for k in KEYS], s["n_words"],
            None, None))
    assert tracker.ctx.launches == launches
    fresh = tracking.Tracker(0)
    with pytest.raises(lib.MvError, match="no vocabulary"):
        call(tr=fresh)
    assert fresh.ctx.launches == 0
    # released before step_table (and after it, without solve): the context still gives the stored answers
    for steps in (0, 1):
        b = _prep_host(tracker, s, 10, 20, 8)
        if steps:
            tracker.track_landmarks_step_table(b, tracker.landmarks_new(s["n_words"]))
        tracker.track_landmarks_release(b)
    res, nl, table, _, _ = landmarks_host(tracker, s)
    assert (res.tobytes(), nl.tobytes(), table_bytes(table)) == (s["res"], s["nl"].tobytes(), s["table"])


@pytest.mark.gpu
def test_existing_host_calls_unchanged(tracker, lmseq):
    """The depth and landmark host calls on a fresh context: results, byte counts and launches per call are the same
    before and after a prepare_host on that context."""
    s, h = lmseq, lmseq["h"]
    tr = _second(tracker, s)

    def both():
        out = []
        n0 = tr.ctx.launches
        r = tr.track_sequence_host(s["p"], h["semi"], h["sscale"], h["desc"], h["depth"])
        out.append((r[0].tobytes(), r[1], r[2], tr.ctx.launches - n0))
        n0 = tr.ctx.launches
        res, nl, table, up, down = landmarks_host(tr, s)
        out.append((res.tobytes(), nl.tobytes(), table_bytes(table), up, down, tr.ctx.launches - n0))
        return out

    both()   # first calls on the context: modules, scratch
    before = both()
    assert before[1][:3] == (s["res"], s["nl"].tobytes(), s["table"])
    tr.track_landmarks_release(_prep_host(tr, s, 5, 40, 16))
    assert both() == before


# ------------------------------------------------------------------ ranks
def _gpu_worker(rank, world, port, out_dir, n_warm, weighted):
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
    s = landmark_sequence(tr, synth, host=True)
    counts = None
    if weighted:
        counts = [c for _, c in tracking.shard_pairs_weighted(N_FRAMES - 1, [1.0 + 2.0 * r for r in range(world)])]
    table = tr.landmarks_new(s["n_words"])
    rec, nl, _, up = tracking.track_sequence_landmarks_host_sharded(tr, s["p"], tuple(s["h"].values()), table,
                                                                    first_frame=s["first"], n_warm=n_warm,
                                                                    counts=counts)
    ok = (rec.cpu().numpy().tobytes() == s["res"].tobytes() and bool((nl.cpu().numpy() == s["nl"]).all())
          and table_bytes(table) == s["table"] and up > 0)
    open(os.path.join(out_dir, f"rank{rank}_{n_warm}_{weighted}.txt"), "w").write("ok" if ok else "differs")
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 4])
def test_host_sharded_equals_one_gpu(tmp_path, world):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    for weighted in (False, True):
        for n_warm in (0, 16):
            mp.spawn(_gpu_worker, args=(world, free_port(), str(tmp_path), n_warm, weighted), nprocs=world, join=True)
            for r in range(world):
                assert open(tmp_path / f"rank{r}_{n_warm}_{weighted}.txt").read() == "ok", (r, n_warm, weighted)


COUNTS = {1: [11], 3: [2, 6, 3], 4: [5, 0, 4, 2]}


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
    rec, nl, rw, up = tracking.track_sequence_landmarks_host_sharded(HostStandIn(), p, frames, table, first_frame=10,
                                                                     n_warm=4, counts=COUNTS[world])
    np.savez(os.path.join(out_dir, f"rank{rank}.npz"), rec=rec.numpy(), nl=nl.numpy(), table=table.numpy(),
             rw=rw.numpy(), up=np.array(up))
    dist.destroy_process_group()


def test_host_relay_order_uneven_cpu(tmp_path):
    """Uneven blocks (one of them empty): rank r steps the table rank r - 1 sent, in rank order; records and counts
    land in pair order on every rank with the padding rows dropped; the last rank's table is broadcast."""
    import torch
    import torch.multiprocessing as mp
    n_pairs = 11
    for world, counts in COUNTS.items():
        mp.spawn(_relay_worker, args=(world, free_port(), n_pairs, str(tmp_path)), nprocs=world, join=True)
        st = StandIn()
        chain = torch.arange(128, dtype=torch.uint8).reshape(2, 64).clone()
        want_rec = np.zeros((n_pairs, 64), np.uint8)
        first = 0
        for c in counts:
            st.track_landmarks_step_table({"first": first, "n_pairs": c, "n_warm": 0, "frame": 10 + first}, chain)
            for i in range(c):
                want_rec[first + i] = (chain.reshape(-1)[:64] + i).numpy()
            first += c
        for r in range(world):
            got = np.load(tmp_path / f"rank{r}.npz")
            first = sum(counts[:r])
            assert (got["table"] == chain.numpy()).all(), (world, r)
            assert (got["rec"] == want_rec).all(), (world, r)
            assert (got["nl"] == 10 + np.arange(n_pairs)).all(), (world, r)
            w = min(4, first)
            assert int(got["rw"][0]) == (w if counts[r] else 0), (world, r)
            assert int(got["up"]) == (1000 * (w + counts[r] + 1) if counts[r] else 0), (world, r)
