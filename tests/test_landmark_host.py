"""The landmark sequence path from host buffers (mv_track_sequence_landmarks_host): the staging pipeline of
mv_track_sequence_host with the landmark table carried from chunk to chunk on the device.

The reference is the device-resident call mv_track_sequence_landmarks (itself checked against the composition of
public calls and the oracle in tests/test_landmark_sequence.py): results, matches with a landmark and the final table
must be byte-equal whatever the chunk size and staging mode.  The byte count is checked against what the staging
needs, computed here from the public detector outputs.
The device one-call is itself held to a CPU reference of the whole path, tests/landmark_reference.py
(tests/test_landmark_reference.py)."""
import ctypes as C

import numpy as np
import pytest

from helpers import FIRST, N_FRAMES, landmark_sequence, landmarks_host, table_bytes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lmseq(tracker, synth):
    """A 66-frame KITTI-shaped sequence, its pinned host copies, and the device landmark path's answer from an
    empty table at frame 500."""
    s = landmark_sequence(tracker, synth, host=True)
    return dict(s, res=s["res"].tobytes())


def _assert_equal_device(s, res, nl, table, what=""):
    assert res.tobytes() == s["res"], what
    assert nl.tobytes() == s["nl"].tobytes(), what
    assert table_bytes(table) == s["table"], what


def test_host_equals_device(tracker, lmseq):
    res, nl, table, _, down = landmarks_host(tracker, lmseq)
    _assert_equal_device(lmseq, res, nl, table)
    assert down == 68 * (N_FRAMES - 1)
    assert (nl > 0).all()


@pytest.mark.parametrize("chunk", ["1", "7", "40"])
def test_chunk_size_changes_nothing(tracker, lmseq, monkeypatch, chunk):
    # 1: one-pair chunks (every chunk a single table step); 7: a short last chunk of 2; 40: 40 + 25
    monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", chunk)
    res, nl, table, _, _ = landmarks_host(tracker, lmseq)
    _assert_equal_device(lmseq, res, nl, table, chunk)


def test_pageable_and_unaligned_staging_change_nothing(tracker, lmseq, monkeypatch):
    """Pageable buffers (plain staged copies) and a pinned depth buffer off a 16-byte boundary give the pinned
    path's answer; pageable staging moves whole descriptor planes, the row gather fewer bytes."""
    import torch
    h, chunk = lmseq["h"], 9
    monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", str(chunk))
    _, _, _, up_gather, _ = landmarks_host(tracker, lmseq)
    pageable = {k: v.numpy().copy() for k, v in h.items()}
    res, nl, table, up_pageable, _ = landmarks_host(tracker, lmseq, h=pageable)
    _assert_equal_device(lmseq, res, nl, table, "pageable")
    # pageable staging moves whole descriptor planes: every byte of a chunk's frames, the halo frame included
    n, cells = h["depth"].shape
    frame = cells * (65 + 4 + 256) + 4 + 4
    assert up_pageable == sum((min(chunk, n - 1 - p0) + 1) * frame for p0 in range(0, n - 1, chunk))
    # a depth buffer 4 bytes off a 16-byte boundary
    buf = torch.empty(n * cells + 4, dtype=torch.float32, pin_memory=True)
    odd = buf[1:1 + n * cells].view(n, cells)
    odd.copy_(h["depth"])
    assert odd.data_ptr() % 16 == 4
    res, nl, table, up_odd, _ = landmarks_host(tracker, lmseq, h=dict(h, depth=odd))
    _assert_equal_device(lmseq, res, nl, table, "unaligned depth")
    assert up_odd == up_gather < up_pageable


def test_resume_and_halo(tracker, lmseq):
    from maveric_slam_b200 import tracking
    s, d, k = lmseq, lmseq["d"], 30
    # a non-empty table: the device path over frames [0, k], then the host path over [k, n-1]
    table = tracker.landmarks_new(s["n_words"])
    res_a, nl_a = tracker.track_sequence_landmarks(s["p"], d["semi"][:k + 1], d["sscale"][:k + 1], d["desc"][:k + 1],
                                                   d["dscale"][:k + 1], d["depth"][:k + 1], table, first_frame=FIRST)
    res_b, nl_b, table, _, _ = landmarks_host(tracker, s, first=FIRST + k, lo=k, table=table)
    res = np.concatenate([res_a.cpu().numpy().reshape(-1), res_b.view(np.uint8).reshape(-1)])
    _assert_equal_device(s, res, np.concatenate([nl_a.cpu().numpy(), nl_b]), table, "device then host")
    # two host calls sharing a halo frame
    table = tracker.landmarks_new(s["n_words"])
    res_a, nl_a, table, _, _ = landmarks_host(tracker, s, hi=k + 1, table=table)
    res_b, nl_b, table, _, _ = landmarks_host(tracker, s, first=FIRST + k, lo=k, table=table,
                                     p=tracking.kitti_track_params(hypotheses=256, first_pair=k))
    _assert_equal_device(s, np.concatenate([res_a, res_b]), np.concatenate([nl_a, nl_b]), table, "host then host")


def test_byte_accounting(tracker, lmseq, monkeypatch):
    """h2d: per chunk, the logits, depth and both scales of every frame and 256 B for every frame's
    candidate-or-query cell (the word assignment reads query rows only)."""
    s, p, chunk = lmseq, lmseq["p"], 9
    monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", str(chunk))
    res, nl, _, up, down = landmarks_host(tracker, s)
    assert res.tobytes() == s["res"]
    idx, prob, _ = tracker.softmax(s["d"]["semi"], s["d"]["sscale"])
    qp, _, _, qc, _ = tracker.top_n(idx, prob, p.top_n, p.max_valid)
    idx, prob, qp, qc = (t.cpu().numpy() for t in (idx, prob, qp, qc))
    n, cells = idx.shape
    need = (idx != 64) & ~(prob.astype(np.float64) < p.match.min_prob0)
    for f in range(n):
        need[f, qp[f, :min(int(qc[f]), p.top_n)]] = True
    rows_per_frame = need.sum(1)
    want, n_pairs = 0, n - 1
    for p0 in range(0, n_pairs, chunk):
        nf = min(chunk, n_pairs - p0) + 1
        want += nf * (cells * (65 + 4) + 4 + 4) + 256 * int(rows_per_frame[p0:p0 + nf].sum())
    assert up == want
    assert down == 68 * n_pairs
    # without the landmark counts only the records come back
    table = tracker.landmarks_new(s["n_words"])
    h = s["h"]
    out = np.zeros(n_pairs, dtype=res.dtype)
    u, dn = C.c_ulonglong(0), C.c_ulonglong(0)
    inputs = (C.c_void_p(h[k].data_ptr()) for k in ("semi", "sscale", "desc", "dscale", "depth"))
    tracker.ctx.check(tracker.lib.mv_track_sequence_landmarks_host(
        tracker.ctx.h, C.byref(p), n, FIRST, *inputs, s["n_words"], tracker._d(table), out.ctypes.data_as(C.c_void_p),
        None, C.byref(u), C.byref(dn)))
    assert out.tobytes() == s["res"] and u.value == up and dn.value == 64 * n_pairs
    assert table_bytes(table) == s["table"]


def test_degenerate_frames(tracker, synth):
    """Frames without keypoints (2, 3), with saturated (5) and zero (7) descriptors, at a 24x80 grid: the host path
    equals the device landmark path, from pinned and from pageable buffers."""
    from maveric_slam_b200 import tracking

    def degenerate(semi, desc, depth):
        semi[2:4] = -5
        desc[5] = -128
        desc[7] = 0

    p = tracking.track_params(24, 80, top_n=100, max_valid=1000, max_matches=150, hypotheses=64)
    s = landmark_sequence(tracker, synth, n_frames=9, rows=24, cols=80, seed=2, params=p, first_frame=7,
                          edit=degenerate, host=True)
    want = (s["res"].tobytes(), s["nl"].tobytes(), s["table"])
    assert s["res"][1:4]["num_matches"].tolist() == [0, 0, 0]
    for bufs in (s["h"].values(), [t.cpu().numpy() for t in s["d"].values()]):
        t2 = tracker.landmarks_new(tracker.n_words)
        r2, nl2, _, _ = tracker.track_sequence_landmarks_host(p, *bufs, t2, first_frame=7)
        assert (r2.tobytes(), nl2.tobytes(), table_bytes(t2)) == want


def test_depth_path_untouched(tracker, lmseq):
    from maveric_slam_b200 import tracking
    h = lmseq["h"]
    p = tracking.kitti_track_params(hypotheses=256)
    before = tracker.track_sequence_host(p, h["semi"], h["sscale"], h["desc"], h["depth"])
    landmarks_host(tracker, lmseq)
    after = tracker.track_sequence_host(p, h["semi"], h["sscale"], h["desc"], h["depth"])
    assert before[0].tobytes() == after[0].tobytes() and before[1:] == after[1:]


def test_argument_errors(tracker, lmseq):
    from maveric_slam_b200 import lib, tracking
    s, h = lmseq, lmseq["h"]
    table = tracker.landmarks_new(s["n_words"])
    landmarks_host(tracker, s, hi=4, table=table)          # a non-empty table that must survive every refused call
    before = table_bytes(table)

    def call(tr=tracker, p=None, n=4, n_words=None, tab=table, **over):
        hb = dict(h, **over)
        out = np.zeros(max(n - 1, 1), tracking.PAIR_RESULT_DTYPE)
        nl = np.zeros(max(n - 1, 1), np.int32)
        u, d = C.c_ulonglong(0), C.c_ulonglong(0)
        ptr = [None if hb[k] is None else C.c_void_p(hb[k].data_ptr()) for k in ("semi", "sscale", "desc", "dscale",
                                                                                  "depth")]
        tr.ctx.check(tr.lib.mv_track_sequence_landmarks_host(
            tr.ctx.h, C.byref(p or s["p"]), n, FIRST, *ptr, s["n_words"] if n_words is None else n_words,
            None if tab is None else tr._d(tab), out.ctypes.data_as(C.c_void_p), nl.ctypes.data_as(C.c_void_p),
            C.byref(u), C.byref(d)))

    with pytest.raises(lib.MvError, match="no vocabulary"):
        call(tr=tracking.Tracker(0))
    with pytest.raises(lib.MvError, match="NULL landmark table"):
        call(tab=None)
    for nw in (0, -5):
        with pytest.raises(lib.MvError, match="n_words must be positive"):
            call(n_words=nw)
    for nf in (1, 0, -3):
        with pytest.raises(lib.MvError, match="bad argument"):
            call(n=nf)
    with pytest.raises(lib.MvError, match="bad argument"):
        call(dscale=None)
    for field, val in (("rows", 0), ("cols", -3), ("max_matches", 0), ("top_n", 0), ("max_valid", 0)):
        p = tracking.kitti_track_params(hypotheses=256)
        setattr(p.match if field in ("rows", "cols", "max_matches") else p, field, val)
        with pytest.raises(lib.MvError, match="bad argument"):
            call(p=p)
    # refusals of the PnP and the matcher: checked before the table is stepped, nothing launched
    for part, field, val in (("pnp", "lanes_per_hypothesis", 4), ("pnp", "hypotheses", 0), ("pnp", "sample_size", 0),
                             ("match", "radius", -1)):
        p = tracking.kitti_track_params(hypotheses=256)
        setattr(getattr(p, part), field, val)
        launches = tracker.ctx.launches
        with pytest.raises(lib.MvError, match="bad argument"):
            call(p=p)
        assert tracker.ctx.launches == launches, field
        assert table_bytes(table) == before, field
    assert table_bytes(table) == before
    # the context still works and continues the same table
    res, nl, table, _, _ = landmarks_host(tracker, s, first=FIRST + 3, lo=3, table=table,
                                 p=tracking.kitti_track_params(hypotheses=256, first_pair=3))
    assert res.tobytes() == s["res"][3 * 64:] and nl.tobytes() == s["nl"][3:].tobytes()
    assert table_bytes(table) == s["table"]


def test_oversize_vocabulary_refused_up_front(tracker, lmseq):
    """A vocabulary mv_bow_set_vocabulary accepts but the word-assignment kernel's shared memory cannot hold (64 bases
    of 211 words) is refused by both landmark calls before they launch anything; the depth paths on the same context
    and thread then give their usual answer."""
    from maveric_slam_b200 import lib, tracking
    s, h, d = lmseq, lmseq["h"], lmseq["d"]
    want = tracker.track_sequence(s["p"], d["semi"], d["sscale"], d["desc"], d["depth"]).cpu().numpy().tobytes()
    fresh = tracking.Tracker(0)
    fresh.bow_set_vocabulary(np.zeros((256, 64), np.int8), np.ones(64, np.float32), np.zeros(64, np.float32),
                             np.zeros((64, 211, 4), np.int32))
    table = fresh.landmarks_new(fresh.n_words)
    before, launches = table_bytes(table), fresh.ctx.launches
    with pytest.raises(lib.MvError, match="shared memory"):
        fresh.track_sequence_landmarks(s["p"], d["semi"], d["sscale"], d["desc"], d["dscale"], d["depth"], table)
    with pytest.raises(lib.MvError, match="shared memory"):
        fresh.track_sequence_landmarks_host(s["p"], h["semi"], h["sscale"], h["desc"], h["dscale"], h["depth"], table)
    assert fresh.ctx.launches == launches
    assert table_bytes(table) == before
    assert fresh.track_sequence(s["p"], d["semi"], d["sscale"], d["desc"], d["depth"]).cpu().numpy().tobytes() == want
    res, _, _ = fresh.track_sequence_host(s["p"], h["semi"], h["sscale"], h["desc"], h["depth"])
    assert res.tobytes() == want
