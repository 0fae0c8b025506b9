"""The landmark sequence path from host buffers (mv_track_sequence_landmarks_host): the staging pipeline of
mv_track_sequence_host with the landmark table carried from chunk to chunk on the device.

The reference is the device-resident call mv_track_sequence_landmarks (itself checked against the composition of
public calls and the oracle in tests/test_landmark_sequence.py): results, matches with a landmark and the final table
must be byte-equal whatever the chunk size and staging mode.  The byte count is checked against what the staging
needs, computed here from the public detector outputs."""
import ctypes as C
import os

import numpy as np
import pytest

from test_landmark_sequence import N_FRAMES, _table_bytes

pytestmark = pytest.mark.gpu

ROWS, COLS, FIRST = 47, 155, 500


def _pinned(torch, t):
    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t)
    return h


@pytest.fixture(scope="module")
def lmseq(tracker, synth):
    """A 66-frame KITTI-shaped sequence, its pinned host copies, and the device landmark path's answer from an
    empty table at frame 500."""
    import torch
    from maveric_slam_b200 import tracking
    v = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vocab.npz"))
    tracker.bow_set_vocabulary(v["base_desc"], v["scale"], v["bias"], v["leaves"])
    n = N_FRAMES
    p = tracking.kitti_track_params(hypotheses=256)
    semi, desc, depth = tracker.synth_frames(21, ROWS, COLS, 0, synth.default_offsets(n, 21))
    sscale = torch.full((n,), float(synth.SEMI_SCALE), device=tracker.device)
    dscale = torch.full((n,), 4.3353, device=tracker.device)
    table = tracker.landmarks_new(tracker.n_words)
    res, nl = tracker.track_sequence_landmarks(p, semi, sscale, desc, dscale, depth, table, first_frame=FIRST)
    h = dict(semi=_pinned(torch, semi), sscale=_pinned(torch, sscale), desc=_pinned(torch, desc),
             dscale=_pinned(torch, dscale), depth=_pinned(torch, depth))
    torch.cuda.synchronize()
    return dict(p=p, d=dict(semi=semi, sscale=sscale, desc=desc, dscale=dscale, depth=depth), h=h,
                n_words=tracker.n_words, res=res.cpu().numpy().tobytes(), nl=nl.cpu().numpy(), table=_table_bytes(table))


def _host(tracker, s, h=None, first=FIRST, lo=0, hi=N_FRAMES, table=None, p=None):
    from maveric_slam_b200 import tracking
    h = h or s["h"]
    table = tracker.landmarks_new(s["n_words"]) if table is None else table
    p = p or (s["p"] if lo == 0 else tracking.kitti_track_params(hypotheses=256, first_pair=lo))
    res, nl, up, down = tracker.track_sequence_landmarks_host(
        p, h["semi"][lo:hi], h["sscale"][lo:hi], h["desc"][lo:hi], h["dscale"][lo:hi], h["depth"][lo:hi], table,
        first_frame=first)
    return res, nl, table, up, down


def _assert_equal_device(s, res, nl, table, what=""):
    assert res.tobytes() == s["res"], what
    assert nl.tobytes() == s["nl"].tobytes(), what
    assert _table_bytes(table) == s["table"], what


def test_host_equals_device(tracker, lmseq):
    res, nl, table, _, down = _host(tracker, lmseq)
    _assert_equal_device(lmseq, res, nl, table)
    assert down == 68 * (N_FRAMES - 1)
    assert (nl > 0).all()


@pytest.mark.parametrize("chunk", ["1", "7", "40"])
def test_chunk_size_changes_nothing(tracker, lmseq, monkeypatch, chunk):
    # 1: one-pair chunks (every chunk a single table step); 7: a short last chunk of 2; 40: 40 + 25
    monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", chunk)
    res, nl, table, _, _ = _host(tracker, lmseq)
    _assert_equal_device(lmseq, res, nl, table, chunk)


def test_staging_mode_changes_nothing(tracker, lmseq, monkeypatch):
    import torch
    h = lmseq["h"]
    monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", "9")
    _, _, _, up_gather, _ = _host(tracker, lmseq)
    pageable = {k: v.numpy().copy() for k, v in h.items()}
    res, nl, table, up_pageable, _ = _host(tracker, lmseq, h=pageable)
    _assert_equal_device(lmseq, res, nl, table, "pageable")
    with monkeypatch.context() as m:
        m.setenv("MV_HOST_GATHER", "0")
        res, nl, table, up_copy, _ = _host(tracker, lmseq)
        _assert_equal_device(lmseq, res, nl, table, "MV_HOST_GATHER=0")
    assert up_copy == up_pageable
    # a depth buffer 4 bytes off a 16-byte boundary
    n, cells = lmseq["h"]["depth"].shape
    buf = torch.empty(n * cells + 4, dtype=torch.float32, pin_memory=True)
    odd = buf[1:1 + n * cells].view(n, cells)
    odd.copy_(h["depth"])
    assert odd.data_ptr() % 16 == 4
    res, nl, table, up_odd, _ = _host(tracker, lmseq, h=dict(h, depth=odd))
    _assert_equal_device(lmseq, res, nl, table, "unaligned depth")
    assert up_odd == up_gather < up_copy


def test_resume_and_halo(tracker, lmseq):
    from maveric_slam_b200 import tracking
    s, d, k = lmseq, lmseq["d"], 30
    # a non-empty table: the device path over frames [0, k], then the host path over [k, n-1]
    table = tracker.landmarks_new(s["n_words"])
    res_a, nl_a = tracker.track_sequence_landmarks(s["p"], d["semi"][:k + 1], d["sscale"][:k + 1], d["desc"][:k + 1],
                                                   d["dscale"][:k + 1], d["depth"][:k + 1], table, first_frame=FIRST)
    res_b, nl_b, table, _, _ = _host(tracker, s, first=FIRST + k, lo=k, table=table)
    res = np.concatenate([res_a.cpu().numpy().reshape(-1), res_b.view(np.uint8).reshape(-1)])
    _assert_equal_device(s, res, np.concatenate([nl_a.cpu().numpy(), nl_b]), table, "device then host")
    # two host calls sharing a halo frame
    table = tracker.landmarks_new(s["n_words"])
    res_a, nl_a, table, _, _ = _host(tracker, s, hi=k + 1, table=table)
    res_b, nl_b, table, _, _ = _host(tracker, s, first=FIRST + k, lo=k, table=table,
                                     p=tracking.kitti_track_params(hypotheses=256, first_pair=k))
    _assert_equal_device(s, np.concatenate([res_a, res_b]), np.concatenate([nl_a, nl_b]), table, "host then host")


def test_byte_accounting(tracker, lmseq, monkeypatch):
    """h2d: per chunk, the logits, depth and both scales of every frame and 256 B for every frame's
    candidate-or-query cell (the word assignment reads query rows only)."""
    s, p, chunk = lmseq, lmseq["p"], 9
    monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", str(chunk))
    res, nl, _, up, down = _host(tracker, s)
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
    assert _table_bytes(table) == s["table"]


def test_degenerate_frames(tracker, synth):
    """Frames without keypoints (2, 3), with saturated (5) and zero (7) descriptors, at a 24x80 grid: the host path
    equals the device landmark path, from pinned and from pageable buffers."""
    import torch
    from maveric_slam_b200 import tracking
    v = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vocab.npz"))
    tracker.bow_set_vocabulary(v["base_desc"], v["scale"], v["bias"], v["leaves"])
    rows, cols, n, seed = 24, 80, 9, 2
    semi, desc, depth = tracker.synth_frames(seed, rows, cols, 0, synth.default_offsets(n, seed))
    semi[2:4] = -5
    desc[5] = -128
    desc[7] = 0
    sscale = torch.full((n,), float(synth.SEMI_SCALE), device=tracker.device)
    dscale = torch.full((n,), 4.3353, device=tracker.device)
    p = tracking.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=64)
    table = tracker.landmarks_new(tracker.n_words)
    res, nl = tracker.track_sequence_landmarks(p, semi, sscale, desc, dscale, depth, table, first_frame=7)
    want = (res.cpu().numpy().tobytes(), nl.cpu().numpy().tobytes(), _table_bytes(table))
    assert tracking.results_to_numpy(res)[1:4]["num_matches"].tolist() == [0, 0, 0]
    pinned = [_pinned(torch, t) for t in (semi, sscale, desc, dscale, depth)]
    torch.cuda.synchronize()
    for bufs in (pinned, [t.cpu().numpy() for t in (semi, sscale, desc, dscale, depth)]):
        t2 = tracker.landmarks_new(tracker.n_words)
        r2, nl2, _, _ = tracker.track_sequence_landmarks_host(p, *bufs, t2, first_frame=7)
        assert (r2.tobytes(), nl2.tobytes(), _table_bytes(t2)) == want


def test_depth_path_untouched(tracker, lmseq):
    from maveric_slam_b200 import tracking
    h = lmseq["h"]
    p = tracking.kitti_track_params(hypotheses=256)
    before = tracker.track_sequence_host(p, h["semi"], h["sscale"], h["desc"], h["depth"])
    _host(tracker, lmseq)
    after = tracker.track_sequence_host(p, h["semi"], h["sscale"], h["desc"], h["depth"])
    assert before[0].tobytes() == after[0].tobytes() and before[1:] == after[1:]


def test_argument_errors(tracker, lmseq):
    from maveric_slam_b200 import lib, tracking
    s, h = lmseq, lmseq["h"]
    table = tracker.landmarks_new(s["n_words"])
    _host(tracker, s, hi=4, table=table)          # a non-empty table that must survive every refused call
    before = _table_bytes(table)

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
    assert _table_bytes(table) == before
    # the context still works and continues the same table
    res, nl, table, _, _ = _host(tracker, s, first=FIRST + 3, lo=3, table=table,
                                 p=tracking.kitti_track_params(hypotheses=256, first_pair=3))
    assert res.tobytes() == s["res"][3 * 64:] and nl.tobytes() == s["nl"][3:].tobytes()
    assert _table_bytes(table) == s["table"]
