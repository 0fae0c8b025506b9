"""Every landmark-path entry point against a CPU reference of the whole path (tests/landmark_reference.py), and the
word assignment (mv_bow_assign_batch) against the oracle beyond the reference vocabulary.

The other landmark modules hold each entry point to the device one-call, and the one-call to a composition of the
library's own calls; a bug those share passes them.  Here the reference is built from oracle primitives only, so
the records (byte-equal, NaN equal to NaN), the per-pair landmark counts and the final table (byte-equal) of

  * mv_track_sequence_landmarks,
  * mv_track_sequence_landmarks_host (pinned, chunked and unchunked; pageable),
  * uneven blocks of mv_track_landmarks_prepare / _prepare_host, step_table, solve (prepared in reverse order, with
    and without warm-up frames),
  * tracking.track_sequence_landmarks_sharded / _host_sharded at world 1

are checked on inputs where the fixtures of the other modules are uniform: per-frame semi / desc scales (a negative
and a zero desc_scale among them), frames without keypoints, an overflowing frame, saturated and zero descriptors,
a top_n that is not a multiple of 8, the one-warp K3 form, negative frame numbers, a vocabulary of another shape with
a table larger and smaller than its word count, and a walk that starts from a live table.

Everything that sets a vocabulary does it on a context of its own: the session's `tracker` keeps the reference
vocabulary for the modules that run after this one.  Two contexts with vocabularies of different sizes on one device
share the word-assignment kernel's shared-memory limit (test_bow_assign_two_contexts_on_one_device).
"""
import copy

import numpy as np
import pytest

from helpers import ref_vocab, with_first_pair
from landmark_reference import (bow_check, bow_inputs, bow_vocab, case_inputs, first_difference, landmark_reference,
                                run_entry, track_cfg)

f32 = np.float32
# fx != fy, cx and cy off the KITTI values, K3's gate, damping, iteration counts and sample size off their defaults
CAMERA_PNP = dict(fx=520.0, fy=910.0, cx=300.5, cy=260.25, gate_sq=16.0, damping=1e-3, sample_iters=3, refine_iters=6,
                  sample_size=9)


# ------------------------------------------------------------------ CPU: the reference's plumbing
def test_reference_depth_mode_equals_track_pair(oracle, synth):
    """With the 3-D side from depth, the reference is orc_track_pair, byte for byte, on every pair; where frame 0 of a
    pair overflowed max_valid only the status differs (orc_track_pair flags frame 1 only)."""
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    rows, cols, n, seed = 24, 80, 7, 3
    semi, desc, depth, off = synth.synth_sequence(seed, rows, cols, n)
    semi[4] = synth.synth_frame(seed, rows, cols, 4, int(off[4, 0]), int(off[4, 1]), keypoint_permille=1000)[0]
    p = tracking.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=64, first_pair=9)
    sscale = np.full(n, synth.SEMI_SCALE, f32)
    rec, _, _ = landmark_reference(oracle, None, p, semi, sscale, desc, None, depth, depth_mode=True)
    cfg = track_cfg(p, synth.SEMI_SCALE)
    for q in range(n - 1):
        want = oracle.track_pair(cfg, 9 + q, semi[q], desc[q], depth[q], semi[q + 1], desc[q + 1])
        got = rec[q:q + 1].tobytes()[:52]
        if q == 4:   # frame 0 overflowed
            assert want.status == 0 and rec[q]["status"] == 4
            got = got[:48]
        assert got == bytes(want)[:len(got)], q
    assert rec[3]["status"] == 4 and rec[3]["num_matches"] == 0
    assert (rec["num_matches"][[0, 1, 2, 5]] > 20).all() and rec[4]["num_matches"] > 0
    assert (rec["pad"] == 0).all()


# ------------------------------------------------------------------ GPU: mv_bow_assign_batch against the oracle
@pytest.fixture(scope="module")
def own_tracker():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    return tracking.Tracker(0)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["1x1", "1x9", "3x7", "17x33", "10x1000", "64x8", "64x210", "repeated_leaves",
                                  "zero_leaves", "nonpositive_scores", "equal_bases"])
def test_bow_assign_vocabularies(own_tracker, oracle, name):
    vocab = bow_vocab(name)
    own_tracker.bow_set_vocabulary(*vocab)
    word = bow_check(own_tracker, oracle, vocab, *bow_inputs(7, 37))
    wpb = vocab[3].shape[1]
    used = word[word >= 0]
    if name == "nonpositive_scores":
        assert (used < wpb).all()
    elif name == "equal_bases":
        assert set(np.unique(used // wpb)) == {0, 2}
    elif name == "repeated_leaves":   # the first of equal windows; 19 of the last base reads the zero pad
        assert set(np.unique(used % wpb)) <= {0, 1, 2, 3, 4, 19}
    elif name == "zero_leaves":
        assert (used % wpb == 0).all()
    elif name not in ("1x1", "1x9", "10x1000"):   # the reference vocabulary picks base 0 on random rows
        assert len(np.unique(used // wpb)) > 1


@pytest.mark.gpu
@pytest.mark.parametrize("top_n", [1, 37, 129])
def test_bow_assign_top_n_and_counts(own_tracker, oracle, top_n):
    """top_n not a multiple of 8 (queries of a frame straddle the lanes' groups), and for 129 more queries than the
    persistent CTAs take in one trip (148 x 128), so they loop."""
    vocab = bow_vocab("3x7")
    own_tracker.bow_set_vocabulary(*vocab)
    reps = 4 if top_n == 129 else 1
    desc, dscale, qp, qc = bow_inputs(top_n, top_n, reps=reps)
    assert top_n < 129 or desc.shape[0] * top_n > 148 * 128
    bow_check(own_tracker, oracle, vocab, desc, dscale, qp, qc)


@pytest.mark.gpu
def test_bow_assign_two_contexts_on_one_device(oracle):
    """Two contexts on one device, one with the reference vocabulary (160 KB of shared memory), one with a 1 x 9
    vocabulary, used in turn: each keeps giving the oracle's words.  The kernel's shared-memory limit is state of the
    device, not of a context, so the smaller vocabulary must not lower it under the larger one."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    a, b = tracking.Tracker(0), tracking.Tracker(0)
    va, vb = ref_vocab(), bow_vocab("1x9")
    a.bow_set_vocabulary(*va)
    b.bow_set_vocabulary(*vb)
    inputs = bow_inputs(3, 37)
    for tr, v in ((a, va), (b, vb), (a, va), (b, vb)):
        bow_check(tr, oracle, v, *inputs)


# ------------------------------------------------------------------ GPU: every entry point against the reference
class _References:
    """Each case's inputs and reference, computed once for the module."""

    def __init__(self, oracle, synth):
        self.oracle, self.synth, self.done = oracle, synth, {}

    def __call__(self, name):
        if name not in self.done:
            self.done[name] = self._make(name)
        return self.done[name]

    def _make(self, name):
        o = self.oracle
        if name == "scales_tc0":   # case "scales" through the CUDA-core matcher: the same answer
            c = dict(self("scales"))
            c["p"] = copy.copy(c["p"])
            c["p"].match = copy.copy(c["p"].match)
            c["p"].match.use_tensor_cores = 0
            return c
        if name == "resume":   # case "scales" entered at frame 8 with the reference's table after frames 0 .. 8
            a = self("scales")
            c = dict(a)
            head = landmark_reference(o, o.bow_vocab(*a["vocab"]), a["p"], *[x[:9] for x in a["frames"]],
                                      first_frame=a["first"], n_words=a["n_words"])
            assert head[0].tobytes() == a["rec"][:8].tobytes() and (head[1] == a["nl"][:8]).all()
            c.update(p=with_first_pair(a["p"], 8), frames=[x[8:] for x in a["frames"]], first=a["first"] + 8,
                     entry=head[2], rec=a["rec"][8:], nl=a["nl"][8:])
            assert np.unique(head[2]["word_id"]).size > 100
            return c
        if name == "camera":   # case "scales" with another camera and K3 away from its defaults (only p.pnp changed)
            a = self("scales")
            c = dict(a)
            c["p"] = copy.copy(a["p"])
            c["p"].pnp = copy.copy(a["p"].pnp)
            for k, v in CAMERA_PNP.items():
                setattr(c["p"].pnp, k, v)
            rec, nl, table = landmark_reference(o, o.bow_vocab(*c["vocab"]), c["p"], *c["frames"], table=c["entry"],
                                                first_frame=c["first"], n_words=c["n_words"])
            c.update(rec=rec, nl=nl, table=table)
            _assert_case_reaches(name, c)
            # the back-projected landmarks and the poses are the camera's own
            assert table.tobytes() != a["table"].tobytes()
            assert (rec["q"] != a["rec"]["q"]).any(axis=1).all()
            return c
        c = case_inputs(name, self.synth)
        rec, nl, table = landmark_reference(o, o.bow_vocab(*c["vocab"]), c["p"], *c["frames"], table=c["entry"],
                                            first_frame=c["first"], n_words=c["n_words"])
        c.update(rec=rec, nl=nl, table=table)
        _assert_case_reaches(name, c)
        return c


def _assert_case_reaches(name, c):
    """The case exercises what it was built for (on the reference's answer)."""
    rec, nl = c["rec"], c["nl"]
    nm = rec["num_matches"]
    assert (rec["pad"] == 0).all()
    if name.startswith("scales") or name == "camera":
        assert (nm > 200).all() and (nl > 0).all()
        if name == "camera":
            assert (rec["pnp_inliers"] > 0).all()
    elif name == "degenerate":
        assert (rec["status"] == np.where(np.isin(np.arange(11), (5, 6)), 4, 0)).all()
        assert (nm[[1, 2, 3, 5, 8, 9]] == 0).all() and (nm[[0, 4, 6, 7, 10]] > 0).all()
        assert nl[6] == 0 and (nl[[0, 4, 7, 10]] > 0).all()
    elif name == "odd":
        assert (nm == 16).any() and (nm > 0).all() and (nl > 0).all()
    elif name == "vocab60":
        assert (nl < nm).any() and (nl > 0).all()
    elif name == "vocab200":
        assert (nl > 0).all() and (c["table"]["word_id"] >= 0).sum() <= 91


@pytest.fixture(scope="module")
def refs(oracle, synth):
    return _References(oracle, synth)


@pytest.fixture(scope="module")
def lm_trackers():
    """A context per vocabulary, none of them the session's `tracker`."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    out = {}

    def get(vocab):
        key = vocab[3].shape
        if key not in out:
            out[key] = tracking.Tracker(0)
            out[key].bow_set_vocabulary(*vocab)
        return out[key]
    return get


ALL_ENTRIES = ("device", "host", "host:3", "host:pageable", "blocks:0", "blocks:8", "blocks_host:0", "blocks_host:8",
               "sharded", "host_sharded")
SOME_ENTRIES = ("device", "host:3", "blocks:8")
ENTRY_CASES = [(c, e) for c in ("scales", "scales_tc0", "degenerate") for e in ALL_ENTRIES] + \
              [(c, e) for c in ("odd", "vocab60", "vocab200", "resume", "camera") for e in SOME_ENTRIES]


@pytest.mark.gpu
@pytest.mark.parametrize("case,entry", ENTRY_CASES)
def test_entry_point_equals_reference(refs, lm_trackers, monkeypatch, case, entry):
    c = refs(case)
    monkeypatch.delenv("MV_HOST_CHUNK_PAIRS", raising=False)
    res, nl, table = run_entry(lm_trackers(c["vocab"]), c, entry, monkeypatch)
    assert res == c["rec"].tobytes(), first_difference(c["rec"], res)
    assert (nl == c["nl"]).all(), (nl, c["nl"])
    assert table == c["table"].tobytes()
