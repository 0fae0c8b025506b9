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
import os

import numpy as np
import pytest

from landmark_reference import landmark_reference, track_cfg

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
f32 = np.float32
# fx != fy, cx and cy off the KITTI values, K3's gate, damping, iteration counts and sample size off their defaults
CAMERA_PNP = dict(fx=520.0, fy=910.0, cx=300.5, cy=260.25, gate_sq=16.0, damping=1e-3, sample_iters=3, refine_iters=6,
                  sample_size=9)


def _ref_vocab():
    v = np.load(os.path.join(GOLDEN, "ref_vocab.npz"))
    return v["base_desc"], v["scale"], v["bias"], v["leaves"]


def _random_vocab(rng, n_base, wpb):
    base = rng.integers(-128, 128, (256, n_base)).astype(np.int8)
    scale = rng.uniform(0.5, 2.0, n_base).astype(f32)
    bias = rng.uniform(-0.3, 0.3, n_base).astype(f32)
    leaves = rng.integers(-2 ** 31, 2 ** 31, (n_base, wpb, 4)).astype(np.int32)
    return base, scale, bias, leaves


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
# one frame per (descriptor kind, desc_scale): random, zero, all -128, all 127, one row repeated
BOW_SCALES = (4.3353, -1.5, 0.0, 1e-30, 1e30, np.inf, -np.inf, np.nan)
BOW_KINDS = ("random", "zero", "min", "max", "repeated")


def _bow_vocab(name):
    """(n_base, wpb) shapes with random contents, the reference vocabulary, and vocabularies built to tie."""
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "10x1000":
        return _ref_vocab()
    if "x" in name:
        nb, wpb = (int(x) for x in name.split("x"))
        return _random_vocab(rng, nb, wpb)
    if name == "repeated_leaves":      # leaf w = L[w % 5]: every 8-word window occurs at 4 leaves of different lanes
        base, scale, bias, _ = _random_vocab(rng, 3, 20)
        L = rng.integers(-2 ** 31, 2 ** 31, (5, 4)).astype(np.int32)
        return base, scale, bias, np.ascontiguousarray(np.broadcast_to(L[np.arange(20) % 5], (3, 20, 4)))
    if name == "zero_leaves":          # every window ties
        base, scale, bias, leaves = _random_vocab(rng, 2, 16)
        return base, scale, bias, np.zeros_like(leaves)
    if name == "nonpositive_scores":   # no score exceeds 0: base 0
        base, scale, bias, leaves = _random_vocab(rng, 4, 11)
        scale[:2], bias[:2], bias[2:] = 0.0, 0.0, -1.2
        return base, scale, bias, leaves
    if name == "equal_bases":          # bases 2..4 identical and the only ones that can win: base 2
        base, scale, bias, leaves = _random_vocab(rng, 5, 12)
        base[:, 3] = base[:, 4] = base[:, 2]
        scale[3:] = scale[2]
        bias[3:] = bias[2] = 0.25
        bias[:2] = -1.0
        return base, scale, bias, leaves
    raise KeyError(name)


def _bow_inputs(seed, top_n, cells=48, reps=1):
    """Descriptors of len(BOW_KINDS) x len(BOW_SCALES) x reps frames, their scales, query cells (duplicates
    included) and counts (0 and top_n among them)."""
    rng = np.random.default_rng(seed)
    n = len(BOW_KINDS) * len(BOW_SCALES) * reps
    desc = rng.integers(-128, 128, (n, cells, 256)).astype(np.int8)
    dscale = np.zeros(n, f32)
    for f in range(n):
        kind = BOW_KINDS[(f // len(BOW_SCALES)) % len(BOW_KINDS)]
        dscale[f] = BOW_SCALES[f % len(BOW_SCALES)]
        if kind == "zero":
            desc[f] = 0
        elif kind == "min":
            desc[f] = -128
        elif kind == "max":
            desc[f] = 127
        elif kind == "repeated":
            desc[f] = desc[f, 0]
    qp = rng.integers(0, cells, (n, top_n)).astype(np.int32)
    qp[:, 1::3] = qp[:, 0::3][:, :qp[:, 1::3].shape[1]]       # the same cell queried twice
    qc = rng.integers(1, top_n + 1, n).astype(np.int32)
    qc[::7] = top_n
    qc[3::11] = 0
    for f in range(n):
        qp[f, qc[f]:] = 0
    return desc, dscale, qp, qc


def _bow_check(tr, oracle, vocab, desc, dscale, qp, qc):
    import torch
    v = oracle.bow_vocab(*vocab)
    wpb = vocab[3].shape[1]
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(tr.device)  # noqa: E731
    word, base = tr.bow_assign(d(desc), d(dscale), d(qp), d(qc))
    word, base = word.cpu().numpy(), base.cpu().numpy()
    for f in range(desc.shape[0]):
        k = int(qc[f])
        assert (word[f, k:] == -1).all() and (base[f, k:] == -1).all(), f
        rb, rw = oracle.bow_assign(v, dscale[f], desc[f][qp[f, :k]])
        assert (base[f, :k] == rb).all(), (f, dscale[f])
        assert (word[f, :k] == rb * wpb + rw).all(), (f, dscale[f])
    return word


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
    vocab = _bow_vocab(name)
    own_tracker.bow_set_vocabulary(*vocab)
    word = _bow_check(own_tracker, oracle, vocab, *_bow_inputs(7, 37))
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
    vocab = _bow_vocab("3x7")
    own_tracker.bow_set_vocabulary(*vocab)
    reps = 4 if top_n == 129 else 1
    desc, dscale, qp, qc = _bow_inputs(top_n, top_n, reps=reps)
    assert top_n < 129 or desc.shape[0] * top_n > 148 * 128
    _bow_check(own_tracker, oracle, vocab, desc, dscale, qp, qc)


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
    va, vb = _ref_vocab(), _bow_vocab("1x9")
    a.bow_set_vocabulary(*va)
    b.bow_set_vocabulary(*vb)
    inputs = _bow_inputs(3, 37)
    for tr, v in ((a, va), (b, vb), (a, va), (b, vb)):
        _bow_check(tr, oracle, v, *inputs)


# ------------------------------------------------------------------ GPU: every entry point against the reference
def _case_inputs(name, synth):
    """Host inputs and parameters of one case -> dict(p, frames (semi, semi_scale, desc, desc_scale, depth), first,
    n_words, vocab, entry table or None)."""
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    rng = np.random.default_rng(sum(map(ord, name)))
    vocab = _ref_vocab()
    n_words, first, entry = 10000, 0, None
    if name == "scales":
        rows, cols, n = 47, 155, 20
        semi, desc, depth, _ = synth.synth_sequence(31, rows, cols, n)
        rng = np.random.default_rng(8)
        sscale = (synth.SEMI_SCALE * rng.uniform(0.9, 1.1, n)).astype(f32)
        dscale = (synth.DESC_SCALE * rng.uniform(0.5, 2.0, n)).astype(f32)
        dscale[4], dscale[11] = -dscale[4], 0.0
        p = tracking.kitti_track_params(hypotheses=256)
        first = 500
    elif name == "degenerate":
        rows, cols, n = 24, 80, 12
        semi, desc, depth, off = synth.synth_sequence(5, rows, cols, n)
        semi[2:4, :, :64], semi[2:4, :, 64] = -128, 127                    # no keypoints
        semi[6] = synth.synth_frame(5, rows, cols, 6, int(off[6, 0]), int(off[6, 1]), keypoint_permille=1000)[0]
        desc[8], desc[9] = -128, 0
        sscale = np.full(n, synth.SEMI_SCALE, f32)
        dscale = np.full(n, synth.DESC_SCALE, f32)
        p = tracking.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=64)
    elif name == "odd":
        rows, cols, n = 13, 37, 14
        semi, desc, depth, _ = synth.synth_sequence(9, rows, cols, n, offsets=synth.default_offsets(n, 9, step=0),
                                                    keypoint_permille=300, noise_amp=2)
        sscale = np.full(n, synth.SEMI_SCALE, f32)
        dscale = (synth.DESC_SCALE * rng.uniform(0.5, 2.0, n)).astype(f32)
        # a query has at most one match, so the cap binds only below top_n
        p = tracking.track_params(rows, cols, top_n=37, max_valid=482, max_matches=16, hypotheses=32, radius=6,
                                  shift=(-2, 1), lanes=32)
        first = -20
    elif name in ("vocab60", "vocab200"):
        rows, cols, n = 24, 80, 16
        semi, desc, depth, _ = synth.synth_sequence(13, rows, cols, n)
        sscale = np.full(n, synth.SEMI_SCALE, f32)
        dscale = np.full(n, synth.DESC_SCALE, f32)
        vocab = _random_vocab(np.random.default_rng(77), 7, 13)
        vocab[3][:, 6:9] = vocab[3][:, 2:5]                                  # repeated leaves
        p = tracking.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=64)
        n_words, first = int(name[5:]), 40
    else:
        raise KeyError(name)
    return dict(p=p, frames=[semi, sscale, desc, dscale, depth], first=first, n_words=n_words, vocab=vocab,
                entry=entry)


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
            c["p"] = copy.copy(a["p"])
            c["p"].pnp = copy.copy(a["p"].pnp)
            c["p"].pnp.first_pair = 8
            c.update(frames=[x[8:] for x in a["frames"]], first=a["first"] + 8, entry=head[2],
                     rec=a["rec"][8:], nl=a["nl"][8:])
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
        c = _case_inputs(name, self.synth)
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


def _pinned(torch, a):
    h = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype, pin_memory=True)
    h.copy_(torch.from_numpy(np.ascontiguousarray(a)))
    return h


def _params(p, first_pair):
    q = copy.copy(p)
    q.pnp = copy.copy(p.pnp)
    q.pnp.first_pair = first_pair
    return q


def _blocks(n_pairs, sizes):
    out, lo = [], 0
    for s in sizes:
        if lo < n_pairs:
            out.append((lo, min(s, n_pairs - lo)))
            lo += out[-1][1]
    if lo < n_pairs:
        out.append((lo, n_pairs - lo))
    return out


def _run(tr, c, entry, monkeypatch):
    """Runs one entry point on the case -> (records bytes, n_with_landmark int32, final table bytes)."""
    import torch
    from maveric_slam_b200 import tracking
    p, first, n_words = c["p"], c["first"], c["n_words"]
    host = c["frames"]
    dev = [torch.from_numpy(np.ascontiguousarray(x)).to(tr.device) for x in host]
    n_pairs = host[0].shape[0] - 1
    entry_table = c["entry"] if c["entry"] is not None else None
    if entry_table is None:
        table = tr.landmarks_new(n_words)
    else:
        table = torch.from_numpy(np.ascontiguousarray(entry_table).view(np.uint8).reshape(-1, 56).copy()).to(tr.device)
    kind, _, opt = entry.partition(":")
    if kind == "device":
        res, nl = tr.track_sequence_landmarks(p, *dev, table, first_frame=first)
        res, nl = res.cpu().numpy(), nl.cpu().numpy()
    elif kind == "host":
        if opt == "pageable":
            bufs = [np.ascontiguousarray(x) for x in host]
        else:
            bufs = [_pinned(torch, x) for x in host]
            if opt:
                monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", opt)
        res, nl, _, _ = tr.track_sequence_landmarks_host(p, *bufs, table, first_frame=first)
    elif kind in ("blocks", "blocks_host"):
        n_warm = int(opt)
        bufs = dev if kind == "blocks" else [_pinned(torch, x) for x in host]
        prep = tr.track_landmarks_prepare if kind == "blocks" else tr.track_landmarks_prepare_host
        blocks = _blocks(n_pairs, (1, 5))
        prepared = {}
        for i, (lo, cnt) in reversed(list(enumerate(blocks))):
            w = min(n_warm, lo)
            prepared[i] = prep(_params(p, p.pnp.first_pair + lo), w, first + lo, *[x[lo - w:lo + cnt + 1] for x in bufs],
                               n_words)
        res, nl = [], []
        for i in range(len(blocks)):
            tr.track_landmarks_step_table(prepared[i], table)
            r, n = tr.track_landmarks_solve(prepared[i])
            res.append(r.cpu().numpy()); nl.append(n.cpu().numpy())
            tr.track_landmarks_release(prepared[i])
        res, nl = np.concatenate(res), np.concatenate(nl)
    elif kind == "sharded":
        res, nl, _ = tracking.track_sequence_landmarks_sharded(tr, p, dev, table, first_frame=first, n_warm=8)
        res, nl = res.cpu().numpy(), nl.cpu().numpy()
    elif kind == "host_sharded":
        bufs = [_pinned(torch, x) for x in host]
        res, nl, _, _ = tracking.track_sequence_landmarks_host_sharded(tr, p, bufs, table, first_frame=first, n_warm=8)
        res, nl = res.cpu().numpy(), nl.cpu().numpy()
    else:
        raise KeyError(entry)
    torch.cuda.synchronize()
    return np.ascontiguousarray(res).view(np.uint8).reshape(-1).tobytes(), np.asarray(nl, np.int32), \
        table.cpu().numpy().tobytes()


def _first_difference(want, got):
    """Pair and field of the first differing byte of two record arrays."""
    from maveric_slam_b200 import tracking
    g = np.frombuffer(got, tracking.PAIR_RESULT_DTYPE)
    for q in range(len(want)):
        for f in tracking.PAIR_RESULT_DTYPE.names:
            if want[q][f].tobytes() != g[q][f].tobytes():
                return "pair %d %s: reference %r, got %r" % (q, f, want[q][f], g[q][f])
    return "lengths %d, %d" % (len(want), len(g))


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
    res, nl, table = _run(lm_trackers(c["vocab"]), c, entry, monkeypatch)
    assert res == c["rec"].tobytes(), _first_difference(c["rec"], res)
    assert (nl == c["nl"]).all(), (nl, c["nl"])
    assert table == c["table"].tobytes()
