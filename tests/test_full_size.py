"""Full-size inputs against the CPU oracle: the shapes the product is built and benchmarked for, where the other
modules stop at KITTI-sized or smaller ones.

  * BASELINE configs[4], the stress shape of tools/stress_bench.py (94x310 cells, 85 % of them keypoints, top 16 000,
    up to 16 384 matches in a 33x33 window, 4 096 hypotheses): the depth path on two blocks of 8 pairs through every
    matcher, K3 form and staging of mv_track_sequence / mv_track_sequence_host, and the landmark path on 5 frames.
  * The landmark table's sequence sort with tiles of several frames (lmseq_tiles in bow.cu: t = min(512, 2^24 /
    n_words, n_steps) tiles of fb = ceil(n_steps / t) frames): mv_landmarks_sequence at fb = 9, 2, 8 and 20, the
    speculation over 8 blocks of the bench sequence, and the whole landmark path on the 4 541-frame bench sequence.
"""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from helpers import dev, pinned, ref_vocab, upload_table, with_first_pair
from landmark_reference import (back_project, detect, landmark_reference, orc_landmarks_sequence, pair_record, table_xyz,
                                track_cfg)

THREADS = os.cpu_count() or 1
ROWS, COLS, PERMILLE, SEED = 94, 310, 850, 0     # tools/stress_bench.py
f32 = np.float32


def _stress_params(first_pair=0, tc=True, lanes=1):
    from maveric_slam_b200 import tracking
    return tracking.track_params(ROWS, COLS, top_n=16000, max_valid=32768, max_matches=16384, hypotheses=4096,
                                 radius=16, shift=(4, 4), use_tensor_cores=tc, lanes=lanes, first_pair=first_pair)


def _stress_oracle(oracle, synth, first, n, lanes=1):
    """orc_bench_sequence over pairs first .. first + n - 1 of the stress sequence -> [PairResult]."""
    from oracle import orc
    off = synth.default_offsets(first + n + 1, SEED)
    cfg = track_cfg(_stress_params(first, lanes=lanes), synth.SEMI_SCALE)
    return oracle.bench_sequence(cfg, orc.SynthCfg(SEED, ROWS, COLS, PERMILLE, 6), off[first:first + n + 1], first, n,
                                 THREADS)[1]


def _tiles(n_words, n_steps):
    """lmseq_tiles (bow.cu) -> (tiles, frames per tile)."""
    t = max(1, min(512, (1 << 24) // n_words, n_steps))
    fb = -(-n_steps // t)
    return -(-n_steps // fb), fb


# ------------------------------------------------------------------ CPU: the oracle of the stress legs
def test_bench_sequence_equals_track_pair_at_stress_shape(oracle, synth):
    """The stress legs' oracle is orc_bench_sequence, which makes its frames with the C generator.  At the stress
    config it is orc_track_pair on orc_synth_frame frames, byte for byte, at pairs 0 and 1000."""
    cfg = track_cfg(_stress_params(), synth.SEMI_SCALE)

    def direct(first):
        off = synth.default_offsets(first + 2, SEED)
        f0, f1 = (oracle.synth_frame(SEED, ROWS, COLS, first + i, int(off[first + i, 0]), int(off[first + i, 1]),
                                     PERMILLE) for i in range(2))
        return oracle.track_pair(cfg, first, f0[0], f0[1], f0[2], f1[0], f1[1])

    with ThreadPoolExecutor(4) as ex:
        seq = [ex.submit(_stress_oracle, oracle, synth, first, 1) for first in (0, 1000)]
        one = [ex.submit(direct, first) for first in (0, 1000)]
        for s, o in zip(seq, one):
            got, want = s.result()[0], o.result()
            assert bytes(got) == bytes(want)
            assert want.num_matches > 5000 and want.status == 0


# ------------------------------------------------------------------ A: configs[4] through the depth path
@pytest.fixture(scope="module")
def stress_refs(oracle, synth):
    """The oracle's records of pairs 0 .. 7 and 1000 .. 1007, with one thread and one warp per hypothesis."""
    keys = [(first, lanes) for first in (0, 1000) for lanes in (1, 32)]
    with ThreadPoolExecutor(len(keys)) as ex:
        return dict(zip(keys, ex.map(lambda k: _stress_oracle(oracle, synth, k[0], 8, k[1]), keys)))


def _check_parity(res, ref, what):
    """Counts, status and the selected hypothesis exact, the pose within 1e-5 rad / 1e-5 relative, as bench.py
    measures it."""
    from bench import parity_against_port
    par = parity_against_port(res, ref, len(ref))
    print(what, par)
    assert par["mismatches"] == 0, (what, par)


@pytest.mark.gpu
@pytest.mark.parametrize("first", [0, 1000])
def test_stress_depth_path_vs_oracle(tracker, oracle, synth, stress_refs, monkeypatch, first):
    """8 pairs of the stress sequence from pair `first`: the tcgen05 leg against the oracle; the dp4a matcher and
    the host entry point (pinned, default chunks and chunks of 3 pairs) give its bytes; the one-warp K3 form against
    the oracle's one-warp form."""
    import torch
    from maveric_slam_b200 import tracking
    off = synth.default_offsets(first + 9, SEED)[first:]
    semi, desc, depth = tracker.synth_frames(SEED, ROWS, COLS, first, off, keypoint_permille=PERMILLE)
    # the oracle makes these frames with its own generator
    s, d, z = oracle.synth_frame(SEED, ROWS, COLS, first, int(off[0, 0]), int(off[0, 1]), PERMILLE)
    assert semi[0].cpu().numpy().tobytes() == s.tobytes() and desc[0].cpu().numpy().tobytes() == d.tobytes()
    assert depth[0].cpu().numpy().tobytes() == z.tobytes()
    scale = torch.full((9,), float(synth.SEMI_SCALE), device=tracker.device)

    def run(**kw):
        return tracking.results_to_numpy(tracker.track_sequence(_stress_params(first, **kw), semi, scale, desc, depth))

    want = run()
    ref = stress_refs[(first, 1)]
    assert min(r.num_matches for r in ref) > 5000 and all(r.status == 0 for r in ref)
    _check_parity(want, ref, "tcgen05")
    assert run(tc=False).tobytes() == want.tobytes(), "dp4a"
    _check_parity(run(lanes=32), stress_refs[(first, 32)], "lanes 32")
    host = [pinned(t) for t in (semi, scale, desc, depth)]
    for chunk in (None, "3"):
        if chunk:
            monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", chunk)
        got, _, _ = tracker.track_sequence_host(_stress_params(first), *host)
        assert got.tobytes() == want.tobytes(), ("host", chunk)


# ------------------------------------------------------------------ D: the landmark path at the stress shape
@pytest.fixture(scope="module")
def lm_tracker():
    """A context of its own with the reference vocabulary."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    tr = tracking.Tracker(0)
    tr.bow_set_vocabulary(*ref_vocab())
    return tr


@pytest.mark.gpu
def test_stress_landmark_path_vs_reference(lm_tracker, oracle, synth):
    """5 stress frames through the device and host one-calls (16 000 queries a frame, so each of the 10 000 words
    occurs 1.6 times a frame): records, landmark counts and the final table equal the CPU reference's."""
    import torch
    tr, n = lm_tracker, 5
    semi, desc, depth = tr.synth_frames(SEED, ROWS, COLS, 0, synth.default_offsets(n, SEED), keypoint_permille=PERMILLE)
    sscale = torch.full((n,), float(synth.SEMI_SCALE), device=tr.device)
    dscale = torch.full((n,), float(synth.DESC_SCALE), device=tr.device)
    frames = (semi, sscale, desc, dscale, depth)
    p = _stress_params()
    rec, nl, table = landmark_reference(oracle, oracle.bow_vocab(*ref_vocab()), p,
                                        *[t.cpu().numpy() for t in frames], n_words=10000, threads=THREADS)
    assert (rec["num_matches"] > 5000).all() and (nl > 0).all()
    t_dev = tr.landmarks_new(10000)
    res, got_nl = tr.track_sequence_landmarks(p, *frames, t_dev)
    assert res.cpu().numpy().tobytes() == rec.tobytes()
    assert (got_nl.cpu().numpy() == nl).all() and t_dev.cpu().numpy().tobytes() == table.tobytes()
    t_host = tr.landmarks_new(10000)
    res, got_nl, _, _ = tr.track_sequence_landmarks_host(p, *[pinned(t) for t in frames], t_host)
    assert res.tobytes() == rec.tobytes()
    assert (got_nl == nl).all() and t_host.cpu().numpy().tobytes() == table.tobytes()


# ------------------------------------------------------------------ E: sequence sorts whose tiles span several frames
def _stream(oracle, name):
    """Words, counts and coordinates of one table sequence, its entry table (None: empty) and tiling."""
    n, top_n, n_words, first, seed = {"bench": (4541, 1000, 10000, 7000, 41), "fb2": (513, 300, 10000, 0, 42),
                                      "words_2e21": (60, 1000, 1 << 21, -5, 43),
                                      "words_2e24": (20, 1000, (1 << 24) + 3, 100, 44)}[name]
    rng = np.random.default_rng(seed)
    word = rng.integers(100, n_words + n_words // 150, (n, top_n)).astype(np.int32)   # ids >= n_words among them
    word[rng.random((n, top_n)) < 0.003] = -1
    word[:, ::40] = 7                    # in every frame, 25 times: 113 525 occurrences over the bench case's tiles
    word[:, 20::80] = n_words - 1
    f = np.arange(n)
    for col, (w, gap) in enumerate(((11, 10), (12, 11), (13, 13), (14, 17), (15, 23))):
        word[f % gap == col, 1 + col] = w   # absent for gap - 1 > 8 frames, re-inserted at every place in a tile
    word[f % 3 == 0, 2:4] = 11           # and 11 twice more in every third frame (more duplicates in a frame)
    qc = np.full(n, top_n, np.int32)
    qc[::97] = 0
    qc[1::7] = rng.integers(1, top_n, len(qc[1::7]))
    qc[4::11] = top_n + 500
    qc[n - 1] = 0
    coords = rng.standard_normal((n, top_n, 3), dtype=np.float32)
    entry = None
    if name == "bench":                  # a live entry table: 30 frames before the sequence
        entry = oracle.pool_new(n_words)
        orc_landmarks_sequence(oracle, entry, first - 30, rng.integers(0, n_words, (30, top_n)).astype(np.int32),
                               np.full(30, top_n, np.int32), rng.standard_normal((30, top_n, 3), dtype=np.float32))
    return dict(n_words=n_words, first=first, word=word, qc=qc, coords=coords, entry=entry,
                tiles=_tiles(n_words, n))


class _Streams:
    """Each stream's inputs and the oracle's answer (coords_out, final table), computed once for the module."""

    def __init__(self, oracle):
        self.oracle, self.done = oracle, {}

    def __call__(self, name):
        if name not in self.done:
            c = _stream(self.oracle, name)
            table = self.oracle.pool_new(c["n_words"]) if c["entry"] is None else c["entry"].copy()
            c["out"] = orc_landmarks_sequence(self.oracle, table, c["first"], c["word"], c["qc"], c["coords"])
            c["table"] = table
            self.done[name] = c
        return self.done[name]


@pytest.fixture(scope="module")
def streams(oracle):
    return _Streams(oracle)


def _entry_table(tr, c):
    if c["entry"] is None:
        return tr.landmarks_new(c["n_words"])
    return upload_table(tr, c["entry"])


def _same_table(t_dev, table):
    return np.array_equal(t_dev.cpu().numpy(), table.view(np.uint8).reshape(-1, 56))


@pytest.mark.gpu
@pytest.mark.parametrize("case,tiling", [("bench", (505, 9)), ("fb2", (257, 2)), ("words_2e21", (8, 8)),
                                         ("words_2e24", (1, 20))])
def test_landmarks_sequence_tiles_of_several_frames(tracker, streams, case, tiling):
    """mv_landmarks_sequence against the oracle's table loop where the sort's tiles hold several frames: the bench
    length (4 541 steps, 10 000 words: 505 tiles of 9 frames, the last of 5) from a live table at frame 7000; 513
    steps (the last tile one frame); 2^21 words (8 tiles of 8 frames); 2^24 + 3 words (one tile of all 20 frames, a
    940 MB table).  A word in every frame 25 times (113 525 occurrences in the bench case), words absent for 9 to 22
    frames and re-inserted at every place in a tile, duplicates in a frame, ids -1 and >= n_words, frames with no
    queries and with q_count above top_n."""
    c = streams(case)
    assert c["tiles"] == tiling
    table = _entry_table(tracker, c)
    out = tracker.landmarks_sequence(table, c["first"], dev(tracker, c["word"]), dev(tracker, c["qc"]),
                                     dev(tracker, c["coords"]))
    assert np.array_equal(out.cpu().numpy().view(np.int32), c["out"].view(np.int32))
    assert _same_table(table, c["table"])
    if case == "bench":
        assert (c["word"] == 7).sum() >= 100000 and (c["out"] != 0).any(axis=2).mean() > 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("n_warm", [0, 8, 32])
def test_speculate_resolve_blocks_of_the_bench_stream(tracker, streams, n_warm):
    """The bench-length stream as the 8 blocks of shard_pairs(4540, 8, r) (the last to the stream's end), each a
    speculation of more than 512 steps, so tiles of 2 frames: all speculated first, in reverse order, then resolved
    in order against a running table.  Each block's coords and the final table equal the oracle's."""
    import torch
    from maveric_slam_b200 import tracking
    c = streams("bench")
    n = c["word"].shape[0]
    blocks = [tracking.shard_pairs(n - 1, 8, r)[:2] for r in range(8)]
    blocks[-1] = (blocks[-1][0], n - blocks[-1][0])
    word, qc, coords = (dev(tracker, c[k]) for k in ("word", "qc", "coords"))
    specs = {}
    for r in reversed(range(8)):
        lo, cnt = blocks[r]
        w = min(n_warm, lo)
        assert _tiles(c["n_words"], w + cnt)[1] == 2
        specs[r] = tracker.landmarks_speculate(c["n_words"], c["first"] + lo, w, word[lo - w:lo + cnt],
                                               qc[lo - w:lo + cnt], coords[lo:lo + cnt])
    table = _entry_table(tracker, c)
    rewalked = []
    for r, (lo, cnt) in enumerate(blocks):
        n_rw = torch.full((1,), -1, dtype=torch.int32, device=tracker.device)
        got = tracker.landmarks_resolve(specs[r], table, n_rewalked=n_rw)
        tracker.landmarks_release(specs[r])
        assert np.array_equal(got.cpu().numpy().view(np.int32), c["out"][lo:lo + cnt].view(np.int32)), r
        rewalked.append(int(n_rw.item()))
    assert _same_table(table, c["table"])
    assert min(rewalked) >= 0
    if n_warm == 0:   # the guess is wrong for some words: both the patch and the re-walk ran
        assert max(rewalked) > 0, rewalked


# ------------------------------------------------------------------ E: the whole landmark path on the bench sequence
NF = 4541
# the first 3 pairs, both sides of the boundaries of tiles 1, 2, 100, 251, 400 and 500 (9 frames a tile), four from
# the middle, the last 5
SAMPLED_PAIRS = sorted({0, 1, 2, 1000, 2000, 3000, 4000, *range(NF - 6, NF - 1)}
                       | {9 * k + d for k in (1, 2, 100, 251, 400, 500) for d in (-1, 0)})


@pytest.mark.gpu
def test_landmark_path_bench_sequence(lm_tracker, oracle, synth):
    """mv_track_sequence_landmarks on the 4 541-frame bench sequence (4 540 table steps: tiles of 9 frames), and the
    same sequence as 8 prepared blocks on one context (all prepared, then stepped and solved in order): the blocks
    give the one-call's bytes, and the one-call equals the CPU reference at 24 sampled pairs.

    The reference is built in parts, as the CPU word assignment of 4 541 frames takes minutes: the device's query
    lists and words of every frame, held equal to oracle.top_n / oracle.bow_assign on the sampled pairs' frames and a
    few more (per-frame functions, pinned elsewhere at this shape); coordinates back-projected from them; the oracle
    table walked over all frames; match, RANSAC-E and K3 by the oracle at the sampled pairs only, on frames made by
    oracle.synth_frame."""
    import torch
    from maveric_slam_b200 import tracking
    tr = lm_tracker
    p = tracking.kitti_track_params(top_n=1000, max_valid=8192, max_matches=1024, hypotheses=1024, seed=SEED)
    rows, cols, top_n, n_words, dsc = 47, 155, 1000, 10000, 4.3353
    off = synth.default_offsets(NF, SEED)
    semi, desc, depth = tr.synth_frames(SEED, rows, cols, 0, off)
    sscale = torch.full((NF,), float(synth.SEMI_SCALE), device=tr.device)
    dscale = torch.full((NF,), dsc, device=tr.device)
    frames = (semi, sscale, desc, dscale, depth)
    assert _tiles(n_words, NF - 1) == (505, 9)
    table = tr.landmarks_new(n_words)
    res, nl = tr.track_sequence_landmarks(p, *frames, table)
    res, nl, final = res.cpu().numpy(), nl.cpu().numpy(), table.cpu().numpy()

    blocks = [tracking.shard_pairs(NF - 1, 8, r)[:2] for r in range(8)]
    prepared = [tr.track_landmarks_prepare(with_first_pair(p, lo), 0, lo, *[x[lo:lo + cnt + 1] for x in frames], n_words)
                for lo, cnt in blocks]
    t_blk = tr.landmarks_new(n_words)
    got, got_nl = [], []
    for blk in prepared:
        tr.track_landmarks_step_table(blk, t_blk)
        r, k = tr.track_landmarks_solve(blk)
        got.append(r.cpu().numpy()); got_nl.append(k.cpu().numpy())
        tr.track_landmarks_release(blk)
    assert np.concatenate(got).tobytes() == res.tobytes() and (np.concatenate(got_nl) == nl).all()
    assert t_blk.cpu().numpy().tobytes() == final.tobytes()

    # the reference: the device's per-frame stages, checked on sampled frames
    idx, prob, _ = tr.softmax(semi, sscale)
    qp, qi, _, qc, ov = tr.top_n(idx, prob, top_n, p.max_valid)
    word, _ = tr.bow_assign(desc[:NF - 1], dscale[:NF - 1], qp[:NF - 1], qc[:NF - 1])
    qp, qi, qc, word, hdepth = (t.cpu().numpy() for t in (qp, qi, qc, word, depth))
    del semi, desc, frames
    vocab = oracle.bow_vocab(*ref_vocab())

    def oracle_frame(f):
        return oracle.synth_frame(SEED, rows, cols, f, int(off[f, 0]), int(off[f, 1]))

    def check_frame(f):
        s, d, _ = oracle_frame(f)
        pa, ix, _, o_ov = oracle.top_n(float(synth.SEMI_SCALE), s, top_n, p.max_valid)
        k = int(qc[f])
        assert k == len(pa) and (qp[f, :k] == pa).all() and (qi[f, :k] == ix).all(), f
        base, wid = oracle.bow_assign(vocab, dsc, d[pa])
        assert (word[f, :k] == base * vocab.words_per_base + wid).all(), f

    checked = sorted(set(SAMPLED_PAIRS) | {250, 500, 1500, 2500, 3500, 4200})
    with ThreadPoolExecutor(THREADS) as ex:
        list(ex.map(check_frame, checked))
    assert len(checked) >= 30
    o_table = oracle.pool_new(n_words)
    snaps = {}
    for f in range(NF - 1):
        k = int(qc[f])
        oracle.pool_observe(o_table, f, word[f, :k], back_project(p, qp[f, :k], qi[f, :k], hdepth[f]))
        oracle.pool_remove_old(o_table, f)
        if f in SAMPLED_PAIRS:
            snaps[f] = o_table.copy()
    assert o_table.tobytes() == final.tobytes()

    def pair(q):
        (s0, d0, _), (s1, d1, _) = oracle_frame(q), oracle_frame(q + 1)
        det0, det1 = detect(oracle, p, np.stack([s0, s1]), np.full(2, synth.SEMI_SCALE, f32))
        k = int(qc[q])
        return pair_record(oracle, p, det0, det1, d0, d1, q, table_xyz(det0[2], word[q, :k], snaps[q], n_words))

    with ThreadPoolExecutor(THREADS) as ex:
        for q, (r, k) in zip(SAMPLED_PAIRS, ex.map(pair, SAMPLED_PAIRS)):
            assert res[q:q + 1].tobytes() == r.tobytes() and nl[q] == k, (q, res[q], r, nl[q], k)
            assert r["num_matches"] > 100 and k > 0
