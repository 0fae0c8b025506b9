"""Loop closure away from the shapes it was built with: the idf weights at their rounding ties, the candidates at
the tile kernel's 128-frame tiles and 64-word k-blocks, at the limits include/maveric_b200.h states and after larger
calls on the same context, and every branch of mv_detect_loops' selection rule.

The candidates and weights are held byte for byte to tests/lcd_oracle.c; mv_detect_loops is held to the library's
separate calls (loop_reference.verify_by_parts) on all of its slots and, on a few frames, to the CPU oracle chain
(detector, match, depth correspondences and K3 of oracle/).
"""
import math

import numpy as np
import pytest

import lcd_oracle
from helpers import dev, ref_vocab, same_bits
from landmark_reference import depth_xyz, detect, match_cfg, pnp_cfg
from loop_reference import (COLS, ROWS, frames, idf, loop_offsets, random_weights, random_words, ref_word_weights,
                            run_candidates, select, small_params, verify_by_parts)

INT_MAX, INT_MIN = 2 ** 31 - 1, -2 ** 31


def cyclic_words(n, dfs, stride=7):
    """Word w held by frames {(w * stride + t) mod n : t < dfs[w]}: every frame's list stays short whatever the
    document frequencies.  -> (word int32 [n, top_n] padded with -1, q_count int32 [n] = top_n)."""
    rows = np.concatenate([(w * stride + np.arange(d)) % n for w, d in enumerate(dfs)])
    ids = np.concatenate([np.full(d, w, np.int32) for w, d in enumerate(dfs)])
    order = np.argsort(rows, kind="stable")
    rows, ids = rows[order], ids[order]
    count = np.bincount(rows, minlength=n)
    top_n = int(count.max())
    pos = np.arange(len(rows)) - np.repeat(np.cumsum(count) - count, count)
    word = np.full((n, top_n), -1, np.int32)
    word[rows, pos] = ids
    return word, np.full(n, top_n, np.int32)


def tie_dfs(m, seed):
    """Document frequencies of a call over n = m^2 frames: word 0 at df = m (the tie), then 1, 2, n - 1, n and a
    spread of others."""
    n = m * m
    rng = np.random.default_rng(seed)
    return [m, 1, 2, n - 1, n, m - 1, m + 1, 3, max(n // 2, 1), n // 3 + 1] + rng.integers(1, n + 1, 6).tolist()


def limit_dfs():
    """Document frequencies at the 65 535-frame limit: 255 (65 025 = 255^2 is not the count here), 256, the ends,
    and a geometric spread."""
    n = 65535
    return [255, 256, 1, 2, n - 1, n] + sorted({int(round(x)) for x in np.geomspace(3, n - 2, 40)})


# ------------------------------------------------------------------ A. word weights at the rounding ties
def test_idf_ties_on_the_host():
    """At df^2 = n the weight is exactly 63.5, which rounds to even: 64.  Evaluated in double it can land an ulp either
    side (with the C library's log it does for m = 11, 13, 21, ...), so the oracle and the restatement decide the tie
    in integers; both give 64 to the tie word at every m of 2 .. 255 and agree on the cyclic lists."""
    plain = [m for m in range(2, 256) if round(127.0 * math.log(m) / math.log(m * m)) != 64]
    print("m where rint of the double value is not 64:", plain)
    for m in range(2, 256):
        n = m * m
        assert idf(n, m) == 64, m
        dfs = tie_dfs(m, m)
        word, q_count = cyclic_words(n, dfs)
        want = lcd_oracle.word_weights(word, q_count, len(dfs))
        assert want[0] == 64, m
        assert want.tolist() == [idf(n, d) for d in dfs], m
        if m <= 40:
            assert ref_word_weights(word, q_count, len(dfs)).tobytes() == want.tobytes(), m


def test_idf_at_the_frame_limit_on_the_host():
    dfs = limit_dfs()
    word, q_count = cyclic_words(65535, dfs, stride=257)
    assert lcd_oracle.word_weights(word, q_count, len(dfs)).tolist() == [idf(65535, d) for d in dfs]


@pytest.mark.gpu
def test_word_weights_at_rounding_ties(tracker):
    """n = m^2 frames for every m of 2 .. 255 (65 025 = 255^2 the last), word 0 held by m of them."""
    bad = []
    for m in range(2, 256):
        dfs = tie_dfs(m, m)
        word, q_count = cyclic_words(m * m, dfs)
        want = lcd_oracle.word_weights(word, q_count, len(dfs))
        got = tracker.lcd_word_weights(dev(tracker, word), dev(tracker, q_count), n_words=len(dfs)).cpu().numpy()
        if got.tobytes() != want.tobytes():
            bad.append((m, got.tolist(), want.tolist()))
    assert not bad, "m, device, oracle: %s" % bad


@pytest.mark.gpu
def test_word_weights_at_the_frame_limit(tracker):
    dfs = limit_dfs()
    word, q_count = cyclic_words(65535, dfs, stride=257)
    got = tracker.lcd_word_weights(dev(tracker, word), dev(tracker, q_count), n_words=len(dfs)).cpu().numpy()
    assert got.tobytes() == lcd_oracle.word_weights(word, q_count, len(dfs)).tobytes()


# ------------------------------------------------------------------ B. candidates at tile and k-block edges
def check_candidates(tracker, word, q_count, n_words, weight, min_gap, k, min_score, first_frame):
    got = run_candidates(tracker, word, q_count, n_words, weight, min_gap, k, min_score, first_frame)
    want = lcd_oracle.candidates(word, q_count, n_words, weight, min_gap, k, min_score, first_frame)
    case = (word.shape, n_words, weight is not None, min_gap, k, min_score, first_frame)
    assert got[0].tobytes() == want[0].tobytes(), case
    assert got[1].tobytes() == want[1].tobytes(), case
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("n_words", [63, 64, 65, 129, 192, 193, 257, 320])
@pytest.mark.parametrize("n", [127, 128, 129, 255, 256, 257])
def test_candidates_at_tile_and_kblock_edges(tracker, n, n_words):
    """Frame counts either side of one and two 128-frame tiles, 1 .. 5 k-blocks of 64 words (the ring has 4 stages),
    and min_gap at the column-tile edges; k, weights, min_score and the first frame vary with the case."""
    rng = np.random.default_rng(n * 1000 + n_words)
    word, q_count = random_words(rng, n, 24, n_words)
    weight = random_weights(rng, n_words)
    for c, min_gap in enumerate([0, 1, 127, 128, 129, n - 1, n]):
        k = (c + n + n_words) % 8 + 1
        check_candidates(tracker, word, q_count, n_words, weight if (c + n_words) % 2 else None, min_gap, k,
                         (1, 0, 2)[c % 3], (0, -n - 3, 11)[(c + n) % 3])


def hub_inputs(n, shares, n_hub=6):
    """Frame f holds a private word (n_hub + f) and the first shares.get(f, 0) of n_hub hub words.
    -> (word, q_count, n_words)."""
    word = np.full((n, n_hub + 1), -1, np.int32)
    word[:, 0] = n_hub + np.arange(n)
    for f, s in shares.items():
        word[f, 1:1 + s] = np.arange(s)
    return word, np.full(n, n_hub + 1, np.int32), n_hub + n


@pytest.mark.gpu
def test_candidates_tie_truncation_and_merge(tracker):
    """More than k (and more than the 8 a tile keeps) equal best scores inside one tile, and equal best scores spread
    over three tiles: the earlier frames win in both."""
    n, q = 300, 299
    in_tile = [3, 9, 17, 40, 41, 42, 100, 126, 127]
    spread = [5, 60, 127, 128, 130, 200, 255, 256, 270]
    for tied in (in_tile, spread):
        shares = {f: 6 for f in tied + [q]}
        shares.update({2: 5, 129: 5, 150: 4})
        word, q_count, n_words = hub_inputs(n, shares)
        for weighted in (False, True):
            weight = np.full(n_words, 3, np.int8) if weighted else None
            for k in range(1, 9):
                for min_gap in (0, 29):
                    cand, _ = check_candidates(tracker, word, q_count, n_words, weight, min_gap, k, 1, 0)
                    # at min_gap 0 the frame itself (the hub and its own word) comes first
                    best = [q] * (min_gap == 0) + [j for j in tied if j <= q - min_gap]
                    assert len(best) > k
                    assert cand[q].tolist() == best[:k], (tied, k, min_gap)


@pytest.mark.gpu
@pytest.mark.parametrize("n,i,min_gap", [(300, 299, 40), (256, 255, 128), (257, 256, 129), (129, 128, 1),
                                         (300, 299, 0), (257, 256, 0)])
def test_candidates_best_at_the_last_allowed_column(tracker, n, i, min_gap):
    """Frame i's unique best is frame i - min_gap, in the last column tile i may see; frame i - min_gap + 1 would
    score higher but is not allowed."""
    word = np.full((n, 8), -1, np.int32)
    word[:, 0] = 0                          # one word every frame holds
    word[:, 1] = 8 + np.arange(n)           # a private word
    j = i - min_gap
    word[i, 2:8] = np.arange(1, 7)
    word[j, 2:6] = np.arange(1, 5)
    if j + 1 < n and j + 1 != i:
        word[j + 1, 2:8] = np.arange(1, 7)
    q_count = np.full(n, 8, np.int32)
    for weight in (None, np.full(8 + n, 127, np.int8)):
        cand, score = check_candidates(tracker, word, q_count, 8 + n, weight, min_gap, 8, 1, -5)
        assert cand[i, 0] == -5 + j


@pytest.mark.gpu
@pytest.mark.parametrize("min_gap", [0, 1, 128])
def test_candidates_largest_scores(tracker, min_gap):
    """Every weight 127 on dense lists: scores up to 127 * 320."""
    n, n_words = 257, 320
    rng = np.random.default_rng(min_gap)
    word = np.tile(np.arange(n_words, dtype=np.int32), (n, 1))
    word[rng.random(word.shape) < 0.02] = -1
    q_count = np.full(n, n_words, np.int32)
    _, score = check_candidates(tracker, word, q_count, n_words, np.full(n_words, 127, np.int8), min_gap, 8, 1, 0)
    assert score.max() > 127 * 290


@pytest.mark.gpu
def test_candidates_zero_weights_and_negative_min_score(tracker):
    """All weights 0: with min_score 0 every allowed frame ties at 0 (the first k allowed frames), with 1 there are
    none.  A negative min_score admits every allowed frame."""
    n, n_words = 200, 150
    rng = np.random.default_rng(5)
    word, q_count = random_words(rng, n, 30, n_words)
    zero = np.zeros(n_words, np.int8)
    for min_gap, k in [(0, 8), (3, 5), (129, 2)]:
        cand, score = check_candidates(tracker, word, q_count, n_words, zero, min_gap, k, 0, 7)
        for i in range(n):
            hi = i - min_gap + 1
            want = (7 + np.arange(min(max(hi, 0), k))).tolist()
            assert cand[i, :len(want)].tolist() == want and (cand[i, len(want):] == -1).all(), i
        assert (score == 0).all()
        cand, _ = check_candidates(tracker, word, q_count, n_words, zero, min_gap, k, 1, 7)
        assert (cand == -1).all()
        for weight in (None, random_weights(rng, n_words)):
            cand, _ = check_candidates(tracker, word, q_count, n_words, weight, min_gap, k, -3, 100)
            assert (cand[min_gap + k - 1:] >= 100).all()


@pytest.mark.gpu
def test_candidates_after_larger_calls_on_one_context(tracker):
    """Shrinking calls on one context, whose presence and per-tile scratch hold the larger call's contents: each
    equals the oracle and a fresh context."""
    from maveric_slam_b200 import tracking
    steps = [(4541, 1000, 10000, True, 30, 4, 1, 0), (37, 13, 100, False, 0, 8, 1, 5),
             (300, 50, 10000, True, 129, 8, 2, 0), (129, 40, 10000, True, 1, 3, 1, -129)]
    for c, (n, top_n, n_words, weighted, min_gap, k, min_score, first_frame) in enumerate(steps):
        rng = np.random.default_rng(c)
        word, q_count = random_words(rng, n, top_n, n_words)
        weight = random_weights(rng, n_words) if weighted else None
        args = (word, q_count, n_words, weight, min_gap, k, min_score, first_frame)
        want = check_candidates(tracker, *args)
        fresh = run_candidates(tracking.Tracker(0), *args)
        assert fresh[0].tobytes() == want[0].tobytes() and fresh[1].tobytes() == want[1].tobytes(), n


# ------------------------------------------------------------------ C. the stated limits
@pytest.mark.gpu
def test_candidates_at_the_frame_limit(tracker):
    """65 535 frames (512 row tiles, 131 328 tiles, 2.1 GB of per-tile lists at k = 8) with idf weights.  Frame
    65 534's best is frame 0 and its second frame 65 434 = 65 534 - min_gap, in the last row tile's last allowed
    column tile."""
    n, top_n, n_words, min_gap = 65535, 8, 10000, 100
    rng = np.random.default_rng(65535)
    word = rng.integers(16, n_words, size=(n, top_n)).astype(np.int32)    # words 0 .. 15 are planted only
    word[n - 1, :6] = np.arange(6)
    word[0, :4] = np.arange(4)
    word[n - 1 - min_gap, :2] = (4, 5)
    q_count = np.full(n, top_n, np.int32)
    weight = lcd_oracle.word_weights(word, q_count, n_words)
    got_w = tracker.lcd_word_weights(dev(tracker, word), dev(tracker, q_count), n_words=n_words).cpu().numpy()
    assert got_w.tobytes() == weight.tobytes()
    cand, _ = check_candidates(tracker, word, q_count, n_words, weight, min_gap, 8, 1, 0)
    assert cand[n - 1, :2].tolist() == [0, n - 1 - min_gap]


@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True])
def test_candidates_at_the_word_limit(tracker, weighted):
    """n_words = 2^24: P is 4.3 GB (twice that with weights), the last k-block's TMA coordinate is 2^24 - 64, and the
    words come from both ends of the range, the last k-block's among them."""
    n, n_words = 200, 1 << 24
    rng = np.random.default_rng(24)
    word = np.concatenate([rng.integers(0, 2000, (n, 15)), rng.integers(n_words - 2000, n_words, (n, 15)),
                           rng.integers(n_words - 64, n_words, (n, 10))], 1).astype(np.int32)
    q_count = np.full(n, word.shape[1], np.int32)
    q_count[::9] = 25
    weight = random_weights(rng, n_words) if weighted else None
    cand, score = check_candidates(tracker, word, q_count, n_words, weight, 3, 8, 1, 0)
    assert (cand[50:] >= 0).all()
    if weighted:
        got_w = tracker.lcd_word_weights(dev(tracker, word), dev(tracker, q_count), n_words=n_words).cpu().numpy()
        assert got_w.tobytes() == lcd_oracle.word_weights(word, q_count, n_words).tobytes()


@pytest.mark.gpu
def test_candidates_at_the_first_frame_limits(tracker):
    """first_frame = INT_MAX - n + 1 is accepted and frame n - 1 (INT_MAX) is its own candidate at min_gap 0;
    first_frame = INT_MIN numbers the candidates from INT_MIN."""
    n, n_words = 150, 500
    rng = np.random.default_rng(31)
    word, q_count = random_words(rng, n, 40, n_words)
    q_count[-1] = 40
    weight = random_weights(rng, n_words)
    for first_frame in (INT_MAX - n + 1, INT_MIN):
        cand, _ = check_candidates(tracker, word, q_count, n_words, weight, 0, 8, 1, first_frame)
        assert (cand[cand != -1] - first_frame >= 0).all()
        if first_frame > 0:
            assert cand[n - 1, 0] == INT_MAX


# ------------------------------------------------------------------ D. mv_detect_loops: every branch of the record
@pytest.fixture(scope="module")
def vocab_tracker(tracker):
    tracker.bow_set_vocabulary(*ref_vocab())
    return tracker


def records(tr, p, args, weight=None, first_frame=0):
    from maveric_slam_b200 import tracking
    return tracking.loop_results_to_numpy(tr.detect_loops(p, *args, weight=weight, first_frame=first_frame))


def expected(p, parts, first_frame=0):
    return select(p, first_frame, parts["cand"], parts["score"], parts["cnt"], parts["pose"], parts["stats"],
                  parts["ov"])


def oracle_slots(oracle, synth, p, args, cand, slots):
    """The CPU oracle chain on the given slots: detector of the frames involved, match, depth correspondences and K3
    keyed on pnp.first_pair + i * k + r.  -> (cnt, pose, stats by slot, overflow by frame)."""
    semi, _, desc, _, depth = args
    need = sorted({i for i, _ in slots} | {int(cand[i, r]) for i, r in slots})
    det = dict(zip(need, detect(oracle, p, semi[need].cpu().numpy(), np.full(len(need), synth.SEMI_SCALE,
                                                                              np.float32))))
    hd = {f: desc[f].cpu().numpy() for f in need}
    hz = {f: depth[f].cpu().numpy() for f in need}
    cnt, pose, stats = {}, {}, {}
    for i, r in slots:
        j = int(cand[i, r])
        mt = oracle.match(match_cfg(p), hd[j], hd[i], det[j][0], det[j][1], det[i][2], det[i][3])
        nm = mt["n"]
        c5 = np.zeros((5, p.match.max_matches), np.float32)
        c5[:3, :nm] = depth_xyz(p, hz[j])(mt)[0].T
        c5[3, :nm], c5[4, :nm] = mt["pts1"][:, 0], mt["pts1"][:, 1]
        pose[i, r], stats[i, r], _ = oracle.pnp_gn(pnp_cfg(p), c5, nm, pair_index=p.pnp.first_pair + i * p.k + r)
        cnt[i, r] = nm
    return cnt, pose, stats, {f: int(det[f][4]) for f in need}


def check_oracle_slots(oracle, synth, p, args, parts, rows):
    slots = [(i, r) for i, r in parts["slots"] if i in rows]
    assert slots
    cnt, pose, stats, ov = oracle_slots(oracle, synth, p, args, parts["cand"], slots)
    for i, r in slots:
        assert cnt[i, r] == parts["cnt"][i, r], (i, r)
        assert same_bits(pose[i, r], parts["pose"][i, r]) and same_bits(stats[i, r], parts["stats"][i, r]), (i, r)
    for f, o in ov.items():
        assert o == parts["ov"][f], f


def check_candidates_of_parts(tr, p, parts, weight):
    """The call's candidates equal the oracle's on the call's own words."""
    word, qc = parts["word"].cpu().numpy(), parts["qc"].cpu().numpy()
    w = None if weight is None else weight.cpu().numpy()
    cand, score = lcd_oracle.candidates(word, qc, tr.n_words, w, p.min_gap, p.k, p.min_score, 0)
    assert cand.tobytes() == parts["cand"].tobytes() and score.tobytes() == parts["score"].tobytes()
    if w is not None:
        assert w.tobytes() == lcd_oracle.word_weights(word, qc, tr.n_words).tobytes()


@pytest.mark.gpu
def test_detect_loops_at_scale_every_record_filled(vocab_tracker, synth, oracle):
    """300 frames (three row tiles), k = 8, min_inliers 0: every frame with a candidate is accepted, so every field
    of every record is compared.  Equal inlier counts across ranks occur and the better BoW rank wins them."""
    tr = vocab_tracker
    n = 300
    p = small_params(k=8, min_inliers=0, first_pair=1000)
    args = frames(tr, synth, loop_offsets(n, True), seed=3)
    parts = verify_by_parts(tr, p, n, args, "idf")
    res = records(tr, p, args, weight=parts["weight"], first_frame=-50)
    assert res.tobytes() == expected(p, parts, -50).tobytes()
    has = parts["cand"][:, 0] >= 0
    assert has.sum() > n - 10 and ((res["bow_rank"] >= 0) == has).all()
    ties = 0
    for i in np.nonzero(has)[0]:
        inl = [parts["stats"][i, r, 0] for r in range(p.k) if parts["cand"][i, r] >= 0]
        top = [r for r, v in enumerate(inl) if v == max(inl)]
        if len(top) > 1:
            ties += 1
            assert res["bow_rank"][i] == top[0], i
    assert ties > 0, "no frame with equal top inlier counts"
    check_candidates_of_parts(tr, p, parts, parts["weight"])
    check_oracle_slots(oracle, synth, p, args, parts, {3, 100, 128, 200, 256, n - 1})


@pytest.mark.gpu
def test_detect_loops_min_inliers_boundary(vocab_tracker, synth):
    """The planted revisit with I inliers: min_inliers = I accepts it, I + 1 rejects it."""
    from maveric_slam_b200 import tracking
    tr = vocab_tracker
    n = 16
    p = tracking.loop_params(ROWS, COLS, top_n=1000, max_valid=8192, max_matches=1024, hypotheses=256, min_gap=12,
                             k=4, min_inliers=0)
    args = frames(tr, synth, loop_offsets(n, True))
    parts = verify_by_parts(tr, p, n, args, "idf")
    inl = int(parts["stats"][n - 1, :, 0].max())
    assert inl >= 30
    for m, accepted in ((inl, True), (inl + 1, False)):
        p.min_inliers = m
        res = records(tr, p, args, weight=parts["weight"])
        assert res.tobytes() == expected(p, parts).tobytes(), m
        assert (res["bow_rank"][n - 1] >= 0) == accepted and (res["frame"][n - 1] == 2) == accepted, m


def valid_counts(tr, semi, sscale):
    idx, prob, _ = tr.softmax(semi, sscale)
    return ((idx != 64) & (prob > 0.01)).sum(1).cpu().numpy()


@pytest.mark.gpu
def test_detect_loops_overflow_status(vocab_tracker, synth, oracle):
    """Frames 0 .. 3 exceed max_valid, frames 4 .. 11 do not.  Frame 0 overflows and has no candidate; frame 4
    accepts an overflowing frame (min_score 0: the overflowing frames have no words and score 0).  The status equals
    the rule fed with the oracle's overflow flags."""
    import torch
    tr = vocab_tracker
    hi = frames(tr, synth, loop_offsets(4, False), seed=7, keypoint_permille=400)
    lo = frames(tr, synth, loop_offsets(8, False) + 2, seed=8, keypoint_permille=60)
    args = tuple(torch.cat([a, b]) for a, b in zip(hi, lo))
    n = 12
    nv = valid_counts(tr, args[0], args[1])
    assert nv[:4].min() > nv[4:].max() + 2, nv
    p = small_params(max_valid=int(nv[:4].min() + nv[4:].max()) // 2 + 1, min_gap=1, k=3, min_score=0,
                     min_inliers=0)
    parts = verify_by_parts(tr, p, n, args, None)
    ov = parts["ov"]
    assert ov.tolist() == [1] * 4 + [0] * 8
    _, _, _, ov_o = oracle_slots(oracle, synth, p, args, parts["cand"], [(i, 0) for i in range(1, n)])
    ov_o = np.array([ov_o.get(f, 0) for f in range(n)], np.int32)
    assert ov_o.tolist() == ov.tolist()
    res = records(tr, p, args)
    assert res.tobytes() == select(p, 0, parts["cand"], parts["score"], parts["cnt"], parts["pose"],
                                   parts["stats"], ov_o).tobytes()
    assert res["bow_rank"][0] == -1 and res["status"][0] == 4                       # the frame itself
    assert res["bow_rank"][4] >= 0 and ov[res["frame"][4]] and res["status"][4] == 4  # its accepted frame
    assert (res["status"][5:] == 0).any()


@pytest.mark.gpu
def test_detect_loops_frames_without_keypoints(vocab_tracker, synth):
    """Frames whose logits are all negative (no keypoint, no word): an empty record, and the other frames' records
    are those of the call without the appended ones."""
    tr = vocab_tracker
    n = 13
    args = frames(tr, synth, loop_offsets(n, False), seed=4)
    args[0][4] = -100
    args[0][11:] = -100
    p = small_params(min_inliers=0)
    parts = verify_by_parts(tr, p, n, args, None)
    assert (parts["qc"].cpu().numpy()[[4, 11, 12]] == 0).all()
    res = records(tr, p, args)
    assert res.tobytes() == expected(p, parts).tobytes()
    empty = np.zeros(1, res.dtype)[0]
    empty["frame"], empty["bow_rank"] = -1, -1
    for f in (4, 11, 12):
        assert res[f].tobytes() == empty.tobytes(), f
    assert (res["bow_rank"][:11] >= 0).sum() > 3
    assert records(tr, p, tuple(a[:11] for a in args)).tobytes() == res[:11].tobytes()


@pytest.mark.gpu
def test_detect_loops_one_frame(vocab_tracker, synth):
    tr = vocab_tracker
    args = frames(tr, synth, loop_offsets(1, False))
    p = small_params(min_gap=0, min_inliers=0)
    res = records(tr, p, args, first_frame=INT_MAX)
    parts = verify_by_parts(tr, p, 1, args, None)
    assert res.tobytes() == expected(p, parts, INT_MAX).tobytes()
    p.min_gap = 1
    res = records(tr, p, args)
    assert res["frame"][0] == -1 and res["bow_rank"][0] == -1 and res["status"][0] == 0
    assert not res.view(np.int32).reshape(-1)[3:].any()


@pytest.mark.gpu
def test_detect_loops_min_gap_zero(vocab_tracker, synth, oracle):
    """min_gap 0: a frame is its own candidate and the pair (i, i) goes through the matcher and K3."""
    tr = vocab_tracker
    n = 8
    p = small_params(min_gap=0, k=2, min_inliers=0)
    args = frames(tr, synth, loop_offsets(n, False), seed=6)
    parts = verify_by_parts(tr, p, n, args, None)
    cand = parts["cand"]
    selfs = [(i, r) for i, r in parts["slots"] if cand[i, r] == i]
    assert len(selfs) >= n - 1
    res = records(tr, p, args, first_frame=3)
    assert res.tobytes() == expected(p, parts, 3).tobytes()
    assert (res["frame"] == 3 + np.arange(n)).any()
    check_candidates_of_parts(tr, p, parts, None)
    check_oracle_slots(oracle, synth, p, args, parts, set(range(n)))


@pytest.mark.gpu
def test_detect_loops_matcher_choice(vocab_tracker, synth):
    """use_tensor_cores 0, 1 and 2 give byte-identical records at 47 x 155 with a whole-grid radius."""
    tr = vocab_tracker
    n = 14
    args = frames(tr, synth, loop_offsets(n, True))
    out = []
    for utc in (0, 1, 2):
        p = small_params(k=4, min_inliers=0)
        assert p.match.radius >= max(ROWS, COLS)
        p.match.use_tensor_cores = utc
        out.append(records(tr, p, args).tobytes())
    assert out[0] == out[1] == out[2]
    parts = verify_by_parts(tr, p, n, args, None)
    assert out[2] == expected(p, parts).tobytes()


@pytest.mark.gpu
def test_detect_loops_at_the_slot_limit(vocab_tracker, synth):
    """n_frames * k = 65 535 exactly (13 107 frames, k = 5) on an 8 x 16 grid: the candidates of every frame, and
    match and K3 on a sample of frames across the row tiles."""
    tr = vocab_tracker
    n, rows, cols = 13107, 8, 16
    p = small_params(rows, cols, top_n=100, max_matches=64, hypotheses=32, k=5, min_inliers=0)
    args = frames(tr, synth, loop_offsets(n, False), seed=9, rows=rows, cols=cols)
    sample = [0, 3, 4, 127, 128, 129, 4000, 8191, 12800, n - 2, n - 1]
    parts = verify_by_parts(tr, p, n, args, None, frames_verified=sample)
    check_candidates_of_parts(tr, p, parts, None)
    res = records(tr, p, args)
    want = expected(p, parts)
    assert res[sample].tobytes() == want[sample].tobytes()
    acc = np.nonzero(res["bow_rank"] >= 0)[0]
    assert len(acc) > n // 2
    r = res["bow_rank"][acc]
    assert (parts["cand"][acc, r] == res["frame"][acc]).all() and (parts["score"][acc, r] == res["bow_score"][acc]).all()
