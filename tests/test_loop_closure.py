"""Loop closure: BoW candidate scoring on the tensor cores (mv_loop_candidates, mv_lcd_word_weights) and the whole
detection call (mv_detect_loops: candidates, one matcher launch, depth correspondences, one K3 launch, selection).

The score is this library's definition (include/maveric_b200.h, DESIGN §4.7; the reference's lcd_main.c cannot be
run here, parity unpinned).  tests/lcd_oracle.c restates the candidates and the weights as plain loops over sorted
word lists, and the GPU is held to it byte for byte; a numpy restatement of the definition is held to the same
oracle without a GPU.  Verification is the composition of calls that are each held to the CPU oracle elsewhere
(matcher, depth correspondences, K3), and is checked here both against those calls made one by one on the GPU and
against the CPU oracle chain.
"""
import ctypes as C

import numpy as np
import pytest

import lcd_oracle
from helpers import dev, ref_vocab
from landmark_reference import depth_xyz, detect, match_cfg, pnp_cfg
from loop_reference import (COLS, ROWS, frames, loop_offsets, random_weights, random_words, ref_candidates,
                            ref_word_weights, run_candidates, select, small_params, verify_by_parts)


# ------------------------------------------------------------------ 1. candidates
CASES = [
    # n, top_n, n_words, weighted, min_gap, k, min_score, first_frame
    (1, 13, 100, True, 0, 4, 1, 0),
    (2, 13, 100, False, 0, 8, 0, 5),
    (2, 13, 100, True, 1, 3, 1, -7),
    (37, 13, 100, True, 0, 8, 1, -100),
    (37, 29, 1, False, 1, 8, 0, 0),            # one word: scores 0 / 1
    (37, 29, 1, True, 3, 2, 1, 3),
    (37, 13, 100, False, 40, 4, 0, 0),         # min_gap above n_frames: no candidates
    (37, 1000, 64, True, 2, 5, 1, 11),
    (300, 20, 70, False, 0, 8, 1, -1),         # several tiles, many equal scores
    (300, 50, 1000, True, 129, 8, 2, 0),       # min_gap just over a tile
    (4541, 1000, 10000, True, 30, 4, 1, 0),    # the bench sequence's length and the reference vocabulary's size
    (4541, 997, 10000, False, 0, 8, 1, -4541),
]


def case_inputs(n, top_n, n_words, weighted, min_gap):
    rng = np.random.default_rng(n * 7919 + top_n * 31 + n_words + min_gap)
    word, q_count = random_words(rng, n, top_n, n_words)
    return word, q_count, (random_weights(rng, n_words) if weighted else None)


def equal_words_inputs(n=200, top_n=24, n_words=90):
    """Every frame holds the same words: all scores are equal."""
    return np.tile(np.arange(top_n, dtype=np.int32) * 3, (n, 1)), np.full(n, top_n, np.int32)


@pytest.mark.parametrize("n,top_n,n_words,weighted,min_gap,k,min_score,first_frame",
                         [c for c in CASES if c[0] <= 300])
def test_numpy_restatement_equals_oracle(n, top_n, n_words, weighted, min_gap, k, min_score, first_frame):
    word, q_count, weight = case_inputs(n, top_n, n_words, weighted, min_gap)
    args = (word, q_count, n_words, weight, min_gap, k, min_score, first_frame)
    for a, b in zip(ref_candidates(*args), lcd_oracle.candidates(*args)):
        assert a.tobytes() == b.tobytes()
    want = lcd_oracle.word_weights(word, q_count, n_words)
    assert ref_word_weights(word, q_count, n_words).tobytes() == want.tobytes()


def test_oracle_tie_order():
    word, q_count = equal_words_inputs()
    cand, score = lcd_oracle.candidates(word, q_count, 90, None, 2, 8, 0, 10)
    assert (cand[150] == 10 + np.arange(8)).all() and (score[150] == 24).all()
    assert (cand[:2] == -1).all() and (cand[5, :4] == 10 + np.arange(4)).all() and (cand[5, 4:] == -1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("n,top_n,n_words,weighted,min_gap,k,min_score,first_frame", CASES)
def test_candidates_equal_reference(tracker, n, top_n, n_words, weighted, min_gap, k, min_score, first_frame):
    word, q_count, weight = case_inputs(n, top_n, n_words, weighted, min_gap)
    got = run_candidates(tracker, word, q_count, n_words, weight, min_gap, k, min_score, first_frame)
    want = lcd_oracle.candidates(word, q_count, n_words, weight, min_gap, k, min_score, first_frame)
    assert got[0].tobytes() == want[0].tobytes()
    assert got[1].tobytes() == want[1].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True])
def test_candidates_tie_order(tracker, weighted):
    """All scores equal: the earlier frames come first."""
    word, q_count = equal_words_inputs()
    weight = np.full(90, 5, np.int8) if weighted else None
    got = run_candidates(tracker, word, q_count, 90, weight, 2, 8, 0, 10)
    want = lcd_oracle.candidates(word, q_count, 90, weight, 2, 8, 0, 10)
    assert got[0].tobytes() == want[0].tobytes() and got[1].tobytes() == want[1].tobytes()
    assert (got[0][150] == 10 + np.arange(8)).all()


@pytest.mark.gpu
def test_candidates_refusals_enqueue_nothing(tracker):
    from maveric_slam_b200 import lib
    word, q_count = random_words(np.random.default_rng(1), 8, 16, 50)
    w, q = dev(tracker, word), dev(tracker, q_count)
    neg = np.ones(50, np.int8)
    neg[17] = -1
    bad = [dict(k=0), dict(k=9), dict(min_gap=-1), dict(n_words=0), dict(first_frame=2 ** 31 - 4),
           dict(weight=dev(tracker, neg))]
    for b in bad:
        kw = dict(weight=None, min_gap=0, k=4, min_score=1, first_frame=0, n_words=50)
        kw.update(b)
        before = tracker.ctx.launches
        with pytest.raises(lib.MvError, match="bad argument"):
            tracker.loop_candidates(w, q, **kw)
        assert tracker.ctx.launches == before, b


# ------------------------------------------------------------------ 2. word weights
@pytest.mark.gpu
@pytest.mark.parametrize("n,top_n,n_words", [(2, 13, 100), (37, 29, 1), (37, 100, 70), (300, 50, 1000),
                                             (4541, 1000, 10000)])
def test_word_weights_equal_reference(tracker, n, top_n, n_words):
    rng = np.random.default_rng(n + n_words)
    word, q_count = random_words(rng, n, top_n, n_words)
    got = tracker.lcd_word_weights(dev(tracker, word), dev(tracker, q_count), n_words=n_words).cpu().numpy()
    assert got.tobytes() == lcd_oracle.word_weights(word, q_count, n_words).tobytes()


# ------------------------------------------------------------------ 3. the whole call equals its parts
@pytest.fixture(scope="module")
def vocab_tracker(tracker):
    tracker.bow_set_vocabulary(*ref_vocab())
    return tracker


@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True])
def test_detect_loops_equals_its_parts(vocab_tracker, synth, oracle, weighted):
    from maveric_slam_b200 import tracking
    tr = vocab_tracker
    n, first_pair = 14, 77
    p = small_params()
    p.pnp.first_pair = first_pair
    args = frames(tr, synth, loop_offsets(n, True))
    semi, _, desc, _, depth = args
    parts = verify_by_parts(tr, p, n, args, "idf" if weighted else None)
    weight = parts["weight"]
    cand, score, K = parts["cand"], parts["score"], p.k
    assert parts["slots"], "the planted sequence must give candidates"
    # first frame numbers: positive, all negative, and one that makes an accepted frame global frame -1 -- the value
    # that marks an empty slot in mv_loop_candidates' own output
    local = select(p, 0, cand, score, parts["cnt"], parts["pose"], parts["stats"], parts["ov"])
    i_acc = int(np.nonzero(local["bow_rank"] >= 0)[0][0])
    j_acc = int(local["frame"][i_acc])
    first_frames = (1000, -100, -1 - j_acc)
    res = {}
    for ff in first_frames:
        res[ff] = tracking.loop_results_to_numpy(tr.detect_loops(p, *args, weight=weight, first_frame=ff))
        want = select(p, ff, cand, score, parts["cnt"], parts["pose"], parts["stats"], parts["ov"])
        assert res[ff].tobytes() == want.tobytes(), ff
        # mv_loop_candidates at the caller's first_frame: the same list shifted
        cand_g = tr.loop_candidates(parts["word"], parts["qc"], weight, p.min_gap, K, p.min_score, ff)[0]
        assert (cand_g.cpu().numpy() == np.where(cand >= 0, cand + ff, -1)).all(), ff
    r = res[-1 - j_acc][i_acc]
    assert r["frame"] == -1 and r["bow_rank"] >= 0 and r["num_matches"] > 0, "global frame -1 accepted as a loop"

    # the CPU oracle chain: detector, words, the oracle's candidates, match, depth correspondences, K3
    hs, hd, hz = semi.cpu().numpy(), desc.cpu().numpy(), depth.cpu().numpy()
    det = detect(oracle, p, hs, np.full(n, synth.SEMI_SCALE, np.float32))
    voc = oracle.bow_vocab(*ref_vocab())
    words = np.full((n, p.top_n), -1, np.int32)
    q_count = np.zeros(n, np.int32)
    for f in range(n):
        qpf = det[f][2]
        q_count[f] = len(qpf)
        words[f, :len(qpf)] = oracle.bow_assign(voc, synth.DESC_SCALE, hd[f][qpf])[1]
    w_ref = lcd_oracle.word_weights(words, q_count, tr.n_words) if weighted else None
    cand_o, score_o = lcd_oracle.candidates(words, q_count, tr.n_words, w_ref, p.min_gap, K, p.min_score, 0)
    assert cand_o.tobytes() == cand.tobytes() and score_o.tobytes() == score.tobytes()
    cnt_o = np.zeros((n, K), np.int32)
    pose_o = np.zeros((n, K, 7), np.float32)
    stats_o = np.zeros((n, K, 4), np.float32)
    for i, r in parts["slots"]:
        j = cand_o[i, r]
        mt = oracle.match(match_cfg(p), hd[j], hd[i], det[j][0], det[j][1], det[i][2], det[i][3])
        nm = mt["n"]
        c5 = np.zeros((5, p.match.max_matches), np.float32)
        c5[:3, :nm] = depth_xyz(p, hz[j])(mt)[0].T
        c5[3, :nm], c5[4, :nm] = mt["pts1"][:, 0], mt["pts1"][:, 1]
        pose, stats, _ = oracle.pnp_gn(pnp_cfg(p), c5, nm, pair_index=first_pair + i * K + r)
        cnt_o[i, r], pose_o[i, r], stats_o[i, r] = nm, pose, stats
    ov_o = np.array([d[4] for d in det], np.int32)
    for ff in first_frames:
        assert select(p, ff, cand_o, score_o, cnt_o, pose_o, stats_o, ov_o).tobytes() == res[ff].tobytes(), ff


# ------------------------------------------------------------------ 4. a planted loop, end to end
# Most of the revisit's matches are PnP inliers.  The synthetic world's depth is random per cell, so the pose is
# not asserted.  The fraction is fixed from the first B200 run of this test: 263 inliers of 400 matches (0.66).
MIN_INLIER_FRACTION = 0.6
# The revisit against every candidate of the frames that revisit nothing, on the same B200 runs: 400 matches and 263
# inliers against at most 212 matches and 1 inlier (217 and 1 without the revisit).  A whole-grid search finds many
# false matches between unrelated frames; the geometry rejects them, so the inliers separate the loop by far more
# than the matches do.
MATCH_MARGIN, INLIER_MARGIN = 1.5, 20


@pytest.mark.gpu
def test_planted_loop_is_found(vocab_tracker, synth):
    """first_frame -3: the revisited frame 2 is global frame -1."""
    from maveric_slam_b200 import tracking
    tr = vocab_tracker
    n, first_frame = 16, -3
    # min_gap 12: frames 12 apart are 48 cells apart, more than the grid's 47 rows, and share no world cell
    p = tracking.loop_params(ROWS, COLS, top_n=1000, max_valid=8192, max_matches=1024, hypotheses=256, min_gap=12,
                             k=4, min_inliers=30)
    for returns in (True, False):
        args = frames(tr, synth, loop_offsets(n, returns))
        parts = verify_by_parts(tr, p, n, args, "idf")
        res = tracking.loop_results_to_numpy(tr.detect_loops(p, *args, weight=parts["weight"],
                                                             first_frame=first_frame))
        # every verified candidate of the frames that do not revisit: the rejected ones the loop must stand above
        others = [(i, r) for i, r in parts["slots"] if i != n - 1 or not returns]
        o_matches = max([int(parts["cnt"][i, r]) for i, r in others], default=0)
        o_inliers = max([float(parts["stats"][i, r, 0]) for i, r in others], default=0.0)
        print("returns=%s frames %s ranks %s matches %s inliers %s; best non-revisit candidate: %d matches, %g "
              "inliers" % (returns, res["frame"].tolist(), res["bow_rank"].tolist(), res["num_matches"].tolist(),
                           res["pnp_inliers"].tolist(), o_matches, o_inliers))
        assert len(others) > 0
        if not returns:
            assert (res["bow_rank"] == -1).all() and (res["frame"] == -1).all()
            continue
        assert (res["bow_rank"][:-1] == -1).all()
        loop = res[-1]
        assert loop["bow_rank"] >= 0 and loop["frame"] == first_frame + 2
        assert loop["num_matches"] > MATCH_MARGIN * max(o_matches, 1)
        assert loop["pnp_inliers"] > INLIER_MARGIN * max(o_inliers, 1.0)
        assert loop["pnp_inliers"] >= MIN_INLIER_FRACTION * loop["num_matches"]


# ------------------------------------------------------------------ 5. edge contracts
@pytest.mark.gpu
def test_detect_loops_refusals_enqueue_nothing(vocab_tracker, synth):
    from maveric_slam_b200 import lib
    tr = vocab_tracker
    args = frames(tr, synth, loop_offsets(4, False))
    neg = np.ones(tr.n_words, np.int8)
    neg[5] = -3
    for kw, weight in [(dict(k=0), None), (dict(k=9), None), (dict(min_gap=-1), None), (dict(top_n=0), None),
                       (dict(hypotheses=0), None), (dict(), dev(tr, neg))]:
        before = tr.ctx.launches
        with pytest.raises(lib.MvError, match="bad argument"):
            tr.detect_loops(small_params(**kw), *args, weight=weight)
        assert tr.ctx.launches == before, kw
    # 8 candidates for each of 8192 frames: more pairs than one batched matcher call takes (refused before any read)
    p = small_params(k=8)
    before = tr.ctx.launches
    with pytest.raises(lib.MvError, match="n_frames \\* k"):
        tr.ctx.check(tr.lib.mv_detect_loops(tr.ctx.h, C.byref(p), 8192, 0, *[tr._d(a) for a in args], None,
                                            tr._d(args[0])))
    assert tr.ctx.launches == before


@pytest.mark.gpu
def test_detect_loops_without_vocabulary_is_refused(tracker, synth):
    from maveric_slam_b200 import lib, tracking
    tr = tracking.Tracker(0)
    args = frames(tr, synth, loop_offsets(4, False))
    before = tr.ctx.launches
    with pytest.raises(lib.MvError, match="no vocabulary"):
        tr.detect_loops(small_params(), *args)
    assert tr.ctx.launches == before


@pytest.mark.gpu
def test_detect_loops_on_a_callers_stream(vocab_tracker, synth):
    """A tracker bound to another stream gives the same records."""
    import torch
    from maveric_slam_b200 import tracking
    tr = vocab_tracker
    args = frames(tr, synth, loop_offsets(14, True))
    p = small_params()
    want = tracking.loop_results_to_numpy(tr.detect_loops(p, *args))
    s = torch.cuda.Stream(device=tr.device)
    s.wait_stream(torch.cuda.current_stream(tr.device))
    with torch.cuda.stream(s):
        other = tracking.Tracker(0)
        other.bow_set_vocabulary(*ref_vocab())
        out = other.detect_loops(p, *args)
    s.synchronize()
    assert tracking.loop_results_to_numpy(out).tobytes() == want.tobytes()
