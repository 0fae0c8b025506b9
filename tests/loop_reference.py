"""Inputs and helpers of the loop-closure modules (tests/test_loop_closure.py, tests/test_loop_closure_edges.py).

presence, ref_candidates and ref_word_weights restate the definition of DESIGN §4.7 in numpy; random_words draws
word lists for mv_loop_candidates and mv_lcd_word_weights; frames, loop_offsets and small_params give
mv_detect_loops its synthetic sequence and parameters; select restates mv_detect_loops' selection rule, and
verify_by_parts runs every candidate slot through the library's separate GPU calls.
"""
import copy
import math

import numpy as np

from helpers import dev

STATUS_TOO_MANY_VALID = 4
ROWS, COLS = 47, 155


def presence(word, q_count, n_words):
    n, top_n = word.shape
    P = np.zeros((n, n_words), np.float32)
    for f in range(n):
        w = word[f, :min(max(int(q_count[f]), 0), top_n)]
        P[f, w[(w >= 0) & (w < n_words)]] = 1
    return P


def ref_candidates(word, q_count, n_words, weight, min_gap, k, min_score, first_frame):
    """-> (cand int32 [n, k], score int32 [n, k]).  Scores in float32 are exact: every partial sum is an integer
    below 127 * top_n < 2^24."""
    assert 127 * word.shape[1] < 2 ** 24
    P = presence(word, q_count, n_words)
    W = P if weight is None else P * weight.astype(np.float32)
    S = (W @ P.T).astype(np.int64)
    n = len(P)
    cand = np.full((n, k), -1, np.int32)
    score = np.zeros((n, k), np.int32)
    for i in range(n):
        hi = i - min_gap + 1
        if hi <= 0:
            continue
        s = S[i, :hi]
        j = np.nonzero(s >= min_score)[0]
        order = j[np.lexsort((j, -s[j]))][:k]
        cand[i, :len(order)] = first_frame + order
        score[i, :len(order)] = s[order]
    return cand, score


def idf(n, df):
    """One weight: 0 for df 0, 64 for the exact tie df^2 = n (63.5, to even), else the value in double rounded to
    the nearest integer (Python's log is the C library's)."""
    if not df:
        return 0
    if df * df == n:
        return 64
    return round(127.0 * math.log(n / df) / math.log(n))


def ref_word_weights(word, q_count, n_words):
    P = presence(word, q_count, n_words)
    n = len(P)
    df = P.sum(0).astype(np.int64)
    return np.array([idf(n, int(d)) for d in df], np.int8)


def random_words(rng, n, top_n, n_words, bad=True):
    """Word lists with duplicates, ids -1 and >= n_words, and query counts 0 and above top_n."""
    word = rng.integers(0, n_words, size=(n, top_n)).astype(np.int32)
    if bad:
        word[rng.random((n, top_n)) < 0.05] = -1
        word[rng.random((n, top_n)) < 0.05] = n_words + 3
    q_count = rng.integers(0, top_n + 4, size=n).astype(np.int32)
    q_count[::7] = 0
    q_count[1::5] = top_n + 9
    return word, q_count


def random_weights(rng, n_words):
    w = rng.integers(0, 128, size=n_words).astype(np.int8)
    w[rng.random(n_words) < 0.1] = 0
    return w


def run_candidates(tracker, word, q_count, n_words, weight, min_gap, k, min_score, first_frame):
    cand, score = tracker.loop_candidates(dev(tracker, word), dev(tracker, q_count),
                                          None if weight is None else dev(tracker, weight), min_gap=min_gap, k=k,
                                          min_score=min_score, first_frame=first_frame, n_words=n_words)
    return cand.cpu().numpy(), score.cpu().numpy()


def loop_offsets(n, returns):
    """A (4, 4) cells/frame drift; with `returns`, the last frame comes back next to frame 2's offset (one cell
    off): the planted revisit of DESIGN §4.7's probe."""
    off = np.array([(4 * f, 4 * f) for f in range(n)], np.int32)
    if returns:
        off[-1] = (9, 8)
    return off


def frames(tracker, synth, off, seed=0, rows=ROWS, cols=COLS, keypoint_permille=140):
    semi, desc, depth = tracker.synth_frames(seed, rows, cols, 0, off, keypoint_permille=keypoint_permille)
    n = off.shape[0]
    sscale = dev(tracker, np.full(n, synth.SEMI_SCALE, np.float32))
    dscale = dev(tracker, np.full(n, synth.DESC_SCALE, np.float32))
    return semi, sscale, desc, dscale, depth


def select(params, first_frame, cand, score, cnt, pose, stats, ov):
    """The selection rule of mv_detect_loops, restated, from candidates as indices within the call (-1: empty slot)
    -> LOOP_RESULT_DTYPE [n]."""
    from maveric_slam_b200 import tracking
    n, k = cand.shape
    out = np.zeros(n, tracking.LOOP_RESULT_DTYPE)
    for i in range(n):
        best = -1
        for r in range(k):
            if cand[i, r] >= 0 and (best < 0 or stats[i, r, 0] > stats[i, best, 0]):
                best = r
        rec = out[i]
        rec["frame"], rec["bow_rank"] = -1, -1
        accepted = best >= 0 and stats[i, best, 0] >= np.float32(params.min_inliers)
        if accepted:
            rec["frame"], rec["bow_score"], rec["bow_rank"] = first_frame + cand[i, best], score[i, best], best
            rec["num_matches"] = cnt[i, best]
            rec["pnp_inliers"], rec["pnp_cost"] = stats[i, best, 0], stats[i, best, 1]
            rec["q"], rec["t"] = pose[i, best, :4], pose[i, best, 4:]
        rec["status"] = STATUS_TOO_MANY_VALID if (ov[i] or (accepted and ov[cand[i, best]])) else 0
    return out


def small_params(rows=ROWS, cols=COLS, **kw):
    from maveric_slam_b200 import tracking
    d = dict(top_n=300, max_valid=8192, max_matches=150, hypotheses=64, min_gap=3, k=2, min_score=1, min_inliers=20)
    d.update(kw)
    return tracking.loop_params(rows, cols, **d)


def verify_by_parts(tr, p, n, args, weight, frames_verified=None):
    """Every candidate of every frame through the separate GPU calls: detector, words, mv_loop_candidates (first frame
    0: indices within the call), mv_match_batch over the explicit list of real candidate pairs only,
    mv_build_corr_batch and one mv_pnp_gn_batch per pair keyed on pnp.first_pair + i * k + r.
    frames_verified: only the candidates of these frames go through the matcher and PnP (the others keep zeros).
    -> dict of cand, score [n, k] and per slot cnt [n, k], pose [n, k, 7], stats [n, k, 4], and ov [n]."""
    semi, sscale, desc, dscale, depth = args
    idx, prob, _ = tr.softmax(semi, sscale)
    qp, qi, _, qc, ov = tr.top_n(idx, prob, p.top_n, p.max_valid)
    word, _ = tr.bow_assign(desc, dscale, qp, qc)
    if weight == "idf":
        weight = tr.lcd_word_weights(word, qc)
    cand, score = tr.loop_candidates(word, qc, weight, p.min_gap, p.k, p.min_score, 0)
    cand, score = cand.cpu().numpy(), score.cpu().numpy()
    K = p.k
    out = dict(cand=cand, score=score, ov=ov.cpu().numpy(), weight=weight, word=word, qc=qc,
               cnt=np.zeros((n, K), np.int32), pose=np.zeros((n, K, 7), np.float32),
               stats=np.zeros((n, K, 4), np.float32))
    rows = range(n) if frames_verified is None else sorted(set(frames_verified))
    slots = [(i, r) for i in rows for r in range(K) if cand[i, r] >= 0]
    out["slots"] = slots
    if not slots:
        return out
    f0 = dev(tr, np.array([cand[i, r] for i, r in slots], np.int32))
    f1 = dev(tr, np.array([i for i, r in slots], np.int32))
    pts, cnt, cell0, _, _ = tr.match(p.match, desc, idx, prob, qp, qi, qc, f0=f0, f1=f1)
    corr = tr.build_corr(pts, cnt, cell0, depth, (p.pnp.fx, p.pnp.fy, p.pnp.cx, p.pnp.cy), p.match.rows, f0=f0)
    cnt_h = cnt.cpu().numpy()
    for m, (i, r) in enumerate(slots):
        pnp = copy.copy(p.pnp)
        pnp.first_pair = p.pnp.first_pair + i * K + r
        pose, stats, _ = tr.pnp_gn(pnp, corr[m:m + 1].contiguous(), cnt[m:m + 1])
        out["cnt"][i, r], out["pose"][i, r] = cnt_h[m], pose.cpu().numpy()[0]
        out["stats"][i, r] = stats.cpu().numpy()[0]
    return out
