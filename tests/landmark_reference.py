"""The landmark sequence path on the CPU: mv_track_sequence_landmarks (and every entry point that shares its
semantics) composed from the oracle's primitives and numpy float32 operations, nothing of the library's.

It follows the semantics list of DESIGN §4.6 ("Words", "Inserted coordinates", "Table steps", "Correspondences",
"The rest") and the record layout of include/maveric_b200.h:
  * detector per frame with that frame's semi_scale (orc_softmax, orc_top_n; an overflowing frame has no queries);
  * words of frame p's queries with frame p's desc_scale (orc_bow_assign), word = base * words_per_base + leaf;
  * each query back-projected with frame p's depth at pixel x = (cell / rows) * 8 + idx % 8,
    y = (cell % rows) * 8 + idx / 8, by the RN float32 operations of build_corr_kernel;
  * table step p = orc_pool_observe(first_frame + p) then orc_pool_remove_old(first_frame + p), frames 0 .. n-2;
  * pair p: orc_match, orc_ransac_identity (cap min(max_matches, 1000)), the 3-D side of match j from the table right
    after step p (the matched frame-0 cell's query, its word in [0, n_words) with a live record; NaN otherwise, and
    only the former counted in n_with_landmark), orc_pnp_gn keyed on pnp.first_pair + p;
  * status 4 (MV_ERR_TOO_MANY_VALID) where either frame of the pair overflowed max_valid.
"""
import numpy as np

from oracle import orc

STATUS_TOO_MANY_VALID = 4
f32 = np.float32


def orc_landmarks_sequence(oracle, table, first_frame, word, q_count, coords, snapshots=None):
    """The semantics of mv_landmarks_sequence on the oracle's table (updated in place): step f observes the first
    q_count[f] words of frame first_frame + f, then removes old frames; returns each occurrence's lookup right after
    its step (0 where the word has no record or q >= q_count)."""
    n_steps, top_n = word.shape
    out = np.zeros((n_steps, top_n, 3), np.float32)
    for f in range(n_steps):
        k = min(int(q_count[f]), top_n)
        oracle.pool_observe(table, first_frame + f, word[f, :k], coords[f, :k])
        oracle.pool_remove_old(table, first_frame + f)
        for q in range(k):
            w = int(word[f, q])
            if 0 <= w < len(table) and table[w]["word_id"] == w:
                out[f, q] = table[w]["coords"]
        if snapshots is not None:
            snapshots.append(table.copy())
    return out


def match_cfg(params):
    m = params.match
    return orc.MatchCfg(m.rows, m.cols, m.shift_x, m.shift_y, m.radius, m.max_matches, m.match_threshold, m.min_prob0)


def pnp_cfg(params):
    k = params.pnp
    return orc.pnp_cfg(k.fx, k.fy, k.cx, k.cy, k.hypotheses, k.sample_size, k.sample_iters, k.refine_iters, k.gate_sq,
                       k.min_depth, k.damping, k.seed, k.lanes_per_hypothesis)


def track_cfg(params, semi_scale):
    """orc_track_pair's configuration for these parameters, one semi_scale for both frames."""
    return orc.TrackCfg(match_cfg(params), pnp_cfg(params), params.top_n, params.max_valid, params.ransac_iterations,
                        params.ransac_threshold, float(semi_scale))


def back_project(params, cell, idx, depth):
    """Pixel (x, y) of keypoint `idx` of `cell`, back-projected with `depth` [cells] at that cell -> float32 [n, 3]."""
    k, rows = params.pnp, params.match.rows
    x = (cell // rows * 8 + idx % 8).astype(f32)
    y = (cell % rows * 8 + idx // 8).astype(f32)
    z = depth[cell].astype(f32)
    return np.stack([(x - f32(k.cx)) / f32(k.fx) * z, (y - f32(k.cy)) / f32(k.fy) * z, z], -1).astype(f32)


def detect(oracle, params, semi, semi_scale):
    """Per frame: (max_idx, probs, query cells, query indices, overflow)."""
    out = []
    for f in range(semi.shape[0]):
        idx, prob, _ = oracle.softmax(float(semi_scale[f]), semi[f])
        qp, qi, _, ov = oracle.top_n(float(semi_scale[f]), semi[f], params.top_n, params.max_valid)
        out.append((idx, prob, qp, qi, ov))
    return out


def pair_record(oracle, params, det0, det1, desc0, desc1, pair_index, xyz_of_cell):
    """Pair (frame 0, frame 1) from the two frames' detect() outputs: match, RANSAC-E, correspondences, K3 and the
    status.  xyz_of_cell(cell0 int32 [nm]) -> (float32 [nm, 3] 3-D side, matches with a landmark or None).
    -> (record PAIR_RESULT_DTYPE, n_with_landmark or None)."""
    from maveric_slam_b200 import tracking
    idx0, prob0, _, _, ov0 = det0
    _, _, qp1, qi1, ov1 = det1
    M = params.match.max_matches
    m = oracle.match(match_cfg(params), desc0, desc1, idx0, prob0, qp1, qi1)
    nm = m["n"]
    ninl = 0
    if params.ransac_iterations > 0:
        _, _, ninl, _ = oracle.ransac_identity(m["pts0"], m["pts1"], params.ransac_iterations,
                                               params.ransac_threshold, cap=min(M, 1000))
    corr = np.zeros((5, M), np.float32)
    xyz, n_with = xyz_of_cell(m)
    corr[:3, :nm] = xyz.T
    corr[3, :nm] = m["pts1"][:, 0]
    corr[4, :nm] = m["pts1"][:, 1]
    pose, stats, _ = oracle.pnp_gn(pnp_cfg(params), corr, nm, pair_index=pair_index)
    r = np.zeros(1, tracking.PAIR_RESULT_DTYPE)[0]
    r["q"], r["t"] = pose[:4], pose[4:]
    r["pnp_inliers"], r["pnp_cost"], r["best_hypothesis"] = stats[0], stats[1], int(stats[2])
    r["num_matches"], r["ransac_inliers"] = nm, ninl
    r["status"] = STATUS_TOO_MANY_VALID if (ov0 or ov1) else 0
    return r, n_with


def depth_xyz(params, depth0):
    """The 3-D side of each match from frame 0's depth at its cell (orc_track_pair's, build_corr_kernel's)."""
    k = params.pnp

    def xyz(m):
        d = depth0[m["cell0"]].astype(f32)
        return np.stack([(m["pts0"][:, 0] - f32(k.cx)) / f32(k.fx) * d, (m["pts0"][:, 1] - f32(k.cy)) / f32(k.fy) * d,
                         d], -1), None
    return xyz


def table_xyz(qp0, words, table, n_words):
    """The 3-D side of each match from the table: the matched frame-0 cell's query, its word in [0, n_words) with a
    live record; NaN otherwise, and only the former counted."""
    def xyz(m):
        nm = m["n"]
        out = np.full((nm, 3), np.nan, np.float32)
        n_with = 0
        pos = np.searchsorted(qp0, m["cell0"])
        for j in range(nm):
            if pos[j] < len(qp0) and qp0[pos[j]] == m["cell0"][j]:
                w = int(words[pos[j]])
                if 0 <= w < n_words and table[w]["word_id"] == w:
                    out[j] = table[w]["coords"]
                    n_with += 1
        return out, n_with
    return xyz


def landmark_reference(oracle, vocab, params, semi, semi_scale, desc, desc_scale, depth, table=None, first_frame=0,
                       n_words=None, depth_mode=False, threads=1):
    """The landmark path over frames 0 .. n-1 (host numpy arrays: semi int8 [n, cells, 65], semi_scale float32 [n],
    desc int8 [n, cells, 256], desc_scale float32 [n], depth float32 [n, cells]).

    vocab: an oracle.bow_vocab handle; table: the entry table (oracle.pool_new layout, not modified), default empty
    of n_words records; n_words defaults to len(table).  Returns (records PAIR_RESULT_DTYPE [n-1], n_with_landmark
    int32 [n-1], final table).  depth_mode: the 3-D side of each match from frame p's depth at its cell instead of
    the table (orc_track_pair's), no words and no table steps; n_with_landmark and the table are then None.
    threads: oracle calls of different frames and pairs run on that many threads (they release the GIL); only the
    table steps are sequential."""
    from concurrent.futures import ThreadPoolExecutor
    from maveric_slam_b200 import tracking
    n = semi.shape[0]
    if not depth_mode:
        table = oracle.pool_new(n_words) if table is None else np.array(table, copy=True)
        n_words = len(table) if n_words is None else n_words
        assert len(table) == n_words
    with ThreadPoolExecutor(threads) as ex:
        frames = list(ex.map(lambda f: detect(oracle, params, semi[f:f + 1], semi_scale[f:f + 1])[0], range(n)))
        if depth_mode:
            xyz = [depth_xyz(params, depth[p]) for p in range(n - 1)]
        else:
            def words_of(p):
                base, wid = oracle.bow_assign(vocab, float(desc_scale[p]), desc[p][frames[p][2]])
                return (base * vocab.words_per_base + wid).astype(np.int32)
            words = list(ex.map(words_of, range(n - 1)))
            xyz = []
            for p in range(n - 1):   # table step p
                oracle.pool_observe(table, first_frame + p, words[p], back_project(params, frames[p][2], frames[p][3],
                                                                                   depth[p]))
                oracle.pool_remove_old(table, first_frame + p)
                xyz.append(table_xyz(frames[p][2], words[p], table.copy(), n_words))
        out = list(ex.map(lambda p: pair_record(oracle, params, frames[p], frames[p + 1], desc[p], desc[p + 1],
                                                params.pnp.first_pair + p, xyz[p]), range(n - 1)))
    rec = np.zeros(n - 1, tracking.PAIR_RESULT_DTYPE)
    for p, (r, _) in enumerate(out):
        rec[p] = r
    if depth_mode:
        return rec, None, None
    return rec, np.array([k for _, k in out], np.int32).reshape(n - 1), table
