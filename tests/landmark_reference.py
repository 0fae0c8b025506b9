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

Below the reference: the inputs of the cases the modules hold to it, the word-assignment checks beyond the reference
vocabulary, and run_entry, which runs one of the library's landmark-path entry points on a case.
"""
import numpy as np

from helpers import blocks_then_rest, dev, pinned, ref_vocab, upload_table, with_first_pair
from oracle import orc

STATUS_TOO_MANY_VALID = 4
f32 = np.float32


def orc_landmarks_sequence(oracle, table, first_frame, word, q_count, coords, snapshots=None):
    """The semantics of mv_landmarks_sequence on the oracle's table (updated in place): step f observes the first
    q_count[f] words of frame first_frame + f, then removes old frames; returns each occurrence's lookup right after
    its step (0 where the word has no record or q >= q_count).  snapshots: a list that receives a copy of the table
    after every step."""
    n_steps, top_n = word.shape
    out = np.zeros((n_steps, top_n, 3), np.float32)
    for f in range(n_steps):
        k = min(int(q_count[f]), top_n)
        w = word[f, :k]
        oracle.pool_observe(table, first_frame + f, w, coords[f, :k])
        oracle.pool_remove_old(table, first_frame + f)
        ok = (w >= 0) & (w < len(table))
        wc = np.where(ok, w, 0)
        ok &= table["word_id"][wc] == wc
        out[f, :k][ok] = table["coords"][wc[ok]]
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


# ------------------------------------------------------------------ the reference's cases and the calls held to it
def random_vocab(rng, n_base, wpb):
    base = rng.integers(-128, 128, (256, n_base)).astype(np.int8)
    scale = rng.uniform(0.5, 2.0, n_base).astype(f32)
    bias = rng.uniform(-0.3, 0.3, n_base).astype(f32)
    leaves = rng.integers(-2 ** 31, 2 ** 31, (n_base, wpb, 4)).astype(np.int32)
    return base, scale, bias, leaves


# one frame per (descriptor kind, desc_scale): random, zero, all -128, all 127, one row repeated
BOW_SCALES = (4.3353, -1.5, 0.0, 1e-30, 1e30, np.inf, -np.inf, np.nan)
BOW_KINDS = ("random", "zero", "min", "max", "repeated")


def bow_vocab(name):
    """(n_base, wpb) shapes with random contents, the reference vocabulary, and vocabularies built to tie."""
    rng = np.random.default_rng(sum(map(ord, name)))
    if name == "10x1000":
        return ref_vocab()
    if "x" in name:
        nb, wpb = (int(x) for x in name.split("x"))
        return random_vocab(rng, nb, wpb)
    if name == "repeated_leaves":      # leaf w = L[w % 5]: every 8-word window occurs at 4 leaves of different lanes
        base, scale, bias, _ = random_vocab(rng, 3, 20)
        L = rng.integers(-2 ** 31, 2 ** 31, (5, 4)).astype(np.int32)
        return base, scale, bias, np.ascontiguousarray(np.broadcast_to(L[np.arange(20) % 5], (3, 20, 4)))
    if name == "zero_leaves":          # every window ties
        base, scale, bias, leaves = random_vocab(rng, 2, 16)
        return base, scale, bias, np.zeros_like(leaves)
    if name == "nonpositive_scores":   # no score exceeds 0: base 0
        base, scale, bias, leaves = random_vocab(rng, 4, 11)
        scale[:2], bias[:2], bias[2:] = 0.0, 0.0, -1.2
        return base, scale, bias, leaves
    if name == "equal_bases":          # bases 2..4 identical and the only ones that can win: base 2
        base, scale, bias, leaves = random_vocab(rng, 5, 12)
        base[:, 3] = base[:, 4] = base[:, 2]
        scale[3:] = scale[2]
        bias[3:] = bias[2] = 0.25
        bias[:2] = -1.0
        return base, scale, bias, leaves
    raise KeyError(name)


def bow_inputs(seed, top_n, cells=48, reps=1):
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


def bow_check(tr, oracle, vocab, desc, dscale, qp, qc):
    """mv_bow_assign_batch on tr against oracle.bow_assign, frame by frame -> the device's words."""
    v = oracle.bow_vocab(*vocab)
    wpb = vocab[3].shape[1]
    word, base = tr.bow_assign(dev(tr, desc), dev(tr, dscale), dev(tr, qp), dev(tr, qc))
    word, base = word.cpu().numpy(), base.cpu().numpy()
    for f in range(desc.shape[0]):
        k = int(qc[f])
        assert (word[f, k:] == -1).all() and (base[f, k:] == -1).all(), f
        rb, rw = oracle.bow_assign(v, dscale[f], desc[f][qp[f, :k]])
        assert (base[f, :k] == rb).all(), (f, dscale[f])
        assert (word[f, :k] == rb * wpb + rw).all(), (f, dscale[f])
    return word


def case_inputs(name, synth):
    """Host inputs and parameters of one case -> dict(p, frames (semi, semi_scale, desc, desc_scale, depth), first,
    n_words, vocab, entry table or None)."""
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import tracking
    rng = np.random.default_rng(sum(map(ord, name)))
    vocab = ref_vocab()
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
        vocab = random_vocab(np.random.default_rng(77), 7, 13)
        vocab[3][:, 6:9] = vocab[3][:, 2:5]                                  # repeated leaves
        p = tracking.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=64)
        n_words, first = int(name[5:]), 40
    else:
        raise KeyError(name)
    return dict(p=p, frames=[semi, sscale, desc, dscale, depth], first=first, n_words=n_words, vocab=vocab,
                entry=entry)


def run_entry(tr, c, entry, monkeypatch):
    """Runs one entry point on the case -> (records bytes, n_with_landmark int32, final table bytes)."""
    import torch
    from maveric_slam_b200 import tracking
    p, first, n_words = c["p"], c["first"], c["n_words"]
    host = c["frames"]
    dframes = [dev(tr, x) for x in host]
    n_pairs = host[0].shape[0] - 1
    table = tr.landmarks_new(n_words) if c["entry"] is None else upload_table(tr, c["entry"])
    kind, _, opt = entry.partition(":")
    if kind == "device":
        res, nl = tr.track_sequence_landmarks(p, *dframes, table, first_frame=first)
        res, nl = res.cpu().numpy(), nl.cpu().numpy()
    elif kind == "host":
        if opt == "pageable":
            bufs = [np.ascontiguousarray(x) for x in host]
        else:
            bufs = [pinned(x) for x in host]
            if opt:
                monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", opt)
        res, nl, _, _ = tr.track_sequence_landmarks_host(p, *bufs, table, first_frame=first)
    elif kind in ("blocks", "blocks_host"):
        n_warm = int(opt)
        bufs = dframes if kind == "blocks" else [pinned(x) for x in host]
        prep = tr.track_landmarks_prepare if kind == "blocks" else tr.track_landmarks_prepare_host
        blocks = blocks_then_rest(n_pairs, (1, 5))
        prepared = {}
        for i, (lo, cnt) in reversed(list(enumerate(blocks))):
            w = min(n_warm, lo)
            prepared[i] = prep(with_first_pair(p, p.pnp.first_pair + lo), w, first + lo,
                               *[x[lo - w:lo + cnt + 1] for x in bufs], n_words)
        res, nl = [], []
        for i in range(len(blocks)):
            tr.track_landmarks_step_table(prepared[i], table)
            r, n = tr.track_landmarks_solve(prepared[i])
            res.append(r.cpu().numpy()); nl.append(n.cpu().numpy())
            tr.track_landmarks_release(prepared[i])
        res, nl = np.concatenate(res), np.concatenate(nl)
    elif kind == "sharded":
        res, nl, _ = tracking.track_sequence_landmarks_sharded(tr, p, dframes, table, first_frame=first, n_warm=8)
        res, nl = res.cpu().numpy(), nl.cpu().numpy()
    elif kind == "host_sharded":
        bufs = [pinned(x) for x in host]
        res, nl, _, _ = tracking.track_sequence_landmarks_host_sharded(tr, p, bufs, table, first_frame=first, n_warm=8)
        res, nl = res.cpu().numpy(), nl.cpu().numpy()
    else:
        raise KeyError(entry)
    torch.cuda.synchronize()
    return np.ascontiguousarray(res).view(np.uint8).reshape(-1).tobytes(), np.asarray(nl, np.int32), \
        table.cpu().numpy().tobytes()


def first_difference(want, got):
    """Pair and field of the first differing byte of two record arrays."""
    from maveric_slam_b200 import tracking
    g = np.frombuffer(got, tracking.PAIR_RESULT_DTYPE)
    for q in range(len(want)):
        for f in tracking.PAIR_RESULT_DTYPE.names:
            if want[q][f].tobytes() != g[q][f].tobytes():
                return "pair %d %s: reference %r, got %r" % (q, f, want[q][f], g[q][f])
    return "lengths %d, %d" % (len(want), len(g))
