"""The landmark table over a whole sequence in one call (mv_landmarks_sequence) and the sequence path that takes the
3-D side of PnP from it (mv_track_sequence_landmarks).

References, all composed from pieces pinned elsewhere (tests/test_bow.py):
  * the per-frame loop of the existing kernels mv_landmarks_observe / mv_landmarks_remove_old, with
    mv_landmarks_lookup after each step -- the final table must be byte-equal, stale slots included;
  * orc_landmarks_sequence (tests/landmark_reference.py): the same loop on the oracle's table (orc_pool_observe / orc_pool_remove_old),
    itself checked against the contents of the host pool, which is pinned to the reference's header;
  * for the sequence path, the public calls softmax -> top_n -> bow_assign, the per-frame table loop,
    match -> ransac_identity, build_corr_landmarks per pair against its snapshot, pnp_gn; and the oracle's K3.
The whole path against a CPU reference built from the oracle alone: tests/test_landmark_reference.py.
"""
import numpy as np
import pytest

from helpers import N_FRAMES, dev, drive_host_pool, landmark_sequence, table_bytes, table_contents, upload_table
from landmark_reference import orc_landmarks_sequence

CAM = (718.856, 718.856, 607.1928, 185.2157)


# ------------------------------------------------------------------ CPU
def test_oracle_sequence_equals_pool_contents(oracle):
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib
    snaps = drive_host_pool(lib.load())
    word = np.stack([s[0] for s in snaps]).astype(np.int32)
    coords = np.stack([s[1] for s in snaps]).astype(np.float32)
    table = oracle.pool_new(10000)
    tabs = []
    out = orc_landmarks_sequence(oracle, table, 0, word, np.full(len(snaps), word.shape[1], np.int32), coords, tabs)
    for f, (ids, _, want) in enumerate(snaps):
        assert table_contents(tabs[f]) == want, f
        for q, w in enumerate(ids):
            assert tuple(float(c) for c in out[f, q]) == want[int(w)][1], (f, q)
    assert len(snaps[-1][2]) > 500


# ------------------------------------------------------------------ GPU: mv_landmarks_sequence
def _per_frame_loop(tracker, table, first_frame, word, q_count, coords):
    """The existing kernels, one frame at a time; lookups after each step."""
    n_steps, top_n = word.shape
    out = np.zeros((n_steps, top_n, 3), np.float32)
    for f in range(n_steps):
        k = min(int(q_count[f]), top_n)
        if k:
            tracker.landmarks_observe(table, first_frame + f, dev(tracker, word[f, :k]), dev(tracker, coords[f, :k]))
        tracker.landmarks_remove_old(table, first_frame + f)
        if k:
            c, _ = tracker.landmarks_lookup(table, dev(tracker, word[f, :k]))
            out[f, :k] = c.cpu().numpy()
    return out


def _cases():
    rng = np.random.default_rng(11)
    cases = {}
    # the 60-frame churn of the reference driver (helpers.drive_host_pool, pinned in tests/test_bow.py)
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib
    snaps = drive_host_pool(lib.load())
    word = np.stack([s[0] for s in snaps]).astype(np.int32)
    cases["churn"] = dict(n_words=10000, first=0, word=word, qc=np.full(len(snaps), 200, np.int32),
                          coords=np.stack([s[1] for s in snaps]).astype(np.float32), init=None)
    # duplicates (one word 20 times in a frame: the ring overflows inside it), ids -1 and >= n_words, short and
    # empty frames, words absent for more than 8 frames (deleted, re-inserted with new coordinates)
    n, top_n = 40, 300
    word = rng.integers(-3, 520, (n, top_n)).astype(np.int32)
    word[5, 10:30] = 77
    word[:, :4] = 3
    word[word == 42] = 43
    word[np.arange(n) % 13 < 2, 4] = 42           # word 42: present 2 frames of 13, absent 11
    qc = np.full(n, top_n, np.int32)
    qc[7], qc[9], qc[21] = 0, 150, 1000           # empty, short, larger than top_n
    cases["churn_dups"] = dict(n_words=500, first=0, word=word, qc=qc,
                               coords=rng.normal(size=(n, top_n, 3)).astype(np.float32), init=None)
    # a non-zero first frame and a non-empty initial table (the oracle's state after 25 other frames)
    from oracle import orc
    o = orc.Oracle()
    init = o.pool_new(500)
    w0 = rng.integers(0, 500, (25, 200)).astype(np.int32)
    orc_landmarks_sequence(o, init, 975, w0, np.full(25, 200, np.int32), rng.normal(size=(25, 200, 3)).astype(np.float32))
    word = rng.integers(0, 520, (30, 200)).astype(np.int32)
    cases["resume"] = dict(n_words=500, first=1000, word=word, qc=np.full(30, 200, np.int32),
                           coords=rng.normal(size=(30, 200, 3)).astype(np.float32), init=init)
    # one word for every query of every frame: the longest possible list
    cases["one_word"] = dict(n_words=10000, first=3, word=np.full((24, 1000), 9999, np.int32),
                             qc=np.full(24, 1000, np.int32), coords=rng.normal(size=(24, 1000, 3)).astype(np.float32),
                             init=None)
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["churn", "churn_dups", "resume", "one_word"])
def test_landmarks_sequence_equals_per_frame_loop_and_oracle(tracker, oracle, case):
    c = _cases()[case]
    word, qc, coords, n_words, first = c["word"], c["qc"], c["coords"], c["n_words"], c["first"]
    init = c["init"] if c["init"] is not None else oracle.pool_new(n_words)
    t_loop = upload_table(tracker, init)
    want = _per_frame_loop(tracker, t_loop, first, word, qc, coords)
    t_seq = upload_table(tracker, init)
    got = tracker.landmarks_sequence(t_seq, first, dev(tracker, word), dev(tracker, qc), dev(tracker, coords))
    got = got.cpu().numpy()
    assert table_bytes(t_seq) == table_bytes(t_loop)
    assert got.view(np.int32).tobytes() == want.view(np.int32).tobytes()
    o_table = init.copy()
    o_out = orc_landmarks_sequence(oracle, o_table, first, word, qc, coords)
    assert table_bytes(t_seq) == o_table.tobytes()
    assert got.tobytes() == o_out.tobytes()
    if case == "churn_dups":   # word 42 really was deleted and re-inserted with the coordinates of its new frame
        rec = t_seq.cpu().numpy().view(oracle.pool_new(1).dtype).reshape(-1)[42]
        last_ins = max(f for f in range(word.shape[0]) if f % 13 == 0)
        assert rec["word_id"] == 42 and (rec["coords"] == coords[last_ins, 4]).all()


@pytest.mark.gpu
def test_landmarks_sequence_split_equals_one_call(tracker, oracle):
    c = _cases()["churn_dups"]
    word, qc, coords = c["word"], c["qc"], c["coords"]
    one = upload_table(tracker, oracle.pool_new(500))
    out1 = tracker.landmarks_sequence(one, 0, dev(tracker, word), dev(tracker, qc), dev(tracker, coords)).cpu().numpy()
    for k in (1, 17, 39):
        two = upload_table(tracker, oracle.pool_new(500))
        a = tracker.landmarks_sequence(two, 0, dev(tracker, word[:k]), dev(tracker, qc[:k]), dev(tracker, coords[:k]))
        b = tracker.landmarks_sequence(two, k, dev(tracker, word[k:]), dev(tracker, qc[k:]), dev(tracker, coords[k:]))
        assert table_bytes(two) == table_bytes(one), k
        assert np.concatenate([a.cpu().numpy(), b.cpu().numpy()]).tobytes() == out1.tobytes(), k


# ------------------------------------------------------------------ GPU: mv_track_sequence_landmarks
@pytest.fixture(scope="module")
def seq(tracker, synth):
    """A KITTI-shaped synthetic sequence, the path's results, and the composition of public calls."""
    import torch
    s = landmark_sequence(tracker, synth)
    semi, sscale, desc, dscale, depth = s["d"].values()
    p, first, n_words, rows, n = s["p"], s["first"], s["n_words"], 47, N_FRAMES
    # the composition
    idx, prob, _ = tracker.softmax(semi, sscale)
    qp, qi, _, qc, ov = tracker.top_n(idx, prob, p.top_n, p.max_valid)
    word, _ = tracker.bow_assign(desc[:n - 1], dscale[:n - 1], qp[:n - 1], qc[:n - 1])
    hq, hi_, hz = qp.cpu().numpy(), qi.cpu().numpy(), depth.cpu().numpy()
    f32 = np.float32
    x = (hq // rows * 8 + hi_ % 8).astype(f32)
    y = (hq % rows * 8 + hi_ // 8).astype(f32)
    dz = np.take_along_axis(hz, hq, axis=1)
    coords = np.stack([(x - f32(CAM[2])) / f32(CAM[0]) * dz, (y - f32(CAM[3])) / f32(CAM[1]) * dz, dz], -1).astype(f32)
    hw, hc = word.cpu().numpy(), qc.cpu().numpy()
    ref_table = tracker.landmarks_new(n_words)
    snaps = []
    for f in range(n - 1):
        k = min(int(hc[f]), p.top_n)
        tracker.landmarks_observe(ref_table, first + f, dev(tracker, hw[f, :k]), dev(tracker, coords[f, :k]))
        tracker.landmarks_remove_old(ref_table, first + f)
        snaps.append(ref_table.clone())
    pts, cnt, cell0, _, _ = tracker.match(p.match, desc, idx, prob, qp, qi, qc)
    rin, _, _ = tracker.ransac_identity(pts, cnt, p.ransac_iterations, p.ransac_threshold)
    corr, nls = [], []
    for pair in range(n - 1):
        c, l = tracker.build_corr_landmarks(snaps[pair], pts[pair:pair + 1], cnt[pair:pair + 1], cell0[pair:pair + 1],
                                            qp, qc, word, f0=torch.tensor([pair], dtype=torch.int32, device=tracker.device))
        corr.append(c); nls.append(l)
    corr = torch.cat(corr)
    pose, stats, _ = tracker.pnp_gn(p.pnp, corr, cnt)
    return dict(s, **s["d"], ref_table=table_bytes(ref_table), pose=pose.cpu().numpy(), stats=stats.cpu().numpy(),
                cnt=cnt.cpu().numpy(), rin=rin.cpu().numpy(), ov=ov.cpu().numpy(), nls=torch.cat(nls).cpu().numpy(),
                corr=corr.cpu().numpy())


@pytest.mark.gpu
def test_track_sequence_landmarks_equals_composition(seq):
    r = seq["res"]
    assert seq["table"] == seq["ref_table"]
    assert r["q"].view(np.int32).tobytes() == seq["pose"][:, :4].view(np.int32).tobytes()
    assert r["t"].view(np.int32).tobytes() == seq["pose"][:, 4:].view(np.int32).tobytes()
    assert r["pnp_inliers"].view(np.int32).tobytes() == seq["stats"][:, 0].copy().view(np.int32).tobytes()
    assert r["pnp_cost"].view(np.int32).tobytes() == seq["stats"][:, 1].copy().view(np.int32).tobytes()
    assert (r["best_hypothesis"] == seq["stats"][:, 2].astype(np.int32)).all()
    assert (r["num_matches"] == seq["cnt"]).all() and (r["ransac_inliers"] == seq["rin"]).all()
    ov = seq["ov"]
    assert (r["status"] == np.where((ov[:-1] != 0) | (ov[1:] != 0), 4, 0)).all()
    assert (seq["nl"] == seq["nls"]).all()
    assert (seq["nl"] > 0.5 * seq["cnt"]).all() and (seq["stats"][:, 3] == 1).all()


@pytest.mark.gpu
def test_k3_on_landmark_correspondences_equals_oracle(seq, oracle):
    from oracle import orc
    p = seq["p"]
    cfg = orc.pnp_cfg(hypotheses=p.pnp.hypotheses, seed=p.pnp.seed, lanes=1)
    r = seq["res"]
    for pair in range(0, N_FRAMES - 1, 8):
        pose, stats, _ = oracle.pnp_gn(cfg, seq["corr"][pair], int(seq["cnt"][pair]), pair_index=p.pnp.first_pair + pair)
        assert np.concatenate([r["q"][pair], r["t"][pair]]).view(np.int32).tobytes() == pose.view(np.int32).tobytes(), pair
        assert r["pnp_inliers"][pair].view(np.int32) == stats[:1].view(np.int32)[0], pair
        assert r["pnp_cost"][pair].view(np.int32) == stats[1:2].view(np.int32)[0], pair
        assert r["best_hypothesis"][pair] == int(stats[2]), pair


@pytest.mark.gpu
def test_track_sequence_landmarks_halo_split_equals_one_call(tracker, seq):
    from maveric_slam_b200 import tracking
    k = 29
    table = tracker.landmarks_new(seq["n_words"])
    parts, nls = [], []
    for lo, hi in ((0, k + 1), (k, N_FRAMES)):
        p = tracking.kitti_track_params(hypotheses=256, first_pair=lo)
        res, nl = tracker.track_sequence_landmarks(p, seq["semi"][lo:hi], seq["sscale"][lo:hi], seq["desc"][lo:hi],
                                                   seq["dscale"][lo:hi], seq["depth"][lo:hi], table,
                                                   first_frame=seq["first"] + lo)
        parts.append(tracking.results_to_numpy(res)); nls.append(nl.cpu().numpy())
    assert np.concatenate(parts).tobytes() == seq["res"].tobytes()
    assert (np.concatenate(nls) == seq["nl"]).all()
    assert table_bytes(table) == seq["table"]


@pytest.mark.gpu
def test_depth_path_untouched_by_landmark_path(tracker, seq):
    p, semi, sscale, desc, depth = seq["p"], seq["semi"], seq["sscale"], seq["desc"], seq["depth"]
    before = tracker.track_sequence(p, semi, sscale, desc, depth).cpu().numpy().tobytes()
    table = tracker.landmarks_new(seq["n_words"])
    tracker.track_sequence_landmarks(p, semi, sscale, desc, seq["dscale"], depth, table)
    after = tracker.track_sequence(p, semi, sscale, desc, depth).cpu().numpy().tobytes()
    assert before == after


@pytest.mark.gpu
def test_track_sequence_landmarks_argument_errors(tracker, seq):
    import torch
    from maveric_slam_b200 import lib, tracking
    p, semi, sscale, desc, dscale, depth = (seq[k] for k in ("p", "semi", "sscale", "desc", "dscale", "depth"))
    table = tracker.landmarks_new(seq["n_words"])
    fresh = tracking.Tracker(0)          # a context without a vocabulary
    with pytest.raises(lib.MvError, match="no vocabulary"):
        fresh.track_sequence_landmarks(p, semi[:3], sscale[:3], desc[:3], dscale[:3], depth[:3], table)
    with pytest.raises(lib.MvError, match="NULL landmark table"):
        tracker.ctx.check(tracker.lib.mv_track_sequence_landmarks(
            tracker.ctx.h, tracking.C.byref(p), 3, 0, tracker._d(semi), tracker._d(sscale), tracker._d(desc),
            tracker._d(dscale), tracker._d(depth), seq["n_words"], None, tracker._d(torch.empty((2, 64), dtype=torch.uint8,
                                                                                                   device=tracker.device)), None))
    with pytest.raises(lib.MvError, match="bad argument"):
        tracker.track_sequence_landmarks(p, semi[:1], sscale[:1], desc[:1], dscale[:1], depth[:1], table)
    n, cells = 3, desc.shape[1]
    buf = torch.empty(n * cells * 256 + 16, dtype=torch.int8, device=tracker.device)
    odd = buf[1:1 + n * cells * 256].view(n, cells, 256)
    odd.copy_(desc[:n])
    with pytest.raises(lib.MvError, match="16-byte aligned"):
        tracker.track_sequence_landmarks(p, semi[:n], sscale[:n], odd, dscale[:n], depth[:n], table)
    with pytest.raises(lib.MvError, match="n_words must be positive"):
        tracker.ctx.check(tracker.lib.mv_landmarks_sequence(tracker.ctx.h, 0, tracker._d(table), 0, 1, 1, None, None,
                                                            None, None))
    # refusals of the PnP and the matcher: checked before the table is stepped, nothing launched
    before = table_bytes(table)
    for part, field, val in (("pnp", "lanes_per_hypothesis", 4), ("pnp", "hypotheses", 0), ("pnp", "sample_size", 0),
                             ("match", "radius", -1)):
        bad = tracking.kitti_track_params(hypotheses=256)
        setattr(getattr(bad, part), field, val)
        launches = tracker.ctx.launches
        with pytest.raises(lib.MvError, match="bad argument"):
            tracker.track_sequence_landmarks(bad, semi, sscale, desc, dscale, depth, table, first_frame=seq["first"])
        assert tracker.ctx.launches == launches, field
        assert table_bytes(table) == before, field
    # the context still works and the table gives the stored answer
    res, nl = tracker.track_sequence_landmarks(p, semi, sscale, desc, dscale, depth, table, first_frame=seq["first"])
    assert tracking.results_to_numpy(res).tobytes() == seq["res"].tobytes() and (nl.cpu().numpy() == seq["nl"]).all()
    assert table_bytes(table) == seq["table"]
