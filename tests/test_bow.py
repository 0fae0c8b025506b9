"""SURVEY §8f rank 3: BoW word assignment (src/bow_main.c:62-125) and the landmark table that holds the contents
of the reference's local feature pool (include/local_feature_pool.h).

What is pinned and what is not:
  * bow_main.c crashes as shipped (tests/test_scope_evidence.py) and feeds every stage memory of the wrong type,
    so the word assignment AS A WHOLE follows the definition stated in oracle/mv_oracle.h -- PARITY UNPINNED;
  * its two helper functions are well defined when handed ints, and the oracle's orc_bow_binarize /
    orc_bow_matching_bits equal the reference's own get_binary_descriptor / count_matching_bits bit for bit
    (compiled from src/bow_main.c where it lies: oracle/_ref/libmaveric_ref_bow.so);
  * the vocabulary is the reference's (tests/golden/ref_vocab.npz, read out of that library);
  * the landmark table's contents equal the contents of the reference's pool (the product's host pool is
    pinned to the reference's header by test_local_feature_pool_matches_reference) under the per-frame
    sequence of src/local_feature_matching.c:153-163.
GPU tests: the CUDA kernels against the oracle, through the C ABI.
"""
import numpy as np
import pytest

from conftest import RECORD_T1, T1Calls
from helpers import drive_host_pool, ref_vocab, table_contents
from oracle import orc


@pytest.fixture(scope="module")
def vocab_np():
    return ref_vocab()


@pytest.fixture(scope="module")
def ref_bow_live():
    orc.build()
    if orc.have_ref_bow():
        return orc.ReferenceBow()
    if RECORD_T1:
        from golden.make_golden_t1 import StandInReferenceBow
        return StandInReferenceBow()
    return None


@pytest.fixture
def ref_bow(ref_bow_live, t1):
    """bow_main.c's helpers (T1): called where built, else their stored answers (tests/conftest.py)."""
    return T1Calls(ref_bow_live, t1)


# ------------------------------------------------------------------ CPU: oracle vs the reference's own code
def test_golden_vocabulary_is_the_references(ref_bow_live, vocab_np):
    if not isinstance(ref_bow_live, orc.ReferenceBow):
        pytest.skip("oracle/_ref/libmaveric_ref_bow.so not built (oracle/Makefile, from the reference's sources)")
    base, scale, bias, leaves = ref_bow_live.vocabulary()
    assert base.shape == (256, 10) and leaves.shape == (10, 1000, 4)
    for a, b in zip((base, scale, bias, leaves), vocab_np):
        assert a.dtype == b.dtype and a.tobytes() == b.tobytes()


def test_binarize_and_matching_bits_equal_reference_functions(oracle, ref_bow):
    """bow_main.c:13-41 and :43-55 on random descriptors (zeros, +-1 and extremes included), both signs of
    the scale, and on random words -- the oracle's restatements against the reference's functions."""
    rng = np.random.default_rng(2)
    for trial in range(200):
        d = rng.integers(-128, 128, 256).astype(np.int8)
        d[rng.random(256) < 0.2] = 0
        for scale in (4.3353, 1e-3, 0.0, -2.0):
            want = ref_bow.get_binary_descriptor(scale, d.astype(np.int32), 8)
            got = oracle.bow_binarize(scale, d)
            assert (want == got).all(), (trial, scale)
    for trial in range(500):
        a = rng.integers(-2**31, 2**31, 8).astype(np.int32)
        b = rng.integers(-2**31, 2**31, 8).astype(np.int32)
        if trial % 5 == 0:
            b = a.copy(); b[rng.integers(0, 8)] ^= np.int32(1 << int(rng.integers(0, 31)))
        assert oracle.bow_matching_bits(a, b) == ref_bow.count_matching_bits(a, b)
        assert oracle.bow_matching_bits(a[:4], b[:4]) == ref_bow.count_matching_bits(a[:4], b[:4])


def test_oracle_word_assignment_follows_its_definition(oracle, vocab_np, image0):
    """The stated definition in numpy (int64 sums, the same fp32 operations) on the reference fixture's own
    descriptors (quantized_image0.h): base node and leaf of 300 keypoint cells."""
    base_desc, scale, bias, leaves = vocab_np
    v = oracle.bow_vocab(base_desc, scale, bias, leaves)
    desc = image0["desc"].reshape(-1, 256)[::6][:300]
    ds = float(image0["desc_scale"])
    b, w = oracle.bow_assign(v, ds, desc)
    flat = np.concatenate([leaves.reshape(-1), np.zeros(4, np.int32)])
    for i in range(desc.shape[0]):
        raw = desc[i].astype(np.int64) @ base_desc.astype(np.int64)
        m = np.clip(np.rint(np.float32(ds) * raw.astype(np.float32) * np.float32(1 / 256)), -128, 127).astype(np.float32)
        score = scale * m + np.float32(256) * bias
        sel, best = 0, np.float32(0)
        for j in range(10):
            if score[j] > best:
                best, sel = score[j], j
        bits = np.packbits((desc[i] > 0) if ds > 0 else (desc[i] <= 0)).view(">u4").astype(np.uint32)
        cand = np.stack([flat[(sel * 1000 + k) * 4:(sel * 1000 + k) * 4 + 8].view(np.uint32) for k in range(1000)])
        match = 256 - np.unpackbits((cand ^ bits).view(np.uint8), axis=1).sum(1)
        assert (b[i], w[i]) == (sel, int(np.argmax(match))), i
    assert len(set(zip(b.tolist(), w.tolist()))) > 50      # it does discriminate


# ------------------------------------------------------------------ CPU: landmark table == contents of the pool
def test_oracle_landmark_table_equals_pool_contents(oracle):
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib
    snaps = drive_host_pool(lib.load())
    table = oracle.pool_new(10000)
    for f, (ids, coords, want) in enumerate(snaps):
        oracle.pool_observe(table, f, ids, coords)
        oracle.pool_remove_old(table, f)
        assert table_contents(table) == want, f
    assert len(snaps[-1][2]) > 500


# ------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_gpu_word_assignment_vs_oracle(tracker, oracle, synth, vocab_np, image0):
    """mv_bow_assign_batch against the oracle: the reference fixture's frame (24x80 cells, its own descriptor
    scale) and two synthetic KITTI-shaped frames, every query of each; plus a negative scale (the <= 0 branch of
    get_binary_descriptor) and a frame without queries."""
    import torch
    base_desc, scale, bias, leaves = vocab_np
    tracker.bow_set_vocabulary(base_desc, scale, bias, leaves)
    v = oracle.bow_vocab(base_desc, scale, bias, leaves)
    cases = []
    semi = image0["semi"].reshape(1, -1, 65)
    cases.append((24, 80, semi, image0["desc"].reshape(1, -1, 256), [float(image0["desc_scale"])], 100))
    s2, d2 = [], []
    for f in range(3):
        s, d, _ = synth.synth_frame(11, 47, 155, f, 3 * f, -2 * f)
        s2.append(s); d2.append(d)
    s2[2] = np.full_like(s2[2], -100)             # a frame without keypoints
    cases.append((47, 155, np.stack(s2), np.stack(d2), [4.3353, -1.5, 2.0], 1000))
    for rows, cols, semi, desc, dscale, N in cases:
        n = semi.shape[0]
        dsemi = torch.from_numpy(semi).to(tracker.device); ddesc = torch.from_numpy(desc).to(tracker.device)
        sscale = torch.full((n,), float(synth.SEMI_SCALE), device=tracker.device)
        idx, prob, _ = tracker.softmax(dsemi, sscale)
        qp, qi, _, qc, _ = tracker.top_n(idx, prob, N, rows * cols + 1)
        word, base = tracker.bow_assign(ddesc, torch.tensor(dscale, dtype=torch.float32, device=tracker.device), qp, qc)
        word, base, qp, qc = word.cpu().numpy(), base.cpu().numpy(), qp.cpu().numpy(), qc.cpu().numpy()
        for f in range(n):
            k = int(qc[f])
            assert (word[f, k:] == -1).all() and (base[f, k:] == -1).all()
            if k == 0:
                continue
            rb, rw = oracle.bow_assign(v, dscale[f], desc[f][qp[f, :k]])
            assert (base[f, :k] == rb).all(), f
            assert (word[f, :k] == rb * 1000 + rw).all(), f
    assert qc[2] == 0


@pytest.mark.gpu
def test_gpu_landmark_table_equals_pool_contents(tracker, oracle):
    """mv_landmarks_observe / remove_old / lookup against the contents of the host pool (the reference's) over 60
    frames of the reference driver's churn, and against the oracle table with duplicate words inside a frame."""
    import torch
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib, tracking
    snaps = drive_host_pool(lib.load())
    table = tracker.landmarks_new(10000)
    for f, (ids, coords, want) in enumerate(snaps):
        tracker.landmarks_observe(table, f, torch.from_numpy(ids).to(tracker.device), torch.from_numpy(coords).to(tracker.device))
        tracker.landmarks_remove_old(table, f)
        if f % 7 == 0 or f == len(snaps) - 1:
            got = table_contents(table.cpu().numpy().view(tracking.LANDMARK_DTYPE).reshape(-1))
            assert got == want, f
    # lookup: the 3-D side of correspondences
    ids, _, want = snaps[-1]
    probe = np.concatenate([ids[:50], np.array([-1, 10000, 9999], np.int32)]).astype(np.int32)
    c, found = tracker.landmarks_lookup(table, torch.from_numpy(probe).to(tracker.device))
    c, found = c.cpu().numpy(), found.cpu().numpy()
    for i, w in enumerate(probe):
        if int(w) in want:
            assert found[i] == 1 and tuple(float(x) for x in c[i]) == want[int(w)][1]
        else:
            assert found[i] == 0 and (c[i] == 0).all()
    # duplicates of a word inside one frame's list, ids out of range, an empty list: against the oracle table
    rng = np.random.default_rng(4)
    t2, o2 = tracker.landmarks_new(500), oracle.pool_new(500)
    for f in range(30):
        ids = rng.integers(-3, 520, 300).astype(np.int32)       # many duplicates, some out of range
        coords = rng.normal(size=(300, 3)).astype(np.float32)
        if f == 9:
            ids, coords = ids[:0], coords[:0]
        oracle.pool_observe(o2, f, ids, coords)
        oracle.pool_remove_old(o2, f)
        if len(ids):
            tracker.landmarks_observe(t2, f, torch.from_numpy(ids).to(tracker.device), torch.from_numpy(coords).to(tracker.device))
        tracker.landmarks_remove_old(t2, f)
        got = t2.cpu().numpy().view(tracking.LANDMARK_DTYPE).reshape(-1)
        assert table_contents(got) == table_contents(o2), f


@pytest.mark.gpu
def test_gpu_landmarks_supply_the_3d_side_of_pnp(tracker, oracle, synth, vocab_np):
    """The loop SURVEY §8f rank 3 closes: queries -> words -> landmark table -> coords_3D of the matched frame-0
    keypoints -> Gauss-Newton PnP.  The landmarks of frame f are its query keypoints back-projected with the frame's
    depth (the same fp32 operations as mv_build_corr_batch).  Where the matched frame-0 keypoint is a query of its
    frame and the first keypoint of its word, the landmark correspondence equals the depth correspondence bit for
    bit; elsewhere it is NaN (no landmark) or another keypoint's landmark (a word collision, an outlier to the
    solver); the pose solved from the landmark correspondences agrees with the depth-based one."""
    import torch
    from maveric_slam_b200 import tracking
    rows, cols, n_frames, N, M = 47, 155, 3, 1000, 1024
    base_desc, scale, bias, leaves = vocab_np
    tracker.bow_set_vocabulary(base_desc, scale, bias, leaves)
    off = synth.default_offsets(n_frames, 5)
    semi, desc, depth = tracker.synth_frames(5, rows, cols, 0, off)
    sscale = torch.full((n_frames,), float(synth.SEMI_SCALE), device=tracker.device)
    idx, prob, _ = tracker.softmax(semi, sscale)
    qp, qi, _, qc, _ = tracker.top_n(idx, prob, N, 8192)
    dscale = torch.full((n_frames,), 4.3353, device=tracker.device)
    word, _ = tracker.bow_assign(desc, dscale, qp, qc)
    p = tracking.kitti_track_params()
    pts, cnt, cell0, _, _ = tracker.match(p.match, desc, idx, prob, qp, qi, qc)
    cam = (p.pnp.fx, p.pnp.fy, p.pnp.cx, p.pnp.cy)
    corr_d = tracker.build_corr(pts, cnt, cell0, depth, cam, rows)
    hq, hi_, hc, hw, hz = (t.cpu().numpy() for t in (qp, qi, qc, word, depth))
    f32 = np.float32
    poses = []
    for pair in range(n_frames - 1):
        f0 = pair
        k = int(hc[f0])
        cells = hq[f0, :k]
        x = (cells // rows * 8 + hi_[f0, :k] % 8).astype(f32)
        y = (cells % rows * 8 + hi_[f0, :k] // 8).astype(f32)
        dz = hz[f0, cells]
        coords = np.stack([(x - f32(cam[2])) / f32(cam[0]) * dz, (y - f32(cam[3])) / f32(cam[1]) * dz, dz], 1).astype(f32)
        table = tracker.landmarks_new(10000)
        tracker.landmarks_observe(table, f0, torch.from_numpy(hw[f0, :k].copy()).to(tracker.device),
                                  torch.from_numpy(coords).to(tracker.device))
        corr_l, nl = tracker.build_corr_landmarks(table, pts[pair:pair + 1], cnt[pair:pair + 1], cell0[pair:pair + 1], qp, qc,
                                                  word, f0=torch.tensor([f0], dtype=torch.int32, device=tracker.device))
        n = int(cnt[pair])
        cl, cd, c0 = corr_l[0].cpu().numpy(), corr_d[pair].cpu().numpy(), cell0[pair].cpu().numpy()
        assert (cl[3:, :n].view(np.int32) == cd[3:, :n].view(np.int32)).all()     # the 2-D side is the match
        first_of_word = {}
        for q in range(k):
            first_of_word.setdefault(int(hw[f0, q]), q)
        exact = nan = other = 0
        for j in range(n):
            q = int(np.searchsorted(cells, c0[j]))
            if q >= k or cells[q] != c0[j]:
                assert np.isnan(cl[:3, j]).all()
                nan += 1
            elif first_of_word[int(hw[f0, q])] == q:
                assert (cl[:3, j].view(np.int32) == cd[:3, j].view(np.int32)).all(), (pair, j)
                exact += 1
            else:
                assert (cl[:3, j].view(np.int32) == coords[first_of_word[int(hw[f0, q])]].view(np.int32)).all()
                other += 1
        assert int(nl[0]) == exact + other and exact > 0.5 * n, (exact, other, nan, n)
        pose_l, stats_l, _ = tracker.pnp_gn(p.pnp, corr_l, cnt[pair:pair + 1])
        pose_d, stats_d, _ = tracker.pnp_gn(p.pnp, corr_d[pair:pair + 1].contiguous(), cnt[pair:pair + 1])
        pl, pd = pose_l.cpu().numpy()[0], pose_d.cpu().numpy()[0]
        ang = 2 * np.arccos(min(1.0, abs(float(np.dot(pl[:4], pd[:4]))) / (np.linalg.norm(pl[:4]) * np.linalg.norm(pd[:4]))))
        # (a sanity bound: the two solves see different correspondence subsets -- word collisions are outliers here)
        assert stats_l.cpu().numpy()[0, 3] == 1 and ang < 5e-3 and np.linalg.norm(pl[4:] - pd[4:]) < 0.3, (ang, pl, pd)
        assert stats_l.cpu().numpy()[0, 0] >= 0.3 * stats_d.cpu().numpy()[0, 0]
        poses.append(ang)
