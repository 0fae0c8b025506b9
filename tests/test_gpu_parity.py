"""GPU parity: every kernel of the hot path, called through the C ABI of
libmaveric_b200.so, against the CPU oracle (pinned to the reference by
test_oracle_vs_ref.py) and against the golden vectors produced by the reference itself.
Bit-exact for integers, indices, candidate/match lists (incl. tie order) and the fp32 of
the detector / RANSAC / SVD; the Gauss-Newton PnP is held to 1e-5 rad / 1e-5 relative
against its (reference-unpinned) oracle."""
import numpy as np
import pytest

from conftest import bits
from helpers import pnp_params
from oracle import orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def tk(tracker):
    from maveric_slam_b200 import tracking
    return tracking


def rot_angle(q1, q2):
    q1 = np.asarray(q1, np.float64); q2 = np.asarray(q2, np.float64)
    q1 = q1 / np.linalg.norm(q1); q2 = q2 / np.linalg.norm(q2)
    # angle of the relative rotation, from the vector part (well conditioned near zero)
    w = abs(float(np.dot(q1, q2)))
    v = np.array([q1[0] * q2[1] - q1[1] * q2[0] - q1[2] * q2[3] + q1[3] * q2[2],
                  q1[0] * q2[2] + q1[1] * q2[3] - q1[2] * q2[0] - q1[3] * q2[1],
                  q1[0] * q2[3] - q1[1] * q2[2] + q1[2] * q2[1] - q1[3] * q2[0]])
    return 2.0 * np.arctan2(np.linalg.norm(v), w)


# ------------------------------------------------------------------ synthetic generator
def test_cuda_generator_equals_numpy(tracker, synth):
    off = synth.default_offsets(3, 5)
    semi, desc, depth = tracker.synth_frames(5, 24, 80, 0, off)
    for f in range(3):
        s, d, z = synth.synth_frame(5, 24, 80, f, int(off[f, 0]), int(off[f, 1]))
        assert (semi[f].cpu().numpy() == s).all()
        assert (desc[f].cpu().numpy() == d).all()
        assert (bits(depth[f].cpu().numpy()) == bits(z)).all()


# ------------------------------------------------------------------ detector
def test_legacy_softmax_topn_on_reference_fixture(tk, image0, kat):
    idx, pr, nv = tk.compute_softmax(image0["semi_scale"], image0["semi"], legacy=True)
    assert nv == 410 and (idx == kat["img0_softmax_idx"]).all()
    assert (bits(pr) == bits(kat["img0_softmax_prob"])).all()
    pa, ix, pp = tk.compute_top_N(image0["semi_scale"], image0["semi"], 100, legacy=True)
    assert (pa == kat["img0_top100_patch"]).all() and (ix == kat["img0_top100_idx"]).all()
    assert (bits(pp) == bits(kat["img0_top100_prob"])).all()


@pytest.mark.parametrize("rows,cols,permille,N", [(24, 80, 140, 100), (47, 155, 140, 1000), (47, 155, 550, 4000),
                                                  (94, 310, 550, 16000), (5, 7, 300, 3)])
def test_softmax_topn_ex_vs_oracle(tk, oracle, synth, rows, cols, permille, N):
    s, d, z = synth.synth_frame(3, rows, cols, 0, 11, -7, permille)
    scale = float(synth.SEMI_SCALE)
    i1, p1, n1 = tk.compute_softmax(scale, s)
    i2, p2, n2 = oracle.softmax(scale, s)
    assert n1 == n2 and (i1 == i2).all() and (bits(p1) == bits(p2)).all()
    mv = rows * cols + 1
    a = tk.compute_top_N(scale, s, N, max_valid=mv)
    b = oracle.top_n(scale, s, N, max_valid=mv)
    assert len(a[0]) == len(b[0])
    assert (a[0] == b[0]).all() and (a[1] == b[1]).all() and (bits(a[2]) == bits(b[2])).all()


def test_topn_overflow_is_reported(tk, oracle, synth):
    from maveric_slam_b200 import lib
    s, _, _ = synth.synth_frame(3, 47, 155, 0, 0, 0, 550)
    assert oracle.top_n(float(synth.SEMI_SCALE), s, 100, max_valid=1000)[3] == 1
    with pytest.raises(lib.MvError):
        tk.compute_top_N(float(synth.SEMI_SCALE), s, 100, max_valid=1000)


def test_softmax_batch_unaligned_and_counts(tracker, oracle, synth):
    import torch
    semi, desc, depth, off = synth.synth_sequence(9, 24, 80, 3)
    buf = torch.zeros(semi.size + 64, dtype=torch.int8, device=tracker.device)
    view = buf[3:3 + semi.size].view(3, 1920, 65)            # deliberately not 16-byte aligned
    view.copy_(torch.from_numpy(semi))
    scale = torch.tensor([0.3562, 0.30, 0.41], dtype=torch.float32, device=tracker.device)
    idx, prob, nv = tracker.softmax(view, scale)
    for f in range(3):
        i2, p2, n2 = oracle.softmax(float(scale[f].item()), semi[f])
        assert int(nv[f]) == n2 and (idx[f].cpu().numpy() == i2).all() and (bits(prob[f].cpu().numpy()) == bits(p2)).all()


@pytest.mark.parametrize("seed", range(6))
def test_detector_on_adversarial_logits(tk, oracle, seed):
    """tests/adversarial.py:adversarial_logits (ties inside cells, 127 under large scales, dustbin-only
    and all-negative cells, probability ties at the top-N cut) through compute_softmax_ex /
    compute_top_N_ex against T2, which test_t2_equals_t1_on_adversarial_logits pins to T1
    (top_N.c:22-49 first-wins argmax, :77 threshold, :108-133 first N in patch order)."""
    from adversarial import adversarial_logits
    semi = adversarial_logits(seed)
    for scale in (0.01, 0.35622698, 1.0, 3.0):
        i1, p1, n1 = tk.compute_softmax(scale, semi)
        i2, p2, n2 = oracle.softmax(scale, semi)
        assert n1 == n2 and (i1 == i2).all() and (bits(p1) == bits(p2)).all()
        for N in (100, 37, 1):
            a = tk.compute_top_N(scale, semi, N, max_valid=1000)
            b = oracle.top_n(scale, semi, N, max_valid=1000)
            assert len(a[0]) == len(b[0])
            assert (a[0] == b[0]).all() and (a[1] == b[1]).all() and (bits(a[2]) == bits(b[2])).all()


# ------------------------------------------------------------------ matcher
def _oracle_pair(oracle, rows, cols, s0, d0, s1, d1, N, M, radius=4, shift=(4, 4), scale=None, max_valid=None):
    scale = float(scale)
    idx, pr, _ = oracle.softmax(scale, s0)
    pa, ix, _, ov = oracle.top_n(scale, s1, N, max_valid or rows * cols + 1)
    cfg = orc.MatchCfg(rows, cols, shift[0], shift[1], radius, M, 0.9, 0.2)
    return idx, pr, pa, ix, oracle.match(cfg, d0, d1, idx, pr, pa, ix)


@pytest.mark.parametrize("rows,cols,permille,N,M,radius,shift", [
    (24, 80, 140, 100, 150, 4, (4, 4)),
    (24, 80, 400, 100, 150, 4, (4, 4)),
    (47, 155, 140, 1000, 1024, 4, (4, 4)),
    (47, 155, 550, 4000, 4096, 4, (4, 4)),
    (47, 155, 140, 1000, 64, 4, (4, 4)),        # cap on matches binds
    (47, 155, 300, 2000, 2048, 16, (0, 0)),      # wide window
    (24, 80, 300, 200, 256, 30, (-3, 5)),        # window larger than the grid in y
    (24, 80, 300, 200, 256, 0, (1, 1)),          # single-cell window
    (24, 80, 300, 200, 256, 2, (200, 0)),        # window entirely off-grid: no matches
    (94, 310, 550, 16000, 16384, 16, (4, 4)),    # BASELINE configs[4] shape: 16k keypoints, 33x33 window
    (94, 155, 550, 8000, 8192, 4, (4, 4)),       # configs[1] sweep, 8k keypoints
    (13, 300, 300, 500, 512, 5, (-2, 1)),        # short columns: a 32-cell block spans 3+ cell columns
    (200, 40, 300, 700, 1024, 6, (2, -3)),       # tall columns: one cell column per TMA box
])
@pytest.mark.parametrize("tc", [False, True], ids=["dp4a", "tcgen05"])
def test_match_pair_vs_oracle(tk, oracle, synth, rows, cols, permille, N, M, radius, shift, tc):
    off = synth.default_offsets(2, 21)
    s0, d0, _ = synth.synth_frame(21, rows, cols, 0, int(off[0, 0]), int(off[0, 1]), permille)
    s1, d1, _ = synth.synth_frame(21, rows, cols, 1, int(off[1, 0]), int(off[1, 1]), permille)
    idx, pr, pa, ix, ref = _oracle_pair(oracle, rows, cols, s0, d0, s1, d1, N, M, radius, shift, synth.SEMI_SCALE)
    p = tk.match_params(rows, cols, shift[0], shift[1], radius, M, use_tensor_cores=tc)
    got = tk.match_pair(p, d0, d1, idx, pr, pa, ix)
    assert got["n"] == ref["n"]
    assert (got["pts0"] == ref["pts0"]).all() and (got["pts1"] == ref["pts1"]).all()
    assert (got["cell0"] == ref["cell0"]).all() and (bits(got["score"]) == bits(ref["score"])).all()


@pytest.mark.parametrize("tc", [False, True], ids=["dp4a", "tcgen05"])
def test_match_zero_descriptors_and_ties(tk, oracle, synth, tc):
    rows, cols = 24, 80
    s0, d0, _ = synth.synth_frame(2, rows, cols, 0, 0, 0, 400)
    s1, d1, _ = synth.synth_frame(2, rows, cols, 1, 4, 4, 400)
    d0 = d0.copy()
    d0[::2] = 0                       # sticky zero norm: several leading candidates go the 256-d way
    d0[1::4] = d0[1]                  # identical descriptors: exact score ties, first must win
    idx, pr, pa, ix, ref = _oracle_pair(oracle, rows, cols, s0, d0, s1, d1, 100, 150, scale=synth.SEMI_SCALE)
    got = tk.match_pair(tk.match_params(rows, cols, use_tensor_cores=tc), d0, d1, idx, pr, pa, ix)
    assert got["n"] == ref["n"] > 0
    assert (got["cell0"] == ref["cell0"]).all() and (bits(got["score"]) == bits(ref["score"])).all()
    assert (got["pts0"] == ref["pts0"]).all()


@pytest.mark.parametrize("tc", [False, True], ids=["dp4a", "tcgen05"])
@pytest.mark.parametrize("seed", range(4))
def test_detector_and_match_on_adversarial_pairs(tk, oracle, synth, seed, tc):
    """The inputs of test_t2_equals_t1_on_adversarial_descriptors (tests/adversarial.py: wrapping products,
    exact ties, runs of zero descriptors, sign flips, probability ties at the top-N threshold) -- where
    the restatement is checked against the reference's own code -- through the library's detector
    and both matchers: same query lists, matches, candidate cells and score bits."""
    from adversarial import adversarial_pair
    scale, s0, d0, s1, d1 = adversarial_pair(oracle, synth, seed)
    idx, pr, pa, ix, ref = _oracle_pair(oracle, 24, 80, s0, d0, s1, d1, 100, 150, scale=scale, max_valid=1000)
    gi, gp, _ = tk.compute_softmax(scale, s0)
    assert (gi == idx).all() and (bits(gp) == bits(pr)).all()
    ga = tk.compute_top_N(scale, s1, 100, max_valid=1000)
    assert (ga[0] == pa).all() and (ga[1] == ix).all()
    got = tk.match_pair(tk.match_params(24, 80, use_tensor_cores=tc), d0, d1, gi, gp, ga[0], ga[1])
    assert got["n"] == ref["n"] > 0
    assert (got["cell0"] == ref["cell0"]).all() and (bits(got["score"]) == bits(ref["score"])).all()
    assert (got["pts0"] == ref["pts0"]).all() and (got["pts1"] == ref["pts1"]).all()


@pytest.mark.parametrize("tc", [False, True], ids=["dp4a", "tcgen05"])
def test_match_self_pair_golden(tk, image0, kat, tc):
    idx, pr, _ = tk.compute_softmax(image0["semi_scale"], image0["semi"], legacy=True)
    pa, ix, _ = tk.compute_top_N(image0["semi_scale"], image0["semi"], 100, legacy=True)
    got = tk.match_pair(tk.match_params(24, 80, use_tensor_cores=tc), image0["desc"], image0["desc"], idx, pr, pa, ix)
    assert got["n"] == 93
    assert (got["pts0"] == kat["self_pts0"]).all() and (got["pts1"] == kat["self_pts1"]).all()


@pytest.mark.parametrize("tc", [False, True], ids=["dp4a", "tcgen05"])
def test_match_no_queries(tk, synth, tc):
    s0, d0, _ = synth.synth_frame(2, 24, 80, 0, 0, 0)
    idx, pr, _ = tk.compute_softmax(float(synth.SEMI_SCALE), s0)
    got = tk.match_pair(tk.match_params(24, 80, use_tensor_cores=tc), d0, d0, idx, pr, np.zeros(0, np.int32), np.zeros(0, np.int32))
    assert got["n"] == 0


# ------------------------------------------------------------------ pose (legacy RANSAC-E)
def test_ransac_legacy_symbol(tk, oracle, kat):
    rng = np.random.default_rng(3)
    p1 = rng.integers(0, 640, size=(150, 2)).astype(np.float32)
    p2 = p1 + rng.integers(-1, 2, size=(150, 2)).astype(np.float32)
    K = np.eye(3, dtype=np.float32)
    E, inl, n = tk.ransac_essential_matrix(p1, p2, K)
    E2, inl2, n2, _ = oracle.ransac_identity(p1, p2)
    assert n == n2 > 0 and (inl == inl2).all() and (E == E2).all()
    E, inl, n = tk.ransac_essential_matrix(p1, p1 + 5, K)     # no inlier: defined as E=I, 0
    assert n == 0 and (E == np.eye(3)).all()
    R1, R2, t = tk.recover_pose_from_essential_matrix(np.eye(3, dtype=np.float32))
    assert (bits(R1) == bits(kat["pose_R1"])).all() and (bits(R2) == bits(kat["pose_R2"])).all()
    assert (bits(t) == bits(kat["pose_t"])).all()
    for A, usv in zip(kat["svd_in"][2:8], kat["svd_usv"][2:8]):
        r1, r2, tt = tk.recover_pose_from_essential_matrix(A)
        o1, o2, ot = oracle.recover_pose(A)
        assert (bits(r1) == bits(o1)).all() and (bits(r2) == bits(o2)).all() and (bits(tt) == bits(ot)).all()


def test_ransac_batch_device_pose(tracker, oracle, kat):
    import torch
    rng = np.random.default_rng(5)
    P, M = 7, 200
    pts = np.zeros((P, M, 4), np.float32)
    cnt = rng.integers(0, M, size=P).astype(np.int32)
    cnt[0] = 0
    for p in range(P):
        a = rng.integers(0, 600, size=(M, 2)).astype(np.float32)
        pts[p, :, :2] = a
        pts[p, :, 2:] = a + rng.integers(-1, 2, size=(M, 2))
    ninl, inl, pose = tracker.ransac_identity(torch.from_numpy(pts).to(tracker.device),
                                              torch.from_numpy(cnt).to(tracker.device))
    for p in range(P):
        E, ref_inl, n, _ = oracle.ransac_identity(pts[p, :cnt[p], :2], pts[p, :cnt[p], 2:], cap=M)
        assert int(ninl[p]) == n and (inl[p, :n].cpu().numpy() == ref_inl).all()
        got = pose[p].cpu().numpy()
        assert (bits(got[:9]) == bits(kat["pose_R1"].reshape(-1))).all() and (bits(got[9:]) == bits(kat["pose_t"])).all()


def test_ransac_batch_inlier_cap(tracker, oracle):
    """pnp_solver.c:107,:146,:152: the inlier array holds 1000 entries.  Pairs of 1024 points with 0, 7,
    999, 1000, 1001 and 1024 inliers, and pairs of 16384 points (BASELINE configs[4]'s match cap) with 0, 1000,
    1001, 9000 and 16384: counts and the ordered inlier lists against T2 with cap = 1000 (T2 == T1 on the
    1024-point shapes: test_ransac_cap_and_empty_cases_vs_reference)."""
    import torch
    rng = np.random.default_rng(9)
    for M, wants in ((1024, [0, 7, 999, 1000, 1001, 1024]), (16384, [0, 1000, 1001, 9000, 16384])):
        P = len(wants)
        pts = np.zeros((P, M, 4), np.float32)
        for p, k in enumerate(wants):
            a = (rng.random((M, 2)) * np.array([1241, 376])).astype(np.float32)
            inl = np.zeros(M, bool)
            inl[rng.permutation(M)[:k]] = True
            off = np.where(inl[:, None], rng.random((M, 2)) * 1.2 - 0.6, 4.0 + rng.random((M, 2)))
            pts[p, :, :2] = a
            pts[p, :, 2:] = a + off.astype(np.float32)
        cnt = np.full(P, M, np.int32)
        ninl, inl, _ = tracker.ransac_identity(torch.from_numpy(pts).to(tracker.device),
                                               torch.from_numpy(cnt).to(tracker.device))
        for p, k in enumerate(wants):
            E, ref_inl, n, _ = oracle.ransac_identity(pts[p, :, :2], pts[p, :, 2:], cap=1000)
            assert n == min(k, 1000) == int(ninl[p]), (M, k)
            assert (inl[p, :n].cpu().numpy() == ref_inl).all(), (M, k)


def test_matmul_shim(tk, kat):
    A, B = kat["mm_A"].copy(), kat["mm_B"].copy()
    C1 = kat["mm_C0"].copy()
    tk.matmul(A, B, C1, 5, 6, 6, 7, 6, 5, 0.5, 1.25)
    assert (bits(C1) == bits(kat["mm_C1"])).all()
    At, Bt = np.ascontiguousarray(A.T), np.ascontiguousarray(B.T)
    C2 = np.zeros((7, 6), np.float32)
    tk.matmul2(At, Bt, kat["mm_C0"].copy(), C2, 7, 5, 6, 6, 7, 6, 5, 1.5, -0.75, 2.0, True, True)
    assert (bits(C2) == bits(kat["mm2_C"])).all()
    # in place: D aliases C (local_bundle_adjustment.c:232-245)
    C3 = kat["mm_C0"].copy()
    tk.matmul2(At, Bt, C3, C3, 7, 5, 6, 6, 7, 6, 5, 1.5, -0.75, 2.0, True, True)
    assert (bits(C3) == bits(kat["mm2_C"])).all()


# ------------------------------------------------------------------ Gauss-Newton PnP
# lanes = 1: one thread per hypothesis (two-phase kernel for n <= 480, streaming kernel above); lanes = 32: one warp
# per hypothesis.
def _pnp_lane_forms():
    return [(1, 8), (1, 7), (32, 8)]


def _oracle_pnp(oracle, cfg, corr, n, want_hyp=True):
    """oracle.pnp_gn of every pair of corr [P, 5, stride], the pairs on threads of their own (the oracle releases the
    GIL) -> [(pose, stats, hypotheses)]."""
    import os
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(min(len(corr), os.cpu_count() or 1)) as ex:
        return list(ex.map(lambda p: oracle.pnp_gn(cfg, corr[p], n, pair_index=p, want_hyp=want_hyp), range(len(corr))))


# H = 288 spans CTAs with a partial last one in both CTA sizes: 128 + 128 + 32 (MV_PNP_GPW=1) and 256 + 32 (=2).
# n above 4096 walks the streaming kernel's staging chunks past 8 x 512; 16384 is BASELINE configs[4]'s match cap.
# The lengths around 32 (a warp), 480 (the two-phase kernel's limit), 512 and 1024 (staging chunks) sit on either side
# of a kernel boundary.
@pytest.mark.parametrize("lanes,sample_size", _pnp_lane_forms())
@pytest.mark.parametrize("n,stride", [(1000, 1024), (37, 64), (330, 1024), (480, 512), (1500, 1536), (2049, 2304), (8, 8),
                                      (4100, 4608), (6900, 16384), (16384, 16384),
                                      (1, 1), (31, 32), (32, 32), (33, 64), (479, 480), (481, 512), (511, 512),
                                      (512, 512), (513, 1024), (1023, 1024), (1024, 1024), (1025, 1536)])
def test_pnp_gn_vs_oracle(tracker, tk, oracle, synth, monkeypatch, lanes, sample_size, n, stride):
    import torch
    H, P = 288, 3
    corr = np.zeros((P, 5, stride), np.float32)
    truth = []
    for p in range(P):
        c, pose, mask = synth.synth_pnp_problem(100 + p, n, stride=stride)
        corr[p] = c
        truth.append(pose)
    cnt = np.full(P, n, np.int32)
    prm = pnp_params(H, lanes, seed=4, sample_size=sample_size)
    cfg = orc.pnp_cfg(hypotheses=H, seed=4, lanes=lanes, sample_size=sample_size)
    want = _oracle_pnp(oracle, cfg, corr, n)
    for gpw in ("1", "2"):
        monkeypatch.setenv("MV_PNP_GPW", gpw)
        pose, stats, hyp = tracker.pnp_gn(prm, torch.from_numpy(corr).to(tracker.device),
                                          torch.from_numpy(cnt).to(tracker.device), want_hyp=True)
        pose, stats, hyp = pose.cpu().numpy(), stats.cpu().numpy(), hyp.cpu().numpy()
        for p in range(P):
            rp, rs, rh = want[p]
            # Every hypothesis, bit for bit: the kernel follows the oracle operation for operation (explicit RN
            # ops, -fmad=false), so pose and inlier count of all H hypotheses are identical -- including the
            # chaotic ones that never found a consensus.  A hypothesis that diverged to NaN is NaN in both
            # (payload and sign of a NaN are not part of the contract).
            g, r = hyp[p], rh
            same = (g.view(np.int32) == r.view(np.int32)) | (np.isnan(g) & np.isnan(r))
            bad = np.nonzero(~same.all(axis=1))[0]
            assert bad.size == 0, (lanes, n, gpw, "hypotheses that differ:", bad[:8].tolist(),
                                   g[bad[:3]].tolist(), r[bad[:3]].tolist())
            # the 1e-5 rad / 1e-5 relative tolerance of BASELINE.json is therefore met with zero error;
            # kept as a statement of the contract on the hypotheses that found a consensus
            good = rh[:, 7] >= 0.3 * n
            assert good.sum() >= 1
            ang = np.array([rot_angle(hyp[p, h, :4], rh[h, :4]) for h in np.nonzero(good)[0]])
            dt = (np.linalg.norm(hyp[p, good, 4:7] - rh[good, 4:7], axis=1)
                  / np.maximum(1.0, np.linalg.norm(rh[good, 4:7], axis=1)))
            assert (ang < 1e-5).all() and (dt < 1e-5).all()
            # selected pose: tolerance stated in BASELINE.json north_star
            assert stats[p, 0] == rs[0] and stats[p, 3] == rs[3]
            assert rot_angle(pose[p, :4], rp[:4]) < 1e-5
            assert np.linalg.norm(pose[p, 4:] - rp[4:]) <= 1e-5 * max(1.0, np.linalg.norm(rp[4:]))
            if n >= 37:  # and it actually solves the problem
                assert rot_angle(pose[p, :4], truth[p][:4]) < 2e-3
                assert np.linalg.norm(pose[p, 4:] - truth[p][4:]) < 0.05


def test_pnp_gn_4096_hypotheses_vs_oracle(tracker, tk, oracle, synth):
    """BASELINE configs[4]'s K3 at its largest: 4096 hypotheses on 16384 correspondences, 32 CTAs of 128 or 16 of
    256 per pair.  The selected pose and stats against the oracle."""
    import torch
    H, n, P = 4096, 16384, 2
    corr = np.stack([synth.synth_pnp_problem(200 + p, n)[0] for p in range(P)])
    pose, stats, _ = tracker.pnp_gn(pnp_params(H, 1, seed=4), torch.from_numpy(corr).to(tracker.device),
                                    torch.full((P,), n, dtype=torch.int32, device=tracker.device))
    pose, stats = pose.cpu().numpy(), stats.cpu().numpy()
    for p, (rp, rs, _) in enumerate(_oracle_pnp(oracle, orc.pnp_cfg(hypotheses=H, seed=4, lanes=1), corr, n,
                                               want_hyp=False)):
        assert stats[p, 0] == rs[0] and stats[p, 2] == rs[2] and stats[p, 3] == rs[3], (p, stats[p], rs)
        assert abs(stats[p, 1] - rs[1]) <= 1e-5 * abs(rs[1]), (p, stats[p], rs)
        assert rot_angle(pose[p, :4], rp[:4]) < 1e-5
        assert np.linalg.norm(pose[p, 4:] - rp[4:]) <= 1e-5 * max(1.0, np.linalg.norm(rp[4:]))
        assert rs[0] >= 0.5 * n


def test_pnp_gn_empty_and_init(tracker, tk, oracle):
    import torch
    corr = torch.zeros((2, 5, 16), device=tracker.device)
    cnt = torch.zeros((2,), dtype=torch.int32, device=tracker.device)
    init = torch.tensor([[1, 0, 0, 0, 0.1, 0.2, 0.3], [1, 0, 0, 0, 0, 0, 0]], dtype=torch.float32, device=tracker.device)
    pose, stats, _ = tracker.pnp_gn(pnp_params(32, 1), corr, cnt, init_pose=init)
    assert (pose.cpu().numpy() == init.cpu().numpy()).all() and (stats.cpu().numpy()[:, 3] == 0).all()


# ------------------------------------------------------------------ whole path
# A camera with fx != fy and cx, cy off the KITTI values, with K3's gate, damping, iteration counts and sample size
# away from their defaults: the back-projection (build_corr_kernel) and K3 both take the camera from the parameters.
CAMERA_PNP = dict(fx=520.0, fy=910.0, cx=300.5, cy=260.25, gate_sq=16.0, damping=1e-3, sample_iters=3, refine_iters=6,
                  sample_size=9)


@pytest.mark.parametrize("rows,cols,N,M,mv,H,pnp", [
    pytest.param(24, 80, 100, 150, 1000, 64, {}, id="24-80-100-150-1000-64"),
    pytest.param(47, 155, 1000, 1024, 8192, 64, {}, id="47-155-1000-1024-8192-64"),
    pytest.param(47, 155, 1000, 1024, 8192, 288, CAMERA_PNP, id="camera"),
])
def test_track_sequence_vs_oracle(tracker, tk, oracle, synth, monkeypatch, rows, cols, N, M, mv, H, pnp):
    import torch
    n_frames, seed = 4, 13
    off = synth.default_offsets(n_frames, seed)
    semi, desc, depth = tracker.synth_frames(seed, rows, cols, 0, off)
    scale = torch.full((n_frames,), float(synth.SEMI_SCALE), device=tracker.device)
    p = tk.track_params(rows, cols, top_n=N, max_valid=mv, max_matches=M, hypotheses=H)
    for k, v in pnp.items():
        setattr(p.pnp, k, v)
    res = tk.results_to_numpy(tracker.track_sequence(p, semi, scale, desc, depth))
    hs, hd, hz = semi.cpu().numpy(), desc.cpu().numpy(), depth.cpu().numpy()
    # same through host buffers (the e2e entry point)
    res_h, up, down = tracker.track_sequence_host(p, hs, np.full(n_frames, synth.SEMI_SCALE, np.float32), hd, hz)
    assert res_h.tobytes() == res.tobytes() and down == 64 * (n_frames - 1)
    monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", "2")     # chunked staging must not change any result
    res_c, _, _ = tracker.track_sequence_host(p, hs, np.full(n_frames, synth.SEMI_SCALE, np.float32), hd, hz)
    assert res_c.tobytes() == res.tobytes()
    cfg = orc.TrackCfg(orc.MatchCfg(rows, cols, 4, 4, 4, M, 0.9, 0.2), orc.pnp_cfg(hypotheses=H, seed=0, lanes=1, **pnp),
                       N, mv, 10, 1.1, float(synth.SEMI_SCALE))
    for pi in range(n_frames - 1):
        ref = oracle.track_pair(cfg, pi, hs[pi], hd[pi], hz[pi], hs[pi + 1], hd[pi + 1])
        got = res[pi]
        assert got["status"] == 0 and got["num_matches"] == ref.num_matches > 0
        assert got["ransac_inliers"] == ref.ransac_inliers
        # every stage of the path is bit-exact, K3's pose and stats included
        assert got["pnp_inliers"] == ref.pnp_inliers > 0 and got["best_hypothesis"] == ref.best_h
        assert (bits(got["pnp_cost"]) == bits(np.float32(ref.pnp_cost))).all(), (pi, got["pnp_cost"], ref.pnp_cost)
        assert (bits(got["q"]) == bits(np.array(list(ref.q), np.float32))).all(), (pi, got["q"], list(ref.q))
        assert (bits(got["t"]) == bits(np.array(list(ref.t), np.float32))).all(), (pi, got["t"], list(ref.t))


def test_gpu_pose_agrees_with_cv2_on_bench_pairs(tracker, tk, synth):
    """An independent solver on the GPU's own output at the bench shape (the Gauss-Newton PnP is parity-unpinned
    by the reference, so this is the outside check of what the B200 returns, not only of the oracle): 128
    pairs of the bench sequence (47x155 cells, top-1000 queries, 1024 hypotheses).  For every pair
    cv2.solvePnP(ITERATIVE), started from nothing, on the consensus set of the GPU pose must land on the
    same pose to 3e-3 rad / 0.05 (the data's noise level: 3-px gate, ~40 % inliers, poses of ~0.05 rad /
    ~0.15; the GPU pose is 10 gated Gauss-Newton steps, cv2 the minimum on the final set) and the GPU pose's
    reprojection RMS on that set is within 25 % of cv2's optimum (measured on
    these 128 pairs with the bit-identical CPU oracle: worst 2.3e-3 rad, 0.025, 1.17x).  The records of mv_track_sequence carry
    the same pose bytes."""
    cv2 = pytest.importorskip("cv2")
    import torch
    rows, cols, n_frames = 47, 155, 129
    off = synth.default_offsets(n_frames, 0)
    semi, desc, depth = tracker.synth_frames(0, rows, cols, 0, off)
    scale = torch.full((n_frames,), float(synth.SEMI_SCALE), device=tracker.device)
    p = tk.kitti_track_params(top_n=1000, max_valid=8192, max_matches=1024, hypotheses=1024)
    res = tk.results_to_numpy(tracker.track_sequence(p, semi, scale, desc, depth))
    idx, prob, _ = tracker.softmax(semi, scale)
    qp, qi, _, qc, _ = tracker.top_n(idx, prob, 1000, 8192)
    pts, cnt, cell0, _, _ = tracker.match(p.match, desc, idx, prob, qp, qi, qc)
    cam = (p.pnp.fx, p.pnp.fy, p.pnp.cx, p.pnp.cy)
    corr = tracker.build_corr(pts, cnt, cell0, depth, cam, rows)
    pose, stats, _ = tracker.pnp_gn(p.pnp, corr, cnt)
    pose, stats, corr, cnt = pose.cpu().numpy(), stats.cpu().numpy(), corr.cpu().numpy(), cnt.cpu().numpy()
    K = np.array([[cam[0], 0, cam[2]], [0, cam[1], cam[3]], [0, 0, 1]], np.float64)

    def q2R(q):
        w, x, y, z = q
        return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                         [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                         [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])

    def project(R, t, X):
        Xc = X @ R.T + t
        return np.stack([cam[0] * Xc[:, 0] / Xc[:, 2] + cam[2], cam[1] * Xc[:, 1] / Xc[:, 2] + cam[3]], 1)

    checked = 0
    for i in range(n_frames - 1):
        assert res[i]["num_matches"] == cnt[i]
        assert np.array_equal(bits(res[i]["q"]), bits(pose[i, :4])) and np.array_equal(bits(res[i]["t"]), bits(pose[i, 4:]))
        n = int(cnt[i])
        if stats[i, 3] != 1 or stats[i, 0] < 30:
            continue
        X, z = corr[i, :3, :n].T.astype(np.float64), corr[i, 3:5, :n].T.astype(np.float64)
        R, t = q2R(pose[i, :4].astype(np.float64)), pose[i, 4:].astype(np.float64)
        cons = ((project(R, t, X) - z) ** 2).sum(1) < p.pnp.gate_sq
        assert abs(int(cons.sum()) - int(stats[i, 0])) <= 2      # float64 re-evaluation of the fp32 gate
        ok, rvec, tvec = cv2.solvePnP(X[cons], z[cons], K, None, flags=cv2.SOLVEPNP_ITERATIVE)
        assert ok
        Rcv, _ = cv2.Rodrigues(rvec)
        ang = np.arccos(np.clip((np.trace(Rcv @ R.T) - 1) / 2, -1, 1))
        assert ang < 3e-3 and np.linalg.norm(tvec.ravel() - t) < 0.05, (i, ang, tvec.ravel(), t)
        rms_gpu = np.sqrt(((project(R, t, X[cons]) - z[cons]) ** 2).sum(1).mean())
        rms_cv = np.sqrt(((project(Rcv, tvec.ravel(), X[cons]) - z[cons]) ** 2).sum(1).mean())
        assert rms_gpu <= 1.25 * rms_cv + 1e-6, (i, rms_gpu, rms_cv)
        checked += 1
    assert checked >= 100, checked


def test_track_sequence_tensor_core_matcher_same_bytes(tracker, tk, synth):
    """The tcgen05 matcher inside the whole path: byte-identical result records, many tiles per CTA."""
    import torch
    rows, cols, n_frames, seed = 47, 155, 40, 3
    off = synth.default_offsets(n_frames, seed)
    semi, desc, depth = tracker.synth_frames(seed, rows, cols, 0, off)
    scale = torch.full((n_frames,), float(synth.SEMI_SCALE), device=tracker.device)
    out = []
    for tc in (False, True):
        p = tk.track_params(rows, cols, top_n=1000, max_valid=8192, max_matches=1024, hypotheses=32,
                            use_tensor_cores=tc)
        out.append(tk.results_to_numpy(tracker.track_sequence(p, semi, scale, desc, depth)).tobytes())
    assert out[0] == out[1]


def test_track_legacy_symbol(tk, image0, kat):
    f = tk.frame_create(192, 640, 1, None, 24, 80, image0["semi_scale"], image0["semi"], image0["desc_scale"], image0["desc"])
    q, t = tk.track(f, f, 4, 4, 9, 0.9)
    assert (bits(t) == bits(kat["pose_t"])).all()
    R1 = kat["pose_R1"].astype(np.float64)
    w, x, y, z = q
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                  [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                  [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
    assert np.abs(R - R1).max() < 5e-3      # R1 comes from an approximate SVD, not exactly orthonormal
    q0, t0 = tk.track(None, f)
    assert list(q0) == [1, 0, 0, 0] and list(t0) == [0, 0, 0]


# ------------------------------------------------------------------ NMS (src/run_nms.c), SURVEY §8f rank 1
@pytest.mark.parametrize("rows,cols,permille", [(24, 80, 140), (24, 80, 1000), (47, 155, 550), (94, 310, 700),
                                                (5, 7, 900), (40, 3, 900)])
def test_nms_vs_oracle(tracker, tk, oracle, synth, rows, cols, permille):
    import torch
    frames = [synth.synth_frame(31 + f, rows, cols, f, 3 * f, -2 * f, permille)[0] for f in range(3)]
    scale = float(synth.SEMI_SCALE)
    idx = np.stack([oracle.softmax(scale, s)[0] for s in frames])
    pr = np.stack([oracle.softmax(scale, s)[1] for s in frames])
    di, dp = torch.from_numpy(idx.copy()).to(tracker.device), torch.from_numpy(pr.copy()).to(tracker.device)
    tracker.nms(rows, cols, di, dp)
    n_sup = 0
    for f in range(3):
        mi, pp, n = oracle.nms(rows, cols, idx[f], pr[f])
        n_sup += n
        assert (di[f].cpu().numpy() == mi).all() and (bits(dp[f].cpu().numpy()) == bits(pp)).all()
    assert n_sup > 0 or permille < 200
    # host-pointer form
    mi, pp, _ = oracle.nms(rows, cols, idx[0], pr[0])
    hi, hp = tk.run_nms(rows, cols, idx[0], pr[0])
    assert (hi == mi).all() and (bits(hp) == bits(pp)).all()
