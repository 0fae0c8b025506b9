"""GPU parity at BASELINE.json's full sizes, through properties that do not depend on the size
(the oracle would need minutes there): determinism, equality of the kernel forms, independence of
a hypothesis from the number of hypotheses, of a pair from its shard / chunk / batch, and of the
result from the entry point (device-resident vs host buffers).  Everything goes through the C ABI.

  configs[2]  1024 hypotheses x Gauss-Newton over ~1k correspondences
  configs[3]  KITTI-00-shaped sequence (47x155 cells, ~1k keypoints, 1024 hypotheses), sharded
  configs[4]  4096 hypotheses (the 16k-keypoint matcher shape is in test_gpu_parity.py)
"""
import ctypes as C

import numpy as np
import pytest

from helpers import pinned, pnp_params, pnp_problems

pytestmark = pytest.mark.gpu

ROWS, COLS = 47, 155


@pytest.fixture(scope="module")
def tk(tracker):
    from maveric_slam_b200 import tracking
    return tracking


@pytest.mark.parametrize("n,stride", [(1000, 1024), (330, 1024), (480, 480), (481, 512), (513, 640), (31, 32), (3, 1024)])
def test_pnp_forms_return_identical_bytes(tracker, synth, monkeypatch, n, stride):
    """configs[2]: the product's two one-thread-per-hypothesis kernels -- the two-phase kernel (gate every
    slot, re-deal by exact count, packed-FFMA2 walk; pairs of up to 480 correspondences) and the streaming
    kernel (larger pairs; MV_PNP_STREAM=1 forces it for every pair) -- with 128 or 256 hypotheses per CTA:
    same bytes for every one of 1024 hypotheses and for the selected pose."""
    import torch
    P, H = 3, 1024
    corr = torch.from_numpy(pnp_problems(synth, P, n, stride)).to(tracker.device)
    cnt = torch.full((P,), n, dtype=torch.int32, device=tracker.device)

    def run():
        pose, stats, hyp = tracker.pnp_gn(pnp_params(H), corr, cnt, want_hyp=True)
        return (pose.cpu().numpy().tobytes(), stats.cpu().numpy().tobytes(), hyp.cpu().numpy().tobytes())

    want = run()
    for gpw in ("1", "2"):
        with monkeypatch.context() as m:
            m.setenv("MV_PNP_GPW", gpw)
            assert run() == want, ("two-phase", gpw)
            m.setenv("MV_PNP_STREAM", "1")
            assert run() == want, ("streaming", gpw)


def test_pnp_split_launch_returns_identical_bytes(tracker, synth, monkeypatch):
    """How K3 cuts a batch into CTAs does not change a byte: 128-hypothesis CTAs for every pair (short
    launches), 256-hypothesis CTAs for every pair, or the split launch (the shortest pairs of the
    longest-first order as 128-hypothesis CTAs in a programmatic dependent launch) -- on a batch whose pairs differ in
    length, with empty pairs and pairs long enough for the streaming kernel."""
    import torch
    P, stride, H = 11, 1024, 1024
    counts = [330, 5, 0, 480, 600, 17, 330, 1000, 128, 3, 250]
    corr = torch.from_numpy(pnp_problems(synth, P, 1000, stride)).to(tracker.device)
    cnt = torch.tensor(counts, dtype=torch.int32, device=tracker.device)

    def run():
        pose, stats, hyp = tracker.pnp_gn(pnp_params(H), corr, cnt, want_hyp=True)
        return (pose.cpu().numpy().tobytes(), stats.cpu().numpy().tobytes(), hyp.cpu().numpy().tobytes())

    want = run()                                   # 11 pairs: every pair as 128-hypothesis CTAs
    monkeypatch.setenv("MV_PNP_K3_SMALL_BELOW", "0")   # never the short-launch form
    assert run() == want, "split launch, 5 tail pairs"
    for tail in ("0", "1", "3"):
        with monkeypatch.context() as m:
            m.setenv("MV_PNP_TAIL_PAIRS", tail)
            assert run() == want, ("tail pairs", tail)


@pytest.mark.parametrize("lanes", [0, 2, 3, 4, 8, 16, 64])
def test_pnp_refuses_lanes_without_a_kernel(tracker, synth, lanes):
    """lanes_per_hypothesis is 1 (one thread per hypothesis) or 32 (one warp): any other value is
    MV_ERR_BAD_ARG from mv_pnp_gn_batch before anything is launched."""
    import torch
    from maveric_slam_b200 import lib
    P, n, stride = 2, 100, 128
    corr = torch.from_numpy(pnp_problems(synth, P, n, stride)).to(tracker.device)
    cnt = torch.full((P,), n, dtype=torch.int32, device=tracker.device)
    pose = torch.zeros((P, 7), dtype=torch.float32, device=tracker.device)
    stats = torch.zeros((P, 4), dtype=torch.float32, device=tracker.device)
    launches = tracker.ctx.launches
    st = tracker.lib.mv_pnp_gn_batch(tracker.ctx.h, C.byref(pnp_params(64, lanes=lanes)), P, stride,
                                     tracker._d(corr), tracker._d(cnt), None, tracker._d(pose), tracker._d(stats),
                                     None)
    assert st == lib.MV_ERR_BAD_ARG, (lanes, st)
    assert tracker.ctx.launches == launches, lanes


def test_pnp_hypothesis_does_not_depend_on_hypothesis_count(tracker, synth):
    """configs[4]: 4096 hypotheses.  Hypothesis h is a function of (seed, pair, h) alone, so the first
    1024 of a 4096-hypothesis run are the 1024-hypothesis run, bit for bit, and the selected pose is
    the best key (inliers, then cost, then index) over the per-hypothesis records."""
    import torch
    P, n, stride = 2, 1000, 1024
    corr = torch.from_numpy(pnp_problems(synth, P, n, stride)).to(tracker.device)
    cnt = torch.full((P,), n, dtype=torch.int32, device=tracker.device)
    pose4, stats4, hyp4 = tracker.pnp_gn(pnp_params(4096), corr, cnt, want_hyp=True)
    pose1, stats1, hyp1 = tracker.pnp_gn(pnp_params(1024), corr, cnt, want_hyp=True)
    hyp4, hyp1 = hyp4.cpu().numpy(), hyp1.cpu().numpy()
    assert hyp4[:, :1024].tobytes() == hyp1.tobytes()
    stats4, pose4 = stats4.cpu().numpy(), pose4.cpu().numpy()
    for p in range(P):
        inl = hyp4[p, :, 7]
        best = inl.max()
        assert stats4[p, 0] == best and stats4[p, 3] == 1
        h = int(stats4[p, 2])
        assert inl[h] == best and (pose4[p] == hyp4[p, h, :7]).all()
        # a 4096-hypothesis search cannot end below the 1024-hypothesis one
        assert best >= stats1.cpu().numpy()[p, 0]


def test_pnp_pair_does_not_depend_on_batch(tracker, synth):
    """A pair's result depends on its global pair index only: a batch of 6 equals two batches of 3
    with first_pair = 0 and 3 (what sharding across GPUs and chunked staging rely on)."""
    import torch
    P, n, stride, H = 6, 700, 1024, 512
    corr = torch.from_numpy(pnp_problems(synth, P, n, stride)).to(tracker.device)
    cnt = torch.full((P,), n, dtype=torch.int32, device=tracker.device)
    pose, stats, _ = tracker.pnp_gn(pnp_params(H), corr, cnt)
    parts = []
    for first in (0, 3):
        prm = pnp_params(H)
        prm.first_pair = first
        pp, ss, _ = tracker.pnp_gn(prm, corr[first:first + 3].contiguous(), cnt[first:first + 3].contiguous())
        parts.append((pp.cpu().numpy(), ss.cpu().numpy()))
    assert np.concatenate([a for a, _ in parts]).tobytes() == pose.cpu().numpy().tobytes()
    assert np.concatenate([b for _, b in parts]).tobytes() == stats.cpu().numpy().tobytes()


def test_pnp_ragged_counts_and_work_counter(tracker, synth):
    """Pairs of one launch with 0, 1, 8, 511, 512, 513 and 1024 correspondences (empty, below the
    minimal sample, around the staging chunk of 512, full): each equals its own single-pair launch;
    the profile-mode work counter never exceeds hypotheses x correspondences x passes."""
    import torch
    counts = [0, 1, 8, 511, 512, 513, 1024]
    stride, H = 1024, 256
    corr = np.zeros((len(counts), 5, stride), np.float32)
    for p, n in enumerate(counts):
        if n:
            corr[p, :, :n] = synth.synth_pnp_problem(900 + p, n, stride=n)[0]
    dcorr = torch.from_numpy(corr).to(tracker.device)
    dcnt = torch.tensor(counts, dtype=torch.int32, device=tracker.device)
    tracker.ctx.profile(True)
    tracker.ctx.pnp_work()
    pose, stats, hyp = tracker.pnp_gn(pnp_params(H), dcorr, dcnt, want_hyp=True)
    work = tracker.ctx.pnp_work()
    tracker.ctx.profile(False)
    assert 0 < work <= H * sum(counts) * 10
    pose, stats = pose.cpu().numpy(), stats.cpu().numpy()
    assert stats[0, 3] == 0 and (pose[0] == np.array([1, 0, 0, 0, 0, 0, 0], np.float32)).all()
    for p, n in enumerate(counts):
        prm = pnp_params(H)
        prm.first_pair = p
        p1, s1, _ = tracker.pnp_gn(prm, dcorr[p:p + 1].contiguous(), dcnt[p:p + 1].contiguous())
        assert p1.cpu().numpy().tobytes() == pose[p:p + 1].tobytes(), n
        assert s1.cpu().numpy().tobytes() == stats[p:p + 1].tobytes(), n


def test_sequence_full_config_properties(tracker, tk, synth, monkeypatch):
    """configs[3] at its real parameters (47x155 cells, top-1000 queries, 1024 matches, 1024
    hypotheses), 97 frames: two runs are identical (determinism); two shards with one halo frame
    and first_pair = 0 / 48 reproduce the unsharded records (multi-GPU sharding); the host-buffer
    entry point, unchunked and in chunks of 7 pairs, returns the same bytes (e2e path); both
    matchers agree."""
    import torch
    n_frames, seed = 97, 0
    off = synth.default_offsets(n_frames, seed)
    semi, desc, depth = tracker.synth_frames(seed, ROWS, COLS, 0, off)
    scale = torch.full((n_frames,), float(synth.SEMI_SCALE), device=tracker.device)

    def params(first=0, tc=True):
        return tk.kitti_track_params(top_n=1000, max_valid=8192, max_matches=1024, hypotheses=1024, refine_iters=10,
                                     sample_iters=4, seed=0, first_pair=first, lanes=1, use_tensor_cores=tc)

    full = tracker.track_sequence(params(), semi, scale, desc, depth).cpu().numpy()
    again = tracker.track_sequence(params(), semi, scale, desc, depth).cpu().numpy()
    assert full.tobytes() == again.tobytes()
    res = tk.results_to_numpy(torch.from_numpy(full))
    assert (res["status"] == 0).all() and (res["num_matches"] > 100).all() and (res["pnp_inliers"] > 20).all()

    a = tracker.track_sequence(params(0), semi[:49], scale[:49], desc[:49], depth[:49]).cpu().numpy()
    b = tracker.track_sequence(params(48), semi[48:], scale[48:], desc[48:], depth[48:]).cpu().numpy()
    assert np.concatenate([a, b]).tobytes() == full.tobytes()

    dp4a = tracker.track_sequence(params(tc=False), semi, scale, desc, depth).cpu().numpy()
    assert dp4a.tobytes() == full.tobytes()

    hs, hsc, hd, hz = (pinned(t) for t in (semi, scale, desc, depth))
    torch.cuda.synchronize()
    host, up, down = tracker.track_sequence_host(params(), hs, hsc, hd, hz)
    assert host.tobytes() == full.tobytes() and down == 64 * (n_frames - 1)
    # selective staging moves the logits, the depth and only the descriptor rows the matcher reads
    assert up < semi.numel() + 4 * depth.numel() + desc.numel() // 2
    # the chunk size of the staging pipeline must not change a byte (7: a last chunk of 5 pairs; 40: 40 + 40 + 16)
    for chunk_pairs in ("7", "40"):
        monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", chunk_pairs)
        chunked, _, _ = tracker.track_sequence_host(params(), hs, hsc, hd, hz)
        assert chunked.tobytes() == full.tobytes(), chunk_pairs


def test_trajectory_chain_is_associative(tracker, tk):
    """Pose chaining (compute_trajectory.py:76-77: R_k ... R_1, t_1 + ... + t_k) over 4540
    transforms, the length of configs[3]: chaining the whole list equals chaining its second half
    on top of the last pose of its first half."""
    import torch
    rng = np.random.default_rng(5)
    n, cut = 4540, 2000
    T = np.zeros((n, 3, 4))
    for i in range(n):
        w = rng.normal(size=3) * 0.01
        th = np.linalg.norm(w)
        k = w / th
        K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
        T[i, :, :3] = np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K
        T[i, :, 3] = rng.normal(size=3) * 0.5

    def chain(x):
        return tracker.chain_transforms(torch.from_numpy(np.ascontiguousarray(x)).to(tracker.device)).cpu().numpy()

    whole, first, second = chain(T), chain(T[:cut]), chain(T[cut:])
    assert whole.shape == (n + 1, 3, 4) and (whole[0] == np.eye(4)[:3]).all()
    assert np.abs(whole[:cut + 1] - first).max() < 1e-11
    R = second[:, :, :3] @ first[-1, :, :3]
    t = second[:, :, 3] + first[-1, :, 3]
    assert np.abs(whole[cut:, :, :3] - R).max() < 1e-11
    assert np.abs(whole[cut:, :, 3] - t).max() < 1e-9 * max(1.0, np.abs(t).max())


# ------------------------------------------------------------------ edge cases of the whole path
def _oracle_seq(oracle, orc, synth, hs, hd, hz, rows, cols, N, M, mv, H):
    cfg = orc.TrackCfg(orc.MatchCfg(rows, cols, 4, 4, 4, M, 0.9, 0.2), orc.pnp_cfg(hypotheses=H, seed=0, lanes=1),
                       N, mv, 10, 1.1, float(synth.SEMI_SCALE))
    return [oracle.track_pair(cfg, p, hs[p], hd[p], hz[p], hs[p + 1], hd[p + 1]) for p in range(hs.shape[0] - 1)]


def test_sequence_with_empty_and_degenerate_frames(tracker, tk, oracle, synth):
    """A sequence whose frames 2 and 3 have no keypoint at all (every logit negative), whose frame 5
    has every descriptor saturated at -128 (maximal wrap-around of the score products) and whose
    frame 7 has all-zero descriptors (the zero-norm rule of squared_dist): pairs without queries,
    without candidates and without matches return the identity pose and zero counts, everything
    else equals the oracle; the host-buffer path returns the same bytes."""
    import torch
    from oracle import orc
    rows, cols, n_frames, seed = 24, 80, 9, 2
    N, M, mv, H = 100, 150, 1000, 64
    off = synth.default_offsets(n_frames, seed)
    semi, desc, depth = tracker.synth_frames(seed, rows, cols, 0, off)
    semi[2:4] = -5
    desc[5] = -128
    desc[7] = 0
    scale = torch.full((n_frames,), float(synth.SEMI_SCALE), device=tracker.device)
    p = tk.track_params(rows, cols, top_n=N, max_valid=mv, max_matches=M, hypotheses=H)
    res = tk.results_to_numpy(tracker.track_sequence(p, semi, scale, desc, depth))
    hs, hd, hz = semi.cpu().numpy(), desc.cpu().numpy(), depth.cpu().numpy()
    ref = _oracle_seq(oracle, orc, synth, hs, hd, hz, rows, cols, N, M, mv, H)
    for pi, r in enumerate(ref):
        got = res[pi]
        assert got["status"] == 0
        assert got["num_matches"] == r.num_matches, pi
        assert got["ransac_inliers"] == r.ransac_inliers, pi
        assert got["pnp_inliers"] == r.pnp_inliers, pi
        assert np.allclose(got["q"], list(r.q), atol=1e-5) and np.allclose(got["t"], list(r.t), atol=1e-4), pi
    # pairs (1,2): no candidates; (2,3): neither; (3,4): no queries... all without a match
    for pi in (1, 2, 3):
        assert res[pi]["num_matches"] == 0 and res[pi]["pnp_inliers"] == 0
        assert list(res[pi]["q"]) == [1, 0, 0, 0] and list(res[pi]["t"]) == [0, 0, 0]
    assert res[0]["num_matches"] > 0
    host, _, _ = tracker.track_sequence_host(p, hs, np.full(n_frames, synth.SEMI_SCALE, np.float32), hd, hz)
    assert host.tobytes() == res.tobytes()


def test_two_frame_sequence_and_single_pair_batches(tracker, tk, oracle, synth):
    """The smallest sequence (one pair) through both entry points, at the KITTI grid."""
    import torch
    from oracle import orc
    rows, cols, seed = 47, 155, 9
    N, M, mv, H = 1000, 1024, 8192, 32
    off = synth.default_offsets(2, seed)
    semi, desc, depth = tracker.synth_frames(seed, rows, cols, 0, off)
    scale = torch.full((2,), float(synth.SEMI_SCALE), device=tracker.device)
    p = tk.track_params(rows, cols, top_n=N, max_valid=mv, max_matches=M, hypotheses=H)
    res = tk.results_to_numpy(tracker.track_sequence(p, semi, scale, desc, depth))
    hs, hd, hz = semi.cpu().numpy(), desc.cpu().numpy(), depth.cpu().numpy()
    r = _oracle_seq(oracle, orc, synth, hs, hd, hz, rows, cols, N, M, mv, H)[0]
    assert res.shape == (1,) and res[0]["num_matches"] == r.num_matches > 100
    assert res[0]["pnp_inliers"] == r.pnp_inliers
    host, up, down = tracker.track_sequence_host(p, hs, np.full(2, synth.SEMI_SCALE, np.float32), hd, hz)
    assert host.tobytes() == res.tobytes() and down == 64


def test_sequence_calls_reject_nonpositive_sizes(tracker, tk, synth):
    """Status codes instead of the reference's undefined behaviour: a non-positive grid, query count or
    match capacity, a negative match radius and PnP parameters mv_pnp_gn_batch refuses are MV_ERR_BAD_ARG from
    both sequence entry points, before anything is allocated or launched."""
    import torch
    from maveric_slam_b200 import lib
    rows, cols = 24, 80
    off = synth.default_offsets(2, 1)
    semi, desc, depth = tracker.synth_frames(1, rows, cols, 0, off)
    scale = torch.full((2,), float(synth.SEMI_SCALE), device=tracker.device)
    hs, hd, hz = semi.cpu().numpy(), desc.cpu().numpy(), depth.cpu().numpy()
    hsc = np.full(2, synth.SEMI_SCALE, np.float32)

    def broken(**kw):
        p = tk.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=32)
        for k, v in kw.items():
            if k in ("rows", "cols", "max_matches", "radius"):
                setattr(p.match, k, v)
            elif k in ("lanes_per_hypothesis", "hypotheses", "sample_size"):
                setattr(p.pnp, k, v)
            else:
                setattr(p, k, v)
        return p

    want = tracker.track_sequence(broken(), semi, scale, desc, depth).cpu().numpy().tobytes()
    for kw in ({"rows": 0}, {"cols": -3}, {"top_n": 0}, {"max_valid": 0}, {"max_matches": 0},
               {"lanes_per_hypothesis": 4}, {"hypotheses": 0}, {"sample_size": 0}, {"radius": -1}):
        launches = tracker.ctx.launches
        with pytest.raises(lib.MvError, match="bad argument"):
            tracker.track_sequence(broken(**kw), semi, scale, desc, depth)
        with pytest.raises(lib.MvError, match="bad argument"):
            tracker.track_sequence_host(broken(**kw), hs, hsc, hd, hz)
        assert tracker.ctx.launches == launches, kw
    # and the context is still usable afterwards, with the same answer
    res = tk.results_to_numpy(tracker.track_sequence(broken(), semi, scale, desc, depth))
    assert res.shape == (1,) and res.tobytes() == want
    assert tracker.track_sequence_host(broken(), hs, hsc, hd, hz)[0].tobytes() == want


def test_contexts_of_two_gpus_from_one_thread(synth):
    """The device contract of maveric_b200.h: every entry point makes its context's GPU current for the call
    and restores the caller's.  Two contexts on two GPUs used alternately from this one thread, with the
    thread's current device left on GPU 0 throughout, return the bytes a single-GPU run returns."""
    import torch
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from maveric_slam_b200 import tracking
    rows, cols, n_frames = 24, 80, 5
    off = synth.default_offsets(n_frames, 3)
    outs = []
    trackers = [tracking.Tracker(0), tracking.Tracker(1)]
    torch.cuda.set_device(0)
    p = tracking.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=64)
    data = []
    for tr in trackers:
        with torch.cuda.device(tr.device):
            data.append(tr.synth_frames(3, rows, cols, 0, off))
    torch.cuda.set_device(0)
    for rep in range(2):
        for tr, (semi, desc, depth) in zip(trackers, data):
            scale = torch.full((n_frames,), float(synth.SEMI_SCALE), device=tr.device)
            assert torch.cuda.current_device() == 0
            res = tr.track_sequence(p, semi, scale, desc, depth)
            assert torch.cuda.current_device() == 0
            tr.ctx.sync()
            outs.append(res.cpu().numpy().tobytes())
    assert len(set(outs)) == 1


def test_matchers_agree_on_random_shapes(tracker, synth):
    """Differential test of the compacted tcgen05 matcher against the dp4a kernel (itself held to the oracle shape by
    shape in test_gpu_parity.py) on 24 random configurations: odd grids (1-row, 1-column, 255 rows), windows of
    radius 0 ... larger than the grid, shifts that push windows off the grid, query counts around the 128-query
    tile and the match cap, densities from a handful of candidates to every cell, batches in which some frames have
    no keypoint at all, and explicit (f0, f1) pair lists that reuse frames.  Matches, counts, cells, queries and
    score bits must be identical."""
    import torch
    from maveric_slam_b200 import tracking
    rng = np.random.default_rng(77)
    for trial in range(24):
        rows = int(rng.choice([1, 2, 3, 7, 24, 47, 64, 255]))
        cols = int(rng.choice([1, 2, 5, 33, 80, 155])) if rows > 3 else int(rng.choice([40, 200, 700]))
        cells = rows * cols
        permille = int(rng.choice([5, 60, 140, 550, 1000]))
        N = int(rng.choice([1, 7, 127, 128, 129, 300, 1000]))
        M = int(rng.choice([1, 16, 150, 1024]))
        radius = int(rng.choice([0, 1, 4, 9, 40]))
        shift = (int(rng.integers(-6, 7)), int(rng.integers(-6, 7)))
        n_frames = int(rng.integers(2, 6))
        off = synth.default_offsets(n_frames, 100 + trial)
        semi, desc, _ = tracker.synth_frames(100 + trial, rows, cols, 0, off, keypoint_permille=permille)
        if trial % 4 == 1:
            semi[int(rng.integers(0, n_frames))] = -100          # a frame without keypoints
        scale = torch.full((n_frames,), float(synth.SEMI_SCALE), device=tracker.device)
        idx, prob, _ = tracker.softmax(semi, scale)
        qp, qi, _, qc, _ = tracker.top_n(idx, prob, N, cells + 1)
        f0 = f1 = None
        if trial % 3 == 2:                                       # explicit pairs, frames reused, a frame with itself
            pairs = [(int(rng.integers(0, n_frames)), int(rng.integers(0, n_frames))) for _ in range(5)]
            f0 = torch.tensor([a for a, _ in pairs], dtype=torch.int32, device=tracker.device)
            f1 = torch.tensor([b for _, b in pairs], dtype=torch.int32, device=tracker.device)
        outs = []
        for tc in (False, True):
            p = tracking.match_params(rows, cols, shift[0], shift[1], radius, M, use_tensor_cores=tc)
            res = tracker.match(p, desc, idx, prob, qp, qi, qc, f0=f0, f1=f1)
            cnt = res[1].cpu().numpy()
            rec = [cnt.tobytes()]
            for t in (res[0], res[2], res[3], res[4]):            # points, cell0, query, score: the first cnt entries
                a = t.cpu().numpy()
                rec.append(b"".join(a[i, :cnt[i]].tobytes() for i in range(len(cnt))))
            outs.append(rec)
        assert outs[0] == outs[1], (trial, rows, cols, permille, N, M, radius, shift)
