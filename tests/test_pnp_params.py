"""K3 (mv_pnp_gn_batch) away from its default parameters, against orc_pnp_gn.

The other K3 tests run a KITTI camera (fx == fy) with the default gate, depth floor, damping and iteration counts.
Here every case changes one or two of them from a base with a camera whose fx, fy, cx and cy all differ, and runs
through every kernel form that can take it: the two-phase kernel (pairs of up to 480 correspondences) and the
streaming kernel (longer pairs) in one launch, the streaming kernel for every pair (MV_PNP_STREAM=1), the
one-warp-per-hypothesis form, and for H > 128 the slot kernels with 128 and 256 hypotheses per CTA and the split
launch that runs the shortest pairs as 128-hypothesis CTAs behind the main launch.  Every hypothesis record, the
selected pose and the four stats are held to the oracle bit for bit (NaN equal to NaN).

_assert_case_reaches checks, on the oracle's answer, that each case reaches what it was built for; it needs no GPU.
"""
import ctypes as C
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import orc

f32 = np.float32
FLT_MIN = float(np.finfo(f32).tiny)
CAM = (520.0, 910.0, 300.5, 260.25)          # 640 x 480 pixels
BOX = (0.0, 640.0, 0.0, 480.0)
NORM_CAM = (1.0, 1.0, 0.0, 0.0)               # normalised image coordinates of the same view
NORM_BOX = ((0 - CAM[2]) / CAM[0], (640 - CAM[2]) / CAM[0], (0 - CAM[3]) / CAM[1], (480 - CAM[3]) / CAM[1])
DEFAULTS = dict(gate_sq=9.0, min_depth=0.1, damping=1e-4, sample_iters=4, refine_iters=10, sample_size=8)


def pnp_problem(seed, n, cam=CAM, box=BOX, noise=0.5, outlier_frac=0.2, stride=None):
    """synth.synth_pnp_problem with the camera as a parameter: image points uniform in `box`, depth U[4, 40], a
    KITTI-like motion, Gaussian noise of `noise` (image units), a fraction of outliers uniform in `box`.
    -> corr float32 [5, stride] (X, Y, Z, u, v), true pose (qw, qx, qy, qz, tx, ty, tz), inlier mask."""
    fx, fy, cx, cy = cam
    rng = np.random.default_rng(seed)
    stride = stride or n
    u0 = rng.uniform(box[0], box[1], n)
    v0 = rng.uniform(box[2], box[3], n)
    d = rng.uniform(4.0, 40.0, n)
    X = np.stack([(u0 - cx) / fx * d, (v0 - cy) / fy * d, d], axis=1)
    ang = rng.normal(0, 0.01, 3)
    ang[1] += rng.normal(0, 0.02)
    t = np.array([rng.normal(0, 0.03), rng.normal(0, 0.02), -rng.uniform(0.5, 1.2)])
    th = np.linalg.norm(ang)
    ax = ang / th
    q = np.concatenate([[np.cos(th / 2)], np.sin(th / 2) * ax])
    K = np.array([[0, -ax[2], ax[1]], [ax[2], 0, -ax[0]], [-ax[1], ax[0], 0]])
    R = np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K
    Xc = X @ R.T + t
    uv = np.stack([fx * Xc[:, 0] / Xc[:, 2] + cx, fy * Xc[:, 1] / Xc[:, 2] + cy], axis=1)
    uv += rng.normal(0, noise, uv.shape)
    n_out = int(round(outlier_frac * n))
    out_idx = rng.choice(n, n_out, replace=False)
    uv[out_idx] = np.stack([rng.uniform(box[0], box[1], n_out), rng.uniform(box[2], box[3], n_out)], axis=1)
    corr = np.zeros((5, stride), f32)
    corr[0, :n], corr[1, :n], corr[2, :n] = X[:, 0], X[:, 1], X[:, 2]
    corr[3, :n], corr[4, :n] = uv[:, 0], uv[:, 1]
    mask = np.ones(n, bool)
    mask[out_idx] = False
    return corr, np.concatenate([q, t]).astype(f32), mask


# (column, value) edits of one correspondence each, spread over a good pair: every non-finite value in every plane,
# depths at and below the floor, camera-frame z at and above the 1e30 ceiling (the identity start keeps z as is), and
# |X| = 1e20, whose projection overflows.
BAD = [(0, np.nan), (1, np.nan), (2, np.nan), (3, np.nan), (4, np.nan),
       (0, np.inf), (1, -np.inf), (2, np.inf), (2, -np.inf), (3, np.inf), (4, -np.inf),
       (2, 0.0), (2, -5.0), (2, 0.1), (2, 1e30), (2, 3e30), (0, 1e20), (0, -1e20)]


def _spoil(corr, n, bad=BAD):
    """BAD at every len(BAD)+1-th correspondence, then five duplicated correspondences -> indices of the bad ones."""
    step = n // (len(bad) + 1)
    idx = []
    for i, (row, v) in enumerate(bad):
        j = (i + 1) * step
        corr[row, j] = f32(v)
        idx.append(j)
    for j in range(5):
        corr[:, 2 * j + 1] = corr[:, 2 * j]
    return idx


def _behind_pose():
    return np.array([0, 0, 1, 0, 0, 0, 0], f32)      # 180 degrees about y: every point of the problem at z < 0


BASE = dict(cam=CAM, H=288, lengths=(150, 600, 40), prm={}, init=None, first_pair=0, lanes32=True)
CASES = {
    "base": {},
    "normalised": dict(cam=NORM_CAM, prm=dict(gate_sq=1e-5)),
    "gate_0": dict(prm=dict(gate_sq=0.0)),
    "gate_0.25": dict(prm=dict(gate_sq=0.25)),
    "gate_400": dict(prm=dict(gate_sq=400.0)),
    "gate_inf": dict(prm=dict(gate_sq=np.inf)),
    "min_depth_8": dict(prm=dict(min_depth=8.0)),
    "min_depth_flt_min": dict(prm=dict(min_depth=FLT_MIN), subnormal=True),
    "damping_0": dict(prm=dict(damping=0.0)),
    "damping_1": dict(prm=dict(damping=1.0)),
    "damping_1e4": dict(prm=dict(damping=1e4)),
    "sample_iters_0": dict(prm=dict(sample_iters=0)),
    "sample_iters_1": dict(prm=dict(sample_iters=1)),
    "refine_iters_0": dict(prm=dict(refine_iters=0)),
    "refine_iters_1": dict(prm=dict(refine_iters=1)),
    "refine_iters_2": dict(prm=dict(refine_iters=2)),
    "sample_iters_0_refine_iters_1": dict(prm=dict(sample_iters=0, refine_iters=1)),
    **{"sample_size_%d" % s: dict(prm=dict(sample_size=s)) for s in (1, 6, 9, 33, 64, 65, 255)},
    **{"hypotheses_%d" % h: dict(H=h) for h in (1, 31, 33, 100, 129, 257)},
    # the last hypothesis fills the key's 16-bit hypothesis field with 0; the one-warp form is left out because the
    # oracle's lane-by-lane restatement of it takes minutes at this H
    "hypotheses_65536": dict(H=65536, lengths=(24, 40, 481), lanes32=False),
    "init_pose": dict(lengths=(150, 600, 300, 700), init=("truth", "identity", "truth_q_x2", "behind")),
    "first_pair": dict(lengths=(150, 600, 40, 300), first_pair=2 ** 24 - 2),
    "bad_correspondences": dict(lengths=(150, 600), bad=True),
    # every correspondence of a pair one point: normal equations of rank 2, which only a damping of 0 leaves singular
    "singular": dict(lengths=(60, 600, 200), prm=dict(damping=0.0), singular=True),
}


def _case(name):
    c = dict(BASE)
    c.update(CASES[name])
    c["name"] = name
    c["prm"] = dict(DEFAULTS, **c["prm"])
    cam, box, noise = c["cam"], BOX, 0.5
    if cam == NORM_CAM:
        box, noise = NORM_BOX, 0.5 / CAM[0]
    lengths = c["lengths"]
    stride = max(lengths)
    seed0 = sum(map(ord, name))
    corr = np.zeros((len(lengths), 5, stride), f32)
    truth, masks = [], []
    for p, n in enumerate(lengths):
        corr[p], pose, mask = pnp_problem(seed0 + p, n, cam, box, noise, stride=stride)
        truth.append(pose)
        masks.append(mask)
    c["bad_idx"] = []
    if c.get("bad"):
        c["bad_idx"] = [_spoil(corr[p], n) for p, n in enumerate(lengths)]
    if c.get("singular"):
        for p, n in enumerate(lengths):
            corr[p, :, :n] = corr[p, :, p:p + 1]
    if c.get("subnormal"):   # a positive depth below FLT_MIN, straight in front of the camera
        corr[0, :, 7] = [0.0, 0.0, f32(2.0 ** -127), f32(cam[2]), f32(cam[3])]
    init = None
    if c["init"]:
        init = np.zeros((len(lengths), 7), f32)
        for p, kind in enumerate(c["init"]):
            init[p] = {"truth": truth[p], "identity": np.array([1, 0, 0, 0, 0, 0, 0], f32),
                       "truth_q_x2": np.concatenate([2 * truth[p][:4], truth[p][4:]]),
                       "behind": _behind_pose()}[kind]
    c.update(corr=corr, counts=np.array(lengths, np.int32), truth=truth, masks=masks, init_pose=init)
    return c


def _cfg(c, lanes):
    pr = c["prm"]
    return orc.pnp_cfg(*c["cam"], hypotheses=c["H"], sample_size=pr["sample_size"], sample_iters=pr["sample_iters"],
                       refine_iters=pr["refine_iters"], gate_sq=pr["gate_sq"], min_depth=pr["min_depth"],
                       damping=pr["damping"], seed=5, lanes=lanes)


def _oracle(oracle, c, lanes, **over):
    """orc_pnp_gn of every pair (pair index first_pair + p, the case's init_pose), on threads -> [(pose, stats, hyp)]."""
    cfg = _cfg(c, lanes)
    for k, v in over.items():
        setattr(cfg, k, v)
    ip = c["init_pose"]

    def one(p):
        return oracle.pnp_gn(cfg, c["corr"][p], int(c["counts"][p]), pair_index=c["first_pair"] + p,
                             init_pose=None if ip is None else ip[p], want_hyp=True)
    with ThreadPoolExecutor(min(len(c["counts"]), os.cpu_count() or 1)) as ex:
        return list(ex.map(one, range(len(c["counts"]))))


def _same(a, b):
    """Bit-equal, NaN equal to NaN (payload and sign of a NaN are not part of the contract)."""
    a, b = np.asarray(a, f32), np.asarray(b, f32)
    return (a.view(np.int32) == b.view(np.int32)) | (np.isnan(a) & np.isnan(b))


def _alive(hyp):
    return hyp[:, 7] >= 0


def _assert_case_reaches(name, c, ref, oracle):
    """The case exercises what it was built for, on the oracle's (lanes 1) answer."""
    lengths = c["lengths"]
    stats = np.array([r[1] for r in ref])
    hyps = [r[2] for r in ref]
    assert min(lengths) <= 480 < max(lengths) and len(lengths) >= 2      # two-phase and streaming in one batch
    if name in ("base", "normalised", "gate_0.25", "min_depth_flt_min"):
        for p, n in enumerate(lengths):
            assert 0 < stats[p, 0] < n and stats[p, 3] == 1, (p, stats[p])
        if name in ("base", "normalised"):   # and it solves the problem
            assert (stats[:, 0] >= 0.6 * np.array(lengths)).all(), stats
    elif name == "gate_0":       # nothing is accepted: every hypothesis alive with 0 inliers, hypothesis 0 wins
        assert all((h[:, 7] == 0).all() for h in hyps)
        assert (stats == [0, 0, 0, 1]).all(), stats
    elif name == "gate_400":
        for p, n in enumerate(lengths):
            assert 0.75 * n < stats[p, 0] < n, (p, stats[p])
    elif name == "gate_inf":     # every correspondence in front of the camera is accepted
        assert (stats[:, 0] == lengths).all(), stats
    elif name == "min_depth_8":  # rejects correspondences on their depth alone
        near = 0
        for p, n in enumerate(lengths):
            zc = _camera_z(ref[p][0].astype(np.float64), c["corr"][p, :, :n].astype(np.float64))
            near_p = int((zc < 7.99).sum())
            assert stats[p, 0] <= n - near_p and stats[p, 0] > 0.3 * n, (p, near_p, stats[p])
            near += near_p
        assert near >= 0.05 * sum(lengths)
        assert stats[:, 0].sum() < sum(r[1][0] for r in _oracle(oracle, c, 1, min_depth=0.1))
    elif name.startswith("damping"):   # the damping moves the poses
        base = _oracle(oracle, c, 1, damping=1e-4)
        for p in range(len(lengths)):
            assert (~_same(hyps[p], base[p][2]).all(axis=1)).mean() > 0.9, p
    elif name.startswith("sample_iters_0"):   # no draws: every hypothesis starts and ends at the same pose
        for h in hyps:
            assert _same(h, h[:1]).all()
        assert (stats[:, 2] == 0).all()
    elif name.startswith("sample_iters") or name.startswith("refine_iters") or name.startswith("sample_size"):
        for p, h in enumerate(hyps):     # hypotheses that differ, and a consensus among them
            assert np.unique(h[:, :7], axis=0).shape[0] > 1 and stats[p, 0] > 0, (p, stats[p])
        if name.startswith("sample_size"):
            assert c["prm"]["sample_size"] != 8
    elif name.startswith("hypotheses"):
        for p, h in enumerate(hyps):
            assert h.shape[0] == c["H"] and 0 <= stats[p, 2] < c["H"] and stats[p, 3] == 1
        assert (stats[:, 0] > 0).any()
        if c["H"] == 65536:   # the last hypothesis, whose key has 0 in its hypothesis field, is a candidate
            assert any(_alive(h[-1:]).all() for h in hyps)
    elif name == "init_pose":
        assert (stats[:3, 0] > 0.5 * np.array(lengths[:3])).all(), stats
        assert not _same(hyps[2], hyps[0][:, :]).all()            # the unnormalised start is not the true one
        assert (hyps[3][:, 7] == 0).all() and (stats[3] == [0, 0, 0, 1]).all(), stats[3]
        assert _same(ref[3][0], _behind_pose()).all()
    elif name == "first_pair":   # first_pair + pair crosses the sampler's 24-bit field: the pair index wraps
        assert c["first_pair"] < 2 ** 24 <= c["first_pair"] + len(lengths) - 1
        wrapped = _oracle(oracle, dict(c, first_pair=c["first_pair"] - 2 ** 24), 1)
        for p in range(len(lengths)):
            assert _same(hyps[p], wrapped[p][2]).all()
    elif name == "bad_correspondences":
        for p in range(len(lengths)):
            n = lengths[p]
            good = np.ones(n, bool)
            good[c["bad_idx"][p]] = False
            # none of the bad ones is an inlier of the winner; some hypotheses sampled a non-finite one and carry NaN
            # or failed their solve
            pose = ref[p][0].astype(np.float64)
            assert stats[p, 0] <= good.sum() and stats[p, 0] > 0.5 * n, stats[p]
            assert np.isnan(hyps[p][:, :7]).any(axis=1).sum() > 0, p
            assert (~_alive(hyps[p])).sum() > 0, p
            assert np.isfinite(pose).all()
    elif name == "singular":     # solve6's failure branch: every hypothesis dead, none selected
        for p in range(len(lengths)):
            assert (~_alive(hyps[p])).all() and (stats[p] == [0, 0, -1, 0]).all(), (p, stats[p])
            assert _same(ref[p][0], [1, 0, 0, 0, 0, 0, 0]).all()
    else:
        raise KeyError(name)


def _camera_z(pose, corr):
    w, x, y, z = pose[:4] / np.linalg.norm(pose[:4])
    R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                  [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                  [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
    return R[2] @ corr[:3] + pose[6]


class _Refs:
    """Each case and its oracle answers (per lane form), computed once for the module."""

    def __init__(self, oracle):
        self.oracle, self.cases, self.ans = oracle, {}, {}

    def case(self, name):
        if name not in self.cases:
            self.cases[name] = _case(name)
        return self.cases[name]

    def answer(self, name, lanes):
        if (name, lanes) not in self.ans:
            self.ans[name, lanes] = _oracle(self.oracle, self.case(name), lanes)
        return self.ans[name, lanes]


@pytest.fixture(scope="module")
def refs(oracle):
    return _Refs(oracle)


@pytest.mark.parametrize("name", list(CASES))
def test_case_reaches(refs, oracle, name):
    _assert_case_reaches(name, refs.case(name), refs.answer(name, 1), oracle)


def _forms(c):
    """(label, lanes, environment) of every kernel form that takes the case."""
    out = [("two-phase+streaming", 1, {}), ("streaming", 1, {"MV_PNP_STREAM": "1"})]
    if c["lanes32"]:
        out.append(("warp", 32, {}))
    if c["H"] > 128:
        out += [("gpw1", 1, {"MV_PNP_GPW": "1"}), ("gpw2", 1, {"MV_PNP_GPW": "2"}),
                ("split", 1, {"MV_PNP_K3_SMALL_BELOW": "0"})]
    return out


def _params(c, lanes):
    from maveric_slam_b200 import lib
    p = lib.PnpParams()
    lib.load().mv_pnp_params_default(C.byref(p))
    p.fx, p.fy, p.cx, p.cy = c["cam"]
    for k, v in c["prm"].items():
        setattr(p, k, v)
    p.hypotheses, p.lanes_per_hypothesis, p.seed, p.first_pair = c["H"], lanes, 5, c["first_pair"]
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_pnp_params_vs_oracle(tracker, refs, monkeypatch, name):
    import torch
    c = refs.case(name)
    dev = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(tracker.device)  # noqa: E731
    for var in ("MV_PNP_STREAM", "MV_PNP_GPW", "MV_PNP_K3_SMALL_BELOW", "MV_PNP_TAIL_PAIRS", "MV_PNP_ORDER"):
        monkeypatch.delenv(var, raising=False)
    for label, lanes, env in _forms(c):
        want = refs.answer(name, lanes)
        with monkeypatch.context() as m:
            for k, v in env.items():
                m.setenv(k, v)
            pose, stats, hyp = tracker.pnp_gn(_params(c, lanes), dev(c["corr"]), dev(c["counts"]),
                                              init_pose=dev(c["init_pose"]), want_hyp=True)
            pose, stats, hyp = pose.cpu().numpy(), stats.cpu().numpy(), hyp.cpu().numpy()
        for p, (rp, rs, rh) in enumerate(want):
            bad = np.nonzero(~_same(hyp[p], rh).all(axis=1))[0]
            assert bad.size == 0, (label, p, "hypotheses that differ:", bad[:8].tolist(), hyp[p, bad[:2]].tolist(),
                                   rh[bad[:2]].tolist())
            assert _same(pose[p], rp).all(), (label, p, pose[p], rp)
            assert _same(stats[p], rs).all(), (label, p, stats[p], rs)


# ------------------------------------------------------------------ the depth floor's domain
BAD_FLOORS = [0.0, -1.0, float("nan"), 1e-39]


@pytest.mark.gpu
def test_min_depth_below_flt_min_is_refused(tracker, synth):
    """The kernels' reciprocal flushes a subnormal depth to 0, where the oracle's 1 / z is finite: a depth floor below
    FLT_MIN (or NaN) would let the two disagree, so mv_pnp_gn_batch and the sequence calls refuse it, before anything
    is enqueued.  FLT_MIN itself is accepted."""
    import torch
    from maveric_slam_b200 import lib, tracking
    c = _case("base")
    corr = torch.from_numpy(c["corr"]).to(tracker.device)
    cnt = torch.from_numpy(c["counts"]).to(tracker.device)
    rows, cols, n_frames = 24, 80, 3
    off = synth.default_offsets(n_frames, 1)
    semi, desc, depth = tracker.synth_frames(1, rows, cols, 0, off)
    scale = torch.full((n_frames,), float(synth.SEMI_SCALE), device=tracker.device)
    tp = tracking.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=64)
    torch.cuda.synchronize()
    for md in BAD_FLOORS:
        p = _params(c, 1)
        p.min_depth = md
        tp.pnp.min_depth = md
        before = tracker.ctx.launches
        with pytest.raises(lib.MvError, match="min_depth"):
            tracker.pnp_gn(p, corr, cnt)
        with pytest.raises(lib.MvError, match="min_depth"):
            tracker.track_sequence(tp, semi, scale, desc, depth)
        assert tracker.ctx.launches == before, md
    p = _params(c, 1)
    p.min_depth = FLT_MIN
    tp.pnp.min_depth = FLT_MIN
    tracker.pnp_gn(p, corr, cnt)
    tracker.track_sequence(tp, semi, scale, desc, depth)
    torch.cuda.synchronize()
