"""The Gauss-Newton PnP oracle has no reference implementation to be pinned to (PARITY
UNPINNED, see oracle/mv_oracle.h).  These tests tie it to what the reference does define and to
an independent solver:
  * its residual equals the reference's compute_error_ProjectionFactor (src/projection_factor.c:
    27-33) evaluated by the reference's own code,
  * its solution agrees with cv2.solvePnP on the consensus set and with the generating pose,
  * the two summation orders (sequential / warp-butterfly) agree within the stated tolerance."""
import ctypes as C

import numpy as np
import pytest

from oracle import orc


def _angle(q1, q2):
    q1 = np.asarray(q1, np.float64); q2 = np.asarray(q2, np.float64)
    q1 = q1 / np.linalg.norm(q1); q2 = q2 / np.linalg.norm(q2)
    w = abs(float(np.dot(q1, q2)))
    v = np.array([q1[0] * q2[1] - q1[1] * q2[0] - q1[2] * q2[3] + q1[3] * q2[2],
                  q1[0] * q2[2] + q1[1] * q2[3] - q1[2] * q2[0] - q1[3] * q2[1],
                  q1[0] * q2[3] - q1[1] * q2[2] + q1[2] * q2[1] - q1[3] * q2[0]])
    return 2.0 * np.arctan2(np.linalg.norm(v), w)


def _quat_to_R(q):
    w, x, y, z = q
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def test_residual_matches_reference_projection_factor(oracle, t1_lib, t1):
    class V2(C.Structure):
        _fields_ = [("x", C.c_float), ("y", C.c_float)]

    class V3(C.Structure):
        _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]

    class Q(C.Structure):
        _fields_ = [("w", C.c_float), ("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]

    class SE3(C.Structure):
        _fields_ = [("q", Q), ("t", V3)]

    class Cam(C.Structure):
        _fields_ = [("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float)]

    class Factor(C.Structure):
        _fields_ = [("landmark", C.POINTER(V3)), ("pose", C.POINTER(SE3)), ("measurement", V2), ("error", V2),
                    ("camera", Cam)]

    rng = np.random.default_rng(0)
    cam = np.array([718.856, 718.856, 607.1928, 185.2157], np.float32)
    for _ in range(50):
        q = rng.normal(size=4); q /= np.linalg.norm(q)
        pose = np.concatenate([q, rng.normal(size=3)]).astype(np.float32)
        X = (rng.normal(size=3) * 5 + [0, 0, 20]).astype(np.float32)
        z = rng.uniform(0, 600, 2).astype(np.float32)
        lm, se3 = V3(*X), SE3(Q(*pose[:4]), V3(*pose[4:]))
        f = Factor(C.pointer(lm), C.pointer(se3), V2(*z), V2(0, 0), Cam(*cam))

        def t1_error():
            t1_lib.compute_error_ProjectionFactor(C.byref(f))
            return np.array([f.error.x, f.error.y], np.float32)
        want = t1.next("compute_error_ProjectionFactor", (pose, X, z, cam), t1_lib and t1_error)
        err = np.zeros(2, np.float32)
        oracle.lib.orc_projection_error(pose, X, z, cam, err)
        assert err[0] == want[0] and err[1] == want[1]


@pytest.mark.parametrize("seed", range(4))
def test_gn_pnp_recovers_pose_and_agrees_with_cv2(oracle, synth, seed):
    cv2 = pytest.importorskip("cv2")
    n = 600
    corr, truth, inl = synth.synth_pnp_problem(40 + seed, n, outlier_frac=0.2, noise_px=0.5)
    cfg = orc.pnp_cfg(hypotheses=64, seed=seed, lanes=1)
    pose, stats, hyp = oracle.pnp_gn(cfg, corr, n, want_hyp=True)
    assert stats[3] == 1 and stats[0] >= 0.95 * inl.sum()
    assert _angle(pose[:4], truth[:4]) < 1.5e-3 and np.linalg.norm(pose[4:] - truth[4:]) < 0.04
    # independent solver on the consensus set
    K = np.array([[cfg.fx, 0, cfg.cx], [0, cfg.fy, cfg.cy], [0, 0, 1]], np.float64)
    R = _quat_to_R(pose[:4].astype(np.float64))
    Xc = corr[:3, :n].T.astype(np.float64) @ R.T + pose[4:]
    uv = np.stack([cfg.fx * Xc[:, 0] / Xc[:, 2] + cfg.cx, cfg.fy * Xc[:, 1] / Xc[:, 2] + cfg.cy], 1)
    cons = ((uv - corr[3:5, :n].T) ** 2).sum(1) < cfg.gate_sq
    assert cons.sum() == int(stats[0])
    ok, rvec, tvec = cv2.solvePnP(corr[:3, :n].T[cons].astype(np.float64), corr[3:5, :n].T[cons].astype(np.float64),
                                  K, None, flags=cv2.SOLVEPNP_ITERATIVE)
    Rcv, _ = cv2.Rodrigues(rvec)
    dR = Rcv @ R.T
    ang = np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1))
    assert ang < 2e-4 and np.linalg.norm(tvec.ravel() - pose[4:]) < 5e-3


def test_summation_orders_agree(oracle, synth):
    n = 1000
    corr, truth, _ = synth.synth_pnp_problem(5, n, stride=1024)
    a = oracle.pnp_gn(orc.pnp_cfg(hypotheses=48, seed=2, lanes=1), corr, n)
    b = oracle.pnp_gn(orc.pnp_cfg(hypotheses=48, seed=2, lanes=32), corr, n)
    assert a[1][0] == b[1][0]
    assert _angle(a[0][:4], b[0][:4]) < 1e-5 and np.linalg.norm(a[0][4:] - b[0][4:]) < 1e-5


def test_degenerate_inputs(oracle):
    corr = np.zeros((5, 16), np.float32)
    pose, stats, _ = oracle.pnp_gn(orc.pnp_cfg(hypotheses=8), corr, 0)
    assert list(pose) == [1, 0, 0, 0, 0, 0, 0] and stats[3] == 0
    corr[2, :4] = -1.0                                    # all behind the camera: nothing to solve
    pose, stats, _ = oracle.pnp_gn(orc.pnp_cfg(hypotheses=8), corr, 4)
    assert stats[0] == 0
