"""Local bundle adjustment, Schur complement of the landmarks (src/local_bundle_adjustment.c:133-246,
SURVEY §8f rank 4).

  T1  the reference program itself (oracle/_ref): its main() on its own input -- whose result is NaN
      in all 48 x 48 pose entries, the 3 x 3 landmark blocks it builds being singular -- and on
      substituted inputs that stay finite; the matrix it passes to cholesky() is the answer.
  T2  the parametrised restatement (oracle/mv_oracle.c) == T1 bit for bit, == the golden file.
  GPU mv_lba_schur_batch == T2 / the golden file bit for bit (NaNs compared as NaNs).

The solve of the reduced system (the reference's cholesky() is a stub, :88-90,247) is this
repository's definition, PARITY UNPINNED: the restatement is checked against a float64 solve and
the GPU kernel against the restatement bit for bit.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from helpers import same_bits, spd_system
from oracle import orc


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(os.path.join(GOLDEN, "ref_lba.npz")))


def _flat(golden, k):
    return None if k == 0 else golden["flat"][k]


def test_oracle_equals_golden(oracle, golden):
    for k in range(golden["C"].shape[0]):
        J = orc.lba_reference_factors(_flat(golden, k))
        assert same_bits(oracle.lba_schur(J, 4), golden["C"][k]), k
    # the reference's own input: every pose entry NaN, the gradient row finite
    c0 = golden["C"][0]
    assert np.isnan(c0[:48, :48]).all() and np.isfinite(c0[:48, 48]).all() and (c0[48] == 0).all()
    for m, inv in zip(golden["inv_in"], golden["inv_out"]):
        assert oracle.invert_3x3(m).tobytes() == inv.tobytes()


def test_oracle_equals_reference(oracle, reference):
    rng = np.random.default_rng(7)
    for k in range(6):
        flat = None if k == 0 else (rng.normal(size=640) * (1.0 if k < 4 else 100.0)).astype(np.float32)
        assert same_bits(oracle.lba_schur(orc.lba_reference_factors(flat), 4), reference.lba_run(flat)), k
    for _ in range(100):
        m = rng.normal(size=(3, 3)).astype(np.float32)
        assert oracle.invert_3x3(m).tobytes() == reference.invert_3x3(m).tobytes()


def test_oracle_solves_a_real_window(oracle):
    """With Jacobians of full rank the restatement is the textbook reduced camera system:
    C = H_PP - H_PL H_LL^-1 H_LP and the gradient row g_P - H_PL H_LL^-1 g_L (float64 check)."""
    rng = np.random.default_rng(3)
    L, P = 40, 3
    J = rng.normal(size=(L, P, 20)).astype(np.float32)
    C = oracle.lba_schur(J, 4).astype(np.float64)
    Hpp = np.zeros((6 * P + 1, 6 * P + 1))
    S = np.zeros((6 * P + 1, 6 * P + 1))
    for l in range(L):
        Hll = np.zeros((3, 3)); Hpl = np.zeros((6 * P + 1, 3))
        for p in range(P):
            Jf = J[l, p].astype(np.float64).reshape(10, 2).T       # 2 x 10
            H = Jf.T @ Jf
            Hll += H[:3, :3]
            Hpl[6 * p:6 * p + 6] += H[3:9, :3]
            Hpl[6 * P] += H[9, :3]
            Hpp[6 * p:6 * p + 6, 6 * p:6 * p + 6] += H[3:9, 3:9]
            Hpp[6 * P, 6 * p:6 * p + 6] += H[9, 3:9]
        S += Hpl @ np.linalg.inv(Hll) @ Hpl.T
    want = Hpp.copy()
    want[:6 * P, :6 * P] -= S[:6 * P, :6 * P]
    got = C.T                                                      # column-major storage
    scale = np.abs(want).max()
    assert np.abs(got[:6 * P, :6 * P] - want[:6 * P, :6 * P]).max() < 2e-3 * scale
    assert np.abs(got[6 * P, :6 * P] - want[6 * P, :6 * P]).max() < 1e-4 * scale   # gradient row: no Schur term


def test_oracle_solve_against_float64(oracle):
    rng = np.random.default_rng(5)
    for P in (1, 2, 5, 8, 11, 16):
        C, S, g = spd_system(rng, P)
        ok, d = oracle.lba_solve(C, 0.0)
        want = np.linalg.solve(S.astype(np.float64), -g.astype(np.float64))
        assert ok == 1 and np.abs(d - want).max() < 1e-4 * np.abs(want).max(), P
        # only the lower triangle is read
        C2 = C.copy()
        iu = np.triu_indices(6 * P, 1)
        C2[:6 * P, :6 * P].T[iu] = 77.0
        assert oracle.lba_solve(C2, 0.0)[1].tobytes() == d.tobytes()
        # damping = Levenberg-Marquardt scaling of the diagonal
        ok, dd = oracle.lba_solve(C, 0.5)
        Sd = S.astype(np.float64) + 0.5 * np.diag(np.diag(S).astype(np.float64))
        want = np.linalg.solve(Sd, -g.astype(np.float64))
        assert ok == 1 and np.abs(dd - want).max() < 1e-4 * np.abs(want).max(), P


def test_oracle_solve_rejects_what_is_not_positive_definite(oracle, golden):
    rng = np.random.default_rng(6)
    C, S, g = spd_system(rng, 3)
    C[4, 4] = -1.0
    ok, d = oracle.lba_solve(C, 0.0)
    assert ok == 0 and not d.any()
    # the reference's own input: every pose entry is NaN
    ok, d = oracle.lba_solve(golden["C"][0], 0.0)
    assert ok == 0 and not d.any()
    # one pose, 6 x 6: the PnP solve's definition (ascending back substitution differs in order only)
    C, S, g = spd_system(rng, 1)
    ok, d = oracle.lba_solve(C, 1e-3)
    want = np.linalg.solve(S.astype(np.float64) * (np.eye(6) * 1e-3 + 1), -g.astype(np.float64))
    assert ok == 1 and np.abs(d - want).max() < 1e-5 * np.abs(want).max()


# --------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_gpu_equals_golden_and_oracle(tracker, oracle, golden):
    import torch
    # the reference's shape (1000 landmarks, 8 poses, chunks of 4), its own input and substituted ones
    J = np.stack([orc.lba_reference_factors(_flat(golden, k)) for k in range(golden["C"].shape[0])])
    C = tracker.lba_schur(torch.from_numpy(J).to(tracker.device), 4).cpu().numpy()
    for k in range(J.shape[0]):
        assert same_bits(C[k], golden["C"][k]), k
    # general factors, other shapes (ragged against the thread count), incl. huge and zero entries
    rng = np.random.default_rng(11)
    for (L, P, ch, amp) in [(1000, 8, 4, 1.0), (12, 1, 4, 1.0), (64, 3, 2, 1.0), (96, 16, 8, 1.0), (40, 8, 1, 1.0),
                            (48, 5, 16, 1.0), (200, 8, 4, 1e18), (200, 8, 4, 0.0)]:
        Jb = (rng.normal(size=(3, L, P, 20)) * amp).astype(np.float32)
        got = tracker.lba_schur(torch.from_numpy(Jb).to(tracker.device), ch).cpu().numpy()
        for w in range(3):
            assert same_bits(got[w], oracle.lba_schur(Jb[w], ch)), (L, P, ch, amp, w)


@pytest.mark.gpu
def test_gpu_kernel_forms_return_identical_bytes(tracker, oracle):
    """Both Schur kernels equal the oracle bit for bit on the same edge inputs: the specialised one at
    the reference shape (8 poses, chunks of 4) and the generic one at 7 poses, chunks of 4."""
    import torch
    for P in (8, 7):
        rng = np.random.default_rng(12)
        J = rng.normal(size=(5, 200, P, 20)).astype(np.float32)
        J[3, 17] = 0.0                       # zero products: the factor chain of the shim becomes serial
        J[4, 5, 2, 7] = np.inf
        got = tracker.lba_schur(torch.from_numpy(J).to(tracker.device), 4).cpu().numpy()
        for w in range(J.shape[0]):
            assert same_bits(got[w], oracle.lba_schur(J[w], 4)), (P, w)


@pytest.mark.gpu
def test_gpu_window_is_independent_of_the_batch(tracker):
    """Full size: 296 windows of 1000 landmarks x 8 poses in one launch; each equals its own launch."""
    import torch
    g = torch.Generator(device="cpu").manual_seed(5)
    J = torch.randn((296, 1000, 8, 20), generator=g).to(tracker.device)
    C = tracker.lba_schur(J, 4)
    assert torch.isfinite(C).all()
    for w in (0, 147, 295):
        one = tracker.lba_schur(J[w:w + 1].contiguous(), 4)
        assert one.cpu().numpy().tobytes() == C[w:w + 1].cpu().numpy().tobytes()
    again = tracker.lba_schur(J, 4)
    assert again.cpu().numpy().tobytes() == C.cpu().numpy().tobytes()


@pytest.mark.gpu
def test_gpu_solve_equals_oracle(tracker, oracle, golden):
    """mv_lba_solve_batch == the restatement bit for bit: every pose count the library takes, well
    and badly conditioned systems, damping, and the systems that must be refused."""
    import torch
    rng = np.random.default_rng(21)
    for P in (1, 2, 3, 5, 6, 8, 11, 16):
        Cs = []
        for w in range(9):
            C, _, _ = spd_system(rng, P, cond=(1.0, 30.0, 1000.0)[w % 3])
            if w == 4:
                C[2 * P, 2 * P] = -abs(C[2 * P, 2 * P])          # a negative pivot in the middle
            if w == 7:
                C[0, P] = np.nan                                  # column 0, row P: lower triangle
            Cs.append(C)
        Cs = np.stack(Cs)
        for damping in (0.0, 1e-3):
            d, ok = tracker.lba_solve(torch.from_numpy(Cs).to(tracker.device), damping)
            d, ok = d.cpu().numpy(), ok.cpu().numpy()
            for w in range(Cs.shape[0]):
                ok_o, d_o = oracle.lba_solve(Cs[w], damping)
                assert ok[w] == ok_o and same_bits(d[w], d_o), (P, w, damping)
            assert ok[4] == 0 and ok[7] == 0 and ok[0] == 1
    # Schur complement -> step, end to end on the device at the reference's shape; its own input is refused
    J = np.stack([orc.lba_reference_factors(_flat(golden, k)) for k in range(golden["C"].shape[0])])
    Cd = tracker.lba_schur(torch.from_numpy(J).to(tracker.device), 4)
    d, ok = tracker.lba_solve(Cd, 1e-3)
    d, ok = d.cpu().numpy(), ok.cpu().numpy()
    assert ok[0] == 0 and not d[0].any()
    for k in range(J.shape[0]):
        ok_o, d_o = oracle.lba_solve(golden["C"][k], 1e-3)
        assert ok[k] == ok_o and same_bits(d[k], d_o), k


@pytest.mark.gpu
def test_gpu_solve_full_batch_and_residual(tracker):
    """2 368 windows of 8 poses in one launch: each equals its own launch, and the step solves its
    system (float64 residual)."""
    import torch
    rng = np.random.default_rng(22)
    base = np.stack([spd_system(rng, 8)[0] for _ in range(37)])
    Cs = torch.from_numpy(np.tile(base, (64, 1, 1))).to(tracker.device)
    d, ok = tracker.lba_solve(Cs, 0.0)
    assert int(ok.sum()) == Cs.shape[0]
    dn = d.cpu().numpy()
    assert dn[:37].tobytes() == dn[37 * 63:].tobytes()
    for w in (0, 36, 1000, 2367):
        one, _ = tracker.lba_solve(Cs[w:w + 1].contiguous(), 0.0)
        assert one.cpu().numpy().tobytes() == dn[w:w + 1].tobytes()
        S = base[w % 37][:48, :48].T.astype(np.float64)
        S = np.tril(S) + np.tril(S, -1).T
        g = base[w % 37][:48, 48].astype(np.float64)
        assert np.abs(S @ dn[w].astype(np.float64) + g).max() < 1e-3 * np.abs(g).max()


@pytest.mark.gpu
def test_gpu_rejects_bad_shapes(tracker):
    import torch
    J = torch.zeros((1, 10, 2, 20), device=tracker.device)
    with pytest.raises(Exception):
        tracker.lba_schur(J, 4)          # 10 landmarks are not a multiple of 4
    with pytest.raises(Exception):
        tracker.lba_solve(torch.zeros((1, 103, 103), device=tracker.device))   # 17 poses
