"""Writes tests/golden/ref_t1_<module>.xz: the answers of the reference's own code (T1) to every call the
tests make to it, in call order (see T1Answers in tests/conftest.py).

    python tests/golden/make_golden_t1.py

Where oracle/_ref is built (oracle/Makefile, from the reference's sources), the answers are T1's own.
Without it they come from StandInReference below: the restatement (oracle/mv_oracle.c, T2) and the
product library's host functions.  The files in the repository were recorded that way, at a commit
whose oracle/, tests/ and library sources are byte-identical to those of the commit at which these
same tests, on these same inputs, passed live against T1 (bit-exact asserts).  Wherever T1 is built, the
tests still call it and check it against these files.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

MODULES = ["test_oracle_vs_ref", "test_lba", "test_bow", "test_oracle_pnp", "test_abi_and_host",
           "test_legacy_scalar_symbols"]


def product_host_library():
    """A private handle of libmaveric_b200.so: its legacy host symbols were held bit-equal to T1's."""
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib
    lib.load()
    return C.CDLL(lib.SO_PATH)


class _StandInLib:
    def __init__(self, o):
        self.o = o

    def compute_reprojection_error(self, p1, p2, E):
        return float(self.o.lib.orc_reproj_error(p1, p2, E))


class StandInReference:
    """orc.Reference's methods, answered by the restatement."""

    def __init__(self):
        from oracle import orc
        self.orc, self.o = orc, orc.Oracle()
        self.lib = _StandInLib(self.o)

    def softmax(self, scale, semi):
        return self.o.softmax(scale, semi)

    def top_n(self, scale, semi, N):
        return self.o.top_n(scale, semi, N)[:3]

    def tracking_main(self, semi_scale0, semi0, desc0, semi_scale1, semi1, desc1):
        idx, pr, _ = self.o.softmax(semi_scale0, semi0)
        pa, ix, _, _ = self.o.top_n(semi_scale1, semi1, 100)
        m = self.o.match(self.orc.MatchCfg(24, 80, 4, 4, 4, 150, 0.9, 0.2), desc0, desc1, idx, pr, pa, ix)
        E, inl, ni, _ = self.o.ransac_identity(m["pts0"], m["pts1"])
        return dict(n=m["n"], pts0=m["pts0"], pts1=m["pts1"], num_inliers=ni, inliers=inl, best_E=E)

    def ransac(self, pts1, pts2, K, iters=10, thr=1.1):
        E, inl, ni, wrote = self.o.ransac_identity(pts1, pts2, iters, thr)
        if not wrote:   # the reference writes nothing: the caller's zeros and -1 stay
            return np.zeros((3, 3), np.float32), np.zeros(0, np.int32), -1
        return E, inl, ni

    def svd3(self, A):
        return self.o.svd3(A)

    def run_nms(self, semi_scale1, semi1):
        idx, pr, _ = self.o.softmax(float(semi_scale1), semi1)
        mi, _, _, ev = self.o.nms(24, 80, idx, pr, want_events=True)
        cells = np.nonzero(mi != 64)[0]
        kp = np.stack([(cells // 24) * 8 + mi[cells] % 8, (cells % 24) * 8 + mi[cells] // 8], axis=1)
        return ev, kp.astype(np.int32)

    def lba_run(self, flat=None):
        return self.o.lba_schur(self.orc.lba_reference_factors(flat), 4)

    def invert_3x3(self, m, stride=3):
        return self.o.invert_3x3(m, stride)


class StandInReferenceBow:
    """orc.ReferenceBow's helper functions, answered by the restatement."""

    def __init__(self):
        from oracle import orc
        self.o = orc.Oracle()

    def get_binary_descriptor(self, scale, feature_int32, size=8):
        return self.o.bow_binarize(scale, np.asarray(feature_int32).astype(np.int8))

    def count_matching_bits(self, a, b):
        return self.o.bow_matching_bits(a, b)


if __name__ == "__main__":
    env = dict(os.environ, MV_RECORD_T1="1")
    files = [os.path.join(ROOT, "tests", m + ".py") for m in MODULES]
    sys.exit(subprocess.run([sys.executable, "-m", "pytest", "-q", "-m", "not gpu", *files], cwd=ROOT, env=env).returncode)
