"""Every scalar legacy symbol libmaveric_b200.so exports (csrc/api.cu: pnp_solver.h helpers, the nine
types.c functions, the projection factor) called THROUGH the product library and compared bit for bit
with the reference's own code (T1 = oracle/_ref/libmaveric_ref.so, compiled unmodified from
src/pnp_solver.c:28-34,36-86,89-105, src/types.c:3-73, src/projection_factor.c:4-33).

These symbols are host code in the reference and host code in the product library, so the comparison
needs no GPU; it closes SURVEY §8 rows a12-a15 at the ABI (before this file they were only checked to
exist)."""
import ctypes as C

import numpy as np
import pytest


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


def _declare(L):
    f32 = C.c_float
    L.add_Vector2f.argtypes, L.add_Vector2f.restype = [V2, V2, f32], V2
    L.add_Vector3f.argtypes, L.add_Vector3f.restype = [V3, V3, f32], V3
    L.mult_Quaternionf.argtypes, L.mult_Quaternionf.restype = [Q, Q], Q
    L.create_Quaternionf.argtypes, L.create_Quaternionf.restype = [f32] * 4, Q
    L.Quaternionf_from_Vector3f.argtypes, L.Quaternionf_from_Vector3f.restype = [V3], Q
    L.conjugate_Quaternionf.argtypes, L.conjugate_Quaternionf.restype = [Q], Q
    L.Vector3f_from_Quaternionf.argtypes, L.Vector3f_from_Quaternionf.restype = [Q], V3
    L.apply_rotation.argtypes, L.apply_rotation.restype = [Q, V3], V3
    L.apply_transform.argtypes, L.apply_transform.restype = [SE3, V3], V3
    L.project2d.argtypes, L.project2d.restype = [V3], V2
    L.cam_project.argtypes, L.cam_project.restype = [V3, Cam], V2
    L.create_ProjectionFactor.argtypes = [C.POINTER(V3), C.POINTER(SE3), V2, Cam]
    L.create_ProjectionFactor.restype = C.POINTER(Factor)
    L.compute_error_ProjectionFactor.argtypes, L.compute_error_ProjectionFactor.restype = [C.POINTER(Factor)], None
    fp = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
    L.normalize_points.argtypes, L.normalize_points.restype = [C.c_int, fp, fp, fp], None
    L.compute_essential_matrix.argtypes, L.compute_essential_matrix.restype = [C.c_int, fp, fp, fp], None
    L.compute_reprojection_error.argtypes, L.compute_reprojection_error.restype = [fp, fp, fp], C.c_float
    return L


def _b(s):
    """bytes of a ctypes struct / float: the comparison is on bit patterns (-0.0 != +0.0, NaN == NaN)"""
    return bytes(s) if isinstance(s, C.Structure) else np.float32(s).tobytes()


@pytest.fixture(scope="module")
def libs(t1_lib):
    """(product, T1); T1 is None where oracle/_ref is not built: its stored answers are used (tests/conftest.py)."""
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib
    # a private handle so the argtypes above do not clash with lib.load()'s void* declarations
    prod = _declare(C.CDLL(lib.SO_PATH))
    lib.load()   # fails loudly if the product library is not built
    ref = None if t1_lib is None else _declare(C.CDLL(t1_lib._name))
    return prod, ref


def _floats(rng, n, special):
    v = rng.normal(size=n).astype(np.float32) * np.float32(10.0 ** rng.integers(-3, 4))
    if special:
        pool = np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, np.nan, 1e-38, 3e38, 1e-45], np.float32)
        m = rng.random(n) < 0.3
        v[m] = pool[rng.integers(0, len(pool), m.sum())]
    return [float(x) for x in v]


@pytest.mark.parametrize("special", [False, True])
def test_types_c_functions_bit_equal(libs, t1, special):
    """types.c:3-73 -- add_Vector2f/3f, mult_/create_/conjugate_Quaternionf, the two conversions,
    apply_rotation, apply_transform; 400 random argument sets, with and without zeros/infs/NaNs/denormals."""
    prod, ref = libs
    rng = np.random.default_rng(11 + special)
    calls = []
    for _ in range(400):
        f = _floats(rng, 16, special)
        a2, b2 = V2(*f[0:2]), V2(*f[2:4])
        a3, b3 = V3(*f[0:3]), V3(*f[3:6])
        qa, qb = Q(*f[6:10]), Q(*f[10:14])
        s = f[14]
        T = SE3(qa, b3)
        calls += [("add_Vector2f", (a2, b2, s)), ("add_Vector3f", (a3, b3, s)),
                  ("mult_Quaternionf", (qa, qb)), ("create_Quaternionf", tuple(f[6:10])),
                  ("Quaternionf_from_Vector3f", (a3,)), ("conjugate_Quaternionf", (qa,)),
                  ("Vector3f_from_Quaternionf", (qa,)), ("apply_rotation", (qa, a3)),
                  ("apply_transform", (T, a3))]

    def results(L):
        """SHA-256 of every call's result bytes, in order; where special, NaNs canonicalised (NaN payloads
        are not part of the contract)"""
        import hashlib
        h = hashlib.sha256()
        for name, args in calls:
            r = np.frombuffer(_b(getattr(L, name)(*args)), np.float32).copy()
            if special:
                r[np.isnan(r)] = np.float32(np.nan)
            h.update(r.tobytes())
        return h.hexdigest()
    assert results(prod) == t1.next("types.c", [x for _, args in calls for x in args],
                                    None if ref is None else lambda: results(ref))


def test_projection_factor_functions_bit_equal(libs, t1):
    """projection_factor.c:4-33 -- create_ProjectionFactor (field copies, caller frees), project2d,
    cam_project, compute_error_ProjectionFactor, through the product library vs T1."""
    prod, ref = libs
    libc = C.CDLL(None)
    libc.free.argtypes = [C.c_void_p]
    rng = np.random.default_rng(5)
    cam = Cam(718.856, 718.856, 607.1928, 185.2157)
    for i in range(300):
        q = rng.normal(size=4); q /= np.linalg.norm(q)
        pose = SE3(Q(*[float(np.float32(v)) for v in q]), V3(*[float(np.float32(v)) for v in rng.normal(size=3)]))
        X = V3(*[float(np.float32(v)) for v in rng.normal(size=3) * 5 + [0, 0, 20 if i % 7 else 0]])
        z = V2(*[float(np.float32(v)) for v in rng.uniform(0, 1241, 2)])

        def factor_error(L):
            lm, se = V3(X.x, X.y, X.z), SE3(pose.q, pose.t)
            fp = L.create_ProjectionFactor(C.pointer(lm), C.pointer(se), z, cam)
            f = fp.contents
            assert C.addressof(f.landmark.contents) == C.addressof(lm) and C.addressof(f.pose.contents) == C.addressof(se)
            assert _b(f.measurement) == _b(z) and _b(f.camera) == _b(cam)
            L.compute_error_ProjectionFactor(fp)
            err = _b(f.error)
            libc.free(fp)
            return err
        want = t1.next("projection_factor.c", (X, pose, z, cam), None if ref is None else
                       lambda: (_b(ref.project2d(X)), _b(ref.cam_project(X, cam)), factor_error(ref)))
        assert (_b(prod.project2d(X)), _b(prod.cam_project(X, cam)), factor_error(prod)) == want


def test_pnp_solver_scalar_helpers_bit_equal(libs, t1):
    """pnp_solver.c:28-34 normalize_points, :36-86 compute_essential_matrix (the 8-point system is built and
    dropped: E = I for every input), :89-105 compute_reprojection_error -- product library vs T1."""
    prod, ref = libs
    rng = np.random.default_rng(8)
    for trial in range(20):
        n = int(rng.integers(8, 300))
        pts = (rng.random((n, 2)) * np.array([1241, 376])).astype(np.float32)
        pts2 = (pts + rng.normal(size=(n, 2)).astype(np.float32)).astype(np.float32)
        K = np.array([[718.856 + trial, 0, 607.1928], [0, 718.856 - trial, 185.2157], [0, 0, 1]], np.float32)
        a = np.zeros((n, 2), np.float32)
        prod.normalize_points(n, pts, K, a)

        def ref_normalize():
            b = np.zeros((n, 2), np.float32)
            ref.normalize_points(n, pts, K, b)
            return b
        b = t1.next("normalize_points", (n, pts, K), None if ref is None else ref_normalize)
        assert a.tobytes() == b.tobytes()
        a2 = np.zeros((n, 2), np.float32)
        prod.normalize_points(n, pts2, K, a2)
        E1 = np.full((3, 3), 7.0, np.float32)
        prod.compute_essential_matrix(n, a, a2, E1)

        def ref_essential():
            E2 = np.full((3, 3), 7.0, np.float32)
            ref.compute_essential_matrix(n, a, a2, E2)
            return E2
        E2 = t1.next("compute_essential_matrix", (n, a, a2), None if ref is None else ref_essential)
        assert E1.tobytes() == E2.tobytes() == np.eye(3, dtype=np.float32).tobytes()
        # reprojection error under I and under a general E (the function is defined for any E)
        for E in (E1, rng.normal(size=(3, 3)).astype(np.float32)):
            def errors(L):
                return b"".join(_b(L.compute_reprojection_error(pts[i].copy(), pts2[i].copy(), np.ascontiguousarray(E)))
                                for i in range(min(n, 40)))
            assert errors(prod) == t1.next("compute_reprojection_error", (pts, pts2, E),
                                           None if ref is None else lambda: errors(ref))
