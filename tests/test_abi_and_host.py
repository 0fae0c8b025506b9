"""CPU-side checks: the C-ABI library loads and exports every symbol its headers declare, it
refuses to run without a GPU (no fallback), the host-side local feature pool behaves like the
reference's, the numpy generator equals the C one, and the product never touches oracle/."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from helpers import InsertResult, LocalFeature, Pool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions(header):
    text = open(os.path.join(ROOT, "include", header)).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"//[^\n]*", "", text)
    text = re.sub(r"#[^\n]*", "", text)
    text = re.sub(r"typedef\s+(struct|enum)[^{;]*\{.*?\}\s*\w+\s*;", "", text, flags=re.S)
    names = set()
    for m in re.finditer(r"\b([A-Za-z_]\w*)\s*\(([^;{}()]|\([^)]*\))*\)\s*;", text):
        names.add(m.group(1))
    return names - {"defined"}


def test_library_exports_every_declared_symbol():
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib
    L = lib.load()
    new = declared_functions("maveric_b200.h")
    legacy = declared_functions("maveric_slam_compat.h")
    assert "mv_track_sequence_host" in new and "mv_pnp_gn_batch" in new and len(new) >= 24
    assert {"compute_top_N", "compute_softmax", "ransac_essential_matrix", "track", "matmul", "matmul2",
            "local_feature_pool_insert", "frame_create", "recover_pose_from_essential_matrix"} <= legacy
    missing = [s for s in sorted(new | legacy) if not hasattr(L, s)]
    assert not missing, missing
    assert set(lib.NEW_SYMBOLS) <= new and set(lib.LEGACY_SYMBOLS) <= legacy


def test_pnp_has_ab_forms_is_zero():
    # kept exported so that existing callers link; the library has no other PnP kernel forms
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib
    assert lib.load().mv_pnp_has_ab_forms() == 0


def test_forwarding_headers_compile_as_c99(tmp_path):
    # a reference-style C caller: the reference's include names, C99, no C++
    src = tmp_path / "caller.c"
    src.write_text('#include "frame.h"\n#include "pnp_solver.h"\n#include "top_N.h"\n#include "tracking.h"\n'
                   '#include "local_feature_pool.h"\n#include "gemmini_functions_cpu.h"\n#include "projection_factor.h"\n'
                   '#include "maveric_b200.h"\n'
                   'int use(void){ Frame f; SE3 T; frame_create(192,640,1,0,24,80,0.3f,0,4.3f,0,&f);'
                   ' track(0,&f,4,4,9,0.9f,&T); return (int)sizeof(LocalFeaturePool) + (int)sizeof(mv_pair_result); }\n')
    r = subprocess.run(["/usr/bin/gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c",
                        str(src), "-o", str(tmp_path / "caller.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib
    with pytest.raises(lib.MvError, match="no usable CUDA device"):
        lib.Context(0)


def test_product_does_not_reference_oracle():
    pkg = os.path.join(ROOT, "maveric-slam_b200")
    for dp, _, files in os.walk(pkg):
        if "build" in dp.split(os.sep):
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                text = open(os.path.join(dp, f)).read()
                assert "mv_oracle" not in text and "import oracle" not in text and "from oracle" not in text, f


def test_numpy_generator_equals_c_generator(oracle, synth):
    for seed, rows, cols, f, ox, oy, pm in [(0, 24, 80, 0, 0, 0, 140), (7, 47, 155, 9, 36, 41, 140),
                                             (3, 5, 7, 100, -50, 1000, 550)]:
        a = synth.synth_frame(seed, rows, cols, f, ox, oy, pm)
        b = oracle.synth_frame(seed, rows, cols, f, ox, oy, pm)
        assert all((x == y).all() for x, y in zip(a, b))
    off = synth.default_offsets(50, 3)
    d = np.diff(off, axis=0)
    assert (d >= 2).all() and (d <= 6).all()          # true displacement stays inside the r=4 window


# ---------------------------------------------------------------- local feature pool (host side)
def _drive_pool(L, frames=60, per_frame=200, seed=0):
    """The churn of src/local_feature_matching.c:129-170: per frame insert-or-update ids, age out,
    check the invariant.  Returns a trace of (size, occupied slots)."""
    L.local_feature_pool_insert.restype = InsertResult
    L.local_feature_pool_insert.argtypes = [C.POINTER(Pool), C.c_int, LocalFeature]
    L.local_feature_pool_load_factor.restype = C.c_float
    pool = Pool()
    L.init_local_feature_pool(C.byref(pool))
    rng = np.random.default_rng(seed)
    prev = rng.choice(5000, per_frame, replace=False)
    trace = []
    for f in range(frames):
        keep = rng.choice(prev, 75, replace=False)
        fresh = rng.choice(np.setdiff1d(np.arange(5000), keep), per_frame - 75, replace=False)
        ids = np.concatenate([keep, fresh])
        for wid in ids:
            feat = LocalFeature()
            L.init_local_feature_with_id(C.byref(feat), int(wid), f)
            res = L.local_feature_pool_insert(C.byref(pool), int(wid), feat)
            if not res.inserted:
                L.update_local_feature(res.feature, f)
        L.local_feature_pool_remove_old(C.byref(pool), f)
        L.local_feature_pool_check_invariant(C.byref(pool), f, False)
        occ = [(i, e.key, e.value.frame_ptr, e.value.num_frames) for i, e in enumerate(pool.entries) if e.is_occupied]
        trace.append((pool.size, tuple(occ), float(L.local_feature_pool_load_factor(C.byref(pool)))))
        prev = ids
    return trace


def _trace_digest(trace):
    import hashlib
    return hashlib.sha256(repr(trace).encode()).hexdigest()


def test_local_feature_pool_matches_reference(t1_lib, t1):
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import lib
    ours = _drive_pool(lib.load())
    # the stored answer is a digest of T1's trace (the trace itself is 0.4 MB)
    theirs = t1.next("_drive_pool", (), t1_lib and (lambda: _trace_digest(_drive_pool(t1_lib))))
    assert _trace_digest(ours) == theirs
    assert ours[-1][0] > 0
