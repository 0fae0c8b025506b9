"""ctypes bindings of the CPU checkers (TEST INFRASTRUCTURE ONLY).

``T2``  = oracle/libmv_oracle.so, this repository's restatement (oracle/mv_oracle.c).
``T1``  = oracle/_ref/libmaveric_ref.so, the reference's own sources compiled unmodified
          from /root/reference by oracle/Makefile (prebuilt file travels to the GPU box).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_i8p = np.ctypeslib.ndpointer(np.int8, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")


def build(force: bool = False) -> None:
    need = force or not os.path.exists(os.path.join(_HERE, "libmv_oracle.so")) \
        or os.path.getmtime(os.path.join(_HERE, "libmv_oracle.so")) < os.path.getmtime(os.path.join(_HERE, "mv_oracle.c"))
    if need or (os.path.isdir("/root/reference/src") and not os.path.exists(os.path.join(_HERE, "_ref", "libmaveric_ref.so"))):
        subprocess.run(["make", "-C", _HERE, "all"], check=True, capture_output=True)


def _cpu_model() -> str:
    """CPU model name + a checksum of its ISA flag set (what -march=native keys on)."""
    import zlib
    name, flags = "unknown", ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and name == "unknown":
                name = line.split(":", 1)[1].strip()
            elif line.startswith("flags") and not flags:
                flags = line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "%s | %08x" % (name, zlib.crc32(flags.encode()))


def build_fast(out_dir: str | None = None) -> str:
    """libmv_oracle_fast.so is compiled -march=native, so it must be built on the CPU that runs it:
    a sidecar file records the build host's CPU model + flag set and the library is rebuilt when
    they differ.  __graft_entry__.build() builds it in oracle/ (out_dir = oracle/); at run time the
    tree's copy is used when it fits this CPU, else a copy under the temporary directory, so that a
    read-only tree still runs.  Returns the path of the library to load."""
    import atexit
    import shutil
    import tempfile
    here = _cpu_model()
    src_mtime = max(os.path.getmtime(os.path.join(_HERE, f)) for f in ("mv_oracle.c", "mv_oracle.h"))

    def state(d):
        so, tag = os.path.join(d, "libmv_oracle_fast.so"), os.path.join(d, "libmv_oracle_fast.host")
        fresh = os.path.exists(so) and os.path.getmtime(so) >= src_mtime
        return so, tag, fresh, fresh and os.path.exists(tag) and open(tag).read().strip() == here

    if out_dir is None:
        so, _, _, ok = state(_HERE)
        if ok:
            return so
        # a fresh private directory (mode 0700), removed at exit: nothing another user placed is loaded
        out_dir = tempfile.mkdtemp(prefix="mv_oracle_fast-")
        atexit.register(shutil.rmtree, out_dir, True)
    so, tag, fresh, ok = state(out_dir)
    if not ok:
        # -B: an up-to-date file built for another CPU is rebuilt all the same
        subprocess.run(["make", "-C", _HERE] + (["-B"] if fresh else []) + ["FAST_SO=" + so, so],
                       check=True, capture_output=True)
        with open(tag, "w") as f:
            f.write(here)
    return so


class MatchCfg(C.Structure):
    _fields_ = [("rows", C.c_int), ("cols", C.c_int), ("shift_x", C.c_int), ("shift_y", C.c_int),
                ("radius", C.c_int), ("max_matches", C.c_int),
                ("match_threshold", C.c_double), ("min_prob0", C.c_double)]


class MatchStats(C.Structure):
    _fields_ = [("window_cells", C.c_longlong), ("pairs_256", C.c_longlong), ("pairs_64", C.c_longlong)]


class PnpCfg(C.Structure):
    _fields_ = [("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
                ("hypotheses", C.c_int), ("sample_size", C.c_int), ("sample_iters", C.c_int),
                ("refine_iters", C.c_int), ("gate_sq", C.c_float), ("min_depth", C.c_float),
                ("damping", C.c_float), ("seed", C.c_uint64), ("lanes", C.c_int)]


class SynthCfg(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("rows", C.c_int), ("cols", C.c_int),
                ("keypoint_permille", C.c_int), ("noise_amp", C.c_int)]


class TrackCfg(C.Structure):
    _fields_ = [("match", MatchCfg), ("pnp", PnpCfg), ("top_n", C.c_int), ("max_valid", C.c_int),
                ("ransac_iters", C.c_int), ("ransac_thr", C.c_float), ("semi_scale", C.c_float)]


class PairResult(C.Structure):
    _fields_ = [("q", C.c_float * 4), ("t", C.c_float * 3), ("pnp_inliers", C.c_float),
                ("pnp_cost", C.c_float), ("num_matches", C.c_int), ("ransac_inliers", C.c_int),
                ("best_h", C.c_int), ("status", C.c_int)]


def pnp_cfg(fx=718.856, fy=718.856, cx=607.1928, cy=185.2157, hypotheses=64, sample_size=8,
            sample_iters=4, refine_iters=10, gate_sq=9.0, min_depth=0.1, damping=1e-4, seed=0, lanes=1):
    return PnpCfg(fx, fy, cx, cy, hypotheses, sample_size, sample_iters, refine_iters,
                  gate_sq, min_depth, damping, seed, lanes)


class BowVocab(C.Structure):
    _fields_ = [("n_base", C.c_int), ("words_per_base", C.c_int), ("base_desc", C.c_void_p), ("scale", C.c_void_p),
                ("bias", C.c_void_p), ("leaves", C.c_void_p)]


LOCAL_FEATURE_DTYPE = np.dtype([("word_id", "<i4"), ("frame_ptr", "<i4"), ("num_frames", "<i4"), ("frames", "<i4", (8,)),
                                ("coords", "<f4", (3,))])
assert LOCAL_FEATURE_DTYPE.itemsize == 56   # include/local_feature_pool.h:16-22


class Oracle:
    """T2: the parametrised restatement."""

    def __init__(self, fast: bool = False):
        build()
        self.lib = C.CDLL(build_fast() if fast else os.path.join(_HERE, "libmv_oracle.so"))
        L = self.lib
        L.orc_softmax.restype = C.c_int
        L.orc_softmax.argtypes = [C.c_float, _i8p, C.c_int, _i32p, _f32p]
        L.orc_nms.restype = C.c_int
        L.orc_nms.argtypes = [C.c_int, C.c_int, _i32p, _f32p, C.c_void_p, C.c_int]
        L.orc_top_n.restype = C.c_int
        L.orc_top_n.argtypes = [C.c_float, _i8p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), _i32p, _i32p, _f32p]
        L.orc_match.restype = C.c_int
        L.orc_match.argtypes = [C.POINTER(MatchCfg), _i8p, _i8p, _i32p, _f32p, C.c_int, _i32p, _i32p,
                                _f32p, _f32p, _i32p, _i32p, _f32p, C.POINTER(MatchStats)]
        L.orc_svd3.argtypes = [_f32p, _f32p, _f32p, _f32p]
        L.orc_reproj_error.restype = C.c_float
        L.orc_reproj_error.argtypes = [_f32p, _f32p, _f32p]
        L.orc_normalize_points.argtypes = [C.c_int, _f32p, _f32p, _f32p]
        L.orc_ransac_identity.restype = C.c_int
        L.orc_ransac_identity.argtypes = [C.c_int, _f32p, _f32p, C.c_int, C.c_float, C.c_int, _f32p, _i32p,
                                          C.POINTER(C.c_int)]
        L.orc_recover_pose.argtypes = [_f32p, _f32p, _f32p, _f32p]
        L.orc_quat_mul.argtypes = [_f32p, _f32p, _f32p]
        L.orc_apply_transform.argtypes = [_f32p, _f32p, _f32p]
        L.orc_projection_error.argtypes = [_f32p, _f32p, _f32p, _f32p, _f32p]
        L.orc_matmul.argtypes = [C.c_size_t] * 3 + [_f32p, _f32p, _f32p] + [C.c_size_t] * 3 + [C.c_float] * 2 + [C.c_int] * 2
        L.orc_matmul2.argtypes = [C.c_size_t] * 3 + [_f32p, _f32p, C.c_void_p, _f32p] + [C.c_size_t] * 4 + [C.c_float] * 3 + [C.c_int] * 2
        L.orc_invert_3x3.argtypes = [_f32p, C.c_int]
        L.orc_lba_schur.argtypes = [C.c_int, C.c_int, C.c_int, _f32p, _f32p]
        L.orc_lba_solve.restype = C.c_int
        L.orc_lba_solve.argtypes = [C.c_int, C.c_float, _f32p, _f32p]
        L.orc_pnp_gn.argtypes = [C.POINTER(PnpCfg), C.c_int, C.c_int, C.c_int, _f32p, C.c_void_p, _f32p, _f32p, C.c_void_p]
        L.orc_synth_frame.argtypes = [C.POINTER(SynthCfg), C.c_int, C.c_int, C.c_int, _i8p, _i8p, _f32p]
        L.orc_track_pair.argtypes = [C.POINTER(TrackCfg), C.c_int, _i8p, _i8p, _f32p, _i8p, _i8p, C.POINTER(PairResult)]
        L.orc_bow_binarize.argtypes = [C.c_float, _i8p, _i32p]
        L.orc_bow_matching_bits.restype = C.c_int
        L.orc_bow_matching_bits.argtypes = [_i32p, _i32p, C.c_int]
        L.orc_bow_assign.argtypes = [C.POINTER(BowVocab), C.c_float, _i8p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.orc_pool_observe.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _i32p, C.c_void_p]
        L.orc_pool_remove_old.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.orc_bench_sequence.restype = C.c_double
        L.orc_bench_sequence.argtypes = [C.POINTER(TrackCfg), C.POINTER(SynthCfg), _i32p, C.c_int, C.c_int, C.c_int,
                                         C.POINTER(PairResult)]

    # -- detector
    def softmax(self, scale, semi):
        semi = np.ascontiguousarray(semi, np.int8)
        cells = semi.shape[0]
        idx = np.zeros(cells, np.int32)
        pr = np.zeros(cells, np.float32)
        nv = self.lib.orc_softmax(float(scale), semi, cells, idx, pr)
        return idx, pr, nv

    def nms(self, rows, cols, max_idx, probs, want_events=False):
        """src/run_nms.c:65-156 on copies of (max_idx, probs) -> (max_idx, probs, n_suppressed[, events])."""
        mi = np.ascontiguousarray(max_idx, np.int32).copy(); pr = np.ascontiguousarray(probs, np.float32).copy()
        cap = rows * cols
        ev = np.zeros((cap, 4), np.int32)
        n = self.lib.orc_nms(rows, cols, mi, pr, ev.ctypes.data, cap)
        return (mi, pr, n, ev[:n].copy()) if want_events else (mi, pr, n)

    def top_n(self, scale, semi, N, max_valid=1000):
        semi = np.ascontiguousarray(semi, np.int8)
        pa = np.zeros(N, np.int32); ix = np.zeros(N, np.int32); pr = np.zeros(N, np.float32)
        n = C.c_int(0)
        ov = self.lib.orc_top_n(float(scale), semi, semi.shape[0], N, max_valid, C.byref(n), pa, ix, pr)
        return pa[:n.value].copy(), ix[:n.value].copy(), pr[:n.value].copy(), ov

    # -- matcher
    def match(self, cfg: MatchCfg, desc0, desc1, max_idx0, probs0, patches1, indices1):
        M = cfg.max_matches
        p0 = np.zeros((M, 2), np.float32); p1 = np.zeros((M, 2), np.float32)
        c0 = np.zeros(M, np.int32); qq = np.zeros(M, np.int32); sc = np.zeros(M, np.float32)
        st = MatchStats()
        patches1 = np.ascontiguousarray(patches1, np.int32)
        indices1 = np.ascontiguousarray(indices1, np.int32)
        n = self.lib.orc_match(C.byref(cfg), np.ascontiguousarray(desc0, np.int8), np.ascontiguousarray(desc1, np.int8),
                               np.ascontiguousarray(max_idx0, np.int32), np.ascontiguousarray(probs0, np.float32),
                               len(patches1), patches1, indices1, p0, p1, c0, qq, sc, C.byref(st))
        return dict(n=n, pts0=p0[:n].copy(), pts1=p1[:n].copy(), cell0=c0[:n].copy(), query=qq[:n].copy(),
                    score=sc[:n].copy(), window_cells=st.window_cells, pairs_256=st.pairs_256, pairs_64=st.pairs_64)

    # -- pose
    def svd3(self, A):
        A = np.ascontiguousarray(A, np.float32)
        U = np.zeros((3, 3), np.float32); S = np.zeros((3, 3), np.float32); V = np.zeros((3, 3), np.float32)
        self.lib.orc_svd3(A, U, S, V)
        return U, S, V

    def ransac_identity(self, pts1, pts2, iters=10, thr=1.1, cap=1000):
        pts1 = np.ascontiguousarray(pts1, np.float32); pts2 = np.ascontiguousarray(pts2, np.float32)
        n = pts1.shape[0]
        E = np.zeros((3, 3), np.float32); inl = np.zeros(max(cap, 1), np.int32); ni = C.c_int(0)
        wrote = self.lib.orc_ransac_identity(n, pts1, pts2, iters, thr, cap, E, inl, C.byref(ni))
        return E, inl[:ni.value].copy(), ni.value, wrote

    def recover_pose(self, E):
        E = np.ascontiguousarray(E, np.float32)
        R1 = np.zeros((3, 3), np.float32); R2 = np.zeros((3, 3), np.float32); t = np.zeros(3, np.float32)
        self.lib.orc_recover_pose(E, R1, R2, t)
        return R1, R2, t

    def pnp_gn(self, cfg: PnpCfg, corr, n, pair_index=0, init_pose=None, want_hyp=False):
        corr = np.ascontiguousarray(corr, np.float32)
        stride = corr.shape[1]
        pose = np.zeros(7, np.float32); stats = np.zeros(4, np.float32)
        hyp = np.zeros((cfg.hypotheses, 8), np.float32) if want_hyp else None
        ip = None if init_pose is None else np.ascontiguousarray(init_pose, np.float32)
        self.lib.orc_pnp_gn(C.byref(cfg), pair_index, n, stride, corr,
                            None if ip is None else ip.ctypes.data, pose, stats,
                            None if hyp is None else hyp.ctypes.data)
        return pose, stats, hyp

    def lba_schur(self, J, chunk=4):
        """J float32 [n_ldmks, n_poses, 20] -> C float32 [(6P+1), (6P+1)] (column-major storage)."""
        J = np.ascontiguousarray(J, np.float32)
        n_l, n_p, _ = J.shape
        sh = 6 * n_p + 1
        out = np.zeros((sh, sh), np.float32)
        self.lib.orc_lba_schur(n_l, n_p, chunk, J.reshape(-1), out.reshape(-1))
        return out

    def lba_solve(self, Cm, damping=0.0):
        """Cm float32 [(6P+1), (6P+1)] as lba_schur returns it -> (ok, d float32 [6P]): the damped
        Cholesky step S d = -g (this repository's definition; the reference's cholesky() is a stub)."""
        Cm = np.ascontiguousarray(Cm, np.float32)
        n_p = (Cm.shape[0] - 1) // 6
        d = np.zeros(6 * n_p, np.float32)
        ok = self.lib.orc_lba_solve(n_p, float(damping), Cm.reshape(-1), d)
        return int(ok), d

    def invert_3x3(self, m, stride=3):
        m = np.ascontiguousarray(m, np.float32).copy()
        self.lib.orc_invert_3x3(m.reshape(-1), stride)
        return m

    # -- BoW word assignment (parity unpinned as a whole; helpers pinned to bow_main.c's own functions)
    def bow_vocab(self, base_desc, scale, bias, leaves):
        """base_desc int8 [256, n_base], scale/bias float32 [n_base], leaves int32 [n_base, wpb, 4] -> handle"""
        base_desc = np.ascontiguousarray(base_desc, np.int8); scale = np.ascontiguousarray(scale, np.float32)
        bias = np.ascontiguousarray(bias, np.float32)
        n_base, wpb = leaves.shape[0], leaves.shape[1]
        flat = np.zeros(n_base * wpb * 4 + 4, np.int32)
        flat[:-4] = np.ascontiguousarray(leaves, np.int32).reshape(-1)
        v = BowVocab(n_base, wpb, base_desc.ctypes.data, scale.ctypes.data, bias.ctypes.data, flat.ctypes.data)
        v._keep = (base_desc, scale, bias, flat)
        return v

    def bow_binarize(self, scale, feature):
        out = np.zeros(8, np.int32)
        self.lib.orc_bow_binarize(float(scale), np.ascontiguousarray(feature, np.int8), out)
        return out

    def bow_matching_bits(self, a, b):
        a = np.ascontiguousarray(a, np.int32); b = np.ascontiguousarray(b, np.int32)
        return int(self.lib.orc_bow_matching_bits(a, b, len(a)))

    def bow_assign(self, vocab, desc_scale, descs):
        """descs int8 [n, 256] -> (base int32 [n], wid int32 [n])"""
        descs = np.ascontiguousarray(descs, np.int8)
        n = descs.shape[0]
        base = np.zeros(n, np.int32); wid = np.zeros(n, np.int32)
        b, w = C.c_int(0), C.c_int(0)
        for i in range(n):
            self.lib.orc_bow_assign(C.byref(vocab), float(desc_scale), descs[i], C.byref(b), C.byref(w))
            base[i], wid[i] = b.value, w.value
        return base, wid

    # -- landmark table (contents of the reference's local feature pool)
    def pool_new(self, n_words):
        t = np.zeros(n_words, LOCAL_FEATURE_DTYPE)
        t["word_id"] = -1
        return t

    def pool_observe(self, table, frame, word_ids, coords=None):
        word_ids = np.ascontiguousarray(word_ids, np.int32)
        c = None if coords is None else np.ascontiguousarray(coords, np.float32)
        self.lib.orc_pool_observe(table.ctypes.data, len(table), int(frame), len(word_ids), word_ids,
                                  None if c is None else c.ctypes.data)

    def pool_remove_old(self, table, current_frame):
        self.lib.orc_pool_remove_old(table.ctypes.data, len(table), int(current_frame))

    def synth_frame(self, seed, rows, cols, frame, off_x, off_y, keypoint_permille=140, noise_amp=6):
        cfg = SynthCfg(seed, rows, cols, keypoint_permille, noise_amp)
        cells = rows * cols
        semi = np.zeros((cells, 65), np.int8); desc = np.zeros((cells, 256), np.int8); depth = np.zeros(cells, np.float32)
        self.lib.orc_synth_frame(C.byref(cfg), frame, off_x, off_y, semi, desc, depth)
        return semi, desc, depth

    def track_pair(self, cfg: TrackCfg, pair_index, semi0, desc0, depth0, semi1, desc1):
        out = PairResult()
        self.lib.orc_track_pair(C.byref(cfg), pair_index, np.ascontiguousarray(semi0), np.ascontiguousarray(desc0),
                                np.ascontiguousarray(depth0, np.float32), np.ascontiguousarray(semi1),
                                np.ascontiguousarray(desc1), C.byref(out))
        return out

    def bench_sequence(self, cfg: TrackCfg, syn: SynthCfg, offsets, first, n, threads):
        out = (PairResult * n)()
        offsets = np.ascontiguousarray(offsets, np.int32)
        secs = self.lib.orc_bench_sequence(C.byref(cfg), C.byref(syn), offsets, first, n, threads, out)
        return secs, out


def have_ref() -> bool:
    return os.path.exists(os.path.join(_HERE, "_ref", "libmaveric_ref.so"))


class Reference:
    """T1: the reference's own code (native 24x80 shape, N=100, <=150 matches)."""
    CELLS = 1920

    def __init__(self):
        build()
        self.lib = C.CDLL(os.path.join(_HERE, "_ref", "libmaveric_ref.so"))
        L = self.lib
        L.ref_load_pair.argtypes = [C.c_float, _i8p, C.c_float, _i8p, C.c_float, _i8p, C.c_float, _i8p]
        L.ref_run_tracking.restype = C.c_int
        L.ref_run_tracking.argtypes = [_f32p, _f32p, C.POINTER(C.c_int), _i32p, _f32p]
        L.compute_softmax.argtypes = [C.c_float, _i8p, C.POINTER(C.c_int), _i32p, _f32p]
        L.compute_top_N.argtypes = [C.c_float, _i8p, C.c_int, C.POINTER(C.c_int), _i32p, _i32p, _f32p]
        L.ref_ransac_essential_matrix.argtypes = [C.c_int, _f32p, _f32p, _f32p, C.c_int, C.c_float, _f32p, _i32p,
                                                  C.POINTER(C.c_int)]
        L.recover_pose_from_essential_matrix.argtypes = [_f32p, _f32p, _f32p, _f32p]
        L.compute_reprojection_error.restype = C.c_float
        L.compute_reprojection_error.argtypes = [_f32p, _f32p, _f32p]
        L.normalize_points.argtypes = [C.c_int, _f32p, _f32p, _f32p]
        L.svd.argtypes = [C.c_float] * 9 + [C.POINTER(C.c_float)] * 27
        L.ref_run_nms.restype = C.c_int
        L.ref_run_nms.argtypes = [_i32p, C.POINTER(C.c_int), _i32p]
        L.ref_lba_run.restype = C.c_int
        L.ref_lba_run.argtypes = [C.c_void_p, _f32p]
        L.ref_invert_3x3.argtypes = [_f32p, C.c_int]
        L.matmul.argtypes = [C.c_size_t] * 3 + [_f32p, _f32p, _f32p] + [C.c_size_t] * 3 + [C.c_float] * 2 + [C.c_bool] * 2
        L.matmul2.argtypes = [C.c_size_t] * 3 + [_f32p, _f32p, C.c_void_p, _f32p] + [C.c_size_t] * 4 + [C.c_float] * 3 + [C.c_bool] * 2

    def softmax(self, scale, semi):
        semi = np.ascontiguousarray(semi, np.int8); assert semi.shape == (1920, 65)
        idx = np.zeros(1920, np.int32); pr = np.zeros(1920, np.float32); nv = C.c_int(0)
        self.lib.compute_softmax(float(scale), semi, C.byref(nv), idx, pr)
        return idx, pr, nv.value

    def top_n(self, scale, semi, N):
        semi = np.ascontiguousarray(semi, np.int8); assert semi.shape == (1920, 65)
        pa = np.zeros(N, np.int32); ix = np.zeros(N, np.int32); pr = np.zeros(N, np.float32); n = C.c_int(0)
        self.lib.compute_top_N(float(scale), semi, N, C.byref(n), pa, ix, pr)
        return pa[:n.value].copy(), ix[:n.value].copy(), pr[:n.value].copy()

    def tracking_main(self, semi_scale0, semi0, desc0, semi_scale1, semi1, desc1):
        """Runs the reference main() (src/tracking_main.c:68-230) on this pair."""
        self.lib.ref_load_pair(float(semi_scale0), np.ascontiguousarray(semi0, np.int8), 1.0,
                               np.ascontiguousarray(desc0, np.int8), float(semi_scale1),
                               np.ascontiguousarray(semi1, np.int8), 1.0, np.ascontiguousarray(desc1, np.int8))
        p1 = np.zeros((150, 2), np.float32); p2 = np.zeros((150, 2), np.float32)
        ni = C.c_int(0); inl = np.zeros(1000, np.int32); E = np.zeros((3, 3), np.float32)
        n = self.lib.ref_run_tracking(p1, p2, C.byref(ni), inl, E)
        return dict(n=n, pts0=p1[:n].copy(), pts1=p2[:n].copy(), num_inliers=ni.value,
                    inliers=inl[:ni.value].copy(), best_E=E)

    def lba_run(self, flat=None):
        """local_bundle_adjustment.c's main() as shipped; `flat` (640 floats, the 64 x 10
        column-major factor matrix of a chunk) replaces its i*10+j input.  Returns C [49, 49]."""
        out = np.zeros((49, 49), np.float32)
        f = None if flat is None else np.ascontiguousarray(flat, np.float32)
        dim = self.lib.ref_lba_run(None if f is None else f.ctypes.data, out.reshape(-1))
        assert dim == 49
        return out

    def invert_3x3(self, m, stride=3):
        m = np.ascontiguousarray(m, np.float32).copy()
        self.lib.ref_invert_3x3(m.reshape(-1), stride)
        return m

    def run_nms(self, semi_scale1, semi1):
        """Runs the reference's run_nms main() (src/run_nms.c:42-175) on this frame (its image1).
        Returns (suppression events [n,4], surviving keypoints [m,2] in patch order)."""
        z = np.zeros((1920, 256), np.int8)
        self.lib.ref_load_pair(1.0, np.zeros((1920, 65), np.int8), 1.0, z, float(semi_scale1),
                               np.ascontiguousarray(semi1, np.int8), 1.0, z)
        ev = np.zeros((4096, 4), np.int32); kp = np.zeros((1920, 2), np.int32); ne = C.c_int(0)
        nk = self.lib.ref_run_nms(ev, C.byref(ne), kp)
        return ev[:ne.value].copy(), kp[:nk].copy()

    def ransac(self, pts1, pts2, K, iters=10, thr=1.1):
        pts1 = np.ascontiguousarray(pts1, np.float32); pts2 = np.ascontiguousarray(pts2, np.float32)
        E = np.zeros((3, 3), np.float32); inl = np.zeros(1000, np.int32); ni = C.c_int(-1)
        self.lib.ref_ransac_essential_matrix(pts1.shape[0], pts1, pts2, np.ascontiguousarray(K, np.float32),
                                             iters, thr, E, inl, C.byref(ni))
        return E, inl[:max(ni.value, 0)].copy(), ni.value

    def recover_pose(self, E):
        E = np.ascontiguousarray(E, np.float32)
        R1 = np.zeros((3, 3), np.float32); R2 = np.zeros((3, 3), np.float32); t = np.zeros(3, np.float32)
        self.lib.recover_pose_from_essential_matrix(E, R1, R2, t)
        return R1, R2, t

    def svd3(self, A):
        A = np.asarray(A, np.float32)
        outs = [(C.c_float)() for _ in range(27)]
        self.lib.svd(*[float(v) for v in A.reshape(-1)], *[C.byref(o) for o in outs])
        vals = np.array([o.value for o in outs], np.float32)
        return vals[:9].reshape(3, 3), vals[9:18].reshape(3, 3), vals[18:].reshape(3, 3)


def have_ref_bow() -> bool:
    return os.path.exists(os.path.join(_HERE, "_ref", "libmaveric_ref_bow.so"))


class ReferenceBow:
    """bow_main.c compiled by itself (oracle/Makefile): its two helper functions and the vocabulary it includes."""

    def __init__(self):
        build()
        self.lib = C.CDLL(os.path.join(_HERE, "_ref", "libmaveric_ref_bow.so"))
        L = self.lib
        L.get_binary_descriptor.argtypes = [C.c_float, _i32p, _i32p, C.c_int]
        L.count_matching_bits.restype = C.c_int
        L.count_matching_bits.argtypes = [_i32p, _i32p, C.c_int]

    def vocabulary(self):
        """(base_desc int8 [256,10], scale f32 [10], bias f32 [10], leaves int32 [10,1000,4]) from vocabulary.h"""
        L = self.lib
        nb = C.c_int.in_dll(L, "num_base_nodes").value
        wpb = C.c_int.in_dll(L, "words_per_base_node").value
        base = np.ctypeslib.as_array((C.c_int8 * (256 * nb)).in_dll(L, "base_descriptors")).reshape(256, nb).copy()
        scale = np.ctypeslib.as_array((C.c_float * nb).in_dll(L, "scale_arr")).copy()
        bias = np.ctypeslib.as_array((C.c_float * nb).in_dll(L, "bias_arr")).copy()
        leaves = np.ctypeslib.as_array((C.c_int * (nb * wpb * 4)).in_dll(L, "leaf_descriptors")).reshape(nb, wpb, 4).copy()
        return base, scale, bias, leaves

    def get_binary_descriptor(self, scale, feature_int32, size=8):
        f = np.ascontiguousarray(feature_int32, np.int32)
        out = np.zeros(size, np.int32)
        self.lib.get_binary_descriptor(float(scale), f, out, size)
        return out

    def count_matching_bits(self, a, b):
        a = np.ascontiguousarray(a, np.int32); b = np.ascontiguousarray(b, np.int32)
        return int(self.lib.count_matching_bits(a, b, len(a)))


def lba_reference_factors(flat=None, n_ldmks=1000, n_poses=8, chunk=4):
    """The factor blocks main() of local_bundle_adjustment.c actually uses, as the [n_ldmks, n_poses, 20]
    input of the parametrised forms: every chunk re-creates the same 64 x 10 column-major matrix
    (:92-98, i*10+j unless `flat` replaces it) and factor (chunk_i, pose) is the 20 floats at row
    pose * chunk_i of its [32][20] view (:157, the index is a product in the reference)."""
    if flat is None:
        flat = np.zeros(640, np.float32)
        for j in range(10):
            for i in range(64):
                flat[j * 64 + i] = i * 10 + j
    flat = np.asarray(flat, np.float32)
    J = np.zeros((n_ldmks, n_poses, 20), np.float32)
    for l in range(n_ldmks):
        ci = l % chunk
        for p in range(n_poses):
            J[l, p] = flat[20 * (p * ci):20 * (p * ci) + 20]
    return J
