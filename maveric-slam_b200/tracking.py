"""Host-side mirror of the reference's tracking interface, over the C ABI.

Single-pair functions keep the reference's names and argument meaning
(``include/top_N.h:8-13``, ``include/pnp_solver.h:3-22``, ``include/tracking.h:3``,
``include/frame.h:7-47``) and take numpy arrays where the C code takes pointers.
The batched API (:class:`Tracker`) runs on device-resident torch tensors: torch is only
used for device memory, the current stream and ``torch.distributed``.

Everything computes on the GPU through ``libmaveric_b200.so``; nothing here has a CPU path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import lib as _lib

PAIR_RESULT_DTYPE = np.dtype([
    ("q", np.float32, 4), ("t", np.float32, 3), ("pnp_inliers", np.float32), ("pnp_cost", np.float32),
    ("num_matches", np.int32), ("ransac_inliers", np.int32), ("best_hypothesis", np.int32),
    ("status", np.int32), ("pad", np.int32, 3)])
assert PAIR_RESULT_DTYPE.itemsize == 64
LOOP_RESULT_DTYPE = np.dtype([
    ("frame", np.int32), ("bow_score", np.int32), ("bow_rank", np.int32), ("num_matches", np.int32),
    ("pnp_inliers", np.float32), ("pnp_cost", np.float32), ("q", np.float32, 4), ("t", np.float32, 3),
    ("status", np.int32), ("pad", np.int32, 2)])
assert LOOP_RESULT_DTYPE.itemsize == 64


@dataclass
class Frame:
    """include/frame.h:7-30 (the fields frame_create sets)."""
    rows: int
    cols: int
    channels: int
    feature_rows: int
    feature_cols: int
    semi_scale: float
    semi: np.ndarray   # int8 [cells, 65], cell = col*feature_rows + row
    desc_scale: float
    desc: np.ndarray   # int8 [cells, 256]


def frame_create(rows, cols, channels, data, feature_rows, feature_cols, semi_scale, semi, desc_scale, desc) -> Frame:
    """include/frame.h:32-47."""
    del data
    cells = feature_rows * feature_cols
    return Frame(rows, cols, channels, feature_rows, feature_cols, float(semi_scale),
                 np.ascontiguousarray(semi, np.int8).reshape(cells, 65), float(desc_scale),
                 np.ascontiguousarray(desc, np.int8).reshape(cells, 256))


_default_ctx: _lib.Context | None = None


def default_context() -> _lib.Context:
    """The context of the single-pair functions called without one.  It is one context for the whole process and
    not safe to share across threads: a thread of its own passes a :class:`lib.Context` of its own as ``ctx``."""
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = _lib.Context(0)
    return _default_ctx


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _hp(a):
    """Host buffer of a sequence call: a (pinned) CPU tensor or a numpy array."""
    return C.c_void_p(a.data_ptr()) if hasattr(a, "data_ptr") else _p(a)


# --------------------------------------------------------------------------------------
# single-pair, host arrays (reference names)
# --------------------------------------------------------------------------------------
def compute_softmax(scale, semi, ctx: _lib.Context | None = None, legacy: bool = False):
    """src/top_N.c:136-165 -> (max_indices int32[cells], probs f32[cells], num_valid)."""
    semi = np.ascontiguousarray(semi, np.int8)
    cells = semi.shape[0]
    idx = np.zeros(cells, np.int32)
    pr = np.zeros(cells, np.float32)
    nv = C.c_int(0)
    if legacy:
        assert cells == 1920, "the legacy symbol is fixed at 24x80 cells (top_N.c:151)"
        _lib.load().compute_softmax(float(scale), _p(semi), C.byref(nv), _p(idx), _p(pr))
    else:
        ctx = ctx or default_context()
        ctx.check(ctx.lib.compute_softmax_ex(ctx.h, float(scale), _p(semi), cells, C.byref(nv), _p(idx), _p(pr)))
    return idx, pr, nv.value


def compute_top_N(scale, semi, N, max_valid: int = 1000, ctx: _lib.Context | None = None, legacy: bool = False):
    """src/top_N.c:53-134 -> (N_patches, N_indices, N_probs) of length num_selected.
    Raises :class:`lib.MvError` where the reference prints "Exceed max number of features!"
    and exits (the legacy symbol does exit)."""
    semi = np.ascontiguousarray(semi, np.int8)
    cells = semi.shape[0]
    pa = np.zeros(N, np.int32); ix = np.zeros(N, np.int32); pr = np.zeros(N, np.float32)
    n = C.c_int(0)
    if legacy:
        assert cells == 1920
        _lib.load().compute_top_N(float(scale), _p(semi), N, C.byref(n), _p(pa), _p(ix), _p(pr))
    else:
        ctx = ctx or default_context()
        ctx.check(ctx.lib.compute_top_N_ex(ctx.h, float(scale), _p(semi), cells, N, max_valid, C.byref(n),
                                           _p(pa), _p(ix), _p(pr)))
    k = n.value
    return pa[:k].copy(), ix[:k].copy(), pr[:k].copy()


def run_nms(rows, cols, max_indices, probs, ctx: _lib.Context | None = None):
    """src/run_nms.c:65-156 on one frame's detector output -> (max_indices, probs) after suppression
    (suppressed cells: index 64, prob 64.0)."""
    ctx = ctx or default_context()
    mi = np.ascontiguousarray(max_indices, np.int32).copy(); pr = np.ascontiguousarray(probs, np.float32).copy()
    ctx.check(ctx.lib.run_nms_ex(ctx.h, rows, cols, _p(mi), _p(pr)))
    return mi, pr


def match_params(rows, cols, shift_x=4, shift_y=4, radius=4, max_matches=150, match_threshold=0.9,
                 min_prob0=0.2, use_tensor_cores=None) -> _lib.MatchParams:
    p = _lib.MatchParams()
    _lib.load().mv_match_params_default(C.byref(p), rows, cols)
    p.shift_x, p.shift_y, p.radius, p.max_matches = shift_x, shift_y, radius, max_matches
    p.match_threshold, p.min_prob0 = match_threshold, min_prob0
    if use_tensor_cores is not None:      # None keeps the library default (2 = auto)
        p.use_tensor_cores = 1 if use_tensor_cores else 0
    return p


def match_pair(params: _lib.MatchParams, desc0, desc1, max_indices0, probs0, patches1, indices1,
               ctx: _lib.Context | None = None):
    """The match loop of src/tracking_main.c:114-194 for one pair.  Returns a dict with
    ``pts0``/``pts1`` float32 [n,2] (the reference's points1/points2), ``cell0`` and ``score``."""
    ctx = ctx or default_context()
    desc0 = np.ascontiguousarray(desc0, np.int8); desc1 = np.ascontiguousarray(desc1, np.int8)
    mi = np.ascontiguousarray(max_indices0, np.int32); pr = np.ascontiguousarray(probs0, np.float32)
    qp = np.ascontiguousarray(patches1, np.int32); qi = np.ascontiguousarray(indices1, np.int32)
    M = params.max_matches
    p0 = np.zeros((M, 2), np.float32); p1 = np.zeros((M, 2), np.float32)
    c0 = np.zeros(M, np.int32); sc = np.zeros(M, np.float32)
    n = C.c_int(0)
    ctx.check(ctx.lib.mv_match_pair_host(ctx.h, C.byref(params), _p(desc0), _p(desc1), _p(mi), _p(pr), len(qp),
                                         _p(qp), _p(qi), _p(p0), _p(p1), C.byref(n), _p(c0), _p(sc)))
    k = n.value
    return dict(n=k, pts0=p0[:k].copy(), pts1=p1[:k].copy(), cell0=c0[:k].copy(), score=sc[:k].copy())


def ransac_essential_matrix(points1, points2, K, num_iterations=10, inlier_threshold=1.1):
    """src/pnp_solver.c:110-165 (legacy symbol) -> (best_E, best_inliers, num_inliers)."""
    p1 = np.ascontiguousarray(points1, np.float32).reshape(-1, 2)
    p2 = np.ascontiguousarray(points2, np.float32).reshape(-1, 2)
    K = np.ascontiguousarray(K, np.float32)
    E = np.zeros((3, 3), np.float32)
    inl = np.zeros(max(len(p1), 1), np.int32)
    n = C.c_int(0)
    _lib.load().ransac_essential_matrix(len(p1), _p(p1), _p(p2), _p(K), num_iterations, inlier_threshold,
                                        _p(E), _p(inl), C.byref(n))
    return E, inl[:n.value].copy(), n.value


def recover_pose_from_essential_matrix(E):
    """src/pnp_solver.c:168-194 -> (R1, R2, t)."""
    E = np.ascontiguousarray(E, np.float32)
    R1 = np.zeros((3, 3), np.float32); R2 = np.zeros((3, 3), np.float32); t = np.zeros(3, np.float32)
    _lib.load().recover_pose_from_essential_matrix(_p(E), _p(R1), _p(R2), _p(t))
    return R1, R2, t


def matmul(A, B, C_, stride_A, stride_B, stride_C, dim_I, dim_J, dim_K, a_scale=1.0, b_scale=1.0,
           transpose_A=False, transpose_B=False):
    """include/gemmini_functions_cpu.h:14-56; C_ is updated in place."""
    _lib.load().matmul(dim_I, dim_J, dim_K, _p(A), _p(B), _p(C_), stride_A, stride_B, stride_C,
                       a_scale, b_scale, transpose_A, transpose_B)


def matmul2(A, B, D, C_, stride_A, stride_B, stride_D, stride_C, dim_I, dim_J, dim_K, a_scale=1.0, b_scale=1.0,
            d_scale=1.0, transpose_A=False, transpose_B=False):
    """include/gemmini_functions_cpu.h:60-124; D may be None or C_ itself."""
    _lib.load().matmul2(dim_I, dim_J, dim_K, _p(A), _p(B), None if D is None else _p(D), _p(C_), stride_A,
                        stride_B, stride_D, stride_C, a_scale, b_scale, d_scale, transpose_A, transpose_B)


class _CFrame(C.Structure):
    _fields_ = [("rows", C.c_int), ("cols", C.c_int), ("channels", C.c_int), ("data", C.c_char_p),
                ("num_features", C.c_int), ("feature_rows", C.c_int), ("feature_cols", C.c_int),
                ("feature_xs", C.c_void_p), ("feature_ys", C.c_void_p), ("semi_scale", C.c_float),
                ("semi", C.c_void_p), ("desc_scale", C.c_float), ("desc", C.c_void_p)]


def track(last_frame: Frame | None, current_frame: Frame, x_shift=4, y_shift=4, window_size=9, threshold=0.9):
    """include/tracking.h:3 with the semantics of src/tracking_main.c:84-218.
    Returns the SE3 as (q[w,x,y,z], t[3])."""
    L = _lib.load()
    L.track.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]
    L.track.restype = None

    def cf(f: Frame):
        return _CFrame(f.rows, f.cols, f.channels, None, 0, f.feature_rows, f.feature_cols, None, None,
                       f.semi_scale, f.semi.ctypes.data, f.desc_scale, f.desc.ctypes.data)
    out = np.zeros(7, np.float32)
    cur = cf(current_frame)
    if last_frame is None:
        L.track(None, C.byref(cur), x_shift, y_shift, window_size, threshold, _p(out))
    else:
        last = cf(last_frame)
        L.track(C.byref(last), C.byref(cur), x_shift, y_shift, window_size, threshold, _p(out))
    return out[:4].copy(), out[4:].copy()


# --------------------------------------------------------------------------------------
# batched, device-resident (torch tensors)
# --------------------------------------------------------------------------------------
def track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=1024, radius=4,
                 shift=(4, 4), refine_iters=10, sample_iters=4, ransac_iterations=10, lanes=1, seed=0,
                 use_tensor_cores=None, first_pair=0) -> _lib.TrackParams:
    p = _lib.TrackParams()
    _lib.load().mv_track_params_default(C.byref(p), rows, cols)
    p.top_n, p.max_valid = top_n, max_valid
    p.match.max_matches, p.match.radius = max_matches, radius
    p.match.shift_x, p.match.shift_y = shift
    if use_tensor_cores is not None:
        p.match.use_tensor_cores = 1 if use_tensor_cores else 0
    p.pnp.hypotheses, p.pnp.refine_iters, p.pnp.sample_iters = hypotheses, refine_iters, sample_iters
    p.pnp.lanes_per_hypothesis, p.pnp.seed, p.pnp.first_pair = lanes, seed, first_pair
    p.ransac_iterations = ransac_iterations
    return p


def kitti_track_params(**kw) -> _lib.TrackParams:
    """KITTI 376x1241 -> 47x155 cells, ~1k keypoints (SURVEY §8 config C1/C4)."""
    d = dict(rows=47, cols=155, top_n=1000, max_valid=8192, max_matches=1024, hypotheses=1024)
    d.update(kw)
    return track_params(**d)


def loop_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=1024, min_gap=30, k=4,
                min_score=1, min_inliers=30, radius=None, shift=(0, 0), refine_iters=10, sample_iters=4, lanes=1, seed=0,
                use_tensor_cores=None, first_pair=0) -> _lib.LoopParams:
    """mv_loop_params_default with these fields set; radius None keeps the default, which covers the grid."""
    p = _lib.LoopParams()
    _lib.load().mv_loop_params_default(C.byref(p), rows, cols)
    p.top_n, p.max_valid = top_n, max_valid
    p.min_gap, p.k, p.min_score, p.min_inliers = min_gap, k, min_score, min_inliers
    p.match.max_matches = max_matches
    if radius is not None:
        p.match.radius = radius
    p.match.shift_x, p.match.shift_y = shift
    if use_tensor_cores is not None:
        p.match.use_tensor_cores = 1 if use_tensor_cores else 0
    p.pnp.hypotheses, p.pnp.refine_iters, p.pnp.sample_iters = hypotheses, refine_iters, sample_iters
    p.pnp.lanes_per_hypothesis, p.pnp.seed, p.pnp.first_pair = lanes, seed, first_pair
    return p


def loop_results_to_numpy(t) -> np.ndarray:
    """uint8 [n, 64] loop records (device or host tensor) -> structured array of LOOP_RESULT_DTYPE."""
    return np.ascontiguousarray(t.cpu().numpy()).view(LOOP_RESULT_DTYPE).reshape(-1)


class Tracker:
    """Batched hot path on one GPU.  Tensors are torch CUDA tensors; calls are asynchronous
    on torch's current stream (bound at construction)."""

    def __init__(self, device: int = 0):
        import torch
        self.torch = torch
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        self.ctx = _lib.Context(device, stream=torch.cuda.current_stream(self.device).cuda_stream)
        self.lib = self.ctx.lib

    @staticmethod
    def _d(t):
        return None if t is None else C.c_void_p(t.data_ptr())

    def synth_frames(self, seed, rows, cols, first_frame, offsets, keypoint_permille=140, noise_amp=6):
        torch = self.torch
        n = offsets.shape[0]
        cells = rows * cols
        off = torch.as_tensor(np.ascontiguousarray(offsets, np.int32), device=self.device)
        semi = torch.empty((n, cells, 65), dtype=torch.int8, device=self.device)
        desc = torch.empty((n, cells, 256), dtype=torch.int8, device=self.device)
        depth = torch.empty((n, cells), dtype=torch.float32, device=self.device)
        sp = _lib.SynthParams(seed, rows, cols, keypoint_permille, noise_amp)
        self.ctx.check(self.lib.mv_synth_frames(self.ctx.h, C.byref(sp), first_frame, n, self._d(off),
                                                self._d(semi), self._d(desc), self._d(depth)))
        return semi, desc, depth

    def softmax(self, semi, semi_scale):
        torch = self.torch
        n, cells, _ = semi.shape
        idx = torch.empty((n, cells), dtype=torch.int32, device=self.device)
        prob = torch.empty((n, cells), dtype=torch.float32, device=self.device)
        nv = torch.empty((n,), dtype=torch.int32, device=self.device)
        self.ctx.check(self.lib.mv_softmax_batch(self.ctx.h, n, cells, self._d(semi), self._d(semi_scale),
                                                 self._d(idx), self._d(prob), self._d(nv)))
        return idx, prob, nv

    def nms(self, rows, cols, max_idx, prob):
        """In-place batched NMS (src/run_nms.c:65-156) of the detector output of every frame."""
        n = max_idx.shape[0]
        self.ctx.check(self.lib.mv_nms_batch(self.ctx.h, n, rows, cols, self._d(max_idx), self._d(prob)))
        return max_idx, prob

    def top_n(self, max_idx, prob, top_n, max_valid):
        torch = self.torch
        n, cells = max_idx.shape
        qp = torch.zeros((n, top_n), dtype=torch.int32, device=self.device)
        qi = torch.zeros((n, top_n), dtype=torch.int32, device=self.device)
        qpr = torch.zeros((n, top_n), dtype=torch.float32, device=self.device)
        qc = torch.zeros((n,), dtype=torch.int32, device=self.device)
        ov = torch.zeros((n,), dtype=torch.int32, device=self.device)
        self.ctx.check(self.lib.mv_top_n_batch(self.ctx.h, n, cells, top_n, max_valid, self._d(max_idx),
                                               self._d(prob), self._d(qp), self._d(qi), self._d(qpr),
                                               self._d(qc), self._d(ov)))
        return qp, qi, qpr, qc, ov

    def match(self, params: _lib.MatchParams, desc, max_idx, prob, q_patch, q_idx, q_count, f0=None, f1=None):
        torch = self.torch
        n_frames = desc.shape[0]
        n_pairs = n_frames - 1 if f0 is None else f0.shape[0]
        top_n = q_patch.shape[1]
        M = params.max_matches
        pts = torch.zeros((n_pairs, M, 4), dtype=torch.float32, device=self.device)
        cnt = torch.zeros((n_pairs,), dtype=torch.int32, device=self.device)
        cell0 = torch.zeros((n_pairs, M), dtype=torch.int32, device=self.device)
        query = torch.zeros((n_pairs, M), dtype=torch.int32, device=self.device)
        score = torch.zeros((n_pairs, M), dtype=torch.float32, device=self.device)
        self.ctx.check(self.lib.mv_match_batch(
            self.ctx.h, C.byref(params), n_frames, n_pairs, top_n, self._d(f0), self._d(f1), self._d(desc),
            self._d(max_idx), self._d(prob), self._d(q_patch), self._d(q_idx), self._d(q_count), self._d(pts),
            self._d(cnt), self._d(cell0), self._d(query), self._d(score)))
        return pts, cnt, cell0, query, score

    def ransac_identity(self, pts, cnt, iterations=10, threshold=1.1):
        torch = self.torch
        n_pairs, M, _ = pts.shape
        ninl = torch.zeros((n_pairs,), dtype=torch.int32, device=self.device)
        inl = torch.zeros((n_pairs, M), dtype=torch.int32, device=self.device)
        pose = torch.zeros((n_pairs, 12), dtype=torch.float32, device=self.device)
        self.ctx.check(self.lib.mv_ransac_identity_batch(self.ctx.h, n_pairs, M, self._d(pts), self._d(cnt),
                                                         iterations, threshold, self._d(ninl), self._d(inl),
                                                         self._d(pose)))
        return ninl, inl, pose

    def build_corr(self, pts, cnt, cell0, depth, cam, rows, f0=None):
        torch = self.torch
        n_pairs, M, _ = pts.shape
        cells = depth.shape[1]
        corr = torch.zeros((n_pairs, 5, M), dtype=torch.float32, device=self.device)
        self.ctx.check(self.lib.mv_build_corr_batch(self.ctx.h, n_pairs, cells, rows, M, self._d(f0),
                                                    self._d(depth), cam[0], cam[1], cam[2], cam[3],
                                                    self._d(pts), self._d(cnt), self._d(cell0), self._d(corr)))
        return corr

    def pnp_gn(self, params: _lib.PnpParams, corr, cnt, init_pose=None, want_hyp=False):
        torch = self.torch
        n_pairs, _, stride = corr.shape
        pose = torch.zeros((n_pairs, 7), dtype=torch.float32, device=self.device)
        stats = torch.zeros((n_pairs, 4), dtype=torch.float32, device=self.device)
        hyp = torch.zeros((n_pairs, params.hypotheses, 8), dtype=torch.float32, device=self.device) if want_hyp else None
        self.ctx.check(self.lib.mv_pnp_gn_batch(self.ctx.h, C.byref(params), n_pairs, stride, self._d(corr),
                                                self._d(cnt), self._d(init_pose), self._d(pose), self._d(stats),
                                                self._d(hyp)))
        return pose, stats, hyp

    def track_sequence(self, params: _lib.TrackParams, semi, semi_scale, desc, depth, out=None):
        """Whole path for pairs (f, f+1) of device-resident frames -> uint8 [n_pairs, 64] tensor
        (view with :func:`results_to_numpy`)."""
        torch = self.torch
        n = semi.shape[0]
        if out is None:
            out = torch.empty((n - 1, 64), dtype=torch.uint8, device=self.device)
        self.ctx.check(self.lib.mv_track_sequence(self.ctx.h, C.byref(params), n, self._d(semi),
                                                  self._d(semi_scale), self._d(desc), self._d(depth),
                                                  self._d(out)))
        return out

    def track_sequence_host(self, params: _lib.TrackParams, semi, semi_scale, desc, depth, out=None):
        """Same, from host tensors/arrays (pinned for full copy bandwidth); blocks until the
        results are on the host.  Returns (results structured array, h2d_bytes, d2h_bytes)."""
        n = semi.shape[0]
        if out is None:
            out = np.zeros(n - 1, PAIR_RESULT_DTYPE)
        up = C.c_ulonglong(0); down = C.c_ulonglong(0)
        self.ctx.check(self.lib.mv_track_sequence_host(self.ctx.h, C.byref(params), n, _hp(semi), _hp(semi_scale),
                                                       _hp(desc), _hp(depth), _hp(out), C.byref(up), C.byref(down)))
        return out, up.value, down.value


    def results_to_transforms(self, results):
        """uint8 [n, 64] result records (device) -> float64 [n, 3, 4] relative transforms [R|t], the
        reference's interchange format (python/pairwise_pnp.py:690-694)."""
        torch = self.torch
        n = results.shape[0]
        T = torch.empty((n, 3, 4), dtype=torch.float64, device=self.device)
        self.ctx.check(self.lib.mv_results_to_transforms(self.ctx.h, n, self._d(results), self._d(T)))
        return T

    def lba_schur(self, J, chunk: int = 4):
        """src/local_bundle_adjustment.c:133-246 for a batch of windows: float32
        [n_windows, n_ldmks, n_poses, 20] factor blocks (device) -> float32
        [n_windows, 6 n_poses + 1, 6 n_poses + 1] reduced camera matrices, stored column-major as in
        the reference (so [w, c, r] is row r, column c)."""
        torch = self.torch
        n_w, n_l, n_p, _ = J.shape
        sh = 6 * n_p + 1
        out = torch.empty((n_w, sh, sh), dtype=torch.float32, device=self.device)
        self.ctx.check(self.lib.mv_lba_schur_batch(self.ctx.h, n_w, n_l, n_p, chunk, self._d(J), self._d(out)))
        return out

    def lba_solve(self, Cm, damping: float = 0.0):
        """The cholesky() step the reference leaves as a stub (local_bundle_adjustment.c:88-90,247):
        float32 [n_windows, 6P+1, 6P+1] reduced camera matrices as lba_schur returns them ->
        (delta float32 [n_windows, 6P], ok int32 [n_windows]); S delta = -g by a damped Cholesky
        factorisation in a fixed summation order (this library's definition, mv_lba_solve_batch)."""
        torch = self.torch
        n_w, sh, _ = Cm.shape
        n_p = (sh - 1) // 6
        delta = torch.empty((n_w, 6 * n_p), dtype=torch.float32, device=self.device)
        ok = torch.empty((n_w,), dtype=torch.int32, device=self.device)
        self.ctx.check(self.lib.mv_lba_solve_batch(self.ctx.h, n_w, n_p, float(damping), self._d(Cm),
                                                   self._d(delta), self._d(ok)))
        return delta, ok

    # -- SURVEY §8f rank 3: BoW word assignment and the landmark table
    def bow_set_vocabulary(self, base_desc, scale, bias, leaves):
        """base_desc int8 [256, n_base], scale / bias float32 [n_base], leaves int32 [n_base, wpb, 4] (host arrays)"""
        base_desc = np.ascontiguousarray(base_desc, np.int8); scale = np.ascontiguousarray(scale, np.float32)
        bias = np.ascontiguousarray(bias, np.float32); leaves = np.ascontiguousarray(leaves, np.int32)
        self.ctx.check(self.lib.mv_bow_set_vocabulary(self.ctx.h, leaves.shape[0], leaves.shape[1], _p(base_desc),
                                                      _p(scale), _p(bias), _p(leaves)))
        self.words_per_base = leaves.shape[1]
        self.n_words = leaves.shape[0] * leaves.shape[1]

    def bow_assign(self, desc, desc_scale, q_patch, q_count):
        """-> (word int32 [n_frames, top_n], base int32 [n_frames, top_n]); word = base * wpb + leaf, -1 = no query"""
        torch = self.torch
        n, cells, _ = desc.shape
        top_n = q_patch.shape[1]
        word = torch.empty((n, top_n), dtype=torch.int32, device=self.device)
        base = torch.empty((n, top_n), dtype=torch.int32, device=self.device)
        self.ctx.check(self.lib.mv_bow_assign_batch(self.ctx.h, n, cells, top_n, self._d(desc), self._d(desc_scale),
                                                    self._d(q_patch), self._d(q_count), self._d(word), self._d(base)))
        return word, base

    # -- loop closure: BoW candidates on the tensor cores, verified by the matcher and the Gauss-Newton PnP
    def lcd_word_weights(self, word, q_count, n_words=None):
        """idf weights int8 [n_words] of the given frames' words (mv_lcd_word_weights):
        rint(127 ln(n / df) / ln(n)), 0 for a word no frame holds."""
        n, top_n = word.shape
        n_words = self.n_words if n_words is None else n_words
        weight = self.torch.empty((n_words,), dtype=self.torch.int8, device=self.device)
        self.ctx.check(self.lib.mv_lcd_word_weights(self.ctx.h, n, top_n, n_words, self._d(word), self._d(q_count),
                                                    self._d(weight)))
        return weight

    def loop_candidates(self, word, q_count, weight=None, min_gap=30, k=4, min_score=1, first_frame=0, n_words=None):
        """The best k earlier frames of every frame by BoW score (mv_loop_candidates): word int32 [n, top_n] and
        q_count int32 [n] as :meth:`bow_assign` / :meth:`top_n` return them, weight int8 [n_words] or None (all 1).
        Returns (cand int32 [n, k] global frame numbers or -1, score int32 [n, k])."""
        torch = self.torch
        n, top_n = word.shape
        n_words = self.n_words if n_words is None else n_words
        cand = torch.empty((n, k), dtype=torch.int32, device=self.device)
        score = torch.empty((n, k), dtype=torch.int32, device=self.device)
        self.ctx.check(self.lib.mv_loop_candidates(self.ctx.h, n, int(first_frame), top_n, n_words, self._d(word),
                                                   self._d(q_count), self._d(weight), int(min_gap), int(k),
                                                   int(min_score), self._d(cand), self._d(score)))
        return cand, score

    def detect_loops(self, params: _lib.LoopParams, semi, semi_scale, desc, desc_scale, depth, weight=None,
                     first_frame=0, out=None):
        """Loop closures of device-resident frames in one call (mv_detect_loops; vocabulary set first with
        :meth:`bow_set_vocabulary`) -> uint8 [n_frames, 64] records (view with :func:`loop_results_to_numpy`)."""
        n = semi.shape[0]
        if out is None:
            out = self.torch.empty((n, 64), dtype=self.torch.uint8, device=self.device)
        self.ctx.check(self.lib.mv_detect_loops(self.ctx.h, C.byref(params), n, int(first_frame), self._d(semi),
                                                self._d(semi_scale), self._d(desc), self._d(desc_scale),
                                                self._d(depth), self._d(weight), self._d(out)))
        return out

    def landmarks_new(self, n_words):
        """Empty device landmark table: uint8 [n_words, 56] (view with LANDMARK_DTYPE after .cpu().numpy())."""
        t = self.torch.empty((n_words, 56), dtype=self.torch.uint8, device=self.device)
        self.ctx.check(self.lib.mv_landmarks_init(self.ctx.h, n_words, self._d(t)))
        return t

    def landmarks_observe(self, table, frame, word_ids, coords=None):
        self.ctx.check(self.lib.mv_landmarks_observe(self.ctx.h, table.shape[0], self._d(table), int(frame),
                                                     word_ids.numel(), self._d(word_ids), self._d(coords)))

    def landmarks_remove_old(self, table, current_frame):
        self.ctx.check(self.lib.mv_landmarks_remove_old(self.ctx.h, table.shape[0], self._d(table), int(current_frame)))

    def landmarks_lookup(self, table, word_ids):
        torch = self.torch
        n = word_ids.numel()
        coords = torch.empty((n, 3), dtype=torch.float32, device=self.device)
        found = torch.empty((n,), dtype=torch.int32, device=self.device)
        self.ctx.check(self.lib.mv_landmarks_lookup(self.ctx.h, table.shape[0], self._d(table), n, self._d(word_ids),
                                                    self._d(coords), self._d(found)))
        return coords, found

    def build_corr_landmarks(self, table, pts, cnt, cell0, q_patch, q_count, word, f0=None):
        """Correspondences [n_pairs, 5, M] whose 3-D side is the landmark of the matched frame-0 keypoint's word
        (NaN where there is none) -> (corr, n_with_landmark int32 [n_pairs])."""
        torch = self.torch
        n_pairs, M, _ = pts.shape
        corr = torch.zeros((n_pairs, 5, M), dtype=torch.float32, device=self.device)
        nl = torch.zeros((n_pairs,), dtype=torch.int32, device=self.device)
        self.ctx.check(self.lib.mv_build_corr_landmarks_batch(
            self.ctx.h, n_pairs, q_patch.shape[1], M, table.shape[0], self._d(table), self._d(f0), self._d(q_patch),
            self._d(q_count), self._d(word), self._d(pts), self._d(cnt), self._d(cell0), self._d(corr), self._d(nl)))
        return corr, nl

    def landmarks_sequence(self, table, first_frame, word, q_count, coords_in, coords_out=None):
        """The table update of a whole sequence in one call (mv_landmarks_sequence): step f observes frame
        first_frame + f (word int32 [n_steps, top_n], the first q_count[f] of them, coordinates float32
        [n_steps, top_n, 3]) and then removes old frames.  `table` is updated in place; returns coords_out float32
        [n_steps, top_n, 3], each occurrence's landmark right after its frame's step (0 where there is none)."""
        n_steps, top_n = word.shape
        if coords_out is None:
            coords_out = self.torch.empty((n_steps, top_n, 3), dtype=self.torch.float32, device=self.device)
        self.ctx.check(self.lib.mv_landmarks_sequence(self.ctx.h, table.shape[0], self._d(table), int(first_frame), n_steps,
                                                      top_n, self._d(word), self._d(q_count), self._d(coords_in),
                                                      self._d(coords_out)))
        return coords_out

    def track_sequence_landmarks(self, params: _lib.TrackParams, semi, semi_scale, desc, desc_scale, depth, table,
                                 first_frame=0, out=None, n_with_landmark=None):
        """:meth:`track_sequence` with the 3-D side of each pair from the landmark table (vocabulary set first with
        :meth:`bow_set_vocabulary`): the table steps over frames 0 .. n-2 (global numbers first_frame + f) and is
        updated in place.  Returns (uint8 [n_pairs, 64] results, int32 [n_pairs] matches with a landmark)."""
        torch = self.torch
        n = semi.shape[0]
        if out is None:
            out = torch.empty((n - 1, 64), dtype=torch.uint8, device=self.device)
        if n_with_landmark is None:
            n_with_landmark = torch.empty((n - 1,), dtype=torch.int32, device=self.device)
        self.ctx.check(self.lib.mv_track_sequence_landmarks(
            self.ctx.h, C.byref(params), n, int(first_frame), self._d(semi), self._d(semi_scale), self._d(desc),
            self._d(desc_scale), self._d(depth), table.shape[0], self._d(table), self._d(out), self._d(n_with_landmark)))
        return out, n_with_landmark

    def track_sequence_landmarks_host(self, params: _lib.TrackParams, semi, semi_scale, desc, desc_scale, depth, table,
                                      first_frame=0, out=None, n_with_landmark=None):
        """:meth:`track_sequence_landmarks` from host tensors/arrays (pinned for full copy bandwidth, as
        :meth:`track_sequence_host`); `table` stays on the device and is updated in place.  Blocks until the results
        are on the host.  Returns (results structured array, int32 [n_pairs] matches with a landmark, h2d_bytes,
        d2h_bytes)."""
        n = semi.shape[0]
        if out is None:
            out = np.zeros(n - 1, PAIR_RESULT_DTYPE)
        if n_with_landmark is None:
            n_with_landmark = np.zeros(n - 1, np.int32)
        up = C.c_ulonglong(0); down = C.c_ulonglong(0)
        self.ctx.check(self.lib.mv_track_sequence_landmarks_host(
            self.ctx.h, C.byref(params), n, int(first_frame), _hp(semi), _hp(semi_scale), _hp(desc), _hp(desc_scale),
            _hp(depth), table.shape[0], self._d(table), _hp(out), _hp(n_with_landmark), C.byref(up), C.byref(down)))
        return out, n_with_landmark, up.value, down.value

    def landmarks_speculate(self, n_words, first_frame, n_warm, word, q_count, coords_in):
        """mv_landmarks_speculate: the table step of block frames first_frame .. from the table that the n_warm
        frames before them give from an empty table.  word int32 [n_warm + n_steps, top_n], q_count int32
        [n_warm + n_steps], coords_in float32 [n_steps, top_n, 3] (kept alive by the returned handle until release).
        Returns a handle for :meth:`landmarks_resolve` / :meth:`landmarks_release`."""
        n_total, top_n = word.shape
        h = C.c_void_p()
        self.ctx.check(self.lib.mv_landmarks_speculate(self.ctx.h, int(n_words), int(first_frame), int(n_warm),
                                                       n_total - int(n_warm), top_n, self._d(word), self._d(q_count),
                                                       self._d(coords_in), C.byref(h)))
        return {"h": h, "n_steps": n_total - int(n_warm), "top_n": top_n, "keep": (word, q_count, coords_in)}

    def landmarks_resolve(self, spec, table, coords_out=None, n_rewalked=None):
        """mv_landmarks_resolve: steps `table` in place exactly as :meth:`landmarks_sequence` over the block would;
        returns coords_out float32 [n_steps, top_n, 3]."""
        if coords_out is None:
            coords_out = self.torch.empty((spec["n_steps"], spec["top_n"], 3), dtype=self.torch.float32,
                                          device=self.device)
        self.ctx.check(self.lib.mv_landmarks_resolve(self.ctx.h, spec["h"], self._d(table), self._d(coords_out),
                                                     self._d(n_rewalked)))
        return coords_out

    def landmarks_release(self, spec):
        if spec["h"]:
            self.lib.mv_lm_spec_release(spec["h"])
            spec["h"] = C.c_void_p()

    def track_landmarks_prepare(self, params: _lib.TrackParams, n_warm, first_frame, semi, semi_scale, desc,
                                desc_scale, depth, n_words):
        """mv_track_landmarks_prepare: everything of :meth:`track_sequence_landmarks` on a block that does not need
        the table.  The inputs hold n_warm warm-up frames, then the block's frames (global numbers first_frame ..);
        they must stay alive until :meth:`track_landmarks_solve`.  Returns a block handle."""
        h = C.c_void_p()
        n = semi.shape[0] - int(n_warm)
        self.ctx.check(self.lib.mv_track_landmarks_prepare(
            self.ctx.h, C.byref(params), int(n_warm), n, int(first_frame), self._d(semi), self._d(semi_scale),
            self._d(desc), self._d(desc_scale), self._d(depth), int(n_words), C.byref(h)))
        return {"h": h, "n_pairs": n - 1, "keep": (semi, semi_scale, desc, desc_scale, depth)}

    def track_landmarks_prepare_host(self, params: _lib.TrackParams, n_warm, first_frame, semi, semi_scale, desc,
                                     desc_scale, depth, n_words):
        """mv_track_landmarks_prepare_host: :meth:`track_landmarks_prepare` from host tensors/arrays (pinned for
        full copy bandwidth, as :meth:`track_sequence_landmarks_host`).  The host buffers are no longer read when it
        returns.  Returns a block handle, as :meth:`track_landmarks_prepare`, whose "h2d_bytes" is the bytes
        staged."""
        h = C.c_void_p()
        up = C.c_ulonglong(0)
        n = semi.shape[0] - int(n_warm)
        self.ctx.check(self.lib.mv_track_landmarks_prepare_host(
            self.ctx.h, C.byref(params), int(n_warm), n, int(first_frame), _hp(semi), _hp(semi_scale), _hp(desc),
            _hp(desc_scale), _hp(depth), int(n_words), C.byref(h), C.byref(up)))
        return {"h": h, "n_pairs": n - 1, "h2d_bytes": up.value}

    def track_landmarks_step_table(self, block, table, n_rewalked=None):
        """mv_track_landmarks_step_table: steps `table` in place over the block's frames."""
        self.ctx.check(self.lib.mv_track_landmarks_step_table(self.ctx.h, block["h"], self._d(table),
                                                              self._d(n_rewalked)))

    def track_landmarks_solve(self, block, out=None, n_with_landmark=None):
        """mv_track_landmarks_solve -> (uint8 [n_pairs, 64] results, int32 [n_pairs] matches with a landmark)."""
        torch = self.torch
        if out is None:
            out = torch.empty((block["n_pairs"], 64), dtype=torch.uint8, device=self.device)
        if n_with_landmark is None:
            n_with_landmark = torch.empty((block["n_pairs"],), dtype=torch.int32, device=self.device)
        self.ctx.check(self.lib.mv_track_landmarks_solve(self.ctx.h, block["h"], self._d(out),
                                                         self._d(n_with_landmark)))
        return out, n_with_landmark

    def track_landmarks_release(self, block):
        if block["h"]:
            self.lib.mv_track_landmarks_release(block["h"])
            block["h"] = C.c_void_p()

    def chain_transforms(self, transforms):
        """python/compute_trajectory.py:49-51,76-77 as a parallel scan: float64 [n, 3, 4] relative
        transforms -> float64 [n+1, 3, 4] frame poses, pose 0 the identity."""
        torch = self.torch
        n = transforms.shape[0]
        traj = torch.empty((n + 1, 3, 4), dtype=torch.float64, device=self.device)
        self.ctx.check(self.lib.mv_chain_transforms(self.ctx.h, n, self._d(transforms), self._d(traj)))
        return traj


# --------------------------------------------------------------------------------------
# trajectory files, in the reference's formats (python/compute_trajectory.py)
# --------------------------------------------------------------------------------------
def save_pose(filename, pose) -> None:
    """compute_trajectory.py:49-51: the 3x4 pose, '%.6f', one row per line."""
    np.savetxt(filename, np.asarray(pose, np.float64)[:3, :], fmt="%.6f")


def write_ply(filename, points) -> None:
    """compute_trajectory.py:6-43: camera centres as an ASCII PLY polyline, first vertex red, last
    black, the others blue."""
    points = [np.asarray(p, np.float64) for p in points]
    n = len(points)
    colors = [[255, 0, 0]] + [[0, 0, 255]] * max(0, n - 2) + [[0, 0, 0]]
    with open(filename, "w") as f:
        f.write("ply\nformat ascii 1.0\n")
        f.write(f"element vertex {n}\n")
        f.write("property float x\nproperty float y\nproperty float z\n")
        f.write("property uchar red\nproperty uchar green\nproperty uchar blue\n")
        f.write(f"element edge {n - 1}\n")
        f.write("property int vertex1\nproperty int vertex2\nend_header\n")
        for pt, c in zip(points, colors):
            f.write(f"{pt[0]} {pt[1]} {pt[2]} {c[0]} {c[1]} {c[2]}\n")
        for i in range(n - 1):
            f.write(f"{i} {i + 1}\n")


def write_trajectory(out_dir, start_frame: int, traj) -> None:
    """The files compute_trajectory.py's main() leaves in out_dir (:53-89): one
    frame-XXXXXX.pose.txt per pose and trajectory_<start>_<end>.ply."""
    import os
    traj = np.asarray(traj, np.float64)
    for i, pose in enumerate(traj):
        save_pose(os.path.join(out_dir, f"frame-{start_frame + i:06d}.pose.txt"), pose)
    end = start_frame + len(traj) - 1
    write_ply(os.path.join(out_dir, f"trajectory_{start_frame:06d}_{end:06d}.ply"), [p[:3, 3] for p in traj])


LANDMARK_DTYPE = np.dtype([("word_id", "<i4"), ("frame_ptr", "<i4"), ("num_frames", "<i4"), ("frames", "<i4", (8,)),
                           ("coords", "<f4", (3,))])   # include/local_feature_pool.h:16-22


def results_to_numpy(t) -> np.ndarray:
    return t.cpu().numpy().view(PAIR_RESULT_DTYPE).reshape(-1)


# --------------------------------------------------------------------------------------
# multi-GPU: frame pairs shard by contiguous block; only the 64-byte results are gathered
# --------------------------------------------------------------------------------------
def shard_pairs(n_pairs: int, world: int, rank: int):
    """Contiguous block of pairs of this rank: [first, first+count)."""
    per = (n_pairs + world - 1) // world
    first = min(rank * per, n_pairs)
    return first, max(0, min(n_pairs, first + per) - first), per


def shard_pairs_weighted(n_pairs: int, weights):
    """Contiguous blocks sized in proportion to `weights` (one per rank) -> [(first, count), ...].

    For the host-buffer path, whose step time is the host link's: on a box where the GPUs do not all see the
    same host-to-device rate (measured on the 8 x B200 pool box: 23 GB/s on GPUs 0-3, 35 GB/s on GPUs 4-7 with
    all eight copying), equal blocks leave the fast ranks idle for a third of the step.  Counts are rounded by
    largest remainder, so they always sum to n_pairs; blocks stay contiguous (pose chaining stays local)."""
    w = [max(0.0, float(x)) for x in weights]
    tot = sum(w)
    if not w or tot <= 0.0:
        raise ValueError("shard_pairs_weighted: weights must hold a positive entry")
    exact = [n_pairs * x / tot for x in w]
    counts = [int(e) for e in exact]
    by_remainder = sorted(range(len(w)), key=lambda r: (exact[r] - counts[r], -r), reverse=True)
    for r in by_remainder[: n_pairs - sum(counts)]:
        counts[r] += 1
    out, first = [], 0
    for cnt in counts:
        out.append((first, cnt))
        first += cnt
    return out


def balance_shards(counts, seconds, tolerance: float = 0.10):
    """New per-rank pair counts from one measured step: `counts[r]` pairs took rank r `seconds[r]`.
    Returns `counts` unchanged when the slowest and fastest rank are within `tolerance` of each other
    (symmetric boxes: no churn from timing noise)."""
    live = [(c, s) for c, s in zip(counts, seconds) if c > 0 and s > 0.0]
    if len(live) < 2:
        return list(counts)
    t = [s for _, s in live]
    if max(t) <= (1.0 + tolerance) * min(t):
        return list(counts)
    rates = [c / s if (c > 0 and s > 0.0) else 0.0 for c, s in zip(counts, seconds)]
    return [cnt for _, cnt in shard_pairs_weighted(sum(counts), rates)]


def gather_results(local, n_pairs: int, world: int, group=None):
    """all_gather of equal, padded shards of 64-byte records -> uint8 [n_pairs, 64] on every rank.
    `local` is uint8 [count, 64] on the rank's device (NCCL) or CPU (gloo).  One-shot form (allocates and
    copies); a loop uses :class:`ResultGather`, whose send buffer the pose kernels write straight into."""
    import torch
    import torch.distributed as dist
    per = (n_pairs + world - 1) // world
    pad = torch.zeros((per, 64), dtype=torch.uint8, device=local.device)
    pad[: local.shape[0]] = local
    out = torch.empty((world * per, 64), dtype=torch.uint8, device=local.device)
    dist.all_gather_into_tensor(out, pad, group=group)
    return out[:n_pairs]


class ResultGather:
    """The only collective of the path (SURVEY §8e): one all_gather of the 64-byte pair records, at most
    291 KB for a KITTI-00-length sequence.  Send and receive buffers are allocated once; ``send`` -- the
    rank's [count, 64] slice of a padded [per, 64] buffer whose padding rows stay zero -- is handed to
    ``Tracker.track_sequence(out=...)`` / ``track_sequence_host``, so the pack kernel writes the records
    straight into the NCCL send buffer and a step adds exactly one collective launch (no pad / zero / copy
    kernels)."""

    def __init__(self, n_pairs: int, world: int, rank: int, device, group=None, counts=None):
        """`counts`: pairs per rank of a weighted partition (:func:`shard_pairs_weighted`); default: the
        equal blocks of :func:`shard_pairs`."""
        import torch
        self.n_pairs, self.world, self.group = n_pairs, world, group
        self._rows = None
        if counts is None:
            first, count, per = shard_pairs(n_pairs, world, rank)
        else:
            if len(counts) != world or sum(counts) != n_pairs or min(counts) < 0:
                raise ValueError("ResultGather: counts must hold one entry per rank and sum to n_pairs")
            first, count, per = sum(counts[:rank]), counts[rank], max(1, max(counts))
            if world > 1:   # where each pair's record lands in the padded receive buffer
                self._rows = torch.cat([torch.arange(r * per, r * per + c, dtype=torch.int64)
                                        for r, c in enumerate(counts)]).to(device)
                self._out = torch.empty((n_pairs, 64), dtype=torch.uint8, device=device)
        self.first, self.count, self.per = first, count, per
        self._send = torch.zeros((per, 64), dtype=torch.uint8, device=device)
        self.send = self._send[:count]
        self._recv = torch.empty((world * per, 64), dtype=torch.uint8, device=device) if world > 1 else None

    def gather(self):
        """-> uint8 [n_pairs, 64] (a view of a buffer this object owns; valid until the next gather)."""
        if self.world == 1:
            return self.send
        import torch
        import torch.distributed as dist
        dist.all_gather_into_tensor(self._recv, self._send, group=self.group)
        if self._rows is None:
            return self._recv[: self.n_pairs]
        torch.index_select(self._recv, 0, self._rows, out=self._out)   # unequal blocks: drop the padding rows
        return self._out


def track_sequence_landmarks_sharded(tracker, params, frames, table, first_frame=0, n_warm=0, group=None,
                                     timings=None):
    """:meth:`Tracker.track_sequence_landmarks` over the whole sequence, its pairs sharded over the ranks of
    `group` in the blocks of :func:`shard_pairs`, with the table relayed from rank to rank.

    frames = (semi, semi_scale, desc, desc_scale, depth): the WHOLE sequence (n frames), on this rank's device;
    each rank reads its block, its halo frame and up to n_warm frames before the block.  table: this rank's
    landmark table, the entry table on rank 0 (it is read there only); on return every rank holds the final
    table.  params.pnp.first_pair is the pair index of the sequence's first pair.  Each rank prepares its block
    (reading no table), receives the table from rank r - 1, steps it, sends it to rank r + 1 and solves; the
    records come back with one all_gather (:class:`ResultGather`), the landmark counts with another, the final
    table with a broadcast from the last rank.  Every exchange is stream-ordered (NCCL on the current stream), so
    nothing waits on the host.  Returns (uint8 [n - 1, 64] records, int32 [n - 1] counts, int32 re-walked words of
    this rank's block).  `timings`: a list that receives this rank's CUDA events (prepare, table wait,
    step_table, solve), for measurement."""
    semi, semi_scale, desc, desc_scale, depth = frames

    def prepare(p, w, ff, lo, hi):
        return tracker.track_landmarks_prepare(p, w, ff, semi[lo:hi], semi_scale[lo:hi], desc[lo:hi],
                                               desc_scale[lo:hi], depth[lo:hi], table.shape[0])
    return _relay_landmarks(tracker, params, semi.shape[0] - 1, table, first_frame, n_warm, group, None, timings,
                            prepare)[:3]


def track_sequence_landmarks_host_sharded(tracker, params, host_frames, table, first_frame=0, n_warm=0, group=None,
                                          counts=None, timings=None):
    """:func:`track_sequence_landmarks_sharded` from host buffers: each rank stages only its block, its halo frame
    and up to n_warm warm-up frames through its own link (:meth:`Tracker.track_landmarks_prepare_host`), then the
    table is relayed as there.

    host_frames = (semi, semi_scale, desc, desc_scale, depth): the WHOLE sequence in host memory (pinned CPU
    tensors or numpy arrays).  `counts`: pairs per rank of a weighted partition (:func:`shard_pairs_weighted`, for
    ranks whose host links differ); default: the equal blocks of :func:`shard_pairs`.  Returns (uint8 [n - 1, 64]
    records, int32 [n - 1] counts, int32 re-walked words of this rank's block, this rank's h2d bytes), the first
    two on this rank's device.  `timings` as :func:`track_sequence_landmarks_sharded` (prepare is the device time
    after the prepare call's start; the call itself returns once staging is done)."""
    def prepare(p, w, ff, lo, hi):
        return tracker.track_landmarks_prepare_host(p, w, ff, *[x[lo:hi] for x in host_frames], table.shape[0])
    return _relay_landmarks(tracker, params, host_frames[0].shape[0] - 1, table, first_frame, n_warm, group, counts,
                            timings, prepare)


def _relay_landmarks(tracker, params, n_pairs, table, first_frame, n_warm, group, counts, timings, prepare):
    """The relay of the sharded landmark calls.  prepare(params, n_warm, first_frame, lo, hi) prepares this rank's
    block from frames [lo, hi) of the sequence (its warm-up frames, its pairs and its halo frame).  Returns
    (records, counts, re-walked words, the block's "h2d_bytes" or 0)."""
    import copy
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    gat = ResultGather(n_pairs, world, rank, tracker.device, group=group, counts=counts)
    first, count = gat.first, gat.count
    nl_send = torch.zeros((gat.per,), dtype=torch.int32, device=tracker.device)
    rewalked = torch.zeros((1,), dtype=torch.int32, device=tracker.device)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)] if timings is not None else None
    if ev:
        ev[0].record()
    block = None
    if count > 0:
        w = min(int(n_warm), first)
        p = copy.copy(params)
        p.pnp = copy.copy(params.pnp)
        p.pnp.first_pair = params.pnp.first_pair + first
        block = prepare(p, w, first_frame + first, first - w, first + count + 1)
    if ev:
        ev[1].record()
    src = _global_rank(group, rank - 1)
    dst = _global_rank(group, rank + 1)
    if rank > 0:
        dist.recv(table, src=src, group=group)
    if ev:
        ev[2].record()
    if block is not None:
        tracker.track_landmarks_step_table(block, table, rewalked)
    if ev:
        ev[3].record()
    if rank + 1 < world:
        dist.send(table, dst=dst, group=group)
    if block is not None:
        tracker.track_landmarks_solve(block, out=gat.send, n_with_landmark=nl_send[:count])
    if ev:
        ev[4].record()
        timings.extend(ev)
    records = gat.gather()
    if world > 1:
        nl_all = torch.empty((world * gat.per,), dtype=torch.int32, device=tracker.device)
        dist.all_gather_into_tensor(nl_all, nl_send, group=group)
        dist.broadcast(table, src=_global_rank(group, world - 1), group=group)
    else:
        nl_all = nl_send
    h2d = 0
    if block is not None:
        h2d = block.get("h2d_bytes", 0)
        tracker.track_landmarks_release(block)
    # equal blocks start at rank * per, so only the tail is padding; weighted ones drop it as the records do
    nl = nl_all[:n_pairs] if gat._rows is None else nl_all.index_select(0, gat._rows)
    return records, nl, rewalked, h2d


def _global_rank(group, r):
    import torch.distributed as dist
    return r if group is None else dist.get_global_rank(group, r)


# --------------------------------------------------------------------------------------
# host side of the host-buffer path: staging memory next to the GPU
# --------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(device_index: int):
    """Restricts this process to the CPUs of the NUMA node GPU `device_index` hangs off, so that the
    pinned staging buffers it allocates afterwards (first touch) are local to that GPU's PCIe root.
    One process per GPU (torchrun) is the intended use.  Returns the node number, or None when the
    platform does not say (single-node hosts, containers without sysfs) -- then nothing changes."""
    import os
    try:
        import torch
        bus = torch.cuda.get_device_properties(device_index).pci_bus_id  # torch >= 2.5
        dom = getattr(torch.cuda.get_device_properties(device_index), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(device_index), "pci_device_id", 0)
        path = "/sys/bus/pci/devices/%04x:%02x:%02x.0/numa_node" % (dom, bus, dev)
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None
