"""Inputs and helpers that several test modules use: one copy of each.

A plain module, imported by name: pytest puts tests/ on sys.path for the test modules, and the multi-rank workers add
it themselves.  Nothing here is a test or a fixture; each module keeps its own fixtures, which call into this one.
"""
import copy
import ctypes as C
import os
import socket

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


# ------------------------------------------------------------------ arrays and buffers
def ref_vocab():
    """The reference's vocabulary (base_desc, scale, bias, leaves)."""
    v = np.load(os.path.join(GOLDEN, "ref_vocab.npz"))
    return v["base_desc"], v["scale"], v["bias"], v["leaves"]


def dev(tracker, a):
    """A numpy array on the tracker's device."""
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(tracker.device)


def pinned(a):
    """A pinned host copy of a torch tensor (on any device) or a numpy array."""
    import torch
    if isinstance(a, np.ndarray):
        a = torch.from_numpy(np.ascontiguousarray(a))
    return torch.empty(a.shape, dtype=a.dtype, pin_memory=True).copy_(a)


def table_bytes(t):
    return t.cpu().numpy().tobytes()


def upload_table(tracker, host_table):
    """A landmark table in the oracle's layout (oracle.pool_new) on the tracker's device."""
    return dev(tracker, host_table.view(np.uint8).reshape(-1, 56))


def same_bits(a, b):
    """float32 arrays equal bit for bit, a NaN equal to any NaN (x86 and CUDA write different NaN bits)."""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and (na == nb).all() and (a[~na].view(np.int32) == b[~nb].view(np.int32)).all()


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


# ------------------------------------------------------------------ parameters and problems
def with_first_pair(p, first_pair):
    """A copy of track parameters p with pnp.first_pair set."""
    q = copy.copy(p)
    q.pnp = copy.copy(p.pnp)
    q.pnp.first_pair = first_pair
    return q


def pnp_params(H, lanes=1, seed=0, refine=10, sample_size=8):
    """mv_pnp_params_default with these fields set (refine_iters 10 and sample_size 8 are the defaults)."""
    from maveric_slam_b200 import lib
    p = lib.PnpParams()
    lib.load().mv_pnp_params_default(C.byref(p))
    p.hypotheses, p.lanes_per_hypothesis, p.seed, p.refine_iters = H, lanes, seed, refine
    p.sample_size = sample_size
    return p


def pnp_problems(synth, P, n, stride):
    """P synthetic PnP problems of n correspondences -> corr float32 [P, 5, stride]."""
    corr = np.zeros((P, 5, stride), np.float32)
    for p in range(P):
        corr[p], _, _ = synth.synth_pnp_problem(500 + p, n, stride=stride)
    return corr


def spd_system(rng, P, cond=1.0):
    """(C as lba_schur lays it out, S, g) for a random SPD pose block."""
    n = 6 * P
    A = rng.normal(size=(n + 24, n)) * np.logspace(0, np.log10(cond), n)
    S = (A.T @ A).astype(np.float32)
    S = np.tril(S) + np.tril(S, -1).T
    g = rng.normal(size=n).astype(np.float32)
    C_ = np.zeros((n + 1, n + 1), np.float32)
    C_[:n, :n] = S.T                    # [column, row]
    C_[:n, n] = g                       # last row
    C_[n, n] = 3.0
    return C_, S, g


def blocks_then_rest(n_pairs, sizes):
    """Blocks (first pair, count) of the given sizes, each once, then one block of the pairs left."""
    out, lo = [], 0
    for s in sizes:
        if lo < n_pairs:
            out.append((lo, min(s, n_pairs - lo)))
            lo += out[-1][1]
    if lo < n_pairs:
        out.append((lo, n_pairs - lo))
    return out


def cycled_blocks(sizes, n_pairs):
    """Blocks (first pair, count) whose sizes cycle through `sizes` to the last pair."""
    out, lo, i = [], 0, 0
    while lo < n_pairs:
        c = min(sizes[i % len(sizes)], n_pairs - lo)
        out.append((lo, c))
        lo, i = lo + c, i + 1
    return out


# ------------------------------------------------------------------ the reference's local feature pool
class LocalFeature(C.Structure):
    _fields_ = [("word_id", C.c_int), ("frame_ptr", C.c_int), ("num_frames", C.c_int), ("frames", C.c_int * 8),
                ("coords_3D", C.c_float * 3)]


class HashEntry(C.Structure):
    _fields_ = [("key", C.c_int), ("value", LocalFeature), ("is_occupied", C.c_bool)]


class Pool(C.Structure):
    _fields_ = [("entries", HashEntry * 3000), ("size", C.c_int), ("capacity", C.c_int)]


class InsertResult(C.Structure):
    _fields_ = [("feature", C.POINTER(LocalFeature)), ("inserted", C.c_bool)]


def frame_ids(rng, prev, per_frame=200, n_words=10000):
    keep = rng.choice(prev, 75, replace=False)
    fresh = rng.choice(np.setdiff1d(np.arange(n_words), keep), per_frame - 75, replace=False)
    return np.concatenate([keep, fresh]).astype(np.int32)


def pool_contents(pool):
    out = {}
    for e in pool.entries:
        if e.is_occupied:
            f = e.value
            out[e.key] = (tuple(f.frames[(f.frame_ptr + k) % 8] for k in range(f.num_frames)), tuple(f.coords_3D))
    return out


def table_contents(table):
    out = {}
    for r in table[table["word_id"] >= 0]:
        assert r["word_id"] >= 0
        out[int(r["word_id"])] = (tuple(int(r["frames"][(r["frame_ptr"] + k) % 8]) for k in range(r["num_frames"])),
                                  tuple(float(c) for c in r["coords"]))
    return out


def drive_host_pool(L, frames=60, seed=0):
    """src/local_feature_matching.c:153-163 on the product's host pool (pinned to the reference's header)."""
    L.local_feature_pool_insert.restype = InsertResult
    L.local_feature_pool_insert.argtypes = [C.POINTER(Pool), C.c_int, LocalFeature]
    pool = Pool()
    L.init_local_feature_pool(C.byref(pool))
    rng = np.random.default_rng(seed)
    prev = rng.choice(10000, 200, replace=False)
    snaps = []
    for f in range(frames):
        ids = frame_ids(rng, prev)
        coords = rng.normal(size=(len(ids), 3)).astype(np.float32)
        for wid, c in zip(ids, coords):
            feat = LocalFeature()
            L.init_local_feature_with_id(C.byref(feat), int(wid), f)
            feat.coords_3D = (C.c_float * 3)(*c)
            res = L.local_feature_pool_insert(C.byref(pool), int(wid), feat)
            if not res.inserted:
                L.update_local_feature(res.feature, f)
        L.local_feature_pool_remove_old(C.byref(pool), f)
        snaps.append((ids, coords, pool_contents(pool)))
        prev = ids
    return snaps


# ------------------------------------------------------------------ the landmark sequence of the landmark modules
N_FRAMES, FIRST = 66, 500
KEYS = ("semi", "sscale", "desc", "dscale", "depth")
WARMS = (0, 1, 7, 8, 16, 64)     # warm-up frame counts of the block tests


def landmark_sequence(tracker, synth, n_frames=N_FRAMES, rows=47, cols=155, seed=21, params=None, first_frame=FIRST,
                      edit=None, host=False):
    """A synthetic sequence (KITTI-shaped by default) and the device landmark path's answer on it, from an empty table
    at first_frame, with the reference vocabulary set on `tracker`.  edit(semi, desc, depth) may change the frames
    before anything runs.  -> dict(p, d: device frames by KEYS, h: pinned host copies by KEYS (host=True) or None,
    first, n_words, res: PAIR_RESULT_DTYPE records, nl: int32 matches with a landmark, table: final table bytes)."""
    import torch
    from maveric_slam_b200 import tracking
    tracker.bow_set_vocabulary(*ref_vocab())
    p = tracking.kitti_track_params(hypotheses=256) if params is None else params
    semi, desc, depth = tracker.synth_frames(seed, rows, cols, 0, synth.default_offsets(n_frames, seed))
    if edit is not None:
        edit(semi, desc, depth)
    sscale = torch.full((n_frames,), float(synth.SEMI_SCALE), device=tracker.device)
    dscale = torch.full((n_frames,), 4.3353, device=tracker.device)
    d = dict(zip(KEYS, (semi, sscale, desc, dscale, depth)))
    table = tracker.landmarks_new(tracker.n_words)
    res, nl = tracker.track_sequence_landmarks(p, *d.values(), table, first_frame=first_frame)
    h = None
    if host:
        h = {k: pinned(t) for k, t in d.items()}
        torch.cuda.synchronize()
    return dict(p=p, d=d, h=h, first=first_frame, n_words=tracker.n_words, res=tracking.results_to_numpy(res),
                nl=nl.cpu().numpy(), table=table_bytes(table))


def landmarks_host(tracker, s, h=None, first=FIRST, lo=0, hi=N_FRAMES, table=None, p=None):
    """mv_track_sequence_landmarks_host on frames lo .. hi-1 of the landmark sequence s (its pinned copies, or the
    buffers h by KEYS) -> (records, matches with a landmark, table, h2d bytes, d2h bytes)."""
    from maveric_slam_b200 import tracking
    h = h or s["h"]
    table = tracker.landmarks_new(s["n_words"]) if table is None else table
    p = p or (s["p"] if lo == 0 else tracking.kitti_track_params(hypotheses=256, first_pair=lo))
    res, nl, up, down = tracker.track_sequence_landmarks_host(p, *[h[k][lo:hi] for k in KEYS], table, first_frame=first)
    return res, nl, table, up, down


# ------------------------------------------------------------------ stand-ins for the relay tests
class StandIn:
    """The block calls of a Tracker on the CPU, with a table step that is not associative: any other order of the
    relay than rank order, or a table read before it arrives, changes the final table and the records."""

    def __init__(self):
        import torch
        self.torch = torch
        self.device = torch.device("cpu")

    def track_landmarks_prepare(self, p, n_warm, first_frame, semi, *rest):
        return {"first": p.pnp.first_pair, "n_pairs": semi.shape[0] - n_warm - 1, "n_warm": n_warm,
                "frame": first_frame}

    def track_landmarks_step_table(self, block, table, n_rewalked=None):
        for i in range(block["n_pairs"]):
            table.copy_(((table.to(self.torch.int64) * 7 + block["first"] + i + 3) % 251).to(self.torch.uint8))
        block["state"] = table.clone()
        if n_rewalked is not None:
            n_rewalked.fill_(block["n_warm"])

    def track_landmarks_solve(self, block, out, n_with_landmark):
        for i in range(block["n_pairs"]):
            out[i] = block["state"].reshape(-1)[:64] + i
            n_with_landmark[i] = block["frame"] + i

    def track_landmarks_release(self, block):
        block.clear()


class HostStandIn(StandIn):
    def track_landmarks_prepare_host(self, p, n_warm, first_frame, semi, *rest):
        b = self.track_landmarks_prepare(p, n_warm, first_frame, semi, *rest)
        b["h2d_bytes"] = 1000 * semi.shape[0]
        return b
