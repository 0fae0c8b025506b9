"""The batched detector stages against the CPU oracle on batches built to sit on their batch logic
(src/top_N.c, src/run_nms.c):

  K0a  mv_softmax_batch  frames whose cells share a 32-lane warp or a 256-cell tile with the next
                         frame's, each frame with its own semi scale (0, 1e-30, 1e10 -> NaN
                         probabilities, negative, NaN); num_valid of every frame
  K0b  mv_top_n_batch    valid counts below, at and above top_n and max_valid in one launch, a cut
                         that ties with the probabilities, and input that NMS rewrote
  NMS  mv_nms_batch      (max_idx, prob) arrays built so that the visiting order, ties, the patch-0
                         quirk and non-finite probabilities show in the answer; edge shapes, batches
                         that are not a multiple of a CTA's 4 frames, and a full-length batch

Bit-exact throughout; NaN probabilities compare as NaN (x86 and CUDA write different NaN bits).
Every builder asserts, on the oracle's answer, that it reaches the case it was built for.  For NMS
that is shown with `nms_emulated`, the reference's loop in Python with its corner order and its two
arg-max scans as parameters (held to the oracle in the reference's order by a CPU test): a built
frame's answer must change when the property it is built for is switched off."""
import functools

import numpy as np
import pytest

from adversarial import adversarial_logits
from helpers import dev, same_bits

F32 = np.float32
FLT_MAX = F32(np.finfo(np.float32).max)
SEMI_SCALE = 0.3562202453613281                              # synth.SEMI_SCALE


# ------------------------------------------------------------------ references
def _cut(v, N):
    """top_N.c:108-109 on the probabilities v of the valid cells (no NaN among them)."""
    hi = max(F32(0), v.max())                                # :69,79-80
    lo = min(FLT_MAX, v.min())
    split = F32(N) / F32(len(v))
    with np.errstate(over="ignore", invalid="ignore"):
        return hi * split + lo * (F32(1) - split)            # float32 scalars: rounded per operation


def top_n_from_cells(max_idx, prob, N, max_valid):
    """top_N.c:53-134 from the softmax stage's (max_idx, prob) instead of the logits.
    -> (patch, idx, prob, count, overflow)."""
    mi = np.asarray(max_idx, np.int32).reshape(-1)
    pr = np.asarray(prob, np.float32).reshape(-1)
    patch = np.flatnonzero((mi != 64) & (pr.astype(np.float64) > 0.01))     # :77, a double compare
    nv = len(patch)
    if nv >= max_valid:                                      # :91-94: the reference exits
        return patch[:0], mi[:0], pr[:0], 0, 1
    if nv > N:                                               # :108-121
        v = pr[patch]
        patch = patch[v >= _cut(v, N)]
    patch = patch[:N]                                        # first N in patch order
    return patch, mi[patch], pr[patch], len(patch), 0


def nms_emulated(rows, cols, max_idx, prob, order="reference", skip_patch0=True, strict_ties=True):
    """run_nms.c:65-156 in Python.  order="reference": corners x outer, y inner; "x+y": wavefronts
    t = x + y, where corners (x, y) and (x+1, y-1) share a cell, every corner of a wavefront
    gathering before any of them writes (lanes of one warp).  skip_patch0 / strict_ties: the first
    arg-max scan ignores patch 0 (:116) / the second takes a later keypoint only if it is strictly
    stronger (:126).  -> (max_idx, prob, wavefronts t = 2x + y of the corners that suppressed)."""
    mi = [int(v) for v in max_idx]
    pr = [float(v) for v in np.asarray(prob, np.float32)]

    def gather(xi, yi):
        out = []
        for xd in (-1, 0):
            xg = xi + xd
            if xg < 0 or xg >= cols:
                continue
            for yd in (-1, 0):
                yg = yi + yd
                if yg < 0 or yg >= rows:
                    continue
                patch = xg * rows + yg
                index = mi[patch]
                if index == 64:
                    continue
                px, py = index % 8, index // 8
                if (xd == -1 and px < 2) or (xd == 0 and px >= 6) or (yd == -1 and py < 2) or (yd == 0 and py >= 6):
                    continue
                out.append([patch, pr[patch], xg * 8 + px, yg * 8 + py])
        return out

    def decide(kp):
        gone = []
        while True:
            best, bi = 0.0, -1
            for i, k in enumerate(kp):
                if (k[0] > 0 or (not skip_patch0 and k[0] == 0)) and k[1] > best:
                    best, bi = k[1], i
            if bi == -1:
                return gone
            for i, k in enumerate(kp):
                if k[0] >= 0 and (k[1] > best or (not strict_ties and k[1] == best)):
                    best, bi = k[1], i
            for i, k in enumerate(kp):
                if i != bi and k[0] >= 0 and abs(kp[bi][2] - k[2]) < 4 and abs(kp[bi][3] - k[3]) < 4:
                    gone.append(k[0])
                    k[0], k[1] = -1, -1.0
            kp[bi][0], kp[bi][1] = -1, -1.0

    if order == "reference":
        waves = [[(x, y)] for x in range(cols + 1) for y in range(rows + 1)]
    else:
        waves = [[(t - y, y) for y in range(rows + 1) if 0 <= t - y <= cols] for t in range(cols + rows + 1)]
    fired = []
    for wave in waves:
        decided = [(c, decide(gather(*c))) for c in wave]
        for (x, y), gone in decided:
            for p in gone:
                mi[p], pr[p] = 64, 64.0
            if gone:
                fired.append(2 * x + y)
    return np.array(mi, np.int32), np.array(pr, np.float32), sorted(set(fired))


def _same_nms(a, b):
    return (a[0] == b[0]).all() and same_bits(a[1], b[1])


# ------------------------------------------------------------------ K0a batches
SOFTMAX_CELLS = (1, 31, 33, 255, 257, 1920, 7285)
FRAME_SCALES = (SEMI_SCALE, 0.0, 1e-30, 3.0, 1e10, -0.35, float("nan"))


@functools.lru_cache(maxsize=None)
def softmax_batch(oracle, synth, cells):
    """-> (semi int8 [n, cells, 65], scale float32 [n], oracle (idx, prob, nv) per frame).  At least 3
    tiles of 256 cells and a frame per scale; contents alternate adversarial_logits palettes (rolled, cut or tiled to size)
    and synthetic frames; scales cycle through FRAME_SCALES."""
    n = max(len(FRAME_SCALES), -(-3 * 256 // cells))
    semi = np.empty((n, cells, 65), np.int8)
    for f in range(n):
        if f % 3 == 2:
            semi[f] = synth.synth_frame(50 + f, 1, cells, f, 0, 0, 400)[0]
        else:
            semi[f] = np.resize(np.roll(adversarial_logits((5 * f + f // 7) % 6), -37 * f, axis=0), (cells, 65))
    scale = np.array([FRAME_SCALES[f % len(FRAME_SCALES)] for f in range(n)], np.float32)
    ref = [oracle.softmax(float(scale[f]), semi[f]) for f in range(n)]

    # reaches: valid cells of two frames in one warp (where a frame's cells are not a multiple of 32)
    # and in one tile, frames of each scale holding valid cells, NaN probabilities among them
    valid = np.concatenate([r[0] != 64 for r in ref])
    frame = np.repeat(np.arange(n), cells)

    def straddles(width):
        return any(np.unique(frame[k:k + width][valid[k:k + width]]).size > 1 for k in range(0, n * cells, width))
    assert straddles(256)
    assert straddles(32) == (cells % 32 != 0)
    for k, s in enumerate(FRAME_SCALES):
        has = sum(r[2] for f, r in enumerate(ref) if f % len(FRAME_SCALES) == k) > 0
        assert has == (s == s), (cells, s)                   # a NaN scale makes every cell the dustbin's
    assert any(np.isnan(r[1][r[0] != 64]).any() for r in ref)
    return semi, scale, ref


# ------------------------------------------------------------------ K0b batches
TOP_N_CELLS = 1920
TOP_N_KS = (1, 100, 300)                                     # 300: two 256-cell rounds of compaction


def _with_valid_count(oracle, semi, scale, target, rng):
    """semi with all but `target` of its valid cells (top_N.c:77) turned into dustbin-only cells."""
    semi = semi.copy()
    idx, pr, _ = oracle.softmax(scale, semi)
    valid = np.flatnonzero((idx != 64) & (pr.astype(np.float64) > 0.01))
    assert len(valid) >= target
    drop = rng.choice(valid, len(valid) - target, replace=False)
    semi[drop, :64] = -1
    semi[drop, 64] = 0
    return semi


def _tied_frame(count, rng):
    """`count` valid cells, every one with 64 zero logits and a dustbin of -1: probability 1/64 each, so
    the cut interpolates between equal hi and lo and lands on that probability."""
    semi = np.full((TOP_N_CELLS, 65), -50, np.int8)
    semi[:, 64] = 60
    semi[rng.choice(TOP_N_CELLS, count, replace=False)] = np.r_[np.zeros(64, np.int8), np.int8(-1)]
    return semi


@functools.lru_cache(maxsize=None)
def top_n_batch(oracle, synth, K):
    """-> (semi [7, 1920, 65], scale [7], max_valid values).  Valid counts K-1, K, K+1, 0, 2K (tied at the
    cut), K+1 (tied) and an unedited adversarial frame, for one launch's top_n = K."""
    rng = np.random.default_rng(300 + K)
    syn = [synth.synth_frame(70 + k, 24, 80, k, 0, 0, 600)[0] for k in range(3)]
    scale = np.array([SEMI_SCALE, SEMI_SCALE, 3.0, SEMI_SCALE, SEMI_SCALE, SEMI_SCALE, 1.0], np.float32)
    frames = [_with_valid_count(oracle, adversarial_logits(0), SEMI_SCALE, K - 1, rng),
              _with_valid_count(oracle, syn[0], SEMI_SCALE, K, rng),
              _with_valid_count(oracle, syn[1], 3.0, K + 1, rng),
              _with_valid_count(oracle, syn[2], SEMI_SCALE, 0, rng),
              _tied_frame(2 * K, rng),
              _tied_frame(K + 1, rng),
              adversarial_logits(4)]
    semi = np.stack(frames)
    max_valids = (K, K + 1, TOP_N_CELLS + 1)

    # reaches: the valid counts; overflowing and normal frames in one launch at max_valid K and K+1;
    # probabilities equal to the cut among the cells taken
    nv = []
    for f in range(len(frames)):
        idx, pr, _ = oracle.softmax(float(scale[f]), semi[f])
        nv.append(int(((idx != 64) & (pr.astype(np.float64) > 0.01)).sum()))
    assert nv[:6] == [K - 1, K, K + 1, 0, 2 * K, K + 1] and nv[6] > K
    for mv in max_valids[:2]:
        ov = [oracle.top_n(float(scale[f]), semi[f], K, mv)[3] for f in range(len(frames))]
        assert 0 < sum(ov) < len(frames), (mv, ov)
    pa, ix, pp, ov = oracle.top_n(float(scale[4]), semi[4], K, TOP_N_CELLS + 1)
    assert ov == 0 and len(pa) == K and (pp == _cut(np.full(2 * K, 1 / 64, np.float32), K)).all()
    return semi, scale, max_valids


# ------------------------------------------------------------------ NMS frames
NMS_SHAPES = ((1, 1), (1, 97), (97, 1), (31, 40), (32, 40), (33, 40), (63, 9), (64, 9), (65, 9), (24, 80), (47, 155))
NMS_KINDS = ("chain_diag", "patch0", "chain_rows", "chain_cols", "ties", "special", "dense")
SPECIAL_PROBS = np.array([0.0, -0.0, -1.0, 1e-40, 0.5, 1.0, 64.0, np.inf, np.nan], np.float32)


def _index(px, py):
    return py * 8 + px


def _nms_frame(kind, rows, cols, seed):
    rng = np.random.default_rng(seed)
    cells = rows * cols
    x, y = np.divmod(np.arange(cells), rows)
    mi = np.full(cells, 64, np.int32)
    pr = np.full(cells, -1.0, np.float32)
    if kind in ("dense", "special", "ties"):
        on = rng.random(cells) < 0.8
        mi[on] = _index(rng.integers(0, 8, on.sum()), rng.integers(0, 8, on.sum()))
        if kind == "dense":
            pr[on] = rng.random(on.sum()).astype(np.float32)
        elif kind == "special":
            pr[on] = SPECIAL_PROBS[rng.integers(0, len(SPECIAL_PROBS), on.sum())]
        else:                                              # ties: two values, four-way ties at most corners
            pr[on] = np.where(rng.random(on.sum()) < 0.8, F32(0.5), F32(0.25))
            mi[0], pr[0] = _index(7, 7), F32(0.5)          # patch 0 ties with the running maximum of corner (1, 1)
    elif kind.startswith("chain"):
        # keypoints in a band of cells at any position (2..5 are gathered by two corners per axis, which
        # carries a suppression from one corner to the next), probabilities rising / falling in patch
        # order; over it, along the band, a chain A > B > C > D whose answer the corner order decides:
        # corner (1, 2) [t = 2x + y = 4] gathers A and B, corner (2, 1) [t = 5] gathers B, C and D.  A
        # suppresses B, so C survives to suppress D; were (2, 1) first, B would suppress C and D survive.
        band = {"chain_rows": (y - rows // 2 + 1) // 3 == 0, "chain_cols": (x - cols // 2 + 1) // 3 == 0,
                "chain_diag": np.abs(x - y) <= 1}[kind]
        band |= min(rows, cols) <= 2                       # a 1- or 2-cell-wide grid: all of it
        mi[band] = _index(rng.integers(0, 8, band.sum()), rng.integers(0, 8, band.sum()))
        ramp = ((np.arange(cells) + 1) / (cells + 1)).astype(np.float32)
        pr[band] = (ramp if kind == "chain_rows" else ramp[::-1])[band]
        if min(rows, cols) >= 3:
            origins = {"chain_rows": [(k, rows // 2 - 1) for k in range(0, cols - 2, 3)],
                       "chain_cols": [(cols // 2 - 1, k) for k in range(0, rows - 2, 3)],
                       "chain_diag": [(k, k) for k in range(0, min(rows, cols) - 2, 3)]}[kind]
            for ox, oy in origins:
                for (cx, cy, px, py, p) in ((1, 2, 2, 0, 0.9), (1, 1, 5, 5, 0.6), (2, 1, 0, 2, 0.3), (2, 0, 0, 7, 0.1)):
                    c = (ox + cx) * rows + (oy + cy)
                    mi[c], pr[c] = _index(px, py), F32(p)
    elif kind == "patch0":
        # patch 0 at pixel (7, 7) with prob 0.9; the first arg-max scan skips it, so its neighbour
        # 1 px away survives while its own prob is <= 0 (0.0 here); patch 1 of a 1-row grid is on its right
        on = rng.random(cells) < 0.5
        mi[on] = _index(rng.integers(0, 8, on.sum()), rng.integers(0, 8, on.sum()))
        pr[on] = rng.random(on.sum()).astype(np.float32)
        near = (x <= 1) & (y <= 1)
        mi[near], pr[near] = 64, -1.0
        mi[0], pr[0] = _index(7, 7), F32(0.9)
        if cells > 1:
            mi[1], pr[1] = (_index(7, 0) if rows > 1 else _index(0, 7)), F32(0.0)
    return mi, pr


@functools.lru_cache(maxsize=None)
def nms_frames(oracle, rows, cols):
    """-> (max_idx [7, cells], prob [7, cells]), one frame of each of NMS_KINDS."""
    built = [_nms_frame(k, rows, cols, 1000 * rows + cols + j) for j, k in enumerate(NMS_KINDS)]
    mi = np.stack([b[0] for b in built])
    pr = np.stack([b[1] for b in built])
    cells = rows * cols
    for j, kind in enumerate(NMS_KINDS):
        ref = oracle.nms(rows, cols, mi[j], pr[j])
        _, _, fired = nms_emulated(rows, cols, mi[j], pr[j])
        if cells == 1:
            continue
        if kind.startswith("chain") and min(rows, cols) >= 3:
            # suppressions on consecutive wavefronts, and an answer the order of the corners decides
            assert any(t + 1 in fired for t in fired), (rows, cols, kind)
            assert not _same_nms(ref, nms_emulated(rows, cols, mi[j], pr[j], order="x+y")), (rows, cols, kind)
        elif kind == "patch0":
            assert ref[0][1] != 64 and not _same_nms(ref, nms_emulated(rows, cols, mi[j], pr[j], skip_patch0=False))
        elif kind == "ties":
            assert not _same_nms(ref, nms_emulated(rows, cols, mi[j], pr[j], strict_ties=False)), (rows, cols)
        elif kind == "special":
            kept = ref[0] != 64
            assert ref[2] > 0 and (np.isnan(ref[1]) & kept).any() and (np.isinf(ref[1]) & kept).any(), (rows, cols)
    return mi, pr


# ------------------------------------------------------------------ CPU: references and builders
def test_top_n_from_cells_equals_oracle_top_n(oracle, synth):
    """top_n_from_cells on the oracle's softmax output == orc.top_n on the logits, overflow included."""
    cases = [(adversarial_logits(s), sc) for s in range(6) for sc in (0.01, 0.35622698, 1.0, 3.0)]
    cases += [(adversarial_logits(s), sc) for s in (0, 3) for sc in FRAME_SCALES]
    cases += [(synth.synth_frame(5, r, c, 0, 3, -2, pm)[0], SEMI_SCALE) for r, c in ((24, 80), (47, 155))
              for pm in (140, 550)]
    n_cut = n_over = 0
    for semi, sc in cases:
        idx, pr, _ = oracle.softmax(sc, semi)
        nv = int(((idx != 64) & (pr.astype(np.float64) > 0.01)).sum())
        for N in sorted({1, 37, 100, nv - 1, nv, nv + 1} - {0, -1}):
            for mv in (len(semi) + 1, nv, nv + 1):
                if mv <= 0:
                    continue
                a = top_n_from_cells(idx, pr, N, mv)
                b = oracle.top_n(sc, semi, N, mv)
                assert a[4] == b[3] and a[3] == len(b[0]), (sc, N, mv)
                assert (a[0] == b[0]).all() and (a[1] == b[1]).all() and same_bits(a[2], b[2]), (sc, N, mv)
                n_cut += a[4] == 0 and 0 < N < nv
                n_over += a[4]
    assert n_cut > 100 and n_over > 100


@pytest.mark.parametrize("rows,cols", NMS_SHAPES)
def test_nms_emulator_equals_oracle(oracle, rows, cols):
    """The emulator the NMS builders reason with == orc.nms in the reference's order (and so is the
    second pass over its own answer)."""
    mi, pr = nms_frames(oracle, rows, cols)
    for f in range(len(mi)):
        ref = oracle.nms(rows, cols, mi[f], pr[f])
        emu = nms_emulated(rows, cols, mi[f], pr[f])
        assert _same_nms(ref, emu), (rows, cols, NMS_KINDS[f])
        assert _same_nms(oracle.nms(rows, cols, ref[0], ref[1]), nms_emulated(rows, cols, emu[0], emu[1]))


def test_builders_reach_their_cases(oracle, synth):
    for cells in SOFTMAX_CELLS:
        softmax_batch(oracle, synth, cells)
    for K in TOP_N_KS:
        top_n_batch(oracle, synth, K)


# ------------------------------------------------------------------ GPU
def _check_top_n(got, want_per_frame):
    qp, qi, qpr, qc, ov = (t.cpu().numpy() for t in got)
    for f, (pa, ix, pp, n, o) in enumerate(want_per_frame):
        assert ov[f] == o and qc[f] == n, (f, ov[f], o, qc[f], n)
        assert (qp[f, :n] == pa).all() and (qi[f, :n] == ix).all() and same_bits(qpr[f, :n], pp), f


@pytest.mark.gpu
@pytest.mark.parametrize("cells,aligned", [(c, True) for c in SOFTMAX_CELLS] + [(7285, False)])
def test_softmax_batch_across_frame_boundaries(tracker, oracle, synth, cells, aligned):
    import torch
    semi, scale, ref = softmax_batch(oracle, synth, cells)
    if aligned:
        dsemi = dev(tracker, semi)
    else:                                                   # not 16-byte aligned: the byte-wise staging path
        buf = torch.zeros(semi.size + 64, dtype=torch.int8, device=tracker.device)
        dsemi = buf[5:5 + semi.size].view(semi.shape)
        dsemi.copy_(torch.from_numpy(semi))
    idx, prob, nv = (t.cpu().numpy() for t in tracker.softmax(dsemi, dev(tracker, scale)))
    for f, (i2, p2, n2) in enumerate(ref):
        assert (idx[f] == i2).all() and same_bits(prob[f], p2) and nv[f] == n2, (cells, f, float(scale[f]))



@pytest.mark.gpu
@pytest.mark.parametrize("K", TOP_N_KS)
def test_top_n_batch_at_count_limits(tracker, oracle, synth, K):
    semi, scale, max_valids = top_n_batch(oracle, synth, K)
    idx, prob, _ = tracker.softmax(dev(tracker, semi), dev(tracker, scale))
    for mv in max_valids:
        want = []
        for f in range(len(semi)):
            pa, ix, pp, ov = oracle.top_n(float(scale[f]), semi[f], K, mv)
            want.append((pa, ix, pp, len(pa), ov))
        _check_top_n(tracker.top_n(idx, prob, K, mv), want)


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols", NMS_SHAPES)
def test_nms_on_built_frames(tracker, oracle, rows, cols):
    """Every batch size 1, 4, 5 and 7 (frames rotated), NMS twice in place at 7, and top-N on the
    rewritten arrays (suppressed cells, 64.0, inf and NaN probabilities among them)."""
    mi, pr = nms_frames(oracle, rows, cols)
    n = len(mi)
    cells = rows * cols
    N = max(1, cells // 10)
    for B in (1, 4, 5, 7):
        sel = [(B + j) % n for j in range(B)]
        di, dp = dev(tracker, mi[sel]), dev(tracker, pr[sel])
        tracker.nms(rows, cols, di, dp)
        gi, gp = di.cpu().numpy(), dp.cpu().numpy()
        once = [oracle.nms(rows, cols, mi[f], pr[f]) for f in sel]
        for j, ref in enumerate(once):
            assert (gi[j] == ref[0]).all() and same_bits(gp[j], ref[1]), (B, NMS_KINDS[sel[j]])
        _check_top_n(tracker.top_n(di, dp, N, cells + 1),
                     [top_n_from_cells(ref[0], ref[1], N, cells + 1) for ref in once])
        if B == 7:
            tracker.nms(rows, cols, di, dp)
            gi, gp = di.cpu().numpy(), dp.cpu().numpy()
            for j, ref in enumerate(once):
                twice = oracle.nms(rows, cols, ref[0], ref[1])
                assert (gi[j] == twice[0]).all() and same_bits(gp[j], twice[1]), NMS_KINDS[sel[j]]


@pytest.mark.gpu
def test_run_nms_ex_off_the_native_shape(tracker, oracle):
    from maveric_slam_b200 import tracking
    mi, pr = nms_frames(oracle, 33, 40)
    for f in (NMS_KINDS.index("chain_diag"), NMS_KINDS.index("special")):
        ref = oracle.nms(33, 40, mi[f], pr[f])
        hi, hp = tracking.run_nms(33, 40, mi[f], pr[f])
        assert (hi == ref[0]).all() and same_bits(hp, ref[1]), NMS_KINDS[f]


@pytest.mark.gpu
def test_nms_full_length_batch(tracker, oracle, synth):
    """4541 frames (KITTI sequence 00) at 47x155: synthetic frames -> softmax -> NMS on the device."""
    import torch
    rows, cols, n = 47, 155, 4541
    semi, desc, depth = tracker.synth_frames(17, rows, cols, 0, synth.default_offsets(n, 17))
    del desc, depth
    scale = torch.full((n,), float(synth.SEMI_SCALE), device=tracker.device)
    di, dp, _ = tracker.softmax(semi, scale)
    mi, pr = di.cpu().numpy(), dp.cpu().numpy()
    for f in (0, n - 1):
        i2, p2, _ = oracle.softmax(float(synth.SEMI_SCALE), semi[f].cpu().numpy())
        assert (mi[f] == i2).all() and same_bits(pr[f], p2), f
    del semi
    tracker.nms(rows, cols, di, dp)
    gi, gp = di.cpu().numpy(), dp.cpu().numpy()
    n_sup = 0
    for f in range(n):
        ref = oracle.nms(rows, cols, mi[f], pr[f])
        n_sup += ref[2]
        assert (gi[f] == ref[0]).all() and same_bits(gp[f], ref[1]), f
    assert n_sup > n


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols,N", [(24, 80, 600), (47, 155, 2160)])     # N splits the frames' valid counts
def test_softmax_nms_top_n_on_the_device(tracker, oracle, synth, rows, cols, N):
    cells = rows * cols
    frames = [np.resize(np.roll(adversarial_logits(s), -101 * s, axis=0), (cells, 65)) for s in range(6)]
    frames += [synth.synth_frame(90 + k, rows, cols, k, 0, 0, pm)[0] for k, pm in enumerate((140, 400, 550))]
    semi = np.stack(frames)
    scale = np.array([SEMI_SCALE, 3.0, 1.0, SEMI_SCALE, 0.01, 1e10, SEMI_SCALE, SEMI_SCALE, 0.5], np.float32)
    mv = cells + 1
    di, dp, _ = tracker.softmax(dev(tracker, semi), dev(tracker, scale))
    tracker.nms(rows, cols, di, dp)
    got = tracker.top_n(di, dp, N, mv)
    gi, gp = di.cpu().numpy(), dp.cpu().numpy()
    want = []
    for f in range(len(frames)):
        i2, p2, _ = oracle.softmax(float(scale[f]), semi[f])
        mi, pr, _ = oracle.nms(rows, cols, i2, p2)
        assert (gi[f] == mi).all() and same_bits(gp[f], pr), f
        want.append(top_n_from_cells(mi, pr, N, mv))
    _check_top_n(got, want)
    assert any(0 < w[3] == N for w in want) and any(0 < w[3] < N for w in want)
