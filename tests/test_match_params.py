"""Both matchers and the whole tracking path away from the default match threshold and candidate gate.

Every other test runs the matcher at match_threshold = 0.9, min_prob0 = 0.2 and RANSAC-E at 10 iterations, 1.1.  At
those defaults a threshold or gate converted to fp32 by round to nearest is the same number as the directed rounding
the kernels use (mv_round_down(0.81) is one ulp below (float)0.81, mv_round_up(0.2) == (float)0.2), and nearly every
score sits far from 0.81, so a key filter of the tensor-core matcher that starts too high loses nothing.  Here:

  * a value grid of thresholds (0 .. 4, negative, 1e20, +inf, NaN) and gates (-inf, -1, 0, NaN, 0.05 .. 1.5) runs
    through mv_match_batch (consecutive pairs, and an explicit f0 / f1 list) and mv_match_pair_host, with the dp4a
    (use_tensor_cores = 0) and the tcgen05 (1) matcher, and auto (2) where it picks differently, on synthetic pairs,
    the four hazards of tests/adversarial.py and a crafted pair whose windows reach all three branches of the
    tensor-core key filter's start (den > 0, den < 0, den == 0, den = n_cand * query 64-d norm as int32);
  * boundary cases put threshold^2 and the gate within one ulp of an achieved score or probability, on either
    side, for a winner that is the query's leading candidate (scored in lead_kernel) and one that is not (scored
    after the key filter): the only inputs on which directed and nearest rounding differ;
  * the whole path (mv_track_sequence, mv_track_sequence_host pinned with the row gather and small chunks, pageable,
    without the gather) and the landmark path (device one-call, host chunks of 3, host-prepared blocks) run with a
    low gate and threshold, a threshold above 1, a gate on one cell's probability and RANSAC-E at 0 / 1 iterations
    and thresholds 0, 0.25, 1e30;
  * use_tensor_cores = 1 with a NaN threshold is refused by every entry point before anything is enqueued.

Matches are held to orc_match bit for bit (count, points, cell0, query, score bits), records to orc_track_pair /
tests/landmark_reference.py byte for byte.  _assert_case_reaches checks on the oracle's answers, without a GPU, that
every case reaches what it was built for.
"""
import copy
import math

import numpy as np
import pytest

from conftest import bits
from helpers import pinned, ref_vocab
from landmark_reference import detect, first_difference, landmark_reference, match_cfg, run_entry
from oracle import orc

f32 = np.float32
INF, NAN = float("inf"), float("nan")
DEFAULT_THR, DEFAULT_GATE = 0.9, 0.2


def _nextafter(x, d):
    return float(np.nextafter(x, d))


def _wrap(v):
    """int32 wrap of a Python int (the reference's -fwrapv products)."""
    return (int(v) + 2 ** 31) % 2 ** 32 - 2 ** 31


# ------------------------------------------------------------------ matcher inputs
def _detect(oracle, scale, semi0, semi1, N, max_valid):
    idx, pr, _ = oracle.softmax(float(scale), semi0)
    qp, qi, _, ov = oracle.top_n(float(scale), semi1, N, max_valid)
    assert ov == 0
    return idx, pr, qp, qi


def _curmax_pair(oracle, synth):
    """A 24x80 synthetic pair with four crafted query windows (norms as int32, leading candidate = first valid cell
    of the window at the default gate):
      A   query 64-d = 256-d norm 65536, lead norm 65536: den (256 and 64) == 2^32 == 0, later scores +-inf / NaN;
      A2  query 256-d norm 65537, 64-d norm 65536, lead norm 65536: the lead scores finite, the rest against 0;
      B   query norm 65536, lead norm 32768: den == 2^31 == INT_MIN, scores n / -2^31;
      D   query norm 65536, lead norm 65537: den == 65536, scores up to 2^15 (above any threshold of the grid).
    Every other window is an ordinary one, of either sign of den."""
    rows, cols = 24, 80
    off = synth.default_offsets(2, 22)
    s0, d0, _ = synth.synth_frame(22, rows, cols, 0, int(off[0, 0]), int(off[0, 1]))
    s1, d1, _ = synth.synth_frame(22, rows, cols, 1, int(off[1, 0]), int(off[1, 1]))
    d0, d1 = d0.copy(), d1.copy()
    idx, pr, qp, qi = _detect(oracle, synth.SEMI_SCALE, s0, s1, 100, 1000)
    g = dict(rows=rows, cols=cols, shift=(4, 4), radius=4)
    used, planted = [], {}
    for kind in ("A", "A2", "B", "D"):
        for q, cell1 in enumerate(qp):
            qx, qy = cell1 // rows, cell1 % rows
            if any(abs(qx - u) < 9 and abs(qy - v) < 9 for u, v in used):   # windows of 9 x 9 cells, disjoint
                continue
            win = _window_valid(g, cell1, idx, pr, DEFAULT_GATE)
            if len(win) < 5:
                continue
            used.append((qx, qy))
            planted[kind] = (q, win[:5])
            lead, c2, c3, c4, c5 = win[:5]
            d1[cell1] = 0
            d1[cell1, :4] = -128
            d0[lead] = 0
            d0[lead, :4] = -128
            if kind == "A2":
                d1[cell1, 100] = 1
            if kind == "B":
                d0[lead, 2:4] = 0
            if kind == "D":
                d0[lead, 200] = 1
            # later candidates: dot = -128 * (sum of their first four entries)
            d0[c2, :4] = -98          # dot 50176: dot^2 wraps negative
            d0[c3, :4] = 0            # dot 0
            d0[c4, :4] = (-1, 0, 0, 0)    # dot 128
            d0[c5, :4] = -95          # dot 48640: dot^2 wraps negative
            break
    assert len(planted) == 4
    return dict(rows=rows, cols=cols, N=100, M=150, scale=float(synth.SEMI_SCALE), semi=[s0, s1], desc=[d0, d1],
                det=[(idx, pr, qp, qi), (None, None, qp, qi)], planted=planted)


def _window_valid(g, cell1, idx, pr, gate):
    """Valid frame-0 cells of the query's window in x-outer / y-inner order (tracking_main.c:135-146)."""
    rows, cols, r = g["rows"], g["cols"], g["radius"]
    qx, qy = cell1 // rows, cell1 % rows
    out = []
    for x in range(max(0, qx + g["shift"][0] - r), min(cols - 1, qx + g["shift"][0] + r) + 1):
        for y in range(max(0, qy + g["shift"][1] - r), min(rows - 1, qy + g["shift"][1] + r) + 1):
            c = x * rows + y
            if idx[c] != 64 and not (float(pr[c]) < gate):
                out.append(c)
    return out


def _make_inputs(oracle, synth):
    """name -> dict(rows, cols, N, M, frames: desc int8 [F, cells, 256], idx, prob [F, cells], qp, qi [F, N],
    qc [F], pairs [(f0, f1)]).  Frame f of a chain is frame 1 of pair f - 1 and frame 0 of pair f."""
    from adversarial import adversarial_pair
    out = {}

    def chain(name, seed, rows, cols, permille, n, N, M):
        semi, desc, _, _ = synth.synth_sequence(seed, rows, cols, n, keypoint_permille=permille)
        dets = [_detect(oracle, synth.SEMI_SCALE, semi[f], semi[f], N, rows * cols + 1) for f in range(n)]
        out[name] = _pack(rows, cols, N, M, desc, dets, [(f, f + 1) for f in range(n - 1)])

    chain("syn24", 21, 24, 80, 140, 3, 100, 150)
    chain("syn47", 23, 47, 155, 550, 3, 4000, 4096)
    for seed in range(4):
        scale, s0, d0, s1, d1 = adversarial_pair(oracle, synth, seed)
        a = _detect(oracle, scale, s0, s1, 100, 1000)
        b = _detect(oracle, scale, s1, s1, 100, 1000)
        out["adv%d" % seed] = _pack(24, 80, 100, 150, np.stack([d0, d1]), [a, b], [(0, 1)])
    c = _curmax_pair(oracle, synth)
    out["curmax"] = _pack(24, 80, 100, 150, np.stack(c["desc"]), c["det"], [(0, 1)])
    out["curmax"]["planted"] = c["planted"]
    return out


def _pack(rows, cols, N, M, desc, dets, pairs):
    """dets[f] = (idx, prob, qp, qi) of frame f (idx / prob as frame 0, qp / qi as frame 1 of a pair)."""
    F, cells = len(dets), rows * cols
    idx = np.full((F, cells), 64, np.int32)
    prob = np.zeros((F, cells), f32)
    qp = np.zeros((F, N), np.int32)
    qi = np.zeros((F, N), np.int32)
    qc = np.zeros(F, np.int32)
    for f, (i, p, a, b) in enumerate(dets):
        if i is not None:
            idx[f], prob[f] = i, p
        qc[f] = len(a)
        qp[f, :len(a)], qi[f, :len(a)] = a, b
    return dict(rows=rows, cols=cols, N=N, M=M, desc=np.ascontiguousarray(desc, np.int8), idx=idx, prob=prob, qp=qp,
                qi=qi, qc=qc, pairs=pairs)


def _oracle_pair(oracle, inp, pair, thr, gate):
    a, b = pair
    cfg = orc.MatchCfg(inp["rows"], inp["cols"], 4, 4, 4, inp["M"], thr, gate)
    k = inp["qc"][b]
    return oracle.match(cfg, inp["desc"][a], inp["desc"][b], inp["idx"][a], inp["prob"][a], inp["qp"][b, :k],
                        inp["qi"][b, :k])


def _lead_of(inp, a, cell1, gate):
    """The query's leading candidate: the first valid cell of its window with a non-zero 256-d norm (-1: none)."""
    g = dict(rows=inp["rows"], cols=inp["cols"], shift=(4, 4), radius=4)
    for c in _window_valid(g, cell1, inp["idx"][a], inp["prob"][a], gate):
        if (inp["desc"][a][c].astype(np.int64) ** 2).sum() != 0:
            return c
    return -1


def _match_kinds(inp, pair, m, gate):
    """Per match: (leading?, den) with den = lead 256-d norm * query 64-d norm as int32."""
    a, b = pair
    out = []
    for j in range(m["n"]):
        cell1 = int(inp["qp"][b, m["query"][j]])
        lead = _lead_of(inp, a, cell1, gate)
        n_cand = int((inp["desc"][a][lead].astype(np.int64) ** 2).sum())
        nq64 = int((inp["desc"][b][cell1, :64].astype(np.int64) ** 2).sum())
        out.append((lead == m["cell0"][j], _wrap(n_cand * nq64)))
    return out


# ------------------------------------------------------------------ settings
# name -> (threshold, gate, inputs or None for all)
GRID = {}
for _t in (0.0, 0.5, 0.9, 0.95, 1.0, 1.5, 4.0, -0.9, 1e20, INF, NAN):
    GRID["thr_%r" % _t] = (_t, DEFAULT_GATE, None)
for _g in (-INF, -1.0, 0.0, NAN, 0.05, 0.2, 0.5, 0.9, 1.0, 1.5):
    GRID["gate_%r" % _g] = (DEFAULT_THR, _g, None)
GRID.update({"joint_0.5_0.05": (0.5, 0.05, None), "joint_1.5_0": (1.5, 0.0, None), "joint_inf_0": (INF, 0.0, None),
             "joint_0_-inf": (0.0, -INF, None), "joint_nan_nan": (NAN, NAN, None), "joint_4_0.5": (4.0, 0.5, None)})
BOUNDARY_SIDES = ("below", "equal", "above")          # threshold^2 just below s*, == s*, just above s*
GATE_SIDES = ("at", "up", "down")                     # gate == p*, nextafter(p*, +inf), nextafter(p*, -inf)
BOUNDARY = ["thr_%s_%s" % (w, s) for w in ("lead", "epi_pos", "epi_neg") for s in BOUNDARY_SIDES] + \
           ["gate_%s_%s" % (w, s) for w in ("cell0", "lead") for s in GATE_SIDES]


def _thresholds_around(s):
    """Doubles t around a positive float score s: below (t*t < s, but (float)(t*t) == s), equal (t*t == s, or None
    where no double squares to s), above (s < t*t < the next float)."""
    s = float(s)
    lo, hi = s - _nextafter(f32(s), f32(-INF)), _nextafter(f32(s), f32(INF)) - s
    t = math.sqrt(s - min(lo, hi) / 4)
    while not t * t < s:
        t = math.nextafter(t, -INF)
    assert float(f32(t * t)) == s and float(f32(s)) == s
    below = t
    equal = None
    t = math.sqrt(s)
    for c in (t, math.nextafter(t, INF), math.nextafter(t, -INF)):
        if c * c == s:
            equal = c
    t = math.sqrt(s + min(lo, hi) / 4)
    while not t * t > s:
        t = math.nextafter(t, INF)
    assert t * t < s + hi
    return dict(below=below, equal=equal, above=t)


class _Refs:
    """Inputs, settings and oracle answers, computed once for the module."""

    def __init__(self, oracle, synth):
        self.oracle, self.synth = oracle, synth
        self.inputs = _make_inputs(oracle, synth)
        self.ans = {}
        self._boundary = None

    def setting(self, name):
        if name in GRID:
            return GRID[name]
        return self.boundary()[name]

    def answer(self, name, inp=None, thr=None, gate=None):
        """[orc_match of every pair] of the input (all inputs: dict) at the setting."""
        if thr is None:
            thr, gate, _ = self.setting(name)
        key = (name, inp, thr, gate)
        if key not in self.ans:
            if inp is None:
                self.ans[key] = {k: self.answer(name, k, thr, gate) for k in self.inputs_of(name)}
            else:
                self.ans[key] = [_oracle_pair(self.oracle, self.inputs[inp], pr, thr, gate)
                                 for pr in self.inputs[inp]["pairs"]]
        return self.ans[key]

    def inputs_of(self, name):
        s = self.setting(name)
        return list(self.inputs) if s[2] is None else s[2]

    def boundary(self):
        """The boundary settings, picked from the oracle's answers at the defaults on syn24 and curmax."""
        if self._boundary is not None:
            return self._boundary
        out = {}
        picks = {}
        for inp in ("syn24", "curmax"):
            I = self.inputs[inp]
            m = self.answer("thr_0.9", inp)[0]
            for j, (lead, den) in enumerate(_match_kinds(I, I["pairs"][0], m, DEFAULT_GATE)):
                s = float(m["score"][j])
                kind = "lead" if lead else ("epi_pos" if den > 0 else ("epi_neg" if den < 0 else None))
                # a winner after the key filter: the one with the smallest |den|, whose key n = s * den lies the
                # closest to accept_gt * den (within 1.5 ulp(s*) * den), far inside the filter start's slack
                if kind and 0 < s < 1e30 and _thresholds_around(s)["equal"] is not None and \
                        (kind not in picks or (kind != "lead" and abs(den) < picks[kind][2])):
                    picks[kind] = (inp, s, abs(den))
        assert sorted(picks) == ["epi_neg", "epi_pos", "lead"], picks
        for kind, (inp, s, _) in picks.items():
            ts = _thresholds_around(s)
            for side in BOUNDARY_SIDES:
                out["thr_%s_%s" % (kind, side)] = (ts[side], DEFAULT_GATE, [inp])
        out.update(self._gate_boundary())
        self._boundary = out
        return out

    def _gate_boundary(self):
        """Gate triples at the probability p* of a matched cell0 and of a leading candidate of syn24's pair 0: the
        lowest such p* above the default gate at which dropping the cell (gate nextafter(p*, +inf)) changes the
        oracle's matches."""
        I = self.inputs["syn24"]
        a, b = I["pairs"][0]
        prob = I["prob"][a]
        m = self.answer("thr_0.9", "syn24")[0]
        leads = {_lead_of(I, a, int(I["qp"][b, q]), DEFAULT_GATE) for q in range(I["qc"][b])} - {-1}
        out = {}
        for kind, cells in (("cell0", set(m["cell0"].tolist())), ("lead", leads - set(m["cell0"].tolist()))):
            for c in sorted(cells, key=lambda c: (float(prob[c]), c)):
                p = float(prob[c])
                if p <= DEFAULT_GATE:
                    continue
                at = _oracle_pair(self.oracle, I, (a, b), DEFAULT_THR, p)
                up = _oracle_pair(self.oracle, I, (a, b), DEFAULT_THR, _nextafter(p, INF))
                if kind == "cell0" and c not in at["cell0"]:
                    continue
                if kind == "lead" and c not in {_lead_of(I, a, int(I["qp"][b, q]), p) for q in range(I["qc"][b])}:
                    continue
                if _same_matches(at, up):
                    continue
                for side, g in zip(GATE_SIDES, (p, _nextafter(p, INF), _nextafter(p, -INF))):
                    out["gate_%s_%s" % (kind, side)] = (DEFAULT_THR, g, ["syn24"])
                break
        assert len(out) == 2 * len(GATE_SIDES), sorted(out)
        return out


def _same_matches(a, b):
    return a["n"] == b["n"] and all(np.array_equal(bits(a[k]) if k == "score" else a[k], bits(b[k]) if k == "score"
                                                   else b[k]) for k in ("pts0", "pts1", "cell0", "query", "score"))


@pytest.fixture(scope="module")
def refs(oracle, synth):
    return _Refs(oracle, synth)


def _all_matches(ans):
    return [m for per in ans.values() for m in per]


def _assert_case_reaches(name, refs):
    """The setting exercises what it was built for, on the oracle's answers."""
    thr, gate, _ = refs.setting(name)
    ans = refs.answer(name)
    ms = _all_matches(ans)
    n = sum(m["n"] for m in ms)
    base = refs.answer("thr_0.9")
    if name == "thr_-0.9":
        assert all(_same_matches(x, y) for x, y in zip(ms, _all_matches(base)))
    elif name == "thr_1e+20":   # accept_gt = FLT_MAX: +inf scores only
        assert n > 0 and all(np.isposinf(m["score"]).all() for m in ms)
    elif name in ("thr_inf", "thr_nan", "joint_nan_nan", "joint_inf_0"):
        assert n == 0
        if name == "thr_inf":   # there were +inf scores to refuse
            assert any(np.isposinf(m["score"]).any() for m in _all_matches(refs.answer("thr_1e+20")))
    elif name.startswith("thr_") and name[4:5].isdigit() or name in ("joint_1.5_0", "joint_4_0.5", "joint_0_-inf"):
        assert n > 0 and all((m["score"].astype(np.float64) > thr * thr).all() for m in ms)
        if thr > 1:
            assert any((m["score"] > 1).any() and np.isfinite(m["score"]).any() for m in ms)
            assert any((np.isfinite(m["score"]) & (m["score"] > thr * thr)).any() for m in ms)
        if thr == 0.0:   # everything with a positive score: more than at the default
            assert n > sum(m["n"] for m in _all_matches(base))
    elif name in ("gate_-inf", "gate_-1.0", "gate_0.0", "gate_nan"):   # every non-dustbin cell a candidate
        ref = refs.answer("gate_-inf")
        assert all(_same_matches(x, y) for x, y in zip(ms, _all_matches(ref)))
        for inp, per in ans.items():
            I = refs.inputs[inp]
            for (a, b), m in zip(I["pairs"], per):
                w = _oracle_pair(refs.oracle, I, (a, b), DEFAULT_THR, 0.2)
                assert m["pairs_256"] + m["pairs_64"] >= w["pairs_256"] + w["pairs_64"]
        assert sum(m["pairs_256"] + m["pairs_64"] for m in ms) > \
            sum(m["pairs_256"] + m["pairs_64"] for m in _all_matches(base))
    elif name.startswith("gate_") and name[5:6].isdigit() or name == "joint_0.5_0.05":
        cand = [m["pairs_256"] + m["pairs_64"] for m in ms]
        if gate == 1.5:
            assert sum(cand) == 0 and n == 0
        elif gate != DEFAULT_GATE:   # another candidate set: the candidate counts move
            assert cand != [m["pairs_256"] + m["pairs_64"] for m in _all_matches(base)]
            fewer = sum(cand) < sum(m["pairs_256"] + m["pairs_64"] for m in _all_matches(base))
            assert fewer == (gate > DEFAULT_GATE)
        if gate < 1.0 and gate != DEFAULT_GATE:
            assert n > 0
    elif name.startswith("thr_") and name.split("_")[-1] in BOUNDARY_SIDES:
        kind = name[4:-len(name.split("_")[-1]) - 1]
        inp = refs.inputs_of(name)[0]
        I = refs.inputs[inp]
        below = refs.answer("thr_%s_below" % kind, inp)[0]
        kinds = _match_kinds(I, I["pairs"][0], below, DEFAULT_GATE)
        s = float(f32(thr * thr)) if name.endswith("_below") else None
        if name.endswith("_below"):   # the winner of that score is kept, and is of its kind
            j = [k for k in range(below["n"]) if below["score"][k] == s]
            assert j, (name, s)
            lead, den = kinds[j[0]]
            assert lead == (kind == "lead") and (kind == "lead" or (den > 0) == (kind == "epi_pos"))
            if kind == "epi_pos":   # the winner's key is within 1.5 ulp(s*) * den < 192 of accept_gt * den
                ulp = _nextafter(f32(s), f32(INF)) - s
                assert abs(den) * ulp < 128, (den, ulp)
            assert float(f32(thr * thr)) == s and thr * thr < s
        else:                          # and lost one ulp or less above
            assert ans[inp][0]["n"] < below["n"]
    elif name.startswith("gate_") and name.split("_")[-1] in GATE_SIDES:
        kind = name.split("_")[1]
        at = refs.answer("gate_%s_at" % kind, "syn24")[0]
        if name.endswith("_up"):
            assert not _same_matches(ans["syn24"][0], at)
        elif name.endswith("_down"):
            assert _same_matches(ans["syn24"][0], at)
    else:
        assert name in ("thr_0.9", "gate_0.2"), name
    if name in ("thr_0.9", "gate_0.2"):   # the crafted windows reach all three branches of the key filter's start
        I = refs.inputs["curmax"]
        m = ans["curmax"][0]
        kinds = _match_kinds(I, I["pairs"][0], m, DEFAULT_GATE)
        epi = [den for lead, den in kinds if not lead]
        assert 0 in epi and -2 ** 31 in epi and any(d > 0 for d in epi) and any(-2 ** 31 < d < 0 for d in epi), epi
        assert any(np.isposinf(m["score"])), m["score"]


def _ids():
    return list(GRID) + BOUNDARY


@pytest.mark.parametrize("name", _ids())
def test_case_reaches(refs, name):
    _assert_case_reaches(name, refs)


# ------------------------------------------------------------------ GPU: both matchers, every entry point
def _mparams(inp, thr, gate, tc):
    from maveric_slam_b200 import tracking
    p = tracking.match_params(inp["rows"], inp["cols"], 4, 4, 4, inp["M"], thr, gate)
    p.use_tensor_cores = tc
    return p


def _modes(thr):
    """dp4a and tcgen05; where the tcgen05 matcher cannot take the threshold (NaN), dp4a and auto."""
    return (0, 2) if math.isnan(thr) else (0, 1)


def _assert_same(got, want, label):
    assert got["n"] == want["n"], (label, got["n"], want["n"])
    for k in ("pts0", "pts1", "cell0", "query", "score"):
        if k in got and got["n"] > 0:
            g, w = (bits(got[k]), bits(want[k])) if k == "score" else (got[k], want[k])
            bad = np.nonzero(np.asarray(g != w).reshape(len(g), -1).any(axis=1))[0]
            assert bad.size == 0, (label, k, bad[:4].tolist(), got[k][bad[:4]].tolist(), want[k][bad[:4]].tolist())


def _batch(tracker, frames, p, f0f1=None):
    """mv_match_batch over stacked frames (desc, idx, prob, qp, qi, qc) -> [match dict per pair]."""
    import torch
    dev = [torch.from_numpy(np.ascontiguousarray(a)).to(tracker.device) for a in frames]
    f0 = f1 = None
    if f0f1 is not None:
        f0, f1 = (torch.tensor([x[i] for x in f0f1], dtype=torch.int32, device=tracker.device) for i in (0, 1))
    pts, cnt, cell0, query, score = (t.cpu().numpy() for t in tracker.match(p, *dev, f0=f0, f1=f1))
    return [dict(n=int(n), pts0=pts[i, :n, :2], pts1=pts[i, :n, 2:], cell0=cell0[i, :n], query=query[i, :n],
                 score=score[i, :n]) for i, n in enumerate(cnt)]


def _frames(inp):
    return [inp[k] for k in ("desc", "idx", "prob", "qp", "qi", "qc")]


@pytest.mark.gpu
@pytest.mark.parametrize("name", _ids())
def test_matchers_vs_oracle(tracker, refs, name):
    """The setting through mv_match_batch (each input's consecutive pairs; the 24x80 inputs stacked and run through
    an explicit f0 / f1 list in reverse order, one pair twice; the 47x155 chain's pairs reversed) and
    mv_match_pair_host, with each matcher."""
    from maveric_slam_b200 import tracking
    thr, gate, _ = refs.setting(name)
    want = refs.answer(name)
    names = refs.inputs_of(name)
    for tc in _modes(thr):
        for k in names:
            I = refs.inputs[k]
            p = _mparams(I, thr, gate, tc)
            for i, g in enumerate(_batch(tracker, _frames(I), p)):
                _assert_same(g, want[k][i], ("batch", tc, k, i))
            for i, (a, b) in enumerate(I["pairs"]):
                q = int(I["qc"][b])
                g = tracking.match_pair(p, I["desc"][a], I["desc"][b], I["idx"][a], I["prob"][a], I["qp"][b, :q],
                                        I["qi"][b, :q], ctx=tracker.ctx)
                _assert_same(g, want[k][i], ("pair", tc, k, i))
        for shape in sorted({refs.inputs[k]["rows"] for k in names}):
            group = [k for k in names if refs.inputs[k]["rows"] == shape]
            stacked, pairs, wants, base = [], [], [], 0
            for k in group:
                I = refs.inputs[k]
                stacked.append(_frames(I))
                pairs += [(a + base, b + base) for a, b in I["pairs"]]
                wants += want[k]
                base += I["desc"].shape[0]
            frames = [np.concatenate([f[j] for f in stacked]) for j in range(6)]
            order = list(range(len(pairs)))[::-1] + [0]
            got = _batch(tracker, frames, _mparams(refs.inputs[group[0]], thr, gate, tc), [pairs[i] for i in order])
            for g, i in zip(got, order):
                _assert_same(g, wants[i], ("f0f1", tc, shape, i))


# ------------------------------------------------------------------ whole path
SEQ_SHAPES = {24: dict(rows=24, cols=80, permille=140, n=10, seed=17, top_n=100, max_valid=1000, max_matches=150),
              47: dict(rows=47, cols=155, permille=550, n=4, seed=19, top_n=4000, max_valid=8192, max_matches=4096)}
SEQ_CASES = {
    "low": dict(shape=24, thr=0.5, gate=0.05),
    "above_1": dict(shape=24, thr=1.05),
    **{"gate_" + s: dict(shape=24, gate=s) for s in GATE_SIDES},
    "ransac_0": dict(shape=47, ransac=(0, 1.1)),
    **{"ransac_1_%r" % t: dict(shape=47, ransac=(1, t)) for t in (0.0, 0.25, 1e30)},
}
SEQ_ENTRIES = ("device", "host_pinned", "host_pageable", "host_pageable_chunk2")


def _seq_params(shape, thr=DEFAULT_THR, gate=DEFAULT_GATE, ransac=(10, 1.1)):
    from maveric_slam_b200 import tracking
    sh = SEQ_SHAPES[shape]
    p = tracking.track_params(sh["rows"], sh["cols"], top_n=sh["top_n"], max_valid=sh["max_valid"],
                              max_matches=sh["max_matches"], hypotheses=32)
    p.match.match_threshold, p.match.min_prob0 = thr, gate
    p.ransac_iterations, p.ransac_threshold = ransac
    return p


def _seq_frames(synth, shape):
    sh = SEQ_SHAPES[shape]
    semi, desc, depth, _ = synth.synth_sequence(sh["seed"], sh["rows"], sh["cols"], sh["n"],
                                                keypoint_permille=sh["permille"])
    return [semi, np.full(sh["n"], synth.SEMI_SCALE, f32), desc, depth]


def _gate_cell(oracle, p, semi, sscale, desc, pair_range):
    """(pair f, cell, p*): a matched frame-0 cell of pair f, not one of frame f's queries (whose rows the gather
    fetches anyway), whose drop (gate nextafter(p*, +inf)) changes pair f's matches at the gate p*.  Of these, the one
    whose probability p* the fewest valid cells of the sequence share, then the lowest p* above the default gate."""
    det = detect(oracle, p, semi, sscale)
    valid = np.concatenate([d[1][d[0] != 64] for d in det])
    vals, counts = np.unique(valid, return_counts=True)
    shared = dict(zip(vals.tolist(), counts.tolist()))
    for f in pair_range:
        q = copy.copy(p)
        q.match = copy.copy(p.match)
        m = oracle.match(match_cfg(q), desc[f], desc[f + 1], det[f][0], det[f][1], det[f + 1][2], det[f + 1][3])
        cells = [c for c in set(m["cell0"].tolist()) if c not in set(det[f][2].tolist())]
        for c in sorted(cells, key=lambda c: (shared[float(det[f][1][c])], float(det[f][1][c]))):
            ps = float(det[f][1][c])
            if ps <= DEFAULT_GATE:
                continue
            out = []
            for g in (ps, _nextafter(ps, INF)):
                q.match.min_prob0 = g
                out.append(oracle.match(match_cfg(q), desc[f], desc[f + 1], det[f][0], det[f][1], det[f + 1][2],
                                        det[f + 1][3]))
            if c in out[0]["cell0"] and not _same_matches(out[0], out[1]):
                return f, c, ps
    raise AssertionError("no gate cell")


class _SeqRefs:
    def __init__(self, oracle, synth):
        self.oracle, self.synth, self.frames, self.done, self.gate = oracle, synth, {}, {}, None

    def inputs(self, shape):
        if shape not in self.frames:
            self.frames[shape] = _seq_frames(self.synth, shape)
        return self.frames[shape]

    def gate_cell(self):
        if self.gate is None:   # frames 6 .. 8 come in the fourth chunk of 2 pairs: the first buffer set's second use
            semi, sscale, desc, _ = self.inputs(24)
            self.gate = _gate_cell(self.oracle, _seq_params(24), semi, sscale, desc, range(6, 9))
        return self.gate

    def params(self, name):
        if name == "default_24" or name == "default_47":
            return _seq_params(int(name[-2:]))
        c = SEQ_CASES[name]
        kw = {k: c[k] for k in ("thr", "ransac") if k in c}
        g = c.get("gate", DEFAULT_GATE)
        if isinstance(g, str):
            ps = self.gate_cell()[2]
            g = {"at": ps, "up": _nextafter(ps, INF), "down": _nextafter(ps, -INF)}[g]
        return _seq_params(c["shape"], gate=g, **kw)

    def records(self, name):
        if name not in self.done:
            shape = int(name[-2:]) if name.startswith("default") else SEQ_CASES[name]["shape"]
            semi, sscale, desc, depth = self.inputs(shape)
            self.done[name] = landmark_reference(self.oracle, None, self.params(name), semi, sscale, desc, None, depth,
                                                 depth_mode=True, threads=8)[0]
        return self.done[name]


@pytest.fixture(scope="module")
def seq_refs(oracle, synth):
    return _SeqRefs(oracle, synth)


def _assert_seq_reaches(name, seq_refs):
    rec = seq_refs.records(name)
    shape = SEQ_CASES[name]["shape"]
    base = seq_refs.records("default_%d" % shape)
    assert rec.tobytes() != base.tobytes()
    assert (rec["status"] == 0).all() and (rec["num_matches"] > 0).all()
    if name == "low":
        assert (rec["num_matches"] >= base["num_matches"]).all() and (rec["num_matches"] > base["num_matches"]).any()
    elif name == "above_1":
        assert (rec["num_matches"] < base["num_matches"]).all()
    elif name.startswith("gate_"):
        f = seq_refs.gate_cell()[0]
        at = seq_refs.records("gate_at")
        if name == "gate_up":     # the one cell's row decides pair f's record
            assert rec[f].tobytes() != at[f].tobytes()
        elif name == "gate_down":
            assert rec.tobytes() == at.tobytes()
    elif name == "ransac_0":
        assert (rec["ransac_inliers"] == 0).all() and (base["ransac_inliers"] > 0).all()
    elif name.startswith("ransac_1_"):
        t = SEQ_CASES[name]["ransac"][1]
        if t == 1e30:           # every match an inlier: the 1000-inlier cap binds
            assert (rec["ransac_inliers"] == 1000).all() and (rec["num_matches"] > 1000).all()
        else:
            assert (rec["ransac_inliers"] < 1000).all()
        assert (rec["ransac_inliers"] != base["ransac_inliers"]).all()
        if t == 0.0:
            assert (rec["ransac_inliers"] <= seq_refs.records("ransac_1_0.25")["ransac_inliers"]).all()
    # matching is the same for every RANSAC-E setting
    if name.startswith("ransac"):
        assert (rec["num_matches"] == base["num_matches"]).all()


@pytest.mark.parametrize("name", list(SEQ_CASES))
def test_sequence_case_reaches(seq_refs, name):
    _assert_seq_reaches(name, seq_refs)


def _run_sequence(tracker, p, frames, entry, monkeypatch):
    import torch
    from maveric_slam_b200 import tracking
    monkeypatch.delenv("MV_HOST_CHUNK_PAIRS", raising=False)
    if entry == "device":
        dev = [torch.from_numpy(np.ascontiguousarray(x)).to(tracker.device) for x in frames]
        return tracking.results_to_numpy(tracker.track_sequence(p, *dev))
    if entry == "host_pageable":
        return tracker.track_sequence_host(p, *[np.ascontiguousarray(x) for x in frames])[0]
    with monkeypatch.context() as m:
        m.setenv("MV_HOST_CHUNK_PAIRS", "2")
        semi, sscale, desc, depth = frames
        # first the same frames with their descriptors in reverse order and every row gathered (gate -inf): every
        # staging buffer row the call below does not gather then holds another frame's descriptor, whatever ran
        # on this context before
        q = copy.copy(p)
        q.match = copy.copy(p.match)
        q.match.min_prob0 = -INF
        reversed_desc = np.ascontiguousarray(desc[::-1])
        tracker.track_sequence_host(q, *[pinned(x) for x in (semi, sscale, reversed_desc, depth)])
        stage = np.ascontiguousarray if entry == "host_pageable_chunk2" else pinned
        return tracker.track_sequence_host(p, *[stage(x) for x in frames])[0]


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SEQ_CASES))
def test_sequence_vs_oracle(tracker, seq_refs, monkeypatch, name):
    """Whole records of every pair, byte for byte, through the device call and the host call from pinned buffers
    (row gather, chunks of 2 pairs: the three staging buffer sets are reused, so a row the gather skipped holds an
    earlier frame's descriptor), and pageable buffers, in the default chunks and in chunks of 2 pairs."""
    want = seq_refs.records(name)
    frames = seq_refs.inputs(SEQ_CASES[name]["shape"])
    p = seq_refs.params(name)
    for entry in SEQ_ENTRIES:
        got = np.ascontiguousarray(_run_sequence(tracker, p, frames, entry, monkeypatch)).tobytes()
        assert got == want.tobytes(), (entry, first_difference(want, got))


# ------------------------------------------------------------------ landmark path
LM_ENTRIES = ("device", "host:3", "blocks_host:8")


class _LmRef:
    """24x80, 12 frames, the reference vocabulary; threshold 0.7, the gate on one cell's probability (a pair of frames
    6 .. 9), RANSAC-E at 1 iteration and 1e30 (every match an inlier)."""

    def __init__(self, oracle, synth):
        self.oracle = oracle
        rows, cols, n = 24, 80, 12
        semi, desc, depth, _ = synth.synth_sequence(41, rows, cols, n)
        sscale = np.full(n, synth.SEMI_SCALE, f32)
        dscale = np.full(n, synth.DESC_SCALE, f32)
        p = _seq_params(24, thr=0.7, ransac=(1, 1e30))
        self.gate = _gate_cell(oracle, p, semi, sscale, desc, range(6, 10))
        p.match.min_prob0 = self.gate[2]
        self.vocab = ref_vocab()
        self.c = dict(p=p, frames=[semi, sscale, desc, dscale, depth], first=0, n_words=10000, vocab=self.vocab,
                      entry=None)
        self.c["rec"], self.c["nl"], self.c["table"] = self.reference(p)

    def reference(self, p):
        o = self.oracle
        return landmark_reference(o, o.bow_vocab(*self.vocab), p, *self.c["frames"], n_words=10000, threads=8)


@pytest.fixture(scope="module")
def lm_ref(oracle, synth):
    return _LmRef(oracle, synth)


def test_landmark_case_reaches(lm_ref):
    from maveric_slam_b200 import tracking
    c = lm_ref.c
    rec, nl = c["rec"], c["nl"]
    assert (rec["num_matches"] > 0).all() and (nl > 0).all() and (rec["status"] == 0).all()
    default = lm_ref.reference(tracking.track_params(24, 80, top_n=100, max_valid=1000, max_matches=150,
                                                     hypotheses=32))
    assert (rec["ransac_inliers"] == rec["num_matches"]).all() and (default[0]["ransac_inliers"] == 0).all()
    assert (rec["num_matches"] != default[0]["num_matches"]).any()
    f = lm_ref.gate[0]
    p = copy.copy(c["p"])
    p.match = copy.copy(c["p"].match)
    p.match.min_prob0 = _nextafter(lm_ref.gate[2], INF)   # dropping the one cell changes pair f
    assert lm_ref.reference(p)[0][f].tobytes() != rec[f].tobytes()


@pytest.fixture(scope="module")
def lm_tracker():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from maveric_slam_b200 import tracking
    tr = tracking.Tracker(0)
    tr.bow_set_vocabulary(*ref_vocab())
    return tr


@pytest.mark.gpu
@pytest.mark.parametrize("entry", LM_ENTRIES)
def test_landmark_path_vs_reference(lm_tracker, lm_ref, monkeypatch, entry):
    c = lm_ref.c
    monkeypatch.delenv("MV_HOST_CHUNK_PAIRS", raising=False)
    res, nl, table = run_entry(lm_tracker, c, entry, monkeypatch)
    assert res == c["rec"].tobytes(), first_difference(c["rec"], res)
    assert (nl == c["nl"]).all(), (nl, c["nl"])
    assert table == c["table"].tobytes()


# ------------------------------------------------------------------ refusals
@pytest.mark.gpu
def test_nan_threshold_with_forced_tensor_cores_is_refused(tracker, lm_tracker, refs, seq_refs, lm_ref, monkeypatch):
    """use_tensor_cores = 1 asks for the tcgen05 matcher, which cannot take a NaN threshold: every entry point refuses
    it with MV_ERR_BAD_ARG before anything is enqueued, and the context then still gives the oracle's answers."""
    import torch
    from maveric_slam_b200 import lib
    I = refs.inputs["syn24"]
    dev = [torch.from_numpy(np.ascontiguousarray(a)).to(tracker.device) for a in _frames(I)]
    frames = seq_refs.inputs(24)
    dframes = [torch.from_numpy(np.ascontiguousarray(x)).to(tracker.device) for x in frames]
    lm = lm_ref.c["frames"]
    lm_dev = [torch.from_numpy(np.ascontiguousarray(x)).to(lm_tracker.device) for x in lm]
    lm_pin = [pinned(x) for x in lm]
    mp = _mparams(I, NAN, DEFAULT_GATE, 1)
    tp = seq_refs.params("low")
    tp.match.match_threshold, tp.match.use_tensor_cores = NAN, 1
    lp = copy.copy(lm_ref.c["p"])
    lp.match = copy.copy(lm_ref.c["p"].match)
    lp.match.match_threshold, lp.match.use_tensor_cores = NAN, 1
    torch.cuda.synchronize()
    calls = [
        ("mv_match_batch", tracker, lambda: tracker.match(mp, *dev)),
        ("mv_track_sequence", tracker, lambda: tracker.track_sequence(tp, *dframes)),
        ("mv_track_sequence_host", tracker,
         lambda: tracker.track_sequence_host(tp, *[pinned(x) for x in frames])),
        ("mv_track_landmarks_prepare", lm_tracker,
         lambda: lm_tracker.track_landmarks_prepare(lp, 0, 0, *lm_dev, 10000)),
        ("mv_track_landmarks_prepare_host", lm_tracker,
         lambda: lm_tracker.track_landmarks_prepare_host(lp, 0, 0, *lm_pin, 10000)),
    ]
    for fn, tr, call in calls:
        before = tr.ctx.launches
        with pytest.raises(lib.MvError, match="bad argument.*tensor"):
            call()
        assert tr.ctx.launches == before, fn
    # the next calls on both contexts give the oracle's bytes
    for i, g in enumerate(_batch(tracker, _frames(I), _mparams(I, DEFAULT_THR, DEFAULT_GATE, 1))):
        _assert_same(g, refs.answer("thr_0.9", "syn24")[i], ("after refusal", i))
    want = seq_refs.records("low")
    got = np.ascontiguousarray(_run_sequence(tracker, seq_refs.params("low"), frames, "host_pinned", monkeypatch))
    assert got.tobytes() == want.tobytes(), first_difference(want, got.tobytes())
    res, nl, table = run_entry(lm_tracker, lm_ref.c, "blocks_host:8", monkeypatch)
    assert res == lm_ref.c["rec"].tobytes() and table == lm_ref.c["table"].tobytes()
