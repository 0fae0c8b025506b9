"""The execution contract of include/maveric_b200.h against the CPU oracle: a context runs on the caller's stream
(mv_ctx_set_stream), a context can be used from any thread, and different contexts are independent.

Every other module builds its Tracker under torch's default stream, so there every device-resident call runs on the
legacy stream 0, which every context on the device shares: a kernel launched on the wrong stream is invisible there,
because the wrong stream and the right one are the same.  Here

  1. a Tracker bound to a non-blocking torch stream runs the depth path (both matchers, the K3 split launch and its
     streaming kernel), the host-buffer pipelines, every landmark-path entry point and the building blocks; each
     answer equals the oracle's and the bytes a default-stream Tracker returns;
  2. eight threads, each with its own stream and context on one GPU, run workloads whose launches need different
     dynamic shared memory of the same kernel (the tcgen05 matcher at three grids, the generic Schur and the solve
     kernel at several pose counts, the word assignment with two vocabularies) at the same time, round after round,
     and every round returns the bytes of a serial run that was held to the oracle first;
  3. a context made on one thread is used from another; contexts of two GPUs are driven from two threads whose
     current devices differ and stay as they were; the legacy symbols run from four threads at once on the shared
     global context, and the `_ex` forms with a context per thread.

Part 2 is a bounded check that concurrent results equal serial ones, not a search for a race.
"""
import os
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import bits
from helpers import dev, pinned, pnp_params, pnp_problems, ref_vocab, same_bits, spd_system, with_first_pair
from landmark_reference import bow_check, bow_inputs, bow_vocab, case_inputs, landmark_reference, orc_landmarks_sequence

pytestmark = pytest.mark.gpu

f32 = np.float32
ROWS, COLS = 47, 155


# ------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import maveric_slam_b200  # noqa: F401
    return torch


@pytest.fixture(scope="module")
def side(torch_cuda):
    """(stream, Tracker bound to it): a non-blocking stream of the caller's, not torch's default stream."""
    from maveric_slam_b200 import tracking
    s = torch_cuda.cuda.Stream(0)
    assert s.cuda_stream != 0 and s.cuda_stream != torch_cuda.cuda.default_stream(0).cuda_stream
    with torch_cuda.cuda.stream(s):
        tr = tracking.Tracker(0)
    return s, tr


@pytest.fixture(scope="module")
def plain(torch_cuda):
    """A Tracker of its own under torch's default stream (the session's `tracker` keeps its vocabulary)."""
    from maveric_slam_b200 import tracking
    assert torch_cuda.cuda.current_stream(0).cuda_stream == 0
    return tracking.Tracker(0)


def _both(side, plain, work, *args):
    """work(tracker, *args) -> dict of bytes, on the caller's stream and on the default stream: the same bytes."""
    import torch
    s, tr = side
    with torch.cuda.stream(s):
        got = work(tr, *args)
    want = work(plain, *args)
    assert got.keys() == want.keys()
    for k in got:
        assert got[k] == want[k], k
    return got


def _b(t):
    return t.cpu().numpy().tobytes()


# ------------------------------------------------------------------ 1. the depth path on the caller's stream
def _depth_params(tc, hypotheses=1024, rows=ROWS, cols=COLS, top_n=1000, max_matches=1024, thr=0.7):
    from maveric_slam_b200 import tracking
    p = tracking.track_params(rows, cols, top_n=top_n, max_valid=rows * cols + 1, max_matches=max_matches,
                              hypotheses=hypotheses, use_tensor_cores=tc)
    p.match.match_threshold = thr
    return p


@pytest.fixture(scope="module")
def depth_case(oracle, synth):
    """8 frames at 47x155, top 1000 queries, 1024 hypotheses, a match threshold of 0.7: pairs of either side of 480
    correspondences, so K3 runs both the two-phase and the streaming kernel.  -> (host frames, oracle records)."""
    n = 8
    semi, desc, depth, _ = synth.synth_sequence(13, ROWS, COLS, n, keypoint_permille=550)
    sscale = np.full(n, synth.SEMI_SCALE, f32)
    frames = (semi, sscale, desc, depth)
    rec, _, _ = landmark_reference(oracle, None, _depth_params(1), semi, sscale, desc, None, depth, depth_mode=True,
                                   threads=os.cpu_count() or 1)
    nm = rec["num_matches"]
    assert (rec["status"] == 0).all() and (nm > 480).any() and (nm <= 480).any(), nm
    return frames, rec.tobytes()


@pytest.mark.parametrize("tc", [0, 1], ids=["dp4a", "tcgen05"])
def test_track_sequence_on_callers_stream(side, plain, depth_case, monkeypatch, tc):
    """mv_track_sequence with K3's split launch (a programmatic dependent launch: the 3 shortest of 7 pairs as
    128-hypothesis CTAs behind the main launch), records byte for byte against the oracle, K3 poses included."""
    (semi, sscale, desc, depth), want = depth_case
    monkeypatch.setenv("MV_PNP_K3_SMALL_BELOW", "0")      # the split launch at 7 pairs

    def work(tr):
        d = [dev(tr, x) for x in (semi, sscale, desc, depth)]
        return {"records": _b(tr.track_sequence(_depth_params(tc), *d))}
    got = _both(side, plain, work)
    assert got["records"] == want


@pytest.mark.parametrize("mode", ["pinned", "pageable", "chunks_of_3"])
def test_track_sequence_host_on_callers_stream(side, plain, depth_case, monkeypatch, mode):
    """mv_track_sequence_host: pinned buffers (the row gather), pageable ones, and staging chunks of 3 pairs."""
    (semi, sscale, desc, depth), want = depth_case
    monkeypatch.setenv("MV_PNP_K3_SMALL_BELOW", "0")
    monkeypatch.delenv("MV_HOST_CHUNK_PAIRS", raising=False)
    if mode == "chunks_of_3":
        monkeypatch.setenv("MV_HOST_CHUNK_PAIRS", "3")

    def work(tr):
        bufs = [np.ascontiguousarray(x) for x in (semi, sscale, desc, depth)] if mode == "pageable" else \
            [pinned(x) for x in (semi, sscale, desc, depth)]
        res, _, down = tr.track_sequence_host(_depth_params(1), *bufs)
        assert down == 64 * (semi.shape[0] - 1)
        return {"records": res.tobytes()}
    got = _both(side, plain, work)
    assert got["records"] == want


# ------------------------------------------------------------------ 1. the landmark path on the caller's stream
@pytest.fixture(scope="module")
def lm_case(oracle, synth):
    """tests/test_landmark_reference.py's "degenerate" case (frames without keypoints, an overflowing frame,
    saturated and zero descriptors) and its reference."""
    c = case_inputs("degenerate", synth)
    rec, nl, table = landmark_reference(oracle, oracle.bow_vocab(*c["vocab"]), c["p"], *c["frames"],
                                        first_frame=c["first"], n_words=c["n_words"])
    return c, rec.tobytes(), nl.tobytes(), table.tobytes()


def _landmark_entry(tr, c, entry):
    """One landmark-path entry point on the case, from an empty table -> dict of bytes."""
    p, first, n_words, host = c["p"], c["first"], c["n_words"], c["frames"]
    tr.bow_set_vocabulary(*c["vocab"])
    table = tr.landmarks_new(n_words)
    n_pairs = host[0].shape[0] - 1
    if entry == "device":
        res, nl = tr.track_sequence_landmarks(p, *[dev(tr, x) for x in host], table, first_frame=first)
        res, nl = _b(res), _b(nl)
    elif entry == "host":
        res, nl, _, _ = tr.track_sequence_landmarks_host(p, *[pinned(x) for x in host], table, first_frame=first)
        res, nl = res.tobytes(), nl.tobytes()
    else:   # two blocks, 8 warm-up frames, prepared in reverse order
        n_warm = 8
        bufs = [dev(tr, x) for x in host] if entry == "blocks" else [pinned(x) for x in host]
        prep = tr.track_landmarks_prepare if entry == "blocks" else tr.track_landmarks_prepare_host
        half = n_pairs // 2
        blocks = [(0, half), (half, n_pairs - half)]
        prepared = {}
        for i, (lo, cnt) in reversed(list(enumerate(blocks))):
            w = min(n_warm, lo)
            prepared[i] = prep(with_first_pair(p, p.pnp.first_pair + lo), w, first + lo,
                               *[x[lo - w:lo + cnt + 1] for x in bufs], n_words)
        rs, ns = [], []
        for i in range(len(blocks)):
            tr.track_landmarks_step_table(prepared[i], table)
            r, k = tr.track_landmarks_solve(prepared[i])
            rs.append(r.cpu().numpy()); ns.append(k.cpu().numpy())
            tr.track_landmarks_release(prepared[i])
        res, nl = np.concatenate(rs).tobytes(), np.concatenate(ns).tobytes()
    return {"records": res, "n_with_landmark": nl, "table": _b(table)}


@pytest.mark.parametrize("entry", ["device", "host", "blocks", "blocks_host"])
def test_landmark_path_on_callers_stream(side, plain, lm_case, monkeypatch, entry):
    c, rec, nl, table = lm_case
    monkeypatch.delenv("MV_HOST_CHUNK_PAIRS", raising=False)
    got = _both(side, plain, _landmark_entry, c, entry)
    assert got == {"records": rec, "n_with_landmark": nl, "table": table}


def _table_walk(tr, oracle, n_words, first, k, n_warm, word, qc, coords):
    """mv_landmarks_sequence over frames 0 .. k-1, then the block k .. by mv_landmarks_sequence and by
    speculate / resolve from the same entry table -> dict of bytes."""
    entry = tr.landmarks_new(n_words)
    head = tr.landmarks_sequence(entry, first, dev(tr, word[:k]), dev(tr, qc[:k]), dev(tr, coords[:k]))
    seq_t = entry.clone()
    seq = tr.landmarks_sequence(seq_t, first + k, dev(tr, word[k:]), dev(tr, qc[k:]), dev(tr, coords[k:]))
    spec = tr.landmarks_speculate(n_words, first + k, n_warm, dev(tr, word[k - n_warm:]), dev(tr, qc[k - n_warm:]),
                                  dev(tr, coords[k:]))
    spec_t = entry.clone()
    res = tr.landmarks_resolve(spec, spec_t)
    out = {"head": _b(head), "entry": _b(entry), "seq": _b(seq), "seq_table": _b(seq_t), "resolve": _b(res),
           "resolve_table": _b(spec_t)}
    tr.landmarks_release(spec)
    return out


def test_landmark_table_calls_on_callers_stream(side, plain, oracle):
    """mv_landmarks_sequence and mv_landmarks_speculate / _resolve (8 warm-up frames) against the oracle's table."""
    rng = np.random.default_rng(17)
    n, top_n, n_words, first, k = 30, 64, 200, 500, 14
    word = rng.integers(-3, 220, (n, top_n)).astype(np.int32)
    word[:, :3] = 5
    qc = np.full(n, top_n, np.int32)
    qc[4], qc[20] = 0, 31
    coords = rng.normal(size=(n, top_n, 3)).astype(f32)
    got = _both(side, plain, _table_walk, oracle, n_words, first, k, 8, word, qc, coords)
    table = oracle.pool_new(n_words)
    head = orc_landmarks_sequence(oracle, table, first, word[:k], qc[:k], coords[:k])
    assert got["head"] == head.tobytes() and got["entry"] == table.tobytes()
    block = orc_landmarks_sequence(oracle, table, first + k, word[k:], qc[k:], coords[k:])
    for name in ("seq", "resolve"):
        assert got[name] == block.tobytes(), name
        assert got[name + "_table"] == table.tobytes(), name


# ------------------------------------------------------------------ 1. the building blocks on the caller's stream
def test_detector_and_matchers_on_callers_stream(side, plain, oracle, synth):
    """Softmax, top-N, NMS and both matchers of a batch, against the oracle frame by frame and pair by pair."""
    from oracle import orc
    rows, cols, n, N, M = 24, 80, 4, 100, 150
    semi, desc, _, _ = synth.synth_sequence(23, rows, cols, n, keypoint_permille=400)
    sscale = (synth.SEMI_SCALE * np.array([1.0, 0.9, 1.1, 1.0])).astype(f32)
    mv = rows * cols + 1

    def work(tr):
        from maveric_slam_b200 import tracking
        out = {}
        idx, prob, nv = tr.softmax(dev(tr, semi), dev(tr, sscale))
        out.update(idx=_b(idx), prob=_b(prob), nv=_b(nv))
        qp, qi, qpr, qc, ov = tr.top_n(idx, prob, N, mv)
        out.update(qp=_b(qp), qi=_b(qi), qpr=_b(qpr), qc=_b(qc), ov=_b(ov))
        for tc in (0, 1):
            m = tr.match(tracking.match_params(rows, cols, use_tensor_cores=tc), dev(tr, desc), idx, prob, qp, qi, qc)
            cnt = m[1].cpu().numpy()
            out["count%d" % tc] = cnt.tobytes()
            for name, t in zip(("pts", "cell0", "query", "score"), (m[0], m[2], m[3], m[4])):
                a = t.cpu().numpy()          # the first count entries of each pair
                out["%s%d" % (name, tc)] = b"".join(a[i, :cnt[i]].tobytes() for i in range(len(cnt)))
        ni, npr = tr.nms(rows, cols, idx.clone(), prob.clone())
        out.update(nms_idx=_b(ni), nms_prob=_b(npr))
        return out
    got = _both(side, plain, work)
    for name in ("count", "pts", "cell0", "query", "score"):
        assert got[name + "0"] == got[name + "1"], name
    idx = np.frombuffer(got["idx"], np.int32).reshape(n, -1)
    prob = np.frombuffer(got["prob"], f32).reshape(n, -1)
    nv, qc = np.frombuffer(got["nv"], np.int32), np.frombuffer(got["qc"], np.int32)
    qp = np.frombuffer(got["qp"], np.int32).reshape(n, N)
    qi = np.frombuffer(got["qi"], np.int32).reshape(n, N)
    ni = np.frombuffer(got["nms_idx"], np.int32).reshape(n, -1)
    npr = np.frombuffer(got["nms_prob"], f32).reshape(n, -1)
    cfg = orc.MatchCfg(rows, cols, 4, 4, 4, M, 0.9, 0.2)
    for f in range(n):
        i2, p2, n2 = oracle.softmax(float(sscale[f]), semi[f])
        assert (idx[f] == i2).all() and (bits(prob[f]) == bits(p2)).all() and nv[f] == n2, f
        pa, ix, _, _ = oracle.top_n(float(sscale[f]), semi[f], N, mv)
        assert qc[f] == len(pa) and (qp[f, :len(pa)] == pa).all() and (qi[f, :len(pa)] == ix).all(), f
        mi, pp, _ = oracle.nms(rows, cols, i2, p2)
        assert (ni[f] == mi).all() and (bits(npr[f]) == bits(pp)).all(), f
    cnt = np.frombuffer(got["count1"], np.int32)
    ends = np.concatenate([[0], np.cumsum(cnt)])
    pts = np.frombuffer(got["pts1"], f32).reshape(-1, 4)
    cell0 = np.frombuffer(got["cell01"], np.int32)
    score = np.frombuffer(got["score1"], f32)
    assert cnt.sum() > 0
    for q in range(n - 1):
        pa, ix, _, _ = oracle.top_n(float(sscale[q + 1]), semi[q + 1], N, mv)
        r = oracle.match(cfg, desc[q], desc[q + 1], idx[q], prob[q], pa, ix)
        lo, hi = ends[q], ends[q + 1]
        assert cnt[q] == r["n"], q
        assert (pts[lo:hi, :2] == r["pts0"]).all() and (pts[lo:hi, 2:] == r["pts1"]).all(), q
        assert (cell0[lo:hi] == r["cell0"]).all() and (bits(score[lo:hi]) == bits(r["score"])).all(), q


def test_ransac_and_pnp_on_callers_stream(side, plain, oracle, synth, monkeypatch):
    """RANSAC-E of a batch, and mv_pnp_gn_batch on test_pnp_split_launch_returns_identical_bytes's batch (pairs of 0 to
    1000 correspondences, the split launch forced): every hypothesis bit for bit against the oracle."""
    from oracle import orc
    monkeypatch.setenv("MV_PNP_K3_SMALL_BELOW", "0")
    rng = np.random.default_rng(5)
    P, M = 5, 300
    pts = np.zeros((P, M, 4), f32)
    cnt = rng.integers(1, M, size=P).astype(np.int32)
    for p in range(P):
        a = rng.integers(0, 600, size=(M, 2)).astype(f32)
        pts[p, :, :2] = a
        pts[p, :, 2:] = a + rng.integers(-1, 2, size=(M, 2))
    counts = np.array([330, 5, 0, 480, 600, 17, 330, 1000, 128, 3, 250], np.int32)
    corr = pnp_problems(synth, len(counts), 1000, 1024)
    H = 1024
    prm = pnp_params(H, 1)

    def work(tr):
        ninl, inl, pose = tr.ransac_identity(dev(tr, pts), dev(tr, cnt))
        kp, ks, kh = tr.pnp_gn(prm, dev(tr, corr), dev(tr, counts), want_hyp=True)
        return {"ninl": _b(ninl), "inl": _b(inl), "pose": _b(pose), "k3_pose": _b(kp), "k3_stats": _b(ks),
                "k3_hyp": _b(kh)}
    got = _both(side, plain, work)
    ninl = np.frombuffer(got["ninl"], np.int32)
    inl = np.frombuffer(got["inl"], np.int32).reshape(P, M)
    for p in range(P):
        _, ref_inl, n, _ = oracle.ransac_identity(pts[p, :cnt[p], :2], pts[p, :cnt[p], 2:], cap=M)
        assert ninl[p] == n and (inl[p, :n] == ref_inl).all(), p
    kp = np.frombuffer(got["k3_pose"], f32).reshape(-1, 7)
    ks = np.frombuffer(got["k3_stats"], f32).reshape(-1, 4)
    kh = np.frombuffer(got["k3_hyp"], f32).reshape(-1, H, 8)
    cfg = orc.pnp_cfg(hypotheses=H, seed=0, lanes=1)
    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:   # the oracle releases the GIL
        want = list(ex.map(lambda p: oracle.pnp_gn(cfg, corr[p], int(counts[p]), pair_index=p, want_hyp=True),
                           range(len(counts))))
    for p, n in enumerate(counts):
        rp, rs, rh = want[p]
        assert ks[p, 0] == rs[0] and ks[p, 3] == rs[3], (p, n, ks[p], rs)
        if n == 0:
            assert ks[p, 3] == 0 and (kp[p] == np.array([1, 0, 0, 0, 0, 0, 0], f32)).all()
            continue
        # every hypothesis bit for bit (a diverged one is NaN in both), so the selected pose is the oracle's
        same = (kh[p].view(np.int32) == rh.view(np.int32)) | (np.isnan(kh[p]) & np.isnan(rh))
        assert same.all(), (p, n, np.nonzero(~same.all(axis=1))[0][:8].tolist())
        if ks[p, 3] == 1:
            assert ks[p, 2] == rs[2] and kp[p].tobytes() == kh[p, int(ks[p, 2]), :7].tobytes(), (p, n)
            assert abs(ks[p, 1] - rs[1]) <= 1e-5 * abs(rs[1]), (p, n, ks[p], rs)


def test_bow_lba_and_trajectory_on_callers_stream(side, plain, oracle):
    """Word assignment (reference vocabulary), the Schur complement (the 8-pose, chunk-4 kernel and the generic one)
    and the solve, pose chaining and results_to_transforms."""
    from oracle import traj_oracle
    from maveric_slam_b200 import tracking
    rng = np.random.default_rng(29)
    vocab = ref_vocab()
    bow_in = bow_inputs(7, 37)
    J = {(P, ch): rng.normal(size=(2, 8 * ch, P, 20)).astype(f32) for P, ch in ((8, 4), (16, 8), (5, 2))}
    Cs = {P: np.stack([spd_system(rng, P)[0] for _ in range(3)]) for P in (16, 12, 3)}
    T = np.zeros((40, 3, 4))
    for k in range(40):
        q = rng.normal(size=4) * [1, 0.01, 0.02, 0.01] + [1, 0, 0, 0]
        T[k] = traj_oracle.quat_t_to_transform(q / np.linalg.norm(q), rng.normal(0, 1, 3))
    rec = np.zeros(20, tracking.PAIR_RESULT_DTYPE)
    q = rng.normal(size=(20, 4))
    rec["q"] = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(f32)
    rec["t"] = rng.normal(size=(20, 3)).astype(f32)

    def work(tr):
        tr.bow_set_vocabulary(*vocab)
        out = {"words": bow_check(tr, oracle, vocab, *bow_in).tobytes()}
        for key, j in J.items():
            out["schur%s" % (key,)] = _b(tr.lba_schur(dev(tr, j), key[1]))
        for P, c in Cs.items():
            d, ok = tr.lba_solve(dev(tr, c), 1e-3)
            out["solve%d" % P] = _b(d) + _b(ok)
        out["chain"] = _b(tr.chain_transforms(dev(tr, T)))
        out["transforms"] = _b(tr.results_to_transforms(dev(tr, rec.view(np.uint8).reshape(20, 64))))
        return out
    got = _both(side, plain, work)
    for (P, ch), j in J.items():
        C = np.frombuffer(got["schur%s" % ((P, ch),)], f32).reshape(2, 6 * P + 1, 6 * P + 1)
        for w in range(2):
            assert same_bits(C[w], oracle.lba_schur(j[w], ch)), (P, ch, w)
    for P, c in Cs.items():
        raw = got["solve%d" % P]
        d = np.frombuffer(raw[:3 * 6 * P * 4], f32).reshape(3, 6 * P)
        ok = np.frombuffer(raw[3 * 6 * P * 4:], np.int32)
        for w in range(3):
            ok_o, d_o = oracle.lba_solve(c[w], 1e-3)
            assert ok[w] == ok_o == 1 and same_bits(d[w], d_o), (P, w)
    traj = np.frombuffer(got["chain"], np.float64).reshape(41, 3, 4)
    ref = traj_oracle.chain_transforms(T)
    assert np.abs(traj - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max()) * 40 ** 0.5
    Tg = np.frombuffer(got["transforms"], np.float64).reshape(20, 3, 4)
    for k in range(20):
        assert np.abs(Tg[k] - traj_oracle.quat_t_to_transform(rec["q"][k], rec["t"][k])).max() <= 1e-15


# ------------------------------------------------------------------ 2. contexts used by several threads at once
ROUNDS = 8


def _run_threads(jobs, rounds=ROUNDS):
    """jobs: [(name, stream, fn)], fn() -> bytes.  Each job on a thread of its own, on its own stream; a barrier at
    the start of every round.  -> {name: [bytes of each round]}; a thread's exception fails the test."""
    import torch
    barrier = threading.Barrier(len(jobs), timeout=300)
    out = {name: [] for name, _, _ in jobs}
    errors = []

    def body(name, s, fn):
        try:
            with torch.cuda.stream(s):
                for _ in range(rounds):
                    barrier.wait()
                    out[name].append(fn())
        except threading.BrokenBarrierError:
            pass
        except BaseException as e:   # an MvError carries mv_last_error's text
            errors.append((name, repr(e)))
            barrier.abort()

    threads = [threading.Thread(target=body, args=job) for job in jobs]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    return out


def _path_job(torch, oracle, synth, rows, cols, seed):
    """The depth path with the tcgen05 matcher forced, on a Tracker of its own stream: (stream, fn, expected bytes);
    the expected bytes are the oracle's."""
    from maveric_slam_b200 import tracking
    n = 3
    semi, desc, depth, _ = synth.synth_sequence(seed, rows, cols, n, keypoint_permille=300)
    sscale = np.full(n, synth.SEMI_SCALE, f32)
    p = _depth_params(1, hypotheses=32, rows=rows, cols=cols, thr=0.9)
    rec, _, _ = landmark_reference(oracle, None, p, semi, sscale, desc, None, depth, depth_mode=True, threads=2)
    assert (rec["status"] == 0).all() and (rec["num_matches"] > 0).all(), rec
    s = torch.cuda.Stream(0)
    with torch.cuda.stream(s):
        tr = tracking.Tracker(0)
        d = [dev(tr, x) for x in (semi, sscale, desc, depth)]
        s.synchronize()
    return s, lambda: _b(tr.track_sequence(p, *d)), rec.tobytes()


def test_contexts_on_several_threads_at_once(torch_cuda, oracle, synth, lm_case):
    """Eight contexts on one GPU, each on a thread and a stream of its own, at the same time for 8 rounds: the
    tcgen05 matcher at 24x80, 47x155 and 94x310 (153 856, 157 696 and 166 912 bytes of dynamic shared memory), the
    generic Schur kernel at 16 poses / chunk 8 and 8 / 8 beside the 8 / 4 kernel, the solve at 16, 12 and 10 poses,
    the word assignment with the reference vocabulary and with a 64 x 210 one, and the landmark one-call from pinned
    buffers.  Every round returns the bytes of the serial run, and those are the oracle's."""
    torch = torch_cuda
    from maveric_slam_b200 import tracking
    jobs, want = [], {}
    for rows, cols, seed in ((24, 80, 3), (47, 155, 4), (94, 310, 5)):
        s, fn, rec = _path_job(torch, oracle, synth, rows, cols, seed)
        jobs.append(("path%dx%d" % (rows, cols), s, fn))
        want[jobs[-1][0]] = rec

    rng = np.random.default_rng(41)
    for name, shapes, solves in (("lba_large", ((16, 8),), (16,)), ("lba_small", ((8, 8), (8, 4)), (12, 10))):
        s = torch.cuda.Stream(0)
        J = [(ch, rng.normal(size=(2, 2 * 8, P, 20)).astype(f32)) for P, ch in shapes]
        Cs = [np.stack([spd_system(rng, P)[0] for _ in range(4)]) for P in solves]
        expect = b"".join(oracle.lba_schur(j[w], ch).tobytes() for ch, j in J for w in range(2))
        for c in Cs:
            sol = [oracle.lba_solve(c[w], 0.0) for w in range(4)]
            assert all(ok == 1 for ok, _ in sol)
            expect += np.stack([d for _, d in sol]).astype(f32).tobytes() + np.ones(4, np.int32).tobytes()
        with torch.cuda.stream(s):
            tr = tracking.Tracker(0)
            dj = [(ch, dev(tr, j)) for ch, j in J]
            dc = [dev(tr, c) for c in Cs]
            s.synchronize()

        def lba(tr=tr, dj=dj, dc=dc):
            out = b"".join(_b(tr.lba_schur(j, ch)) for ch, j in dj)
            for c in dc:
                d, ok = tr.lba_solve(c, 0.0)
                out += _b(d) + _b(ok)
            return out
        jobs.append((name, s, lba))
        want[name] = expect

    bow_in = bow_inputs(7, 37)
    for name, vocab in (("bow_ref", ref_vocab()), ("bow_64x210", bow_vocab("64x210"))):
        s = torch.cuda.Stream(0)
        with torch.cuda.stream(s):
            tr = tracking.Tracker(0)
            tr.bow_set_vocabulary(*vocab)
            words = bow_check(tr, oracle, vocab, *bow_in)     # the serial run, held to the oracle
            d = [dev(tr, x) for x in bow_in]
            s.synchronize()
        jobs.append((name, s, lambda tr=tr, d=d: _b(tr.bow_assign(*d)[0])))
        want[name] = words.tobytes()

    c, rec, nl, table = lm_case
    s = torch.cuda.Stream(0)
    with torch.cuda.stream(s):
        tr = tracking.Tracker(0)
        tr.bow_set_vocabulary(*c["vocab"])
        bufs = [pinned(x) for x in c["frames"]]

    def landmarks(tr=tr, bufs=bufs):
        t = tr.landmarks_new(c["n_words"])
        res, k, _, _ = tr.track_sequence_landmarks_host(c["p"], *bufs, t, first_frame=c["first"])
        return res.tobytes() + k.tobytes() + _b(t)
    jobs.append(("landmarks_host", s, landmarks))
    want["landmarks_host"] = rec + nl + table

    out = _run_threads(jobs)
    for name, rounds in out.items():
        assert len(rounds) == ROUNDS, name
        for r, got in enumerate(rounds):
            assert got == want[name], (name, "round", r)


# ------------------------------------------------------------------ 3. threads and devices
def test_context_made_on_one_thread_used_on_another(torch_cuda, oracle, synth):
    """A Tracker made on this thread (on a stream of its own), driven from a worker thread: the oracle's bytes, as on
    this thread."""
    torch = torch_cuda
    s, fn, want = _path_job(torch, oracle, synth, 24, 80, 7)
    with torch.cuda.stream(s):
        here = fn()
    there = _run_threads([("worker", s, fn)], rounds=2)["worker"]
    assert here == want and there == [want, want]


def test_contexts_of_two_gpus_from_two_threads(torch_cuda, synth):
    """Two threads whose current devices are GPU 0 and GPU 1 each drive a context on either GPU, alternately: the
    bytes of a one-GPU run, and after every call the thread's current device is the one it set."""
    torch = torch_cuda
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from maveric_slam_b200 import tracking
    rows, cols, n = 24, 80, 4
    semi, desc, depth, _ = synth.synth_sequence(3, rows, cols, n)
    sscale = np.full(n, synth.SEMI_SCALE, f32)
    p = _depth_params(None, hypotheses=64, rows=rows, cols=cols, top_n=100, max_matches=150, thr=0.9)
    ctxs = {}
    for t in (0, 1):
        for gpu in (0, 1):
            tr = tracking.Tracker(gpu)
            ctxs[t, gpu] = (tr, [dev(tr, x) for x in (semi, sscale, desc, depth)])
    torch.cuda.set_device(0)
    want = _b(ctxs[0, 0][0].track_sequence(p, *ctxs[0, 0][1]))
    got, errors = {}, []

    def body(t):
        try:
            torch.cuda.set_device(t)
            outs = []
            for _ in range(3):
                for gpu in (0, 1):
                    tr, d = ctxs[t, gpu]
                    res = tr.track_sequence(p, *d)
                    assert torch.cuda.current_device() == t, (t, gpu)
                    tr.ctx.sync()
                    assert torch.cuda.current_device() == t, (t, gpu)
                    outs.append(_b(res))
            got[t] = outs
        except BaseException as e:
            errors.append((t, repr(e)))

    threads = [threading.Thread(target=body, args=(t,)) for t in (0, 1)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    assert got[0] == [want] * 6 and got[1] == [want] * 6


def test_legacy_symbols_and_ex_forms_from_four_threads(torch_cuda, oracle, image0, kat):
    """compute_softmax, compute_top_N, ransac_essential_matrix and track through the legacy symbols (one global
    context behind a mutex) from four threads at once, and the `_ex` forms (detector, NMS, a matcher pair) with a
    context per thread: the reference's stored answers and the oracle's, on every thread and round."""
    from maveric_slam_b200 import lib, tracking
    rng = np.random.default_rng(3)
    p1 = rng.integers(0, 640, size=(150, 2)).astype(f32)
    p2 = p1 + rng.integers(-1, 2, size=(150, 2)).astype(f32)
    E_o, inl_o, n_o, _ = oracle.ransac_identity(p1, p2)
    scale = float(image0["semi_scale"])
    i_o, pr_o, _ = oracle.softmax(scale, image0["semi"])
    nms_o = oracle.nms(24, 80, i_o, pr_o)
    frame = tracking.frame_create(192, 640, 1, None, 24, 80, image0["semi_scale"], image0["semi"],
                                  image0["desc_scale"], image0["desc"])
    errors = []
    barrier = threading.Barrier(4, timeout=300)

    def body(t):
        try:
            ctx = lib.Context(0)
            for _ in range(4):
                barrier.wait()
                idx, pr, nv = tracking.compute_softmax(image0["semi_scale"], image0["semi"], legacy=True)
                assert nv == 410 and (idx == kat["img0_softmax_idx"]).all()
                assert (bits(pr) == bits(kat["img0_softmax_prob"])).all()
                pa, ix, pp = tracking.compute_top_N(image0["semi_scale"], image0["semi"], 100, legacy=True)
                assert (pa == kat["img0_top100_patch"]).all() and (ix == kat["img0_top100_idx"]).all()
                assert (bits(pp) == bits(kat["img0_top100_prob"])).all()
                E, inl, n = tracking.ransac_essential_matrix(p1, p2, np.eye(3, dtype=f32))
                assert n == n_o > 0 and (inl == inl_o).all() and (E == E_o).all()
                q, tt = tracking.track(frame, frame, 4, 4, 9, 0.9)
                assert (bits(tt) == bits(kat["pose_t"])).all()
                # the _ex forms on this thread's context
                ei, ep, en = tracking.compute_softmax(scale, image0["semi"], ctx=ctx)
                assert (ei == i_o).all() and (bits(ep) == bits(pr_o)).all() and en == 410
                ea, ex, _ = tracking.compute_top_N(scale, image0["semi"], 100, ctx=ctx)
                assert (ea == kat["img0_top100_patch"]).all() and (ex == kat["img0_top100_idx"]).all()
                mi, mp = tracking.run_nms(24, 80, ei, ep, ctx=ctx)
                assert (mi == nms_o[0]).all() and (bits(mp) == bits(nms_o[1])).all()
                m = tracking.match_pair(tracking.match_params(24, 80, use_tensor_cores=t % 2), image0["desc"],
                                        image0["desc"], ei, ep, ea, ex, ctx=ctx)
                assert m["n"] == 93 and (m["pts0"] == kat["self_pts0"]).all() and (m["pts1"] == kat["self_pts1"]).all()
            ctx.close()
        except threading.BrokenBarrierError:
            pass
        except BaseException as e:
            errors.append((t, repr(e)))
            barrier.abort()

    threads = [threading.Thread(target=body, args=(t,)) for t in range(4)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
