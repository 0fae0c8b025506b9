#!/usr/bin/env python
"""A small invocation of every kernel of the library, meant to run under compute-sanitizer:

    compute-sanitizer --tool memcheck --error-exitcode 9 python tools/sanitize_path.py
    compute-sanitizer --tool racecheck|synccheck|initcheck ... python tools/sanitize_path.py [stages]

Stages (default all): seq (device-resident sequence, tcgen05 and dp4a matchers, every PnP form),
host (host-buffer sequence with the TMA row gather), nms, traj, lba.  Sizes are small: a tool that
replays every memory access is 10-100x slower than the kernels.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import maveric_slam_b200  # noqa: E402,F401
from maveric_slam_b200 import synth, tracking  # noqa: E402

stages = set(sys.argv[1:]) or {"seq", "host", "nms", "traj", "lba"}
tr = tracking.Tracker(0)
rows, cols, nf = 24, 80, 4
semi, desc, depth = tr.synth_frames(1, rows, cols, 0, synth.default_offsets(nf, 1))
scale = torch.full((nf,), float(synth.SEMI_SCALE), device=tr.device)

if "seq" in stages:
    ref = None
    for tc in (True, False):
        for lanes, hyp in ((1, 300), (32, 32)):     # the two K3 mappings
            p = tracking.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=hyp,
                                      lanes=lanes, use_tensor_cores=tc)
            res = tr.track_sequence(p, semi, scale, desc, depth)
            tr.ctx.sync()
            if lanes == 1:
                b = res.cpu().numpy().tobytes()
                ref = ref or b
                assert b == ref, "matchers disagree"
    for knob in ("MV_PNP_STREAM", "MV_PNP_GPW"):     # streaming kernel for every pair; 128 hypotheses per CTA
        os.environ[knob] = "1"
        p = tracking.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=300)
        assert tr.track_sequence(p, semi, scale, desc, depth).cpu().numpy().tobytes() == ref, knob
        os.environ.pop(knob)
    # KITTI grid: ragged tiles of 128 queries, windows clipped at the border
    s2, d2, z2 = tr.synth_frames(2, 47, 155, 0, synth.default_offsets(3, 2))
    p = tracking.kitti_track_params(hypotheses=256)
    tr.track_sequence(p, s2, torch.full((3,), float(synth.SEMI_SCALE), device=tr.device), d2, z2)
    tr.ctx.sync()
    print("seq ok", flush=True)

if "host" in stages:
    p = tracking.track_params(rows, cols, top_n=100, max_valid=1000, max_matches=150, hypotheses=128)
    pin = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t) for t in (semi, scale, desc, depth)]
    torch.cuda.synchronize()
    out, up, down = tr.track_sequence_host(p, pin[0], pin[1], pin[2], pin[3])
    dev = tracking.results_to_numpy(tr.track_sequence(p, semi, scale, desc, depth))
    assert out.tobytes() == dev.tobytes(), "host path differs from the device path"
    print("host ok", up, down, flush=True)

if "nms" in stages:
    idx, prob, _ = tr.softmax(semi, scale)
    tr.nms(rows, cols, idx, prob)
    tr.ctx.sync()
    print("nms ok", flush=True)

if "traj" in stages:
    T = torch.zeros((1500, 3, 4), dtype=torch.float64, device=tr.device)
    T[:, 0, 0] = T[:, 1, 1] = T[:, 2, 2] = 1.0
    T[:, 2, 3] = 0.5
    P = tr.chain_transforms(T)
    assert abs(float(P[-1, 2, 3]) - 750.0) < 1e-9
    print("traj ok", flush=True)

if "lba" in stages:
    g = torch.Generator(device="cpu").manual_seed(3)
    for (L, P_, ch) in ((40, 8, 4), (24, 3, 2), (32, 16, 8)):
        J = torch.randn((3, L, P_, 20), generator=g).to(tr.device)
        Cm = tr.lba_schur(J, ch)
        d, ok = tr.lba_solve(Cm, 1e-3)
        assert int(ok.sum()) == 3 and bool(torch.isfinite(d).all())
    print("lba ok", flush=True)
print("sanitize_path done")
