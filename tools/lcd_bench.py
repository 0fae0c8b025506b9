#!/usr/bin/env python
"""Loop closure on the bench sequence (4 541 synthetic KITTI-shaped frames, 47 x 155 cells, 1 000 words a frame, the
reference's 10 000-word vocabulary): the candidate scoring (mv_loop_candidates with idf weights) and the whole
mv_detect_loops call.

Times: CUDA events of the context's profile mode ("lcd" = presence + tiles + merge, "lcd_tiles" = the tensor-core
tile kernel alone), and events around whole mv_detect_loops calls.  Work: the tile kernel executes
tiles x 128 x 128 x kpad int8 multiply-adds (kpad = n_words rounded up to 64); it is compared with the measured int8
peak of profiles/int8_peak.json.  The operands (2 x frames x kpad bytes, 91 MB) fit the 126 MB L2.

    python tools/lcd_bench.py [--frames N] [--reps R] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import maveric_slam_b200  # noqa: E402,F401
from maveric_slam_b200 import synth, tracking  # noqa: E402

TILE, KBLOCK = 128, 64


def tiles(n, min_gap):
    """Tiles the candidate stage launches: per row tile, the column tiles that hold a pair j <= i - min_gap."""
    t = 0
    for ti in range((n + TILE - 1) // TILE):
        max_i = min(ti * TILE + TILE - 1, n - 1)
        t += (max_i - min_gap) // TILE + 1 if max_i >= min_gap else 0
    return t


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=4541)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--detect-reps", type=int, default=3)
    ap.add_argument("--min-gap", type=int, default=30)
    ap.add_argument("--k", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    n = a.frames
    tr = tracking.Tracker(0)
    v = np.load(os.path.join(ROOT, "tests", "golden", "ref_vocab.npz"))
    tr.bow_set_vocabulary(v["base_desc"], v["scale"], v["bias"], v["leaves"])
    semi, desc, depth = tr.synth_frames(0, 47, 155, 0, synth.default_offsets(n, 0))
    sscale = torch.full((n,), float(synth.SEMI_SCALE), device=tr.device)
    dscale = torch.full((n,), float(synth.DESC_SCALE), device=tr.device)
    idx, prob, _ = tr.softmax(semi, sscale)
    qp, qi, _, qc, _ = tr.top_n(idx, prob, 1000, 8192)
    word, _ = tr.bow_assign(desc, dscale, qp, qc)
    weight = tr.lcd_word_weights(word, qc)

    # candidate scoring: warm-up, then profiled launches
    for _ in range(3):
        cand, score = tr.loop_candidates(word, qc, weight, a.min_gap, a.k)
    tr.ctx.sync()
    tr.ctx.profile(True)
    for _ in range(a.reps):
        cand, score = tr.loop_candidates(word, qc, weight, a.min_gap, a.k)
    tr.ctx.sync()
    ms_stage = tr.ctx.profile_read("lcd")[0]
    ms_tiles = tr.ctx.profile_read("lcd_tiles")[0]
    tr.ctx.profile(False)

    n_words = tr.n_words
    kpad = (n_words + KBLOCK - 1) // KBLOCK * KBLOCK
    t = tiles(n, a.min_gap)
    ops = 2.0 * t * TILE * TILE * kpad
    peak = json.load(open(os.path.join(ROOT, "profiles", "int8_peak.json")))

    # the whole call
    p = tracking.loop_params(47, 155, top_n=1000, max_valid=8192, max_matches=1024, hypotheses=1024,
                             min_gap=a.min_gap, k=a.k)
    out = tr.detect_loops(p, semi, sscale, desc, dscale, depth, weight)
    tr.ctx.sync()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(a.detect_reps):
        out = tr.detect_loops(p, semi, sscale, desc, dscale, depth, weight)
    ev1.record()
    ev1.synchronize()
    ms_detect = ev0.elapsed_time(ev1) / a.detect_reps
    res = tracking.loop_results_to_numpy(out)

    r = {"gpu": gpu_info(), "frames": n, "n_words": n_words, "top_n": 1000, "min_gap": a.min_gap, "k": a.k,
         "candidates_ms": ms_stage, "tile_kernel_ms": ms_tiles, "tiles": t, "kpad": kpad,
         "executed_int8_tops": ops / (ms_tiles * 1e-3) / 1e12,
         "frac_of_measured_int8_peak": ops / (ms_tiles * 1e-3) / 1e12 / peak["int8_tops"],
         "frac_of_sustained_int8_peak": ops / (ms_tiles * 1e-3) / 1e12 / peak["int8_tops_sustained"],
         "detect_loops_ms": ms_detect, "verified_pairs": int((cand.cpu().numpy() >= 0).sum()),
         "accepted_loops": int((res["frame"] >= 0).sum()), "reps": a.reps, "detect_reps": a.detect_reps}
    line = json.dumps(r)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
