#!/usr/bin/env python
"""BASELINE.json configs[4] end to end: 94x310 cells, 16k keypoints per frame (SURVEY §8d C5; --permille 850:
85 % of the synthetic world's cells are keypoints, of which the detector selects the top 16 000 per frame;
round 1 and the first half of round 2 ran --permille 550 = ~12.2k keypoints), 33x33 search window, up to 16384 matches per pair, 4096 Gauss-Newton hypotheses.  On one B200 or,
under torchrun, sharded by contiguous pair blocks over N B200s with the one all_gather of 64-byte
records (the same sharding as bench.py).  Device-resident frames, CUDA events, max over ranks, 2 warm-ups;
prints one JSON line with the per-kernel breakdown of rank 0.  Also a scale check of the whole path: two
runs must return identical bytes and both matchers must agree; and parity: rank 0's first 8 pairs against the CPU
oracle (orc_bench_sequence on all host cores), compared as bench.py's cpu_baseline.parity (--no-parity skips it).

    python tools/stress_bench.py [--frames F] [--steps K] [--no-parity]
    python -m torch.distributed.run --nproc-per-node 8 --master-addr 127.0.0.1 tools/stress_bench.py --frames 257
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=33)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--permille", type=int, default=850, help="keypoint density of the synthetic world")
    ap.add_argument("--no-parity", action="store_true", help="skip the comparison with the CPU oracle")
    args = ap.parse_args()
    import torch
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import synth, tracking

    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    rows, cols, seed = 94, 310, 0
    n_pairs_all = args.frames - 1
    first, count, per = tracking.shard_pairs(n_pairs_all, world, rank)
    tr = tracking.Tracker(local_rank)
    off = synth.default_offsets(args.frames, seed)
    semi, desc, depth = tr.synth_frames(seed, rows, cols, first, off[first:first + count + 1], keypoint_permille=args.permille)
    scale = torch.full((count + 1,), float(synth.SEMI_SCALE), device=tr.device)
    gat = tracking.ResultGather(n_pairs_all, world, rank, tr.device)

    def params(tc=True):
        return tracking.track_params(rows, cols, top_n=16000, max_valid=32768, max_matches=16384, hypotheses=4096,
                                     radius=16, shift=(4, 4), use_tensor_cores=tc, first_pair=first)

    out = tr.track_sequence(params(), semi, scale, desc, depth)
    ref = out.cpu().numpy().tobytes()
    local = tracking.results_to_numpy(out)
    same = tr.track_sequence(params(), semi, scale, desc, depth).cpu().numpy().tobytes() == ref
    dp4a = tr.track_sequence(params(False), semi, scale, desc, depth).cpu().numpy().tobytes() == ref
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        tr.track_sequence(params(), semi, scale, desc, depth, out=gat.send)
        allres = gat.gather()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / args.steps], dtype=torch.float64, device=tr.device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    tr.ctx.profile(True)
    tr.track_sequence(params(), semi, scale, desc, depth, out=gat.send)
    tr.ctx.sync()
    prof = {t_: tr.ctx.profile_read(t_)[0] for t_ in ["detect", "topn", "match", "emit", "ransac", "gather", "pnp", "pnp_select"]}
    tr.ctx.profile(False)
    out = allres
    res = tracking.results_to_numpy(out)
    idx_, prob_, _ = tr.softmax(semi, scale)
    kp = float(tr.top_n(idx_, prob_, 16000, 32768)[3].float().mean().item())   # query keypoints per frame (rank 0)
    n_pairs = args.frames - 1
    flags = torch.tensor([int(same), int(dp4a)], device=tr.device)
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    parity = None
    if rank == 0 and not args.no_parity:
        import numpy as np
        from bench import parity_against_port
        from oracle import orc
        n_par = min(8, count)
        cfg = orc.TrackCfg(orc.MatchCfg(rows, cols, 4, 4, 16, 16384, 0.9, 0.2),
                           orc.pnp_cfg(hypotheses=4096, seed=0, lanes=1), 16000, 32768, 10, 1.1, float(synth.SEMI_SCALE))
        _, cpu = orc.Oracle().bench_sequence(cfg, orc.SynthCfg(seed, rows, cols, args.permille, 6),
                                             np.ascontiguousarray(off[:n_par + 1]), 0, n_par, os.cpu_count() or 1)
        parity = parity_against_port(local, cpu, n_par)
    if rank == 0:
        print(json.dumps({
            "metric": "frame-pairs/sec (window match + PnP), BASELINE configs[4] stress shape, %d GPU(s)" % world,
            "value": n_pairs / (ms * 1e-3), "unit": "frame-pairs/s", "n_gpus": world, "ms_per_step": ms, "pairs": n_pairs,
            "config": {"grid": [rows, cols], "radius": 16, "top_n": 16000, "max_matches": 16384, "hypotheses": 4096,
                       "keypoint_permille": args.permille, "keypoints_per_frame": kp,
                       "mean_matches_per_pair": float(res["num_matches"].mean()),
                       "mean_pnp_inliers": float(res["pnp_inliers"].mean())},
            "kernel_ms_rank0": prof, "deterministic": bool(flags[0].item()), "dp4a_matcher_same_bytes": bool(flags[1].item()),
            "status_ok": bool((res["status"] == 0).all()), "parity": parity}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
