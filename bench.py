#!/usr/bin/env python
"""bench.py -- frame-pairs/sec of the tracking hot path (window match + PnP).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    (N > 1: launched by torch.distributed.run, one rank per GPU)

Workload (BASELINE.json configs[3], named in config.workload): a KITTI-00-length synthetic
sequence -- 4541 frames = 4540 frame pairs of a 47x155-cell grid (376x1241 px), ~1k keypoints
per frame, radius-4 window search, then per pair the reference's RANSAC-E inlier scan and a
Gauss-Newton PnP RANSAC with 1024 hypotheses x (4 minimal-sample + 10 refinement) iterations
over the pair's correspondences.  A step is one pass over all pairs; pairs shard across ranks
in contiguous blocks (strong scaling) and only the 64-byte per-pair results are all-gathered.

`value`  : device-resident inputs, CUDA-event timed, max over ranks.
`e2e`    : the same work through mv_track_sequence_host with pinned HOST buffers: per step all
           frames go host->device (chunked, overlapped with compute) and results come back.
           At N > 1 the ranks' blocks of this leg are cut by measured rank time before the timed
           steps (tracking.balance_shards: the host links of a box need not be equal); the gathered
           records are compared with the device-resident step's.
`roofline`: the dominant kernel (Gauss-Newton PnP; FP32-issue bound, see DESIGN.md) plus
           `rooflines` for every kernel of the step against its own bound.
`cpu_baseline`: the CPU port of the same path (oracle/, -O3 -march=native, OpenMP) on a bounded
           sample of the same pairs on this host.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROWS, COLS = 47, 155
N_FRAMES = 4541
TOP_N, MAX_VALID, MAX_MATCHES = 1000, 8192, 1024
HYPOTHESES, SAMPLE_ITERS, REFINE_ITERS = 1024, 4, 10
SEED = 0
FLOPS_NORMAL = 127         # FP32 flops of one correspondence in one Gauss-Newton pass (DESIGN.md §4.2; FMA = 2)
FLOPS_SCORE = 32           # ... in the final scoring pass (residual, gate, cost: no normal equations)
WORKLOAD = ("KITTI-00-length synthetic sequence: 4541 frames (4540 pairs), 47x155 cells, ~1k keypoints/frame, "
            "r=4 window match + RANSAC-E + GN-PnP 1024 hyp x (4+10) iters")


def workload_config(n_frames: int) -> dict:
    """The `config` object: the workload and nothing else, identical in both arms (--impl ours | reference).
    What is specific to an arm's run (sharding, matcher, the reference arm's sample size) goes to `run`."""
    return {"workload": WORKLOAD, "frames": n_frames, "pairs": n_frames - 1, "grid": [ROWS, COLS], "top_n": TOP_N,
            "max_matches": MAX_MATCHES, "hypotheses": HYPOTHESES, "gn_iters": [SAMPLE_ITERS, REFINE_ITERS],
            "cache": "a rank's device-resident frames (10.8 GB at N=1, 1.35 GB at N=8) exceed the 126 MB L2; no flush between steps"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured", d.get("sm_max_mhz", 1965.0)
    return 6650.0, "fallback", 1965.0


class ClockSampler:
    """nvidia-smi clocks + throttle reasons streamed during the timed region."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index: int, period_ms: int = 50):
        self.idx = gpu_index
        self.period_ms = period_ms
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.proc = None
        self._th = None

    def _reader(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 6:
                continue
            try:
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
            except ValueError:
                continue
            for n, v in zip(self.NAMES, f[2:6]):
                if v.lower().startswith("active"):
                    self.reasons.add(n)

    def __enter__(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.period_ms)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self._th = threading.Thread(target=self._reader, daemon=True)
            self._th.start()
            time.sleep(0.3)          # first samples land before the timed region starts
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.1)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            if self._th:
                self._th.join(timeout=2)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def track_cfg_for_oracle(orc, synth):
    return orc.TrackCfg(orc.MatchCfg(ROWS, COLS, 4, 4, 4, MAX_MATCHES, 0.9, 0.2),
                        orc.pnp_cfg(hypotheses=HYPOTHESES, sample_iters=SAMPLE_ITERS, refine_iters=REFINE_ITERS,
                                    seed=SEED, lanes=1),
                        TOP_N, MAX_VALID, 10, 1.1, float(synth.SEMI_SCALE))


def cpu_port_throughput(budget_s: float, n_threads: int | None = None):
    """Times the CPU port of the same path (oracle/, fast build) on a bounded sample."""
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import synth
    from oracle import orc
    o = orc.Oracle(fast=True)
    cores = n_threads or len(os.sched_getaffinity(0))
    cfg = track_cfg_for_oracle(orc, synth)
    syn = orc.SynthCfg(SEED, ROWS, COLS, 140, 6)
    offs = synth.default_offsets(N_FRAMES, SEED)
    # calibrate on one pair per thread, then size the sample to the budget
    t1, _ = o.bench_sequence(cfg, syn, offs[:cores + 1], 0, cores, cores)
    per_round = max(t1, 1e-3)
    rounds = int(max(1, min(budget_s / per_round, (N_FRAMES - 1) // cores)))
    n = min(N_FRAMES - 1, cores * rounds)
    secs, out = o.bench_sequence(cfg, syn, offs[:n + 1], 0, n, cores)
    cpu_port_throughput.last_results = out      # the checker's records of pairs [0, n)
    return n / secs, cores, n, secs


def reference_program_leg(tr, synth, tracking, torch, n_pairs=8192, ref_pairs=128):
    """What the reference program itself computes (src/tracking_main.c: 24x80 cells, top-100 queries,
    <= 150 matches, RANSAC-E + pose, no Gauss-Newton PnP): its unmodified sources (oracle/_ref, in process,
    one core -- it is single-threaded) against the library's batched kernels on this GPU, same inputs."""
    from oracle import orc
    if not orc.have_ref():
        return None
    rows, cols = 24, 80
    off = synth.default_offsets(n_pairs + 1, SEED)
    semi, desc, _ = tr.synth_frames(SEED, rows, cols, 0, off)
    scale = torch.full((n_pairs + 1,), float(synth.SEMI_SCALE), device=tr.device)
    mp = tracking.match_params(rows, cols, 4, 4, 4, 150)

    def step():
        idx, prob, _ = tr.softmax(semi, scale)
        qp, qi, _, qc, _ = tr.top_n(idx, prob, 100, 1000)
        pts, cnt, _, _, _ = tr.match(mp, desc, idx, prob, qp, qi, qc)
        ninl, _, _ = tr.ransac_identity(pts, cnt, 10, 1.1)
        return pts, cnt, ninl

    for _ in range(3):
        out = step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    gpu_pairs_s = n_pairs / (e0.elapsed_time(e1) / 5 * 1e-3)
    pts, cnt, ninl = [x[:ref_pairs].cpu().numpy() for x in out]
    ref = orc.Reference()
    hs, hd = semi[:ref_pairs + 1].cpu().numpy(), desc[:ref_pairs + 1].cpu().numpy()
    t0 = time.perf_counter()
    res = [ref.tracking_main(synth.SEMI_SCALE, hs[p], hd[p], synth.SEMI_SCALE, hs[p + 1], hd[p + 1])
           for p in range(ref_pairs)]
    dt = (time.perf_counter() - t0) / ref_pairs
    same = all(r["n"] == cnt[p] and r["num_inliers"] == ninl[p]
               and np.array_equal(r["pts0"], pts[p, :r["n"], :2]) and np.array_equal(r["pts1"], pts[p, :r["n"], 2:])
               for p, r in enumerate(res))
    return {"kind": "reference", "cores": 1, "value": 1.0 / dt, "unit": "frame-pairs/s",
            "workload": "the reference's own program at its native shape: 24x80 cells, N=100, <=150 matches, RANSAC-E + pose "
                        "(no Gauss-Newton PnP); %d pairs through main() of src/tracking_main.c in process" % ref_pairs,
            "gpu_same_workload": {"value": gpu_pairs_s, "unit": "frame-pairs/s", "pairs_per_launch": n_pairs},
            "same_matches_and_inliers": bool(same)}


def parity_against_port(resn, out, n):
    """The timed GPU records of the first n pairs against the CPU port's, in the same run: counts and
    the selected hypothesis exactly, the pose within BASELINE.json's tolerance (1e-5 rad / 1e-5)."""
    bad = 0
    max_ang = max_dt = 0.0
    for p in range(n):
        r, g = out[p], resn[p]
        exact = (g["num_matches"] == r.num_matches and g["ransac_inliers"] == r.ransac_inliers
                 and g["pnp_inliers"] == r.pnp_inliers and g["best_hypothesis"] == r.best_h and g["status"] == r.status)
        q1 = np.asarray(g["q"], np.float64); q2 = np.asarray(list(r.q), np.float64)
        q1 = q1 / np.linalg.norm(q1); q2 = q2 / np.linalg.norm(q2)
        # angle of the relative rotation from the vector part of q1 * conj(q2) (well conditioned near zero)
        vx = q1[0] * q2[1] - q1[1] * q2[0] - q1[2] * q2[3] + q1[3] * q2[2]
        vy = q1[0] * q2[2] + q1[1] * q2[3] - q1[2] * q2[0] - q1[3] * q2[1]
        vz = q1[0] * q2[3] - q1[1] * q2[2] + q1[2] * q2[1] - q1[3] * q2[0]
        ang = 2.0 * float(np.arctan2(np.sqrt(vx * vx + vy * vy + vz * vz), abs(float(np.dot(q1, q2)))))
        t2 = np.asarray(list(r.t), np.float64)
        dt = float(np.linalg.norm(np.asarray(g["t"], np.float64) - t2) / max(1.0, np.linalg.norm(t2)))
        if r.num_matches > 0:
            max_ang, max_dt = max(max_ang, ang), max(max_dt, dt)
        if not exact or ang > 1e-5 or dt > 1e-5:
            bad += 1
    return {"pairs_checked": int(n), "mismatches": int(bad), "max_rotation_error_rad": max_ang,
            "max_translation_error_rel": max_dt,
            "what": "num_matches, ransac_inliers, pnp_inliers, best hypothesis exact; pose within 1e-5 rad / 1e-5"}


def dump_outputs(out_dir: str, recs) -> None:
    """One .npy per field of the pair records a caller of mv_track_sequence receives (all pairs, 64 B each):
    float fields as float32, integer fields as float64 (exact)."""
    os.makedirs(out_dir, exist_ok=True)
    for name in recs.dtype.names:
        if name == "pad":
            continue
        a = recs[name]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32 if a.dtype.kind == "f" else np.float64))


def run_reference(args, rank: int):
    if rank != 0:
        return
    vals = []
    n = cores = 0
    for i in range(args.warmup + args.steps):
        # each step: a bounded sample, the whole run about a minute (MV_BENCH_REF_BUDGET_S: test hook)
        budget = float(os.environ.get("MV_BENCH_REF_BUDGET_S", max(4.0, 60.0 / max(1, args.steps + args.warmup))))
        v, cores, n, secs = cpu_port_throughput(budget_s=budget)
        if i >= args.warmup:
            vals.append((v, secs))
    value = float(np.mean([v for v, _ in vals]))
    line = {
        "impl": "reference", "metric": "frame-pairs/sec (window match + PnP)", "value": value, "unit": "frame-pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": float(np.mean([s for _, s in vals]) * 1e3), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "int8 match / fp32 PnP", "data": "synthetic",
        "config": workload_config(args.frames),
        "run": {"sample_pairs_per_step": n, "note": "each step times the first sample_pairs_per_step pairs of the configured "
                                                    "sequence on all host cores and reports pairs/s"},
        "cpu_baseline": {"value": value, "unit": "frame-pairs/s", "cores": cores, "kind": "port",
                         "sample": f"first {n} pairs of the same synthetic sequence per step, OpenMP over pairs, "
                                   "oracle/mv_oracle.c built -O3 -march=native (the reference itself is fixed at 24x80 "
                                   "cells / N=100 and has no PnP, so its CPU path is timed through the port that is "
                                   "bit-pinned to it)"},
        "e2e": {"value": value, "unit": "frame-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--frames", type=int, default=N_FRAMES, help="sequence length (default: KITTI-00, 4541)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--matcher", default="tcgen05", choices=["tcgen05", "dp4a"],
                    help="windowed matcher: tcgen05 tile GEMM (default) or the dp4a warp-per-query kernel")
    ap.add_argument("--tensor-cores", action="store_true", help="same as --matcher tcgen05")
    ap.add_argument("--lanes", type=int, default=1,
                    help="PnP summation lanes per hypothesis (1: one thread; 2: one thread, packed FFMA2; 4..32: threads)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the per-pair results of the last timed step as DIR/<field>.npy (float32 / float64), "
                         "so that two builds can be compared on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    args.tensor_cores = args.tensor_cores or args.matcher == "tcgen05"
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    import maveric_slam_b200  # noqa: F401
    from maveric_slam_b200 import synth, tracking

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    n_frames = args.frames
    n_pairs = n_frames - 1
    first, count, per = tracking.shard_pairs(n_pairs, world, rank)
    tr = tracking.Tracker(local_rank)
    params = tracking.kitti_track_params(top_n=TOP_N, max_valid=MAX_VALID, max_matches=MAX_MATCHES,
                                         hypotheses=HYPOTHESES, refine_iters=REFINE_ITERS,
                                         sample_iters=SAMPLE_ITERS, seed=SEED, first_pair=first, lanes=args.lanes,
                                         use_tensor_cores=args.tensor_cores)

    # ---- inputs: this rank's frames [first, first+count] generated on the device (setup, untimed)
    offs = synth.default_offsets(n_frames, SEED)
    my_frames = count + 1
    semi, desc, depth = tr.synth_frames(SEED, ROWS, COLS, first, offs[first:first + my_frames])
    scale = torch.full((my_frames,), float(synth.SEMI_SCALE), device=dev)
    # the pack kernel writes the rank's records straight into the persistent, padded NCCL send buffer
    gat = tracking.ResultGather(n_pairs, world, rank, dev)
    out = gat.send
    torch.cuda.synchronize()
    in_bytes = semi.numel() + desc.numel() + depth.numel() * 4

    def step():
        tr.track_sequence(params, semi, scale, desc, depth, out=out)
        return gat.gather()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = tr.ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        barrier()
        e0.record()
        for _ in range(args.steps):
            res = step()
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1)
    launches = tr.ctx.launches - launches0
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    ms_per_step = ms_max / args.steps
    value = n_pairs / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        # `res` is every pair's record as the last timed step gathered it; the passes below overwrite it
        dump_outputs(args.dump_outputs, tracking.results_to_numpy(res))

    # ---- per-kernel device time (CUDA events on the launch stream, separate short pass)
    tr.ctx.profile(True)
    for _ in range(2):
        tr.track_sequence(params, semi, scale, desc, depth, out=out)
    tr.ctx.sync()
    prof = {}
    for tag in ["detect", "topn", "match", "emit", "ransac", "gather", "pnp", "pnp_select"]:
        prof[tag] = tr.ctx.profile_read(tag)[0]
    # the tensor-core matcher's three kernels (inside "match"; not added to the step sum a second time)
    match_parts = {tag: tr.ctx.profile_read(tag)[0] for tag in ["match_compact", "match_lead", "match_gemm"]}
    match_tiles, match_chunks = tr.ctx.match_work() if args.tensor_cores else (0, 0)
    pnp_accepted = tr.ctx.pnp_work() // 2   # accepted correspondence-passes of one step (two profiled steps)
    tr.ctx.profile(False)

    resn = tracking.results_to_numpy(out)
    n_corr = int(resn["num_matches"].sum())
    hbm_peak, peak_src, sm_max = peaks()
    cells = ROWS * COLS
    sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    fp32_nominal = sm_count * 128 * 2 * sm_max * 1e6 / 1e12   # TFLOP/s, FMA = 2 flops
    # ALGORITHMIC flops = what the oracle's Gauss-Newton executes (DESIGN.md 4.2): every correspondence is
    # projected and gated in every pass (FLOPS_SCORE); only an accepted one is accumulated into the normal
    # equations (FLOPS_NORMAL - FLOPS_SCORE more).  `pnp_accepted` is counted by the kernel in profile mode.
    # The dense equivalent (every correspondence updates in every pass) is reported beside it.
    pnp_flops_dense = (count * HYPOTHESES * SAMPLE_ITERS * 8 * FLOPS_NORMAL
                       + HYPOTHESES * n_corr * (REFINE_ITERS * FLOPS_NORMAL + FLOPS_SCORE))
    if pnp_accepted > 0:
        pnp_flops = (count * HYPOTHESES * SAMPLE_ITERS * 8 * FLOPS_NORMAL
                     + HYPOTHESES * n_corr * (REFINE_ITERS + 1) * FLOPS_SCORE
                     + pnp_accepted * (FLOPS_NORMAL - FLOPS_SCORE))
    else:   # kernel forms without the counter (lanes > 1, MV_PNP_FORM=mask|dense)
        pnp_flops = pnp_flops_dense
    pnp_bytes = 20 * n_corr + 64 * count
    pnp_ms = prof["pnp"]

    def hbm_entry(name, tag, bytes_):
        ms_k = prof[tag]
        ach = bytes_ / (ms_k * 1e-3) / 1e9 if ms_k > 0 else None
        return {"kernel": name, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                "frac": ach / hbm_peak if ach else None, "ms_per_launch": ms_k, "algorithmic_bytes": bytes_,
                "peak_source": peak_src}

    # ---- matcher work.  Algorithmic int8 ops (SURVEY §8d: 2*256*sum_q |window_q|, cells valid or not) and
    # algorithmic bytes (SURVEY §8d B_match: descriptors read once + mask/idx + output) from an untimed pass;
    # the tile ops the tensor pipe executed from the library's own count of the chunks it ran.
    idx_t, prob_t, _ = tr.softmax(semi, scale)
    qp_t, _, _, qc_t, _ = tr.top_n(idx_t, prob_t, TOP_N, MAX_VALID)
    qp_h, qc_h = qp_t.cpu().numpy(), qc_t.cpu().numpy()
    n_cand = int(((idx_t != 64) & ~(prob_t < 0.2)).sum().item())     # candidate cells of all frames
    del idx_t, prob_t, qp_t, qc_t
    win_cells = 0
    n_queries = 0
    for f in range(1, my_frames):
        pq = qp_h[f, :min(int(qc_h[f]), TOP_N)].astype(np.int64)
        if pq.size == 0:
            continue
        n_queries += int(pq.size)
        x, y = pq // ROWS, pq % ROWS
        w = np.clip(np.minimum(x + 4 + 4, COLS - 1) - np.maximum(x + 4 - 4, 0) + 1, 0, None)
        h = np.clip(np.minimum(y + 4 + 4, ROWS - 1) - np.maximum(y + 4 - 4, 0) + 1, 0, None)
        win_cells += int((w * h).sum())
    match_alg_ops = 2 * 256 * win_cells
    tile_ops = match_chunks * 2 * 128 * 256 * 64
    # B_match per pair = 256*(N + cells0) + 8*cells0 + 8*N + 16*matches (SURVEY §8d), and the tighter figure
    # with only the cells that are candidates (what an ideal matcher has to read under the reference's rules)
    match_bytes_survey = 256 * (n_queries + count * cells) + 8 * count * cells + 8 * n_queries + 16 * n_corr
    match_bytes_valid = 256 * (n_queries + n_cand) + 8 * count * cells + 8 * n_queries + 16 * n_corr
    ipath = os.path.join(ROOT, "profiles", "int8_peak.json")
    if os.path.exists(ipath):
        ij = json.load(open(ipath))
        int8_peak, int8_src = ij["int8_tops"], ("measured on this pool by tools/int8_peak.py (cuBLASLt s8 GEMM 8192^3, burst; "
                                                "sustained %.0f): profiles/int8_peak.json" % ij["int8_tops_sustained"])
    else:
        int8_peak = 2.0 * (json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops", 1590.0)
                           if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 1590.0)
        int8_src = "ASSUMED 2 x measured dense bf16 (profiles/int8_peak.json absent)"
    match_ms = prof["match"]
    match_entries = []
    if args.tensor_cores:
        gemm_ms = match_parts["match_gemm"]
        match_entries.append(
            {"kernel": "match_tc_kernel (K1 tile GEMM + exact-score epilogue, tcgen05 kind::i8 + TMA)", "bound": "tensor",
             "achieved": tile_ops / (gemm_ms * 1e-3) / 1e12 if gemm_ms else None, "peak": int8_peak, "unit": "TOP/s",
             "frac": (tile_ops / (gemm_ms * 1e-3) / 1e12) / int8_peak if gemm_ms else None, "ms_per_launch": gemm_ms,
             "executed_tile_int8_ops": tile_ops, "tiles": match_tiles, "chunks_128x256x64": match_chunks,
             "algorithmic_int8_ops": match_alg_ops, "executed_over_algorithmic": tile_ops / max(1, match_alg_ops),
             "algorithmic_TOPs_whole_matcher": match_alg_ops / (match_ms * 1e-3) / 1e12 if match_ms else None,
             "peak_source": int8_src,
             "note": "K=64 per tile (the reference scores 64 dims) and an exact-score epilogue: at r=4 the matcher is "
                     "HBM/latency-bound (next entry), the tensor pipe idles; see DESIGN.md 4.1 and profiles/"})
        match_entries.append(
            {"kernel": "matcher K1 = compact_candidates + lead + match_tc kernels (whole)", "bound": "hbm",
             "achieved": match_bytes_survey / (match_ms * 1e-3) / 1e9 if match_ms else None, "peak": hbm_peak, "unit": "GB/s",
             "frac": (match_bytes_survey / (match_ms * 1e-3) / 1e9) / hbm_peak if match_ms else None,
             "ms_per_launch": match_ms, "kernel_ms": match_parts, "algorithmic_bytes": match_bytes_survey,
             "algorithmic_bytes_candidates_only": match_bytes_valid,
             "frac_candidates_only": (match_bytes_valid / (match_ms * 1e-3) / 1e9) / hbm_peak if match_ms else None,
             "peak_source": peak_src,
             "note": "algorithmic_bytes = SURVEY §8d B_match (every cell's descriptor once); candidates_only counts the "
                     "descriptors of candidate cells and queries only"})
    else:
        match_entries.append(hbm_entry("match_queries_kernel (K1a, dp4a)", "match", match_bytes_valid))
    rooflines = [
        {"kernel": ("pnp_gn_twophase_kernel (K3)" if args.lanes == 1 else "pnp_gn_kernel<%d> (K3)" % args.lanes), "bound": "fp32", "achieved": pnp_flops / (pnp_ms * 1e-3) / 1e12 if pnp_ms else None,
         "peak": fp32_nominal, "unit": "TFLOP/s",
         "frac": (pnp_flops / (pnp_ms * 1e-3) / 1e12) / fp32_nominal if pnp_ms else None,
         "ms_per_launch": pnp_ms, "algorithmic_flops": pnp_flops,
         "flops_note": "algorithmic = the oracle's operation count: 32 flop to project and gate every correspondence in "
                       "every pass, 95 more for each accepted one in a normal-equation pass (accepted passes counted by "
                       "the kernel: %d per step = %.1f%% of all); dense_equivalent_flops counts all 127 for every "
                       "correspondence" % (pnp_accepted, 100.0 * pnp_accepted / max(1, HYPOTHESES * n_corr * REFINE_ITERS)),
         "dense_equivalent_flops": pnp_flops_dense,
         "dense_equivalent_TFLOPs": pnp_flops_dense / (pnp_ms * 1e-3) / 1e12 if pnp_ms else None,
         "peak_source": "nominal: SMs x 128 FMA/clk x 2 x clocks.max.sm from MEASURED_PEAKS.json "
                        "(FFMA microbenchmark on this pool: 72.9 TFLOP/s, profiles/r01/ffma_peak.txt)",
         "hbm_achieved_gbs": pnp_bytes / (pnp_ms * 1e-3) / 1e9 if pnp_ms else None},
        hbm_entry("softmax_cells_kernel (K0a)", "detect", my_frames * cells * (65 + 8)),
        # K0b reads idx/prob twice (count + select); the algorithm needs them once
        hbm_entry("top_n_kernel (K0b)", "topn", my_frames * (cells * 8 + TOP_N * 12)),
    ] + match_entries
    step_kernel_ms = sum(v for v in prof.values())
    roofline = dict(rooflines[0])
    roofline["traffic"] = None
    # DRAM traffic of the dominant kernel from its ncu --set full capture (profiles/ncu_traffic.json holds
    # dram__bytes_read.sum + dram__bytes_write.sum of one launch and the pairs that launch processed)
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tpath) and args.lanes == 1:
        tj = json.load(open(tpath))
        per_pair = tj["pnp_gn_dram_bytes_per_launch"] / tj["pairs_per_launch"]
        roofline["traffic"] = int(per_pair * count)
        roofline["traffic_source"] = tj.get("source") + " (scaled by pairs per launch: %d -> %d)" % (tj["pairs_per_launch"], count)
        roofline["algorithmic_bytes"] = pnp_bytes
    roofline["share_of_step"] = pnp_ms / step_kernel_ms if step_kernel_ms else None

    # ---- end to end through the host-buffer entry point
    e2e = None
    if not args.no_e2e:
        if world > 1:   # staging memory on the NUMA node of this rank's GPU (a no-op where the platform does not say)
            tracking.bind_to_gpu_numa_node(local_rank)
        res_device = res.clone()   # all pairs, as the device-resident steps gathered them

        class HostShard:
            """Pinned host copies of frames [first_, first_ + count_] and the parameters of that block."""
            def __init__(self, first_, count_):
                self.first, self.count = first_, count_
                if (first_, count_) == (first, count):
                    s_, d_, z_ = semi, desc, depth
                else:
                    s_, d_, z_ = tr.synth_frames(SEED, ROWS, COLS, first_, offs[first_:first_ + count_ + 1])
                self.semi = torch.empty(s_.shape, dtype=torch.int8, pin_memory=True)
                self.desc = torch.empty(d_.shape, dtype=torch.int8, pin_memory=True)
                self.depth = torch.empty(z_.shape, dtype=torch.float32, pin_memory=True)
                self.scale = torch.full((count_ + 1,), float(synth.SEMI_SCALE), dtype=torch.float32).pin_memory()
                self.semi.copy_(s_); self.desc.copy_(d_); self.depth.copy_(z_)
                torch.cuda.synchronize()
                self.params = params if first_ == first else tracking.kitti_track_params(
                    top_n=TOP_N, max_valid=MAX_VALID, max_matches=MAX_MATCHES, hypotheses=HYPOTHESES,
                    refine_iters=REFINE_ITERS, sample_iters=SAMPLE_ITERS, seed=SEED, first_pair=first_,
                    lanes=args.lanes, use_tensor_cores=args.tensor_cores)
                self.out = np.zeros(count_, tracking.PAIR_RESULT_DTYPE)
                self.up = self.down = 0

            def run(self):
                if self.count > 0:
                    _, self.up, self.down = tr.track_sequence_host(self.params, self.semi, self.scale, self.desc,
                                                                   self.depth, out=self.out)

        def all_ranks(x: float):
            v = torch.full((world,), 0.0, dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_gather_into_tensor(v, torch.tensor([x], dtype=torch.float64, device=dev))
            else:
                v[0] = x
            return [float(a) for a in v.tolist()]

        # Blocks of the host-buffer path follow the ranks' measured step times (tracking.balance_shards): on a
        # box whose GPUs do not share one host-link rate, equal blocks leave the fast ranks idle.  At most three
        # rounds of: every rank runs its block at the same time, times are gathered, blocks are re-cut.  Symmetric
        # boxes (and N = 1) keep the equal blocks.  MV_BENCH_BALANCE=0 switches it off, MV_BENCH_WEIGHTS=a,b,..
        # forces a partition (test hook).
        counts = [tracking.shard_pairs(n_pairs, world, r)[1] for r in range(world)]
        equal_counts = list(counts)
        balance_log = []
        forced = os.environ.get("MV_BENCH_WEIGHTS")
        if world > 1 and forced:
            counts = [c for _, c in tracking.shard_pairs_weighted(n_pairs, [float(x) for x in forced.split(",")])]
        shard = HostShard(sum(counts[:rank]), counts[rank])
        shard.run()
        shard.run()
        if world > 1 and not forced and os.environ.get("MV_BENCH_BALANCE", "1") != "0":
            for _ in range(3):
                best = float("inf")
                for _ in range(2):
                    barrier()
                    t0 = time.perf_counter()
                    shard.run()
                    best = min(best, time.perf_counter() - t0)
                secs = all_ranks(best)
                balance_log.append({"pairs_per_rank": list(counts), "rank_ms": [round(x * 1e3, 3) for x in secs]})
                new_counts = tracking.balance_shards(counts, secs)
                if new_counts == counts:
                    break
                counts = new_counts
                shard = HostShard(sum(counts[:rank]), counts[rank])
                shard.run()
        gat_e = gat if counts == equal_counts else tracking.ResultGather(n_pairs, world, rank, dev, counts=counts)
        barrier()
        t0 = time.perf_counter()
        full = None
        for _ in range(args.steps):
            shard.run()
            if world > 1:
                gat_e.send.copy_(torch.from_numpy(shard.out.view(np.uint8).reshape(-1, 64)), non_blocking=True)
                full = gat_e.gather()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s = float(tt.item()) / args.steps
        up_all, down_all = sum(all_ranks(float(shard.up))), sum(all_ranks(float(shard.down)))
        if world > 1:
            same = bool(torch.equal(full, res_device))
        else:
            same = shard.out.tobytes() == resn.tobytes()
        e2e = {"value": n_pairs / e2e_s, "unit": "frame-pairs/s",
               "h2d_bytes_per_step": int(up_all), "d2h_bytes_per_step": int(down_all),
               "bytes_are": "summed over the ranks", "ms_per_step": e2e_s * 1e3,
               "results_equal_device_path": bool(same),
               "api": "mv_track_sequence_host (pinned host buffers, chunked H2D overlapped with compute)",
               "pairs_per_rank": list(counts)}
        if balance_log:
            e2e["balance_rounds"] = balance_log
        del shard

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, cores, n, secs = cpu_port_throughput(budget_s=15.0)
        cpu = {"value": v, "unit": "frame-pairs/s", "cores": cores, "kind": "port",
               "sample": f"first {n} pairs of the same sequence, {secs:.1f} s, OpenMP over pairs, "
                         "oracle/mv_oracle.c -O3 -march=native",
               "parity": parity_against_port(resn, cpu_port_throughput.last_results, n)}
        try:
            cpu["reference_program"] = reference_program_leg(tr, synth, tracking, torch)
        except Exception as e:   # the main line must not depend on this leg
            cpu["reference_program"] = {"error": str(e)[:200]}

    if rank == 0:
        line = {
            "metric": "frame-pairs/sec (window match + PnP)", "value": value, "unit": "frame-pairs/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int8 match / fp32 PnP", "data": "synthetic",
            "config": workload_config(n_frames),
            "run": {"pnp_lanes_per_hypothesis": args.lanes, "matcher": "tcgen05" if args.tensor_cores else "dp4a",
                    "match_algorithmic_int8_ops_per_step": match_alg_ops,
                    "sharding": f"{world} x contiguous pair blocks, all_gather of 64 B/pair",
                    "cache": f"inputs {in_bytes / 1e9:.2f} GB per rank >> 126 MB L2, no flush needed",
                    "mean_matches_per_pair": n_corr / max(1, count)},
            "clocks": clk.summary(), "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "rooflines": rooflines, "kernel_ms": prof, "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
