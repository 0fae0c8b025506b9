#!/usr/bin/env python
"""The landmark path sharded over GPUs (tracking.track_sequence_landmarks_sharded) on the bench workload (BASELINE
configs[3]: 4 541 KITTI-shaped synthetic frames, 47x155 cells, top_n 1000, 1024 matches, 1024 hypotheses; vocabulary
tests/golden/ref_vocab.npz), device-resident, against the depth path sharded the same way, legs alternated in one
process.

    torchrun --nproc_per_node N tools/landmark_shard_bench.py [frames] [steps] [out.json]
    python tools/landmark_shard_bench.py ...            (one GPU, no torchrun)

Per leg: median pairs/s (host clock around a step that ends in a barrier and a device synchronise on every rank).
One leg is the undivided mv_track_sequence_landmarks over the whole sequence on each rank's GPU: the split's own
cost at N = 1.
For the landmark legs (W = warm-up frames per block: 0 is the plain relay, 8 / 16 / 32 speculate) each rank's
median device times of prepare, the wait for the table, step_table and solve (CUDA events), and the words each rank
walked again.  Checks, on every rank, that the gathered records, landmark counts and final table equal one
mv_track_sequence_landmarks over the whole sequence on that rank's GPU.

Host legs, from pinned host copies of the frames (each rank stages through its own link):
    landmarks_host_one_call     mv_track_sequence_landmarks_host over the whole sequence, on each rank's GPU
    landmarks_host_W<w>         tracking.track_sequence_landmarks_host_sharded (W = 0, 8, 32)
    landmarks_upload_relay      the rank's frames uploaded whole (every descriptor), then the device relay (W = 0)
with each rank's h2d bytes per step, the phase times and re-walked words of the sharded legs, and the same
byte-equality check."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import maveric_slam_b200  # noqa: E402,F401
from maveric_slam_b200 import synth, tracking  # noqa: E402

NF = int(sys.argv[1]) if len(sys.argv) > 1 else 4541
STEPS = int(sys.argv[2]) if len(sys.argv) > 2 else 5
OUT = sys.argv[3] if len(sys.argv) > 3 else None
WARMS = (0, 8, 16, 32)
SEED = 0

world = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))

tr = tracking.Tracker(local)
v = np.load(os.path.join(ROOT, "tests", "golden", "ref_vocab.npz"))
tr.bow_set_vocabulary(v["base_desc"], v["scale"], v["bias"], v["leaves"])
p = tracking.kitti_track_params(top_n=1000, max_valid=8192, max_matches=1024, hypotheses=1024, refine_iters=10,
                                sample_iters=4, seed=SEED)
semi, desc, depth = tr.synth_frames(SEED, 47, 155, 0, synth.default_offsets(NF, SEED))
sscale = torch.full((NF,), float(synth.SEMI_SCALE), device=tr.device)
dscale = torch.full((NF,), 4.3353, device=tr.device)
frames = (semi, sscale, desc, dscale, depth)
n_pairs = NF - 1
table = tr.landmarks_new(tr.n_words)
gat = tracking.ResultGather(n_pairs, world, rank, tr.device)


def barrier():
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()


def depth_step():
    pp = tracking.kitti_track_params(top_n=1000, max_valid=8192, max_matches=1024, hypotheses=1024, refine_iters=10,
                                     sample_iters=4, seed=SEED, first_pair=gat.first)
    if gat.count:
        lo, hi = gat.first, gat.first + gat.count + 1
        tr.track_sequence(pp, semi[lo:hi], sscale[lo:hi], desc[lo:hi], depth[lo:hi], out=gat.send)
    return gat.gather()


last = {}


def landmark_step(w):
    tr.ctx.check(tr.lib.mv_landmarks_init(tr.ctx.h, tr.n_words, tr._d(table)))
    ev = []
    rec, nl, rw = tracking.track_sequence_landmarks_sharded(tr, p, frames, table, first_frame=0, n_warm=w, timings=ev)
    last[w] = (rec, nl, rw, ev)


def timed(fn):
    barrier()
    t0 = time.perf_counter()
    fn()
    barrier()
    return time.perf_counter() - t0


one_table = tr.landmarks_new(tr.n_words)


def one_call_step():   # the undivided call over the whole sequence, for the split's own cost at N = 1
    tr.ctx.check(tr.lib.mv_landmarks_init(tr.ctx.h, tr.n_words, tr._d(one_table)))
    tr.track_sequence_landmarks(p, *frames, one_table, first_frame=0)


# ---- host legs
HOST_WARMS = (0, 8, 32)
host = tuple(torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t) for t in frames)
torch.cuda.synchronize()
h2d = {}
host_last = {}


def host_one_call_step():
    tr.ctx.check(tr.lib.mv_landmarks_init(tr.ctx.h, tr.n_words, tr._d(one_table)))
    _, _, up, _ = tr.track_sequence_landmarks_host(p, *host, one_table, first_frame=0)
    h2d["landmarks_host_one_call"] = up


def host_step(w, key):
    tr.ctx.check(tr.lib.mv_landmarks_init(tr.ctx.h, tr.n_words, tr._d(table)))
    ev = []
    rec, nl, rw, up = tracking.track_sequence_landmarks_host_sharded(tr, p, host, table, first_frame=0, n_warm=w,
                                                                     timings=ev)
    host_last[key] = (rec, nl, rw, ev)
    h2d[key] = up


def upload_relay_step():
    # what a user without prepare_host does: the rank's frames (block and halo) copied whole, then the device relay
    if gat.count:
        lo, hi = gat.first, gat.first + gat.count + 1
        for d, hst in zip(frames, host):
            d[lo:hi].copy_(hst[lo:hi], non_blocking=True)
        h2d["landmarks_upload_relay"] = sum(x[lo:hi].numel() * x.element_size() for x in host)
    landmark_step(0)
    host_last["landmarks_upload_relay"] = last[0]


legs = {"depth": depth_step, "landmarks_one_call": one_call_step}
for w in WARMS:
    legs[f"landmarks_W{w}"] = (lambda w=w: landmark_step(w))
legs["landmarks_host_one_call"] = host_one_call_step
for w in HOST_WARMS:
    legs[f"landmarks_host_W{w}"] = (lambda w=w: host_step(w, f"landmarks_host_W{w}"))
legs["landmarks_upload_relay"] = upload_relay_step

SHARDED = [k for k in legs if k.startswith("landmarks_host_W")] + ["landmarks_upload_relay"]
for fn in legs.values():   # warm-up: modules, scratch, NCCL communicators
    fn()
times = {k: [] for k in legs}
phases = {w: [] for w in WARMS}
rewalked = {w: [] for w in WARMS}
host_phases = {k: [] for k in SHARDED}
host_rewalked = {k: [] for k in SHARDED}
for _ in range(STEPS):
    for k, fn in legs.items():
        times[k].append(timed(fn))
        if k.startswith("landmarks_W"):
            w = int(k[len("landmarks_W"):])
            ev = last[w][3]
            phases[w].append([ev[i].elapsed_time(ev[i + 1]) for i in range(4)])
            rewalked[w].append(int(last[w][2].item()))
        if k in SHARDED:
            ev = host_last[k][3]
            host_phases[k].append([ev[i].elapsed_time(ev[i + 1]) for i in range(4)])
            host_rewalked[k].append(int(host_last[k][2].item()))

# byte-equality with one call over the whole sequence on this rank's GPU
one = tr.landmarks_new(tr.n_words)
res1, nl1 = tr.track_sequence_landmarks(p, *frames, one, first_frame=0)
equal = {}
for w in WARMS:
    landmark_step(w)
    rec, nl, _, _ = last[w]
    equal[w] = bool(rec.cpu().numpy().tobytes() == res1.cpu().numpy().tobytes() and torch.equal(nl, nl1)
                    and torch.equal(table, one))
host_equal = {}
for k in SHARDED:
    legs[k]()
    rec, nl, _, _ = host_last[k]
    host_equal[k] = bool(rec.cpu().numpy().tobytes() == res1.cpu().numpy().tobytes() and torch.equal(nl, nl1)
                         and torch.equal(table, one))
tr.ctx.check(tr.lib.mv_landmarks_init(tr.ctx.h, tr.n_words, tr._d(one_table)))
h_res, h_nl, _, _ = tr.track_sequence_landmarks_host(p, *host, one_table, first_frame=0)
host_equal["landmarks_host_one_call"] = bool(h_res.tobytes() == res1.cpu().numpy().tobytes()
                                             and (h_nl == nl1.cpu().numpy()).all() and torch.equal(one_table, one))

mine = {"rank": rank, "device": torch.cuda.get_device_name(local), "block": [gat.first, gat.count],
        "equal_to_one_gpu": {str(w): equal[w] for w in WARMS},
        "phase_ms_median": {str(w): dict(zip(("prepare", "table_wait", "step_table", "solve"),
                                             np.median(np.array(phases[w]), axis=0).round(4).tolist()))
                            for w in WARMS},
        "rewalked_words": {str(w): rewalked[w][-1] for w in WARMS},
        "host_equal_to_one_gpu": host_equal, "h2d_bytes_per_step": h2d,
        "host_phase_ms_median": {k: dict(zip(("prepare", "table_wait", "step_table", "solve"),
                                             np.median(np.array(v), axis=0).round(4).tolist()))
                                 for k, v in host_phases.items()},
        "host_rewalked_words": {k: v[-1] for k, v in host_rewalked.items()}}
ranks = [None] * world
if world > 1:
    dist.all_gather_object(ranks, mine)
else:
    ranks = [mine]
if rank == 0:
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                                "-i", str(local)], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        power = "not read"
    med = {k: float(np.median(t)) for k, t in times.items()}
    out = {"gpus": world, "frames": NF, "pairs": n_pairs, "steps": STEPS, "gpu": power,
           "pairs_per_s": {k: n_pairs / m for k, m in med.items()}, "median_s": med,
           "all_s": times, "ranks": ranks,
           "all_equal_to_one_gpu": all(all(r["equal_to_one_gpu"].values()) and all(r["host_equal_to_one_gpu"].values())
                                       for r in ranks)}
    s = json.dumps(out, indent=1)
    print(s)
    if OUT:
        os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
        open(OUT, "w").write(s + "\n")
if world > 1:
    dist.destroy_process_group()
