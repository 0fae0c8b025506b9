#!/usr/bin/env python
"""The landmark sequence path (mv_track_sequence_landmarks) on the bench workload (BASELINE configs[3]: 4 541
KITTI-shaped synthetic frames, 47x155 cells, top_n 1000, 1024 matches, 1024 hypotheses; vocabulary
tests/golden/ref_vocab.npz), against the depth path (mv_track_sequence) in the same process, alternated.

Reports device-resident pairs/s of both paths (host clock around work ending in a device synchronise), the per-stage
device times of the landmark path from the context's profile mode (bow, sort, walk, corr), the per-frame loop of
mv_landmarks_observe / mv_landmarks_remove_old over the same words for contrast, the longest word list and the mean
landmarks per pair.

End to end from pinned host buffers (the frames a caller gets off a camera or a file), alternated in one process:
the depth path (mv_track_sequence_host) and the landmark path (mv_track_sequence_landmarks_host); median pairs/s,
h2d bytes and the host-to-device rate they imply.   python tools/landmark_bench.py [frames] [steps] > out.json"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import maveric_slam_b200  # noqa: E402,F401
from maveric_slam_b200 import synth, tracking  # noqa: E402

NF = int(sys.argv[1]) if len(sys.argv) > 1 else 4541
STEPS = int(sys.argv[2]) if len(sys.argv) > 2 else 5
SEED = 0

tr = tracking.Tracker(0)
v = np.load(os.path.join(ROOT, "tests", "golden", "ref_vocab.npz"))
tr.bow_set_vocabulary(v["base_desc"], v["scale"], v["bias"], v["leaves"])
p = tracking.kitti_track_params(top_n=1000, max_valid=8192, max_matches=1024, hypotheses=1024, refine_iters=10,
                                sample_iters=4, seed=SEED)
semi, desc, depth = tr.synth_frames(SEED, 47, 155, 0, synth.default_offsets(NF, SEED))
sscale = torch.full((NF,), float(synth.SEMI_SCALE), device=tr.device)
dscale = torch.full((NF,), 4.3353, device=tr.device)
table = tr.landmarks_new(tr.n_words)
out = torch.empty((NF - 1, 64), dtype=torch.uint8, device=tr.device)
nl = torch.empty((NF - 1,), dtype=torch.int32, device=tr.device)


def depth_step():
    tr.track_sequence(p, semi, sscale, desc, depth, out=out)


def landmark_step():
    tr.ctx.check(tr.lib.mv_landmarks_init(tr.ctx.h, tr.n_words, tr._d(table)))
    tr.track_sequence_landmarks(p, semi, sscale, desc, dscale, depth, table, out=out, n_with_landmark=nl)


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


for fn in (depth_step, landmark_step):   # warm-up: modules, scratch
    fn()
times = {"depth": [], "landmarks": []}
for _ in range(STEPS):
    times["depth"].append(timed(depth_step))
    times["landmarks"].append(timed(landmark_step))
launches0 = tr.ctx.launches
landmark_step()
torch.cuda.synchronize()
launches_landmark = tr.ctx.launches - launches0
launches0 = tr.ctx.launches
depth_step()
torch.cuda.synchronize()
launches_depth = tr.ctx.launches - launches0

# per-stage device times (profile mode, a run of its own)
tr.ctx.profile(True)
for _ in range(3):
    landmark_step()
stages = {t: tr.ctx.profile_read(t)[0] for t in ("detect", "topn", "bow", "sort", "walk", "corr", "match", "ransac", "pnp")}
tr.ctx.profile(False)

# the same table update as the per-frame loop of the existing kernels: 2 calls (3 launches) per frame
idx, prob, _ = tr.softmax(semi, sscale)
qp, qi, _, qc, _ = tr.top_n(idx, prob, 1000, 8192)
word, _ = tr.bow_assign(desc[:NF - 1], dscale[:NF - 1], qp[:NF - 1], qc[:NF - 1])
hc = qc.cpu().numpy()
coords = torch.zeros((NF - 1, 1000, 3), dtype=torch.float32, device=tr.device)
words_f = [word[f, :min(int(hc[f]), 1000)] for f in range(NF - 1)]
coords_f = [coords[f, :min(int(hc[f]), 1000)] for f in range(NF - 1)]
loop_table = tr.landmarks_new(tr.n_words)


def per_frame_loop():
    for f in range(NF - 1):
        tr.landmarks_observe(loop_table, f, words_f[f], coords_f[f])
        tr.landmarks_remove_old(loop_table, f)


def batched():
    tr.landmarks_sequence(seq_table, 0, word, qc[:NF - 1], coords, coords_out)


seq_table = tr.landmarks_new(tr.n_words)
coords_out = torch.empty_like(coords)
per_frame_loop(); batched()
loop_s = min(timed(per_frame_loop) for _ in range(3))
seq_s = min(timed(batched) for _ in range(3))

# end to end from pinned host buffers
def pinned(t):
    return torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t)


hs, hsc, hd, hds, hz = (pinned(t) for t in (semi, sscale, desc, dscale, depth))
host_nl = np.zeros(NF - 1, np.int32)
e2e = {}


def depth_host():
    e2e["depth_host"] = tr.track_sequence_host(p, hs, hsc, hd, hz)


def landmark_host():
    tr.ctx.check(tr.lib.mv_landmarks_init(tr.ctx.h, tr.n_words, tr._d(table)))
    e2e["landmark_host"] = tr.track_sequence_landmarks_host(p, hs, hsc, hd, hds, hz, table, n_with_landmark=host_nl)


legs = {"depth_host": depth_host, "landmark_host": landmark_host}
for fn in legs.values():   # warm-up: pinned pages, scratch of the host pipeline
    fn()
e2e_times = {k: [] for k in legs}
for _ in range(STEPS):
    for k, fn in legs.items():
        e2e_times[k].append(timed(fn))
host_table = table.clone()
landmark_step()
device_res, device_nl = out.cpu().numpy().tobytes(), nl.cpu().numpy()
host_equals_device = (e2e["landmark_host"][0].tobytes() == device_res and (host_nl == device_nl).all()
                      and bool(torch.equal(host_table, table)))
e2e_out = {}
for k in legs:
    med = float(np.median(e2e_times[k]))
    up = e2e[k][-2]
    e2e_out[k] = {"median_s": med, "pairs_per_s": (NF - 1) / med, "h2d_bytes": up, "d2h_bytes": e2e[k][-1],
                  "h2d_GB_per_s": up / med / 1e9, "h2d_bytes_per_frame": up / NF, "all_s": e2e_times[k]}

w = word.cpu().numpy()
valid = w[(w >= 0) & (w < tr.n_words)]
hist = np.bincount(valid, minlength=tr.n_words)
res = tracking.results_to_numpy(out)
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
dt, lt = float(np.median(times["depth"])), float(np.median(times["landmarks"]))
print(json.dumps({
    "gpu": gpu, "frames": NF, "pairs": NF - 1, "steps": STEPS,
    "depth_path": {"median_s": dt, "pairs_per_s": (NF - 1) / dt, "launches": launches_depth, "all_s": times["depth"]},
    "landmark_path": {"median_s": lt, "pairs_per_s": (NF - 1) / lt, "launches": launches_landmark,
                      "all_s": times["landmarks"]},
    "landmark_stage_ms": stages,
    "new_stages_ms": stages["bow"] + stages["sort"] + stages["walk"] + stages["corr"],
    "table_update_per_frame_loop_ms": loop_s * 1e3, "table_update_batched_ms": seq_s * 1e3,
    "tables_equal": bool(torch.equal(loop_table, seq_table)),
    "occurrences": int(valid.size), "distinct_words": int((hist > 0).sum()), "longest_word_list": int(hist.max()),
    "longest_word": int(hist.argmax()), "mean_landmarks_per_pair": float(nl.float().mean().item()),
    "mean_matches_per_pair": float(res["num_matches"].mean()),
    "e2e_pinned": e2e_out, "e2e_landmark_host_equals_device": bool(host_equals_device),
}, indent=1))
