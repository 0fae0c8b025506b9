import sys, os, time, json
sys.path.insert(0, '/root/repo')
import numpy as np, torch
import maveric_slam_b200
from maveric_slam_b200 import synth, tracking
ROWS, COLS, NF = 47, 155, 4541
tr = tracking.Tracker(0)
params = tracking.kitti_track_params(top_n=1000, max_valid=8192, max_matches=1024, hypotheses=1024, refine_iters=10, sample_iters=4, seed=0, first_pair=0, lanes=1, use_tensor_cores=True)
offs = synth.default_offsets(NF, 0)
semi, desc, depth = tr.synth_frames(0, ROWS, COLS, 0, offs)
scale = torch.full((NF,), float(synth.SEMI_SCALE), device=tr.device)
hs = torch.empty(semi.shape, dtype=torch.int8, pin_memory=True).copy_(semi)
hd = torch.empty(desc.shape, dtype=torch.int8, pin_memory=True).copy_(desc)
hz = torch.empty(depth.shape, dtype=torch.float32, pin_memory=True).copy_(depth)
hsc = torch.empty(scale.shape, dtype=torch.float32, pin_memory=True).copy_(scale)
del semi, desc, depth
torch.cuda.synchronize()
out = np.zeros(NF - 1, tracking.PAIR_RESULT_DTYPE)
ref = None
for label, env in [("default", {}), ("chunk185", {"MV_HOST_CHUNK_PAIRS": "185"}), ("chunk740", {"MV_HOST_CHUNK_PAIRS": "740"})]:
    os.environ.pop("MV_HOST_CHUNK_PAIRS", None)
    os.environ.update(env)
    for _ in range(2):
        tr.track_sequence_host(params, hs, hsc, hd, hz, out=out)
    t0 = time.perf_counter()
    for _ in range(5):
        _, up, down = tr.track_sequence_host(params, hs, hsc, hd, hz, out=out)
    dt = (time.perf_counter() - t0) / 5
    if ref is None: ref = out.tobytes()
    print(label, "%.2f ms  %.1f GB/s  %.0f pairs/s same=%s" % (dt * 1e3, up / dt / 1e9, (NF - 1) / dt, out.tobytes() == ref), flush=True)
