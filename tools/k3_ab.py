#!/usr/bin/env python
"""A/B timing of a kernel's environment knobs on the bench workload (4 540 pairs x 1 024
hypotheses): one process, the knob read per call, CUDA-event kernel times from the context's
profile mode (K3_AB_TAG: pnp by default, or match, detect, ...), results compared byte for byte
with the default's.

    python tools/k3_ab.py [ENV=VALUE[,ENV=VALUE] ...]     e.g.  MV_PNP_STREAM=1 MV_PNP_GPW=1 MV_PNP_TAIL_PAIRS=0
    K3_AB_TAG=match python tools/k3_ab.py                 (another kernel's time; K3_AB_FRAMES=569 a shorter sequence)
    MV_LIB_PATH=/path/variant.so python tools/k3_ab.py    (an A/B build of the library: build.py MV_EXTRA_NVCC / MV_OUT)
"""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import maveric_slam_b200  # noqa: E402,F401
from maveric_slam_b200 import synth, tracking  # noqa: E402

NF = int(os.environ.get("K3_AB_FRAMES", "4541"))
TAG = os.environ.get("K3_AB_TAG", "pnp")
tr = tracking.Tracker(0)
params = tracking.kitti_track_params(top_n=1000, max_valid=8192, max_matches=1024, hypotheses=1024, refine_iters=10,
                                     sample_iters=4, seed=0, first_pair=0, lanes=1, use_tensor_cores=True)
semi, desc, depth = tr.synth_frames(0, 47, 155, 0, synth.default_offsets(NF, 0))
scale = torch.full((NF,), float(synth.SEMI_SCALE), device=tr.device)
ref = None
knobs = set()
variants = [{}] + [dict(kv.split("=", 1) for kv in a.split(",")) for a in sys.argv[1:]] + [{}]
for env in variants:
    knobs |= set(env)
for env in variants:
    for k in knobs:
        os.environ.pop(k, None)
    os.environ.update(env)
    for _ in range(2):
        res = tr.track_sequence(params, semi, scale, desc, depth)
    tr.ctx.sync()
    tr.ctx.profile(True)
    for _ in range(3):
        res = tr.track_sequence(params, semi, scale, desc, depth)
    tr.ctx.sync()
    ms = tr.ctx.profile_read(TAG)[0]
    tr.ctx.profile(False)
    b = res.cpu().numpy().tobytes()
    if ref is None:
        ref = b
    print(json.dumps({"env": env, TAG + "_ms": ms, "same_bytes": b == ref, "sha1": hashlib.sha1(b).hexdigest()[:12]}),
          flush=True)   # sha1: compare two libraries (MV_LIB_PATH) across processes
