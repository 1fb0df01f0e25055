#!/usr/bin/env python
"""Times the EPnP initialiser of the 6DoF evaluation flow (epnp_epnp_init_f32) and the evaluation step around it.

    python tools/epnp_bench.py [--out profiles/r3_epnp.jsonl] [--iters 20]

One JSON line per measurement, on stdout and, with --out, appended to that file:
  * kernel: B in {32, 256, 4096}, N = 4096 (64 x 64 maps), q = 0.8 -- CUDA events around `iters` launches after a
    warm-up.  At B = 4096 the inputs are 4096 * 4096 * 28 B = 470 MB, larger than the 126 MB L2; the smaller batches are
    L2-resident after the first pass (said so in the record).
  * step: the evaluation step of EPro-PnP-6DoF/lib/test.py:196-211 -- epnp_pose_init, AdaptiveHuberPnPCost.set_param and
    EProPnP6DoF(...) with fast_mode=True -- host clock around `iters` steps ending in a device synchronise.
  * cv2_loop: the host loop test.py:176-194 replaces (numpy quantile mask, cv2.solvePnP(SOLVEPNP_EPNP), scipy), host
    time per object -- only where cv2 is importable; otherwise the record says "not measured".
The card's name and power limit are read in the same run and go into every record.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "epro-pnp_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np   # noqa: E402
import torch         # noqa: E402


def card():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        _, power, clock = [s.strip() for s in out.split(",")]
        info.update(power_limit=power, max_sm_clock=clock)
    except Exception as e:                                  # noqa: BLE001
        info.update(power_limit=f"not read ({type(e).__name__})")
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("tools/epnp_bench.py measures on a CUDA device; none is available")
    from epropnp.camera import PerspectiveCamera
    from epropnp.cost_fun import AdaptiveHuberPnPCost
    from epropnp.epnp_init import epnp_pose_init
    from epropnp.epropnp import EProPnP6DoF
    from epropnp.levenberg_marquardt import LMSolver
    from epropnp_b200 import native
    from epropnp_b200.synth import make_problem

    dev = torch.device("cuda:0")
    hw = card()
    out = None
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        out = open(args.out, "a")

    def emit(rec):
        rec.update(card=hw)
        line = json.dumps(rec)
        print(line, flush=True)
        if out is not None:
            out.write(line + "\n")
            out.flush()

    N, q = 4096, 0.8
    for B in (32, 256, 4096):
        pc = make_problem(B, N, seed=3, grid2d=True)
        x3d, x2d, w2d, K = (pc[k].to(dev) for k in ("x3d", "x2d", "w2d", "cam_mats"))
        for _ in range(args.warmup):
            native.epnp_init(x3d, x2d, w2d, K, q)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.iters):
            native.epnp_init(x3d, x2d, w2d, K, q)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.iters
        in_bytes = B * N * (3 + 2 + 2) * 4
        emit(dict(what="kernel epnp_epnp_init_f32", B=B, N=N, q=q, iters=args.iters, ms_per_call=ms,
                  us_per_object=1e3 * ms / B, input_bytes=in_bytes,
                  cache="inputs larger than L2" if in_bytes > 126e6 else "inputs L2-resident after the first pass"))

        # the evaluation step (test.py:196-211): EPnP initial pose, set_param, GN fast-mode solve in the 6DoF layer
        camera = PerspectiveCamera(cam_mats=K, z_min=0.01)
        cost_fun = AdaptiveHuberPnPCost(relative_delta=0.1)
        layer = EProPnP6DoF(mc_samples=512, num_iter=4, solver=LMSolver(dof=6, num_iter=10))

        def step():
            pose_init = epnp_pose_init(x3d, x2d, w2d, K, q)
            cost_fun.set_param(x2d, w2d)
            return layer(x3d, x2d, w2d, camera, cost_fun, pose_init=pose_init, fast_mode=True)[0]

        with torch.no_grad():
            for _ in range(args.warmup):
                step()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.iters):
                step()
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / args.iters
        emit(dict(what="evaluation step (epnp_pose_init + set_param + EProPnP6DoF fast_mode)", B=B, N=N, q=q,
                  iters=args.iters, ms_per_step=1e3 * dt, us_per_object=1e6 * dt / B))

    try:
        import cv2
        from scipy.spatial.transform import Rotation
    except ImportError:
        emit(dict(what="cv2 host loop (test.py:176-194)", result="not measured: cv2 is not importable here"))
        return
    B = 32
    pc = make_problem(B, N, seed=3, grid2d=True)
    x3d, x2d, w2d, K = (pc[k].numpy() for k in ("x3d", "x2d", "w2d", "cam_mats"))
    t0 = time.perf_counter()
    conf = w2d.mean(-1)
    mask = conf >= np.quantile(conf.reshape(B, -1), q, axis=1, keepdims=True)
    for b in range(B):
        _, rv, tv = cv2.solvePnP(x3d[b][mask[b]], x2d[b][mask[b]], K[b], np.zeros((4, 1), np.float32),
                                 flags=cv2.SOLVEPNP_EPNP)
        Rotation.from_rotvec(rv.reshape(-1)).as_quat()[[3, 0, 1, 2]]
    dt = time.perf_counter() - t0
    emit(dict(what="cv2 host loop (test.py:176-194)", B=B, N=N, q=q, ms_total=1e3 * dt, us_per_object=1e6 * dt / B,
              cv2=cv2.__version__))


if __name__ == "__main__":
    main()
