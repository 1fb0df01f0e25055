"""Golden vectors of the EPnP initialiser of the 6DoF evaluation flow: cv2 and scipy run exactly as
EPro-PnP-6DoF/lib/test.py:179-194 runs them.  Needs cv2 (only this script imports it).

    python oracle/make_golden_epnp.py          # writes tests/golden/epnp/<case>.npz

Each case stores the fp32 inputs (x3d, x2d, w2d, cam_mats), q, numpy's mask and count, cv2's pose (B, 7), the float64
oracle's pose (oracle/epnp_oracle.py) and a per-object `floor`: the largest change of cv2's pose (max over the seven
components) when the fp32 inputs move by about one ulp, over a few perturbations -- how well the problem itself pins
the answer down.

The dense case (32 objects of 64 x 64 maps, the test.py setting) is too large to keep its inputs in the repository: its
file stores `inputs_sha1` instead, and the inputs are regenerated from the seed by dense_problem() (make_problem draws
everything on the CPU with an explicit torch.Generator); the tests check the hash before they use them.
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "epro-pnp_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from epropnp_b200.synth import make_problem          # noqa: E402
from oracle import epnp_oracle                         # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "epnp")


def cv2_poses(x3d, x2d, w2d, cam_mats, q):
    """test.py:179-194: quantile mask, cv2.solvePnP(EPNP) per object, rotvec -> quaternion (w, i, j, k)."""
    import cv2
    from scipy.spatial.transform import Rotation
    B = x3d.shape[0]
    conf = w2d.mean(-1)
    mask = conf >= np.quantile(conf.reshape(B, -1), q, axis=1, keepdims=True)
    out = np.zeros((B, 7))
    for b in range(B):
        _, rv, tv = cv2.solvePnP(x3d[b][mask[b]], x2d[b][mask[b]], cam_mats[b], np.zeros((4, 1), np.float32),
                                 flags=cv2.SOLVEPNP_EPNP)
        out[b, :3] = tv.reshape(-1)
        out[b, 3:] = Rotation.from_rotvec(rv.reshape(-1)).as_quat()[[3, 0, 1, 2]]
    return out, mask


def floor_of(x3d, x2d, w2d, cam_mats, q, base, trials=16, seed=0):
    rng = np.random.default_rng(seed)
    eps = np.finfo(np.float32).eps
    fl = np.zeros(x3d.shape[0])
    for _ in range(trials):
        p3 = (x3d * (1 + eps * rng.choice([-1.0, 1.0], x3d.shape))).astype(np.float32)
        p2 = (x2d * (1 + eps * rng.choice([-1.0, 1.0], x2d.shape))).astype(np.float32)
        pose, _ = cv2_poses(p3, p2, w2d, cam_mats, q)
        pose[:, 3:] *= np.sign((pose[:, 3:] * base[:, 3:]).sum(1, keepdims=True))
        fl = np.maximum(fl, np.abs(pose - base).max(1))
    return fl


INPUT_KEYS = ("x3d", "x2d", "w2d", "cam_mats")
def dense_problem():
    return make_problem(32, 4096, seed=11, grid2d=True)


REGENERATED = {"dense": dense_problem}          # cases whose inputs are rebuilt from their seed, not stored


def inputs_sha1(arrays):
    h = hashlib.sha1()
    for a in arrays:
        h.update(np.ascontiguousarray(a, np.float32).tobytes())
    return h.hexdigest()


def cases():
    out = {}
    out["dense"] = (dense_problem(), 0.8)
    out["all_points"] = (make_problem(16, 512, seed=12), 0.0)
    pc = make_problem(16, 1024, seed=13)
    g = torch.Generator().manual_seed(13)
    K = pc["cam_mats"].clone()
    K[:, 0, 0] = 500 + 700 * torch.rand(16, generator=g)
    K[:, 1, 1] = K[:, 0, 0] * (0.9 + 0.2 * torch.rand(16, generator=g))
    K[:, 0, 2] = 250 + 150 * torch.rand(16, generator=g)
    K[:, 1, 2] = 180 + 120 * torch.rand(16, generator=g)
    # re-project the points with each object's own camera (same 3D points and pose, same relative pixel noise)
    pc2 = make_problem(16, 1024, seed=13)
    x2d = pc2["x2d"]
    x2d_n = (x2d - pc2["cam_mats"][:, None, :2, 2]) / pc2["cam_mats"][:, None, [0, 1], [0, 1]]
    pc["x2d"] = (x2d_n * K[:, None, [0, 1], [0, 1]] + K[:, None, :2, 2]).float()
    pc["cam_mats"] = K
    out["per_object_K"] = (pc, 0.7)
    pc = make_problem(16, 1024, seed=14)
    pc["w2d"] = (torch.round(pc["w2d"] / pc["w2d"].amax(dim=(1, 2), keepdim=True) * 4) / 4).float()
    out["ties"] = (pc, 0.5)
    pc = make_problem(16, 1024, seed=15)
    # flatten the object: shrink the z extent about the object's own centre and re-project
    x3d = pc["x3d"].clone()
    x3d[..., 2] = x3d[..., 2].mean(1, keepdim=True) + 0.03 * (x3d[..., 2] - x3d[..., 2].mean(1, keepdim=True))
    from epropnp_b200.synth import quat_to_mat_ref
    R = quat_to_mat_ref(pc["pose_gt"][:, 3:])
    cam = x3d @ R.transpose(-1, -2) + pc["pose_gt"][:, None, :3]
    proj = cam @ pc["cam_mats"].transpose(-1, -2)
    x2d_clean = proj[..., :2] / proj[..., 2:]
    g = torch.Generator().manual_seed(15)
    pc["x2d"] = (x2d_clean + 0.5 * torch.randn(x2d_clean.shape, generator=g)).float()
    pc["x3d"] = x3d.float()
    out["thin"] = (pc, 0.8)
    out["minimal"] = (make_problem(8, 26, seed=16), 0.8)     # 26 - ceil(0.8 * 25) = 6 points
    return out


def main():
    os.makedirs(OUT, exist_ok=True)
    for name, (pc, q) in cases().items():
        x3d, x2d, w2d, K = (pc[k].numpy().astype(np.float32) for k in ("x3d", "x2d", "w2d", "cam_mats"))
        pose, mask = cv2_poses(x3d, x2d, w2d, K, q)
        omask, count = epnp_oracle.select(w2d, q)
        assert (omask == mask).all(), name
        orc, _, _ = epnp_oracle.epnp_pose_init(x3d, x2d, w2d, K, q)
        fl = floor_of(x3d, x2d, w2d, K, q, pose)
        inputs = dict(x3d=x3d, x2d=x2d, w2d=w2d, cam_mats=K)
        if name in REGENERATED:
            inputs = dict(inputs_sha1=np.array(inputs_sha1([x3d, x2d, w2d, K])))
        np.savez_compressed(os.path.join(OUT, name + ".npz"), q=np.float32(q), mask=mask, count=count, pose_cv2=pose,
                            pose_oracle=orc, floor=fl, **inputs)
        d = np.abs(orc - pose).max(1)
        print(f"{name:13s} B={x3d.shape[0]:3d} N={x3d.shape[1]:5d} q={q}  n_used {count.min()}..{count.max()}  "
              f"floor median {np.median(fl):.1e} max {fl.max():.1e}  |oracle - cv2| / floor max {np.max(d / fl):.2f}")


if __name__ == "__main__":
    main()
