"""EPnP initialiser of the 6DoF evaluation flow (epnp_epnp_init_f32, epropnp.epnp_init) without a GPU.

The goldens under tests/golden/epnp/ hold what the reference flow computes (EPro-PnP-6DoF/lib/test.py:179-194: numpy
quantile mask, cv2.solvePnP(SOLVEPNP_EPNP), scipy quaternion) and, per object, `floor`: how far cv2's own pose moves
when the fp32 inputs move by one ulp.  Checked here: the float64 oracle against cv2, and the real kernel source under the
SIMT emulator against cv2 with exact point counts."""
import ctypes

import numpy as np
import pytest
import torch

import simt_native
from conftest import GOLDEN_DIR
from epropnp_b200 import capi, native
from oracle import epnp_oracle

CASES = ["dense", "all_points", "per_object_K", "ties", "thin", "minimal"]


def load(name):
    g = np.load(f"{GOLDEN_DIR}/epnp/{name}.npz")
    g = {k: g[k] for k in g.files}
    if "inputs_sha1" in g:          # large case: inputs regenerated from their seed, checked against the stored hash
        from oracle import make_golden_epnp
        pc = make_golden_epnp.REGENERATED[name]()
        g.update({k: pc[k].numpy().astype(np.float32) for k in make_golden_epnp.INPUT_KEYS})
        have = make_golden_epnp.inputs_sha1([g[k] for k in make_golden_epnp.INPUT_KEYS])
        assert have == str(g["inputs_sha1"]), f"{name}: regenerated inputs differ from the ones the golden was made from"
    return g


def pose_errors(pose, ref):
    """Per-object max |pose - ref| over the seven components (both quaternions have w >= 0)."""
    return np.abs(np.asarray(pose, np.float64) - ref).max(1)


def bound(g, rel, k):
    return np.maximum(rel * np.abs(g["pose_cv2"]).max(), k * g["floor"])


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_cv2(name):
    g = load(name)
    mask, count = epnp_oracle.select(g["w2d"], float(g["q"]))
    assert (mask == g["mask"]).all() and (count == g["count"]).all()
    pose, _, _ = epnp_oracle.epnp_pose_init(g["x3d"], g["x2d"], g["w2d"], g["cam_mats"], float(g["q"]))
    err = pose_errors(pose, g["pose_cv2"])
    assert (err <= bound(g, 1e-9, 3)).all(), (err, g["floor"])
    assert (pose[:, 3] >= 0).all()


def test_ties_case_has_ties_at_the_threshold():
    g = load("ties")
    conf = g["w2d"].astype(np.float32).mean(-1)
    thr = np.array([epnp_oracle.quantile_threshold(c, float(g["q"])) for c in conf])
    assert ((conf == thr[:, None]).sum(1) > 1).all()


@pytest.fixture
def emul(monkeypatch):
    return simt_native.install(monkeypatch)


@pytest.mark.parametrize("name", CASES)
def test_kernel_matches_cv2_under_emulation(emul, name):
    g = load(name)
    B = 8 if name == "dense" else g["x3d"].shape[0]          # the emulator runs a CTA at a time: a slice of the big case
    t = lambda k: torch.from_numpy(g[k][:B])
    pose, n_used = native.epnp_init(t("x3d"), t("x2d"), t("w2d"), t("cam_mats"), float(g["q"]), want_count=True)
    assert (n_used.numpy() == g["count"][:B]).all()
    err = pose_errors(pose.numpy(), g["pose_cv2"][:B])
    b = bound({k: g[k][:B] for k in ("pose_cv2", "floor")}, 1e-6, 5)
    assert (err <= b).all(), (err, b)
    assert (pose[:, 3] >= 0).all()
    assert torch.allclose(pose[:, 3:].norm(dim=-1), torch.ones(B), atol=1e-6)


def test_single_camera_matrix_is_broadcast(emul):
    g = load("all_points")
    t = lambda k: torch.from_numpy(g[k][:3])
    a = native.epnp_init(t("x3d"), t("x2d"), t("w2d"), t("cam_mats"), 0.0)
    b = native.epnp_init(t("x3d"), t("x2d"), t("w2d"), torch.from_numpy(g["cam_mats"][0]), 0.0)
    assert torch.equal(a, b)


def test_arguments_are_rejected(emul):
    g = load("all_points")
    x3d, x2d, w2d, K = (torch.from_numpy(g[k][:2]) for k in ("x3d", "x2d", "w2d", "cam_mats"))
    with pytest.raises(native.NativeError, match="bad argument"):         # 8 - ceil(0.8 * 7) = 2 points left
        native.epnp_init(x3d[:, :8], x2d[:, :8], w2d[:, :8], K, 0.8)
    native.epnp_init(x3d[:, :20], x2d[:, :20], w2d[:, :20], K, 0.8)       # 20 - ceil(15.2) = 4: accepted
    for q in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            native.epnp_init(x3d, x2d, w2d, K, q)
    with pytest.raises(ValueError):
        native.epnp_init(x3d, x2d[:, :-1], w2d, K)
    with pytest.raises(ValueError):
        native.epnp_init(x3d, x2d, w2d[..., :1], K)
    with pytest.raises(ValueError):
        native.epnp_init(x3d[..., :2], x2d, w2d, K)
    with pytest.raises(ValueError):
        native.epnp_init(x3d, x2d, w2d, K[:, :2])


def test_c_entry_point_checks_its_arguments(emul):
    lib = capi.lib()
    buf = torch.zeros(16)
    p = ctypes.c_void_p(buf.data_ptr())
    f = lambda q, B, N, pose=p: lib.epnp_epnp_init_f32(p, p, p, p, ctypes.c_float(q), pose, None, B, N, None)
    assert f(0.5, 1, 16384 + 1) == -2                     # EPNP_ERR_TOO_MANY_POINTS
    assert f(1.5, 1, 64) == -1 and f(-0.5, 1, 64) == -1 and f(float("nan"), 1, 64) == -1
    assert f(0.5, 1, 0) == -1 and f(0.5, -1, 64) == -1 and f(0.5, 1, 64, None) == -1
    assert f(1.0, 1, 64) == -1                            # only the maximum is >= the 1.0 quantile
    assert f(0.5, 0, 64) == 0                             # empty batch: nothing to do


def test_product_path_refuses_cpu_tensors():
    g = load("minimal")
    x3d, x2d, w2d, K = (torch.from_numpy(g[k]) for k in ("x3d", "x2d", "w2d", "cam_mats"))
    with pytest.raises(native.NativeError, match="CUDA only"):
        native.epnp_init(x3d, x2d, w2d, K)
    from epropnp.epnp_init import epnp_pose_init
    with pytest.raises(native.NativeError):
        epnp_pose_init(x3d, x2d, w2d, K)


def test_solver_refuses_4dof_and_bad_quantiles():
    from epropnp.epnp_init import EPnPSolver
    with pytest.raises(ValueError):
        EPnPSolver(dof=4)
    with pytest.raises(ValueError):
        EPnPSolver(conf_quantile=1.2)
    assert EPnPSolver().conf_quantile == 0.8


def test_solver_contract_under_emulation(emul):
    """EPnPSolver.solve as LMSolver calls it: (pose, None, cost) with the cost of evaluate_pnp at that pose."""
    from epropnp.camera import PerspectiveCamera
    from epropnp.cost_fun import AdaptiveHuberPnPCost
    from epropnp.epnp_init import EPnPSolver
    g = load("minimal")
    x3d, x2d, w2d, K = (torch.from_numpy(g[k]) for k in ("x3d", "x2d", "w2d", "cam_mats"))
    camera = PerspectiveCamera(cam_mats=K)
    cost_fun = AdaptiveHuberPnPCost(relative_delta=0.1)
    cost_fun.set_param(x2d, w2d)
    pose, cov, cost = EPnPSolver().solve(x3d, x2d, w2d, camera, cost_fun, with_cost=True)
    assert cov is None and pose.shape == (8, 7) and cost.shape == (8,)
    prob = native.Problem(x3d, x2d, w2d, K, None, None, cost_fun.delta)
    assert torch.equal(cost, native.evaluate_cost(prob, pose[None], 6, camera.z_min)[0])
    assert EPnPSolver().solve(x3d, x2d, w2d, camera, cost_fun)[2] is None
