"""EPnP initialiser of the 6DoF evaluation flow on a real GPU (epnp_epnp_init_f32, epropnp.epnp_init): the goldens of
tests/test_epnp_cpu.py on the device, a full-size batch against the float64 oracle, determinism, CUDA-graph capture and
the evaluation flow EPnP -> Gauss-Newton (EPro-PnP-6DoF/lib/test.py:176-211)."""
import numpy as np
import pytest
import torch

from conftest import assert_lm_parity, err_stats, record_parity
from epropnp_b200 import native
from epropnp_b200.synth import make_problem
from oracle import epnp_oracle
from test_epnp_cpu import CASES, bound, load, pose_errors

pytestmark = pytest.mark.gpu


@pytest.fixture
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")


def on(dev, g, *keys):
    return [torch.from_numpy(g[k]).to(dev) for k in keys]


@pytest.mark.parametrize("name", CASES)
def test_device_matches_cv2(dev, name):
    g = load(name)
    x3d, x2d, w2d, K = on(dev, g, "x3d", "x2d", "w2d", "cam_mats")
    pose, n_used = native.epnp_init(x3d, x2d, w2d, K, float(g["q"]), want_count=True)
    pose, n_used = pose.cpu().numpy(), n_used.cpu().numpy()
    assert (n_used == g["count"]).all()
    err = pose_errors(pose, g["pose_cv2"])
    b = bound(g, 1e-6, 5)
    record_parity(f"epnp_init_{name}", vs="cv2.solvePnP(SOLVEPNP_EPNP)", **err_stats(pose, g["pose_cv2"]),
                  max_err_over_floor=float((err / g["floor"]).max()), floor_median=float(np.median(g["floor"])))
    assert (err <= b).all(), (err, b)
    assert (pose[:, 3] >= 0).all()


def test_large_batch_against_oracle(dev):
    """B = 4096 objects of 64 x 64 maps at q = 0.8 (the test.py setting); every 64th object against the float64 oracle."""
    B, N = 4096, 4096
    pc = make_problem(B, N, seed=21, grid2d=True)
    x3d, x2d, w2d, K = (pc[k].to(dev) for k in ("x3d", "x2d", "w2d", "cam_mats"))
    pose, n_used = native.epnp_init(x3d, x2d, w2d, K, 0.8, want_count=True)
    pose, n_used = pose.cpu().numpy(), n_used.cpu().numpy()
    idx = np.arange(0, B, 64)
    ref, _, count = epnp_oracle.epnp_pose_init(pc["x3d"].numpy()[idx], pc["x2d"].numpy()[idx], pc["w2d"].numpy()[idx],
                                               pc["cam_mats"].numpy()[idx], 0.8)
    assert (n_used[idx] == count).all()
    err = pose_errors(pose[idx], ref)
    record_parity("epnp_init_B4096_N4096", vs="float64 oracle, every 64th object", **err_stats(pose[idx], ref))
    assert err.max() <= 1e-6 * np.abs(ref).max() + 1e-6, err.max()


def test_deterministic_and_batch_independent(dev):
    g = load("dense")
    x3d, x2d, w2d, K = on(dev, g, "x3d", "x2d", "w2d", "cam_mats")
    a = native.epnp_init(x3d, x2d, w2d, K, 0.8)
    b = native.epnp_init(x3d, x2d, w2d, K, 0.8)
    assert torch.equal(a, b)
    s = native.epnp_init(x3d[5:17], x2d[5:17], w2d[5:17], K[5:17], 0.8)
    assert torch.equal(s, a[5:17])


def test_cuda_graph_replay(dev):
    """The call enqueues work only (no host synchronisation, no allocation inside the library): it can be captured."""
    g = load("ties")
    x3d, x2d, w2d, K = on(dev, g, "x3d", "x2d", "w2d", "cam_mats")
    eager = native.epnp_init(x3d, x2d, w2d, K, float(g["q"]))
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        native.epnp_init(x3d, x2d, w2d, K, float(g["q"]))         # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = native.epnp_init(x3d, x2d, w2d, K, float(g["q"]))
    out.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager)


def _flow(dev, g):
    from epropnp.camera import PerspectiveCamera
    from epropnp.cost_fun import AdaptiveHuberPnPCost
    x3d, x2d, w2d, K = on(dev, g, "x3d", "x2d", "w2d", "cam_mats")
    camera = PerspectiveCamera(cam_mats=K, z_min=0.01)
    cost_fun = AdaptiveHuberPnPCost(relative_delta=0.1)
    cost_fun.set_param(x2d, w2d)
    return x3d, x2d, w2d, camera, cost_fun


@pytest.mark.parametrize("name", ["dense", "per_object_K"])
def test_evaluation_flow_reaches_the_same_solution(dev, name):
    """test.py:176-211: EPnP initial pose, then the Gauss-Newton solve (fast_mode).  Started from this EPnP or from the
    goldens' cv2 poses, the solve ends at the same poses."""
    from epropnp.epnp_init import EPnPSolver
    from epropnp.levenberg_marquardt import LMSolver
    g = load(name)
    x3d, x2d, w2d, camera, cost_fun = _flow(dev, g)
    solver = LMSolver(dof=6, num_iter=10, init_solver=EPnPSolver(float(g["q"])))
    pose, _, cost = solver.solve(x3d, x2d, w2d, camera, cost_fun, with_cost=True, fast_mode=True)
    cv2_init = torch.from_numpy(g["pose_cv2"]).float().to(dev)
    ref_pose, _, ref_cost = solver.solve(x3d, x2d, w2d, camera, cost_fun, pose_init=cv2_init, with_cost=True,
                                         fast_mode=True)
    flips = assert_lm_parity(pose.cpu(), cost.cpu(), ref_pose.cpu(), ref_cost.cpu(), 1e-4, what=f"epnp flow {name}")
    record_parity(f"epnp_flow_{name}", vs="GN fast mode from the cv2 initial poses", flip_frac=flips,
                  **err_stats(pose.cpu().numpy(), ref_pose.cpu().numpy()))


def test_lm_solver_uses_the_init_solver(dev):
    from epropnp.epnp_init import EPnPSolver, epnp_pose_init
    from epropnp.levenberg_marquardt import LMSolver
    g = load("all_points")
    x3d, x2d, w2d, camera, cost_fun = _flow(dev, g)
    solver = LMSolver(dof=6, num_iter=5, init_solver=EPnPSolver(0.0))
    start = epnp_pose_init(x3d, x2d, w2d, camera.cam_mats, 0.0)
    a = solver.solve(x3d, x2d, w2d, camera, cost_fun, fast_mode=True)[0]
    b = solver.solve(x3d, x2d, w2d, camera, cost_fun, pose_init=start, fast_mode=True)[0]
    assert torch.equal(a, b)
    # force_init_solve: per object, the cheaper of pose_init and the EPnP pose is where the iterations start
    bad = start.clone()
    bad[:, 2] += 3.0
    c = solver.solve(x3d, x2d, w2d, camera, cost_fun, pose_init=bad, force_init_solve=True, fast_mode=True)[0]
    assert torch.equal(c, a)
