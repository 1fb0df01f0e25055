"""Tensor-level entry points of the native library (one function per C-ABI call).

Inputs are torch CUDA tensors; every function validates / normalises them (float32, contiguous,
broadcast scalars), allocates the outputs with torch (the library never allocates) and enqueues
the kernel on the current CUDA stream.  CPU tensors are rejected: there is no fallback path.
"""
import ctypes

import torch

from . import capi
from .capi import NativeError, check, default_params, lib, ptr, stream_ptr


def _need_cuda(t, what):
    if not t.is_cuda:
        raise NativeError(f"{what}: tensor is on {t.device}; the EPro-PnP hot path runs on CUDA only "
                          "(no CPU / PyTorch fallback). Move the inputs to a B200 device.")


def _f32c(t):
    return t.detach().to(torch.float32).contiguous()


def _bounds(lb, ub, B, device):
    """None | float | (B,2)/(2,) tensor -> (B,2) float32 contiguous (or None, None)."""
    if lb is None or ub is None:
        return None, None

    def one(b):
        if torch.is_tensor(b):
            return b.detach().to(device=device, dtype=torch.float32).expand(B, 2).contiguous()
        return torch.full((B, 2), float(b), dtype=torch.float32, device=device)
    return one(lb), one(ub)


def _delta(delta, B, device):
    if torch.is_tensor(delta):
        return delta.detach().to(device=device, dtype=torch.float32).expand(B).contiguous()
    return torch.full((B,), float(delta), dtype=torch.float32, device=device)


def _cam(cam_mats, B, device):
    return cam_mats.detach().to(device=device, dtype=torch.float32).expand(B, 3, 3).contiguous()


class Problem:
    """Validated, contiguous fp32 view of one batch of correspondence sets + camera + Huber delta."""

    def __init__(self, x3d, x2d, w2d, cam_mats, lb, ub, delta):
        _need_cuda(x3d, "x3d")
        if x3d.dim() != 3 or x2d.dim() != 3 or w2d.dim() != 3:
            raise ValueError("x3d/x2d/w2d must be (num_obj, num_pts, 3|2|2)")
        self.B, self.N = x3d.shape[0], x3d.shape[1]
        self.device = x3d.device
        # the kernels read B*N*{3,2,2} floats through raw pointers: anything else must be caught here
        if x3d.shape[2] != 3 or tuple(x2d.shape) != (self.B, self.N, 2):
            raise ValueError(f"x3d must be (B, N, 3) and x2d (B, N, 2); got {tuple(x3d.shape)}, {tuple(x2d.shape)}")
        if w2d.shape[:2] != x2d.shape[:2] or w2d.shape[2] not in (1, 2):
            raise ValueError(f"w2d must be (B, N, 2) (or (B, N, 1), broadcast); got {tuple(w2d.shape)}")
        if x2d.device != self.device or w2d.device != self.device:
            raise ValueError("x3d, x2d and w2d must live on one device")
        if w2d.shape[2] == 1:
            w2d = w2d.expand(self.B, self.N, 2)          # the reference's arithmetic accepts a broadcast weight
        self.x3d, self.x2d, self.w2d = _f32c(x3d), _f32c(x2d), _f32c(w2d)
        self.cam = _cam(cam_mats, self.B, self.device)
        self.lb, self.ub = _bounds(lb, ub, self.B, self.device)
        self.delta = _delta(delta, self.B, self.device)

    def common_ptrs(self):
        return (ptr(self.x3d), ptr(self.x2d), ptr(self.w2d), ptr(self.cam), ptr(self.lb), ptr(self.ub),
                ptr(self.delta))

    def empty(self, *shape):
        return torch.empty(shape, dtype=torch.float32, device=self.device)


def adaptive_delta(x2d, w2d, relative_delta):
    _need_cuda(x2d, "x2d")
    B, N = x2d.shape[0], x2d.shape[1]
    x2d, w2d = _f32c(x2d), _f32c(w2d)
    out = torch.empty(B, dtype=torch.float32, device=x2d.device)
    with torch.cuda.device(x2d.device):
        check(lib().epnp_adaptive_delta_f32(ptr(x2d), ptr(w2d), ctypes.c_float(relative_delta), ptr(out), B, N,
                                            stream_ptr(x2d.device)), "epnp_adaptive_delta_f32")
    return out


def evaluate_cost(prob: Problem, poses, dof, z_min):
    """poses (S, B, D) -> cost (S, B)."""
    S = poses.shape[0]
    _check_pose(poses, (S, prob.B), 7 if dof == 6 else 4, "poses")
    poses = _f32c(poses)
    out = prob.empty(S, prob.B)
    with torch.cuda.device(prob.device):
        check(lib().epnp_evaluate_cost_f32(*prob.common_ptrs(), ptr(poses), ptr(out), S, prob.B, prob.N, dof,
                                           ctypes.c_float(z_min), stream_ptr(prob.device)), "epnp_evaluate_cost_f32")
    return out


def evaluate_full(prob: Problem, pose, dof, z_min, huber_eps, clip_jac, want_residual, want_jac, want_cost):
    pose = _f32c(pose)
    B, N = prob.B, prob.N
    res = prob.empty(B, 2 * N) if want_residual else None
    jac = prob.empty(B, 2 * N, dof) if want_jac else None
    cost = prob.empty(B) if want_cost else None
    with torch.cuda.device(prob.device):
        check(lib().epnp_evaluate_f32(*prob.common_ptrs(), ptr(pose), ptr(res), ptr(jac), ptr(cost), int(clip_jac),
                                      B, N, dof, ctypes.c_float(z_min), ctypes.c_float(huber_eps),
                                      stream_ptr(prob.device)), "epnp_evaluate_f32")
    return res, cost, jac


def _check_pose(pose, lead, D, what):
    if tuple(pose.shape) != tuple(lead) + (D,):
        raise ValueError(f"{what} must be {tuple(lead) + (D,)}; got {tuple(pose.shape)}")


def lm_solve(prob: Problem, pose_init, params, want_cov=False, want_cost=False, want_plus=False,
             want_cost_init=False):
    D = 7 if params.dof == 6 else 4
    B = prob.B
    _check_pose(pose_init, (B,), D, "pose_init")
    pose_init = _f32c(pose_init)
    out = dict(pose_opt=prob.empty(B, D),
               pose_cov=prob.empty(B, params.dof, params.dof) if want_cov else None,
               cost=prob.empty(B) if want_cost else None,
               pose_opt_plus=prob.empty(B, D) if want_plus else None,
               cost_init=prob.empty(B) if want_cost_init else None)
    with torch.cuda.device(prob.device):
        check(lib().epnp_lm_solve_f32(*prob.common_ptrs(), ptr(pose_init), ptr(out["pose_opt"]), ptr(out["pose_cov"]),
                                      ptr(out["cost"]), ptr(out["pose_opt_plus"]), ptr(out["cost_init"]), B, prob.N,
                                      ctypes.byref(params), stream_ptr(prob.device)), "epnp_lm_solve_f32")
    return out


def rslm_draw(x3d, x2d, w2d, cam_mats, P, n, dof, eps=1e-5, seed=0, obj_offset=0, t_init=None, want_t=False):
    """Everything before the solves of the random-sample initialiser in one launch (epnp_rslm_draw_f32): the
    centre-based translation guess (unless t_init (B, 3) is given -- then x3d / x2d / cam_mats may be None), inds
    (P, B, n) int32 (weighted subsets without replacement, per proposal and object) and start (P, B, D) (that translation
    + a uniformly random orientation).  -> inds, start [, t (B, 3) with want_t]."""
    _need_cuda(w2d, "w2d")
    if w2d.dim() != 3 or w2d.shape[-1] != 2:
        raise ValueError(f"w2d must be (B, N, 2), got {tuple(w2d.shape)}")
    B, N = w2d.shape[0], w2d.shape[1]
    dev = w2d.device
    if t_init is not None:
        if tuple(t_init.shape) != (B, 3):
            raise ValueError(f"t_init must be ({B}, 3), got {tuple(t_init.shape)}")
        t_init = _f32c(t_init.to(dev))
        x3d = x2d = cam_mats = None
    else:
        for t, shape, what in ((x3d, (B, N, 3), "x3d"), (x2d, (B, N, 2), "x2d"), (cam_mats, (B, 3, 3), "cam_mats")):
            if t is None or tuple(t.shape) != shape or t.device != dev:
                raise ValueError(f"{what} must be {shape} on {dev}")
        x3d, x2d, cam_mats = _f32c(x3d), _f32c(x2d), _f32c(cam_mats)
    D = 7 if dof == 6 else 4
    w2d = _f32c(w2d)
    inds = torch.empty(P, B, n, dtype=torch.int32, device=dev)
    start = torch.empty(P, B, D, dtype=torch.float32, device=dev)
    t_out = torch.empty(B, 3, dtype=torch.float32, device=dev) if want_t else None
    with torch.cuda.device(dev):
        check(lib().epnp_rslm_draw_f32(ptr(x3d), ptr(x2d), ptr(w2d), ptr(cam_mats), ptr(t_init), ctypes.c_uint64(seed),
                                       ctypes.c_uint32(obj_offset), capi.iptr(inds), ptr(start), ptr(t_out), P, n, B, N, dof,
                                       ctypes.c_float(eps), stream_ptr(dev)), "epnp_rslm_draw_f32")
    return (inds, start, t_out) if want_t else (inds, start)


def epnp_init(x3d, x2d, w2d, cam_mats, conf_quantile=0.8, want_count=False):
    """EPnP initial pose per object (epnp_epnp_init_f32): the points whose confidence mean(w2d, -1) is at or above the
    object's conf_quantile quantile (numpy 'linear'), EPnP on them in fp64.  cam_mats (3, 3) or (B, 3, 3).
    -> pose (B, 7) = x y z w i j k with w >= 0 [, n_used (B) int32 with want_count]."""
    _need_cuda(w2d, "w2d")
    if x3d.dim() != 3 or x3d.shape[-1] != 3:
        raise ValueError(f"x3d must be (B, N, 3), got {tuple(x3d.shape)}")
    B, N = x3d.shape[0], x3d.shape[1]
    dev = x3d.device
    for t, shape, what in ((x2d, (B, N, 2), "x2d"), (w2d, (B, N, 2), "w2d")):
        if tuple(t.shape) != shape or t.device != dev:
            raise ValueError(f"{what} must be {shape} on {dev}, got {tuple(t.shape)} on {t.device}")
    if tuple(cam_mats.shape) not in ((3, 3), (B, 3, 3)) or cam_mats.device != dev:
        raise ValueError(f"cam_mats must be (3, 3) or ({B}, 3, 3) on {dev}, got {tuple(cam_mats.shape)}")
    q = float(conf_quantile)
    if not 0.0 <= q <= 1.0:
        raise ValueError(f"conf_quantile must be in [0, 1], got {q}")
    x3d, x2d, w2d, cam = _f32c(x3d), _f32c(x2d), _f32c(w2d), _cam(cam_mats, B, dev)
    pose = torch.empty(B, 7, dtype=torch.float32, device=dev)
    n_used = torch.empty(B, dtype=torch.int32, device=dev) if want_count else None
    with torch.cuda.device(dev):
        check(lib().epnp_epnp_init_f32(ptr(x3d), ptr(x2d), ptr(w2d), ptr(cam), ctypes.c_float(q), ptr(pose),
                                       None if n_used is None else capi.iptr(n_used), B, N, stream_ptr(dev)),
              "epnp_epnp_init_f32")
    return (pose, n_used) if want_count else pose


def rslm(prob: Problem, inds, start, params, want_all=False):
    """Fused random-sample LM initialiser (epnp_rslm_f32): inds (P, B, n) integer indices within each object, start
    (P, B, D) -> dict(pose (B, D), cost (B), pose_all (P, B, D) | None, cost_all (P, B) | None)."""
    D = 7 if params.dof == 6 else 4
    P, B, n = inds.shape
    assert B == prob.B and start.shape == (P, B, D)
    inds32 = inds.detach().to(device=prob.device, dtype=torch.int32).contiguous()
    start = _f32c(start)
    out = dict(pose=prob.empty(B, D), cost=prob.empty(B),
               pose_all=prob.empty(P, B, D) if want_all else None, cost_all=prob.empty(P, B) if want_all else None)
    with torch.cuda.device(prob.device):
        check(lib().epnp_rslm_f32(*prob.common_ptrs(), capi.iptr(inds32), ptr(start), ptr(out["pose"]), ptr(out["cost"]),
                                  ptr(out["pose_all"]), ptr(out["cost_all"]), P, n, B, prob.N, ctypes.byref(params),
                                  stream_ptr(prob.device)), "epnp_rslm_f32")
    return out


def gn_plus_backward(prob: Problem, pose, grad_pose_plus, dof, z_min, eps, huber_eps, want=(True, True, True, True)):
    """dL/d(x3d, x2d, w2d, delta) of pose_opt_plus = pose (+) gn_step(pose) (epnp_gn_plus_backward_f32)."""
    B, N = prob.B, prob.N
    pose, gp = _f32c(pose), _f32c(grad_pose_plus)
    g3 = prob.empty(B, N, 3) if want[0] else None
    g2 = prob.empty(B, N, 2) if want[1] else None
    gw = prob.empty(B, N, 2) if want[2] else None
    gd = prob.empty(B) if want[3] else None
    with torch.cuda.device(prob.device):
        check(lib().epnp_gn_plus_backward_f32(*prob.common_ptrs(), ptr(pose), ptr(gp), ptr(g3), ptr(g2), ptr(gw), ptr(gd),
                                              B, N, dof, ctypes.c_float(z_min), ctypes.c_float(eps),
                                              ctypes.c_float(huber_eps), stream_ptr(prob.device)),
              "epnp_gn_plus_backward_f32")
    return g3, g2, gw, gd


def _noise_ptrs(noise):
    if noise is None:
        return None, None, None, ()
    n3, c2, n4 = (_f32c(t) for t in noise)
    return ptr(n3), ptr(c2), ptr(n4), (n3, c2, n4)


def amis(prob: Problem, pose_opt, pose_cov, params, noise=None, seed=0, obj_offset=0, want_proposals=False):
    """-> pose_samples (B, M, D), logw (B, M) [object-major], proposals (B, I, 19) | None."""
    D = 7 if params.dof == 6 else 4
    B, M, I = prob.B, params.mc_samples, params.mc_iter
    pose_opt, pose_cov = _f32c(pose_opt), _f32c(pose_cov)
    samples, logw = prob.empty(B, M, D), prob.empty(B, M)
    props = prob.empty(B, I, 19) if want_proposals else None
    p3, p2, p4, keep = _noise_ptrs(noise)
    with torch.cuda.device(prob.device):
        check(lib().epnp_amis_f32(*prob.common_ptrs(), ptr(pose_opt), ptr(pose_cov), p3, p2, p4,
                                  ctypes.c_uint64(seed), ctypes.c_uint32(obj_offset), ptr(samples), ptr(logw),
                                  ptr(props), B, prob.N, ctypes.byref(params), stream_ptr(prob.device)),
              "epnp_amis_f32")
    del keep
    return samples, logw, props


def lm_amis_fused(prob: Problem, pose_init, params, noise=None, seed=0, obj_offset=0, want_cost=False,
                  want_plus=False, want_cost_init=True, want_proposals=False, want_cov=True):
    D = 7 if params.dof == 6 else 4
    B, M, I = prob.B, params.mc_samples, params.mc_iter
    _check_pose(pose_init, (B,), D, "pose_init")
    pose_init = _f32c(pose_init)
    out = dict(pose_opt=prob.empty(B, D), pose_cov=prob.empty(B, params.dof, params.dof) if want_cov else None,
               cost=prob.empty(B) if want_cost else None,
               pose_opt_plus=prob.empty(B, D) if want_plus else None,
               cost_init=prob.empty(B) if want_cost_init else None,
               pose_samples=prob.empty(B, M, D), logw=prob.empty(B, M),
               proposals=prob.empty(B, I, 19) if want_proposals else None)
    p3, p2, p4, keep = _noise_ptrs(noise)
    with torch.cuda.device(prob.device):
        check(lib().epnp_lm_amis_fused_f32(*prob.common_ptrs(), ptr(pose_init), p3, p2, p4,
                                           ctypes.c_uint64(seed), ctypes.c_uint32(obj_offset),
                                           ptr(out["pose_opt"]), ptr(out["pose_cov"]), ptr(out["cost"]),
                                           ptr(out["pose_opt_plus"]), ptr(out["cost_init"]),
                                           ptr(out["pose_samples"]), ptr(out["logw"]), ptr(out["proposals"]),
                                           B, prob.N, ctypes.byref(params), stream_ptr(prob.device)),
              "epnp_lm_amis_fused_f32")
    del keep
    return out


def peer_table(buffers, device):
    """Device array of pointers (int64 tensor) to the peers' buffers: tensors in other GPUs' memory or raw device
    pointers (ints) of IPC-mapped buffers (sharded.raw_ipc_open).  Build it ONCE per set of buffers: creating a device
    tensor from host data is a synchronous copy on the current stream."""
    return torch.tensor([t if isinstance(t, int) else t.data_ptr() for t in buffers] or [0], dtype=torch.int64, device=device)


def lm_amis_fused_push(prob: Problem, pose_init, params, pose_opt_out, logw_out, peer_logw, peer_pose, seed=0,
                       obj_offset=0, want_cost=False, want_cov=False, n_peers=None):
    """Fused solve + in-kernel gather (epnp_lm_amis_fused_push_f32).  pose_opt_out (B, D) / logw_out (B, M): where the
    LOCAL results go (contiguous; normally rows [obj_offset, obj_offset + B) of this rank's own full-batch buffers);
    peer_logw / peer_pose: the full-batch (B_total, M) / (B_total, D) float32 buffers in OTHER GPUs' memory the kernel
    also writes this rank's rows into -- lists (<= 8) of tensors / raw pointers, or, for a steady-state loop, the
    peer_table() of each list built once (then `n_peers` = how many entries are in use).  Returns dict(pose_opt, logw,
    pose_samples, cost, pose_cov) of local tensors."""
    D = 7 if params.dof == 6 else 4
    B, M = prob.B, params.mc_samples
    for t, shape in ((pose_opt_out, (B, D)), (logw_out, (B, M))):
        if tuple(t.shape) != shape or t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError(f"local output must be contiguous float32 {shape}")
    if torch.is_tensor(peer_logw) != torch.is_tensor(peer_pose):
        raise ValueError("peer_logw / peer_pose: both lists or both peer_table() tensors")
    if torch.is_tensor(peer_logw):
        n = int(n_peers if n_peers is not None else peer_logw.numel())
        for t in (peer_logw, peer_pose):
            if t.dtype != torch.int64 or not t.is_contiguous() or t.numel() < max(n, 1) or t.device != prob.device:
                raise ValueError("peer tables: contiguous int64 tensors on the solving device (native.peer_table)")
        tab_lw, tab_ps = peer_logw, peer_pose
    else:
        if len(peer_logw) != len(peer_pose) or len(peer_logw) > 8:
            raise ValueError("peer_logw / peer_pose: equally long lists of at most 8 buffers")
        for lw, ps in zip(peer_logw, peer_pose):
            if isinstance(lw, int) and isinstance(ps, int):      # raw device pointers of IPC-mapped peer buffers
                continue
            if lw.dtype != torch.float32 or ps.dtype != torch.float32 or not lw.is_contiguous() or not ps.is_contiguous() \
                    or lw.dim() != 2 or lw.shape[1] != M or ps.dim() != 2 or ps.shape[1] != D \
                    or lw.shape[0] < obj_offset + B or ps.shape[0] < obj_offset + B:
                raise ValueError("peer buffers must be contiguous float32 (B_total, M) / (B_total, D) with "
                                 "B_total >= obj_offset + B")
        n = len(peer_logw)
        tab_lw, tab_ps = peer_table(peer_logw, prob.device), peer_table(peer_pose, prob.device)
    if n > 8:
        raise ValueError("the kernel pushes to at most 8 peers")
    pose_init = _f32c(pose_init)
    out = dict(pose_opt=pose_opt_out, logw=logw_out, pose_samples=prob.empty(B, M, D),
               cost=prob.empty(B) if want_cost else None,
               pose_cov=prob.empty(B, params.dof, params.dof) if want_cov else None)
    with torch.cuda.device(prob.device):
        check(lib().epnp_lm_amis_fused_push_f32(*prob.common_ptrs(), ptr(pose_init), ctypes.c_uint64(seed),
                                                ctypes.c_uint32(obj_offset), ptr(out["pose_opt"]), ptr(out["pose_cov"]),
                                                ptr(out["cost"]), ptr(out["pose_samples"]), ptr(out["logw"]),
                                                ctypes.c_void_p(tab_lw.data_ptr()), ctypes.c_void_p(tab_ps.data_ptr()), n,
                                                B, prob.N, ctypes.byref(params), stream_ptr(prob.device)),
              "epnp_lm_amis_fused_push_f32")
    if not torch.is_tensor(peer_logw) and tab_lw.is_cuda:
        tab_lw.record_stream(torch.cuda.current_stream(prob.device))       # the kernel reads the tables after we return
        tab_ps.record_stream(torch.cuda.current_stream(prob.device))
    return out


def cost_backward(prob: Problem, dof, z_min, poses_a, grad_a, poses_b=None, grad_b=None,
                  want=(True, True, True, True)):
    """sum_p grad[p] * d cost(pose p) / d (x3d, x2d, w2d, delta) for object-major pose sets
    a: (B, PA, D) / (B, PA) and optional b: (B, PB, D) / (B, PB).  Returns (gx3d, gx2d, gw2d, gdelta), None
    where `want` is False."""
    B, N = prob.B, prob.N
    poses_a, grad_a = _f32c(poses_a), _f32c(grad_a)
    PA = poses_a.shape[1]
    PB = 0
    if poses_b is not None:
        poses_b, grad_b = _f32c(poses_b), _f32c(grad_b)
        PB = poses_b.shape[1]
    gx3d = prob.empty(B, N, 3) if want[0] else None
    gx2d = prob.empty(B, N, 2) if want[1] else None
    gw2d = prob.empty(B, N, 2) if want[2] else None
    gdel = prob.empty(B) if want[3] else None
    with torch.cuda.device(prob.device):
        check(lib().epnp_cost_backward_f32(*prob.common_ptrs(), ptr(poses_a), ptr(grad_a), PA, ptr(poses_b), ptr(grad_b), PB,
                                           ptr(gx3d), ptr(gx2d), ptr(gw2d), ptr(gdel), B, N, int(dof),
                                           ctypes.c_float(z_min), stream_ptr(prob.device)), "epnp_cost_backward_f32")
    return gx3d, gx2d, gw2d, gdel


def fused_workspace_bytes(B, N, params):
    return int(lib().epnp_fused_workspace_bytes(B, N, ctypes.byref(params)))


def lm_amis_fused_host(host, params, workspace, n_chunks=8, seed=0, obj_offset=0, out=None, want_samples=True):
    """End-to-end call with HOST (pinned) tensors: host = dict(x3d, x2d, w2d, cam_mats, lb, ub, delta,
    pose_init) of CPU float32 tensors; `workspace` a CUDA uint8 tensor of fused_workspace_bytes().
    Results land in `out` (pinned CPU tensors, allocated when None).  Work is enqueued on the current
    stream of the workspace's device; synchronise that stream before reading `out`."""
    B, N = host["x3d"].shape[0], host["x3d"].shape[1]
    D = 7 if params.dof == 6 else 4
    M = params.mc_samples
    if out is None:
        pin = dict(dtype=torch.float32, pin_memory=True)
        out = dict(pose_opt=torch.empty(B, D, **pin), pose_cov=torch.empty(B, params.dof, params.dof, **pin),
                   cost=torch.empty(B, **pin), logw=torch.empty(B, M, **pin),
                   pose_samples=torch.empty(B, M, D, **pin) if want_samples else None)
    for k in ("x3d", "x2d", "w2d", "cam_mats", "delta", "pose_init"):
        t = host[k]
        assert (not t.is_cuda) and t.dtype == torch.float32 and t.is_contiguous(), k
    dev = workspace.device
    with torch.cuda.device(dev):
        check(lib().epnp_lm_amis_fused_host_f32(
            ptr(host["x3d"]), ptr(host["x2d"]), ptr(host["w2d"]), ptr(host["cam_mats"]), ptr(host.get("lb")),
            ptr(host.get("ub")), ptr(host["delta"]), ptr(host["pose_init"]), ctypes.c_uint64(seed),
            ctypes.c_uint32(obj_offset), ptr(out["pose_opt"]), ptr(out["pose_cov"]), ptr(out["cost"]),
            ptr(out.get("pose_samples")), ptr(out["logw"]), ctypes.c_void_p(workspace.data_ptr()),
            ctypes.c_size_t(workspace.numel()), int(n_chunks), B, N, ctypes.byref(params), stream_ptr(dev)),
            "epnp_lm_amis_fused_host_f32")
    return out


def mc_epilogue(logw_bm, pose_samples_bmd=None, pose_opt=None, cost_target=None, want_lse=True, want_loss=False,
                want_weights=False, want_score=False):
    """One pass over the object-major AMIS outputs (epnp_mc_epilogue_f32): logw (B, M) [, pose_samples (B, M, D),
    pose_opt (B, D), cost_target (B)] -> dict(lse (B), loss (B), weights (B, M), score_te (B)), absent ones None."""
    _need_cuda(logw_bm, "logw")
    B, M = logw_bm.shape
    logw_bm = _f32c(logw_bm)
    dev = logw_bm.device
    dof = 6
    if want_score:
        if pose_samples_bmd is None or pose_opt is None:
            raise ValueError("the MC score needs pose_samples (B, M, D) and pose_opt (B, D)")
        D = pose_samples_bmd.shape[-1]
        if D not in (4, 7) or tuple(pose_samples_bmd.shape) != (B, M, D) or tuple(pose_opt.shape) != (B, D):
            raise ValueError("pose_samples must be (B, M, D) and pose_opt (B, D) with D = 4 or 7")
        dof = 6 if D == 7 else 4
        pose_samples_bmd, pose_opt = _f32c(pose_samples_bmd), _f32c(pose_opt)
    else:
        pose_samples_bmd = pose_opt = None
    if cost_target is not None:
        cost_target = _f32c(cost_target).expand(B).contiguous()
    new = lambda *s: torch.empty(s, dtype=torch.float32, device=dev)
    out = dict(lse=new(B) if want_lse else None, loss=new(B) if want_loss else None,
               weights=new(B, M) if want_weights else None, score_te=new(B) if want_score else None)
    if B == 0:
        return out
    with torch.cuda.device(dev):
        check(lib().epnp_mc_epilogue_f32(ptr(logw_bm), ptr(pose_samples_bmd), ptr(pose_opt), ptr(cost_target),
                                         ptr(out["lse"]), ptr(out["loss"]), ptr(out["weights"]), ptr(out["score_te"]),
                                         B, M, dof, stream_ptr(dev)), "epnp_mc_epilogue_f32")
    return out


def mc_lse_backward(logw_bm, lse, grad_lse):
    """grad_logw (B, M) = grad_lse[b] * exp(logw[b, m] - lse[b]) (epnp_mc_lse_backward_f32)."""
    _need_cuda(logw_bm, "logw")
    B, M = logw_bm.shape
    logw_bm, lse, grad_lse = _f32c(logw_bm), _f32c(lse), _f32c(grad_lse)
    out = torch.empty_like(logw_bm)
    if B == 0:
        return out
    with torch.cuda.device(logw_bm.device):
        check(lib().epnp_mc_lse_backward_f32(ptr(logw_bm), ptr(lse), ptr(grad_lse), ptr(out), B, M,
                                             stream_ptr(logw_bm.device)), "epnp_mc_lse_backward_f32")
    return out


__all__ = ["Problem", "adaptive_delta", "cost_backward", "evaluate_cost", "evaluate_full", "lm_solve", "amis", "lm_amis_fused",
           "lm_amis_fused_host", "lm_amis_fused_push", "fused_workspace_bytes", "rslm", "epnp_init", "gn_plus_backward", "mc_epilogue", "mc_lse_backward", "default_params", "NativeError", "capi"]
