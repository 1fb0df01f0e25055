"""The step before the solve in the 6DoF evaluation flow (EPro-PnP-6DoF/lib/test.py:176-211):

    epnp_pose_init   per object, the correspondences whose confidence mean(w2d, -1) is at or above the object's
                     `conf_quantile` quantile (numpy's 'linear'), then EPnP on them -- what test.py:179-194 does with
                     .cpu().numpy(), np.quantile, cv2.solvePnP(SOLVEPNP_EPNP) in a Python loop and
                     Rotation.from_rotvec(...).as_quat()[[3, 0, 1, 2]].  Here it is one kernel launch on the device
                     (epnp_epnp_init_f32): no host round trip, no synchronisation, fp64 inside.
    EPnPSolver       the same as an `init_solver` of LMSolver (the `solve` contract LMSolver calls), so
                     LMSolver(dof=6, init_solver=EPnPSolver()) starts its iterations from EPnP when pose_init is None
                     or force_init_solve=True.

6DoF only (x y z w i j k); lens distortion is not modelled (test.py passes zero distortion).  Not differentiable:
the reference's cv2 call is not either.
"""
import torch

from epropnp_b200 import native


def epnp_pose_init(x3d, x2d, w2d, cam_mats, conf_quantile=0.8):
    """x3d (B, N, 3), x2d (B, N, 2) pixels, w2d (B, N, 2), cam_mats (3, 3) or (B, 3, 3) -> pose (B, 7) = x y z w i j k
    with w >= 0, in the dtype of x2d."""
    with torch.no_grad():
        return native.epnp_init(x3d, x2d, w2d, cam_mats, conf_quantile).to(x2d.dtype)


class EPnPSolver:
    """EPnP initial pose as an `init_solver` of LMSolver (levenberg_marquardt.py:115-130 calls
    solve(x3d, x2d, w2d, camera, cost_fun, with_cost=..., fast_mode=...))."""

    def __init__(self, conf_quantile=0.8, dof=6):
        if dof != 6:
            raise ValueError(f"EPnPSolver gives 6DoF poses only, got dof={dof}")
        if not 0.0 <= float(conf_quantile) <= 1.0:
            raise ValueError(f"conf_quantile must be in [0, 1], got {conf_quantile}")
        self.dof = 6
        self.conf_quantile = float(conf_quantile)

    def solve(self, x3d, x2d, w2d, camera, cost_fun, with_cost=False, fast_mode=False, **kwargs):
        """-> pose (B, 7), None, cost (B) | None; the cost is evaluate_pnp's at that pose (epnp_evaluate_cost_f32)."""
        pose = epnp_pose_init(x3d, x2d, w2d, camera.cam_mats, self.conf_quantile)
        cost = None
        if with_cost:
            prob = native.Problem(x3d, x2d, w2d, camera.cam_mats, camera.lb, camera.ub, cost_fun.delta)
            cost = native.evaluate_cost(prob, pose[None], 6, float(camera.z_min))[0].to(x2d.dtype)
        return pose, None, cost


__all__ = ["epnp_pose_init", "EPnPSolver"]
