"""Drop-in replacement of the reference's `epropnp` package (same module and class names) whose
batched hot loops run in hand-written sm_100a CUDA behind libepropnp_b200.so:

    epropnp.epropnp               EProPnP6DoF / EProPnP4DoF / EProPnPBase / cholesky_wrapper
    epropnp.levenberg_marquardt   LMSolver / RSLMSolver
    epropnp.camera                PerspectiveCamera
    epropnp.cost_fun              HuberPnPCost / AdaptiveHuberPnPCost
    epropnp.common                evaluate_pnp, pnp_normalize, pnp_denormalize, rotation helpers
    epropnp.distributions         AngularCentralGaussian / VonMisesUniformMix
    epropnp.monte_carlo_pose_loss MonteCarloPoseLoss (6DoF and detection flavours), mc_logsumexp / mc_sample_weights / mc_score_te
    epropnp.builder               build_pnp / build_camera / build_cost_fun + registries (detection-style configs)
    epropnp.epnp_init             epnp_pose_init / EPnPSolver: the 6DoF evaluation flow's EPnP initialiser, on the device

Put `<repo>/epro-pnp_b200` on sys.path (instead of the reference checkout) and existing imports keep
working.  The solve / Monte-Carlo paths have no CPU or PyTorch fallback: CPU tensors raise.
"""

# Importing the package registers the classes with the builders, and exposes the flat names the detection variant's
# `ops.pnp` package exports (EPro-PnP-Det/epropnp_det/ops/pnp/__init__.py:5-14).
from .builder import build_pnp, build_camera, build_cost_fun      # noqa: E402,F401
from .camera import PerspectiveCamera                              # noqa: E402,F401
from .cost_fun import HuberPnPCost, AdaptiveHuberPnPCost           # noqa: E402,F401
from .common import evaluate_pnp                                   # noqa: E402,F401
from .levenberg_marquardt import LMSolver, RSLMSolver              # noqa: E402,F401
from .epropnp import EProPnP4DoF, EProPnP6DoF                      # noqa: E402,F401

__all__ = ['build_pnp', 'build_camera', 'build_cost_fun', 'PerspectiveCamera', 'HuberPnPCost', 'AdaptiveHuberPnPCost',
           'evaluate_pnp', 'LMSolver', 'RSLMSolver', 'EProPnP4DoF', 'EProPnP6DoF']
