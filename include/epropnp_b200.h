/* epropnp_b200.h -- C ABI of libepropnp_b200.so: the EPro-PnP hot path (batched LM / GN pose solve
 * and the AMIS Monte-Carlo loop) as hand-written sm_100a CUDA.
 *
 * The reference (tjiiv-cprg/EPro-PnP) has NO native interface for this path: it is ~10^3 PyTorch
 * op launches behind Python classes.  This header is therefore the FFI a maintainer would bind
 * underneath those classes; each entry point names the reference code it replaces (file:line under
 * epropnp/ of the reference).  The Python mirror of the reference surface that calls it lives in
 * epro-pnp_b200/epropnp/ ; INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to contiguous row-major fp32 unless the name ends in _host;
 *   - the caller owns and allocates every buffer; the library allocates no memory, is re-entrant, and only enqueues work
 *     on `stream` (a cudaStream_t passed as void*).  Per-host-thread state, exactly two items: the cudaError_t of the
 *     last failed call (epnp_last_cuda_error) and the four helper streams of epnp_lm_amis_fused_host_f32, created on that
 *     thread's first host-buffer call and kept for its lifetime;
 *   - return value: EPNP_OK or a negative EPNP_ERR_* code (never throws, never aborts);
 *     CUDA launch errors come back as EPNP_ERR_CUDA (epnp_last_cuda_error() has the cudaError_t);
 *   - B = objects, N = correspondences per object, D = 7 (dof 6: x y z w i j k) or 4 (dof 4:
 *     x y z yaw), M = mc_samples, I = mc_iter, S = M / I;
 *   - nullable arguments are marked [opt];
 *   - AMIS outputs are OBJECT-MAJOR: pose_samples (B, M, D), logw (B, M).  The reference returns
 *     (M, B, D) / (M, B); the Python layer hands out transposed views.
 */
#ifndef EPROPNP_B200_H
#define EPROPNP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EPNP_ABI_VERSION 2   /* 2: epnp_rslm_draw_f32 added; the push entry point takes DEVICE arrays of peer pointers */
/* epnp_epnp_init_f32 was added within version 2: a new symbol, no existing one changed, so a binding written for
 * version 2 without it keeps working. */

enum {
    EPNP_OK = 0,
    EPNP_ERR_BAD_ARG = -1,       /* null pointer, non-positive size, dof not in {4,6}, M % I != 0 ...  */
    EPNP_ERR_TOO_MANY_POINTS = -2, /* N (and M) do not fit the 227 KB shared memory of one SM       */
    EPNP_ERR_UNSUPPORTED = -3,   /* combination not supported by this build                            */
    EPNP_ERR_CUDA = -4,          /* a CUDA runtime call failed, see epnp_last_cuda_error()             */
    EPNP_ERR_NO_DEVICE = -5      /* no sm_100 device is current                                        */
};

/* Hyper-parameters of the solve.  Defaults (epnp_default_params) are the reference's constructor
 * defaults: LMSolver.__init__ levenberg_marquardt.py:31-53, HuberPnPCost.__init__ cost_fun.py:25-28,
 * PerspectiveCamera.__init__ camera.py:35-43, EProPnPBase/6DoF.__init__ epropnp.py:47-62,273-280. */
typedef struct EpnpParams {
    int32_t dof;                    /* 4 or 6                                                   */
    int32_t lm_iter;                /* LMSolver.num_iter                                        */
    int32_t fast_mode;              /* 1: Gauss-Newton, no trust region, no clip_jac            */
    float   z_min;                  /* PerspectiveCamera.z_min                                  */
    float   min_lm_diagonal;
    float   max_lm_diagonal;
    float   min_relative_decrease;
    float   initial_radius;         /* initial_trust_region_radius                              */
    float   max_radius;             /* max_trust_region_radius                                  */
    float   eps;                    /* LMSolver.eps                                             */
    float   huber_eps;              /* HuberPnPCost.eps                                         */
    int32_t mc_samples;             /* EProPnPBase.mc_samples  (M)                              */
    int32_t mc_iter;                /* EProPnPBase.num_iter    (I)                              */
    float   amis_eps;               /* EProPnPBase.eps                                          */
    int32_t acg_mle_iter;           /* EProPnP6DoF.acg_mle_iter                                 */
    float   acg_dispersion;         /* EProPnP6DoF.acg_dispersion                               */
} EpnpParams;

int         epnp_abi_version(void);
const char* epnp_error_string(int code);
int         epnp_last_cuda_error(void);             /* cudaError_t of the last EPNP_ERR_CUDA    */
void        epnp_default_params(EpnpParams* p, int dof);
/* Largest N one object may have (correspondences are resident in shared memory); mc_samples = 0
 * for the LM-only entry points. */
int         epnp_max_points(int dof, int mc_samples, int mc_iter);

/* AdaptiveHuberPnPCost.set_param (cost_fun.py:123-126):
 *   delta[b] = mean(w2d[b]) * sqrt(sum_xy var_unbiased(x2d[b])) * relative_delta               */
int epnp_adaptive_delta_f32(const float* x2d, const float* w2d, float relative_delta,
                            float* delta /*(B)*/, int B, int N, void* stream);

/* evaluate_pnp(..., out_cost=True) for a stack of poses (common.py:67-100 through camera.py:21-30
 * `project_b` and cost_fun.py:52-59): poses (S, B, D) -> cost (S, B).  S may be 1.
 * lb/ub: [opt] (B, 2) clamp bounds of the projection (both or neither).                        */
int epnp_evaluate_cost_f32(const float* x3d /*(B,N,3)*/, const float* x2d /*(B,N,2)*/,
                           const float* w2d /*(B,N,2)*/, const float* cam_mats /*(B,3,3)*/,
                           const float* lb, const float* ub, const float* delta /*(B)*/,
                           const float* poses, float* cost,
                           int S, int B, int N, int dof, float z_min, void* stream);

/* evaluate_pnp(..., out_jacobian, out_residual, out_cost) at one pose per object (common.py:67-100,
 * camera.py:10-18,64-143, cost_fun.py:33-89): pose (B, D) ->
 * residual [opt] (B, 2N), jac [opt] (B, 2N, dof), cost [opt] (B).                              */
int epnp_evaluate_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                      const float* lb, const float* ub, const float* delta, const float* pose,
                      float* residual, float* jac, float* cost, int clip_jac,
                      int B, int N, int dof, float z_min, float huber_eps, void* stream);

/* Backward of the derivative-regularisation branch: pose_opt_plus = pose (+) gn_step(pose) with the pose detached
 * (LMSolver.forward :66-68, gn_step :243-253, pose_add :255-265, evaluated with autograd on in the reference:
 * camera.py:119-129, cost_fun.py:52-84).  Given dL/d pose_opt_plus (B, D), writes dL/d x3d (B, N, 3), dL/d x2d
 * (B, N, 2), dL/d w2d (B, N, 2) and dL/d delta (B) (each optional).  The forward value is what
 * epnp_lm_solve_f32 returns in pose_opt_plus (lm_iter = 0 evaluates the step at pose_init).                      */
int epnp_gn_plus_backward_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                              const float* lb, const float* ub, const float* delta, const float* pose,
                              const float* grad_pose_plus, float* grad_x3d, float* grad_x2d, float* grad_w2d,
                              float* grad_delta, int B, int N, int dof, float z_min, float eps, float huber_eps,
                              void* stream);

/* Everything RSLMSolver.solve does before its solves (levenberg_marquardt.py:283-324) in one launch:
 *   the centre-based translation guess (center_based_init, :283-298: mean ray direction times the ratio of the 3D spread
 *     to the ray spread), computed per object unless t_init (B, 3) is given; written to t_out [opt] (B, 3);
 *   inds (P, B, n) int32: per (proposal, object) n distinct correspondence indices drawn WITHOUT replacement with
 *     probabilities proportional to mean(w2d, -1) -- torch.multinomial(mean_weight, num_points) (:306-309), by the
 *     same exponential race (the n smallest E_i / w_i, E_i ~ Exp(1)); a weight <= 0 is never drawn while a positive
 *     one is left (the reference raises when fewer than n are positive; here the subset is completed in index order);
 *   start (P, B, D): that translation (:314) + a uniformly random orientation: normalised Gaussian quaternion,
 *     (1,0,0,0) when its norm < eps (:319-324), or a yaw uniform on [0, 2 pi) (:316-317).
 * x3d / x2d / cam_mats may be NULL when t_init is given.
 * Philox-4x32-10 keyed by (seed; obj_offset + object, proposal): a batch shard draws what the whole batch would.   */
int epnp_rslm_draw_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                       const float* t_init, uint64_t seed, uint32_t obj_offset,
                       int* inds, float* start, float* t_out,
                       int P, int n, int B, int N, int dof, float eps, void* stream);

/* EPnP initial pose per object, as EPro-PnP-6DoF/lib/test.py:176-194 computes it with cv2.solvePnP(SOLVEPNP_EPNP):
 *   conf[b,i] = 0.5 * (w2d[b,i,0] + w2d[b,i,1]); points with conf >= the conf_quantile quantile of the object
 *   (numpy's default 'linear' method, evaluated in fp32 as numpy does for float32 data) are used;
 *   pose (B, 7) = x y z w i j k with w >= 0; n_used [opt] (B) int32 = number of points used.
 * EPnP (Lepetit, Moreno-Noguer, Fua, IJCV 2009) in pixels with fx, fy, cx, cy of cam_mats (skew ignored), fp64 inside.
 * Rejects (EPNP_ERR_BAD_ARG) conf_quantile outside [0, 1] and N - ceil(q (N-1)) < 4;
 * N > 16384 (a 128 x 128 map) returns EPNP_ERR_TOO_MANY_POINTS.  No lens distortion.                             */
int epnp_epnp_init_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                       float conf_quantile, float* pose, int* n_used, int B, int N, void* stream);

/* RSLMSolver.solve after the hypotheses are drawn (levenberg_marquardt.py:300-353): for every object, P starting
 * poses, each refined by LM / GN on its own n sampled correspondences, scored on all N correspondences, cheapest
 * kept.  Replaces the reference's gather of (P*B, n, .) mini-problems, the P-fold repeated camera / cost objects,
 * the solve of P*B tiny problems and the stacked evaluate_pnp (:326-352).
 *   inds (P, B, n) int32: sampled correspondence indices WITHIN the object (the torch.multinomial draw, :310-312)
 *   start (P, B, D): starting poses (centre-based translation + random orientation, :314-324)
 *   pose_best (B, D), cost_best (B); pose_all [opt] (P, B, D), cost_all [opt] (P, B)                          */
int epnp_rslm_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                  const float* lb, const float* ub, const float* delta, const int* inds, const float* start,
                  float* pose_best, float* cost_best, float* pose_all, float* cost_all,
                  int P, int n, int B, int N, const EpnpParams* p, void* stream);

/* LMSolver.solve with a given pose_init (levenberg_marquardt.py:80-190, _lm_iter :192-241, GN
 * fast mode :136-152) plus, when pose_opt_plus != NULL, the extra Gauss-Newton step of
 * LMSolver.forward (:66-68, gn_step :243-253, pose_add :255-265).
 *   pose_opt (B, D); pose_cov [opt] (B, dof, dof) = inverse(J^T J + eps I); cost [opt] (B);
 *   cost_init [opt] (B) = cost at pose_init (what monte_carlo_forward returns, epropnp.py:121-124) */
int epnp_lm_solve_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                      const float* lb, const float* ub, const float* delta, const float* pose_init,
                      float* pose_opt, float* pose_cov, float* cost, float* pose_opt_plus,
                      float* cost_init, int B, int N, const EpnpParams* p, void* stream);

/* The AMIS loop of EProPnPBase.monte_carlo_forward (epropnp.py:132-182) for EProPnP6DoF
 * (initial_fit :288-302, gen_new/old_distr :304-315, estimate_params :317-342; proposals from
 * distributions.py:15-52 and pyro MultivariateStudentT), starting from a given local solution.
 *   noise_*: [opt] injected base noise, object-major, m = iteration * S + s:
 *            noise_normal (B, M, 3), noise_chi2 (B, M), noise_rot (B, M, 4) for dof 6; for dof 4
 *            (EProPnP4DoF, epropnp.py:199-260, distributions.py:55-79) noise_rot is (B, M) and holds the
 *            YAW DRAWS themselves (the reference samples yaw with numpy on the host).  All three or none;
 *            when NULL the kernel draws Philox-4x32-10 noise keyed by (seed, obj_offset + b, m),
 *            so a sharded batch reproduces the unsharded one.
 *   proposals [opt] (B, I, 19): mode[3], L_t[6] (row-major lower), L_r[10] per AMIS iteration
 *            (dof 4: mode[3], L_t[6], yaw mode, kappa, 0...).                                     */
int epnp_amis_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                  const float* lb, const float* ub, const float* delta,
                  const float* pose_opt, const float* pose_cov,
                  const float* noise_normal, const float* noise_chi2, const float* noise_rot,
                  uint64_t seed, uint32_t obj_offset,
                  float* pose_samples /*(B,M,D)*/, float* logw /*(B,M)*/, float* proposals,
                  int B, int N, const EpnpParams* p, void* stream);

/* monte_carlo_forward with pose_init given and no init solver (epropnp.py:87-196 with force_init_solve=False):
 * LM solve + covariance + AMIS in ONE call = two launches on `stream`, no host round trip -- the warp-per-object LM
 * kernel (epnp_lm_solve_f32's), then the CTA-per-object AMIS kernel (epnp_amis_f32's); each stages the object's
 * correspondence set once into shared memory by TMA bulk copies.  (As a single kernel the LM half ran latency-bound:
 * DESIGN.md section 0.)  pose_cov [opt]: when NULL, the covariance travels between the two kernels through the first
 * dof^2 floats of each object's -- not yet written -- pose_samples rows (needs M * D >= dof^2).                      */
int epnp_lm_amis_fused_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                           const float* lb, const float* ub, const float* delta, const float* pose_init,
                           const float* noise_normal, const float* noise_chi2, const float* noise_rot,
                           uint64_t seed, uint32_t obj_offset,
                           float* pose_opt, float* pose_cov, float* cost, float* pose_opt_plus,
                           float* cost_init, float* pose_samples, float* logw, float* proposals,
                           int B, int N, const EpnpParams* p, void* stream);

/* Multi-GPU form of epnp_lm_amis_fused_f32 (one process per GPU, one NVLink / NVSwitch node): the solve AND the gather
 * of its small results in one kernel (the AMIS kernel).  Every CTA, when its object is finished, additionally stores the object's
 * pose_opt row and its M log-weights into row (obj_offset + b) of `n_peers` (<= 8) full-batch buffers that live in
 * OTHER GPUs' memory -- peer_logw[r] (B_total, M), peer_pose[r] (B_total, D), device pointers the caller obtained with
 * cudaIpcOpenMemHandle(..., cudaIpcMemLazyEnablePeerAccess) WHILE THIS DEVICE WAS CURRENT (a mapping opened under the
 * exporting device's index is not dereferenceable by this device's kernels) -- with plain stores over NVLink, object
 * by object underneath the remaining math.  peer_logw / peer_pose themselves are DEVICE arrays of n_peers pointers (in
 * this device's memory, like a batched-BLAS pointer array; the kernel reads them when an object finishes): built once
 * per set of buffers, they must stay valid until the launch has completed.
 * There is no gather kernel and no copy afterwards (what replaces the NCCL all-gather of SURVEY.md section 8e); the
 * caller needs one rendezvous of the ranks before it reads its own full-batch buffer.  pose_opt / logw are the LOCAL
 * outputs as before -- typically the local slice [obj_offset, obj_offset + B) of this rank's own full-batch buffers.
 * obj_offset doubles as the global object index of the Philox stream, so the assembled batch is bit-identical to the
 * single-GPU run.  Injected noise, pose_opt_plus, cost_init and proposals are not offered by this entry point. */
int epnp_lm_amis_fused_push_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                                const float* lb, const float* ub, const float* delta, const float* pose_init,
                                uint64_t seed, uint32_t obj_offset,
                                float* pose_opt, float* pose_cov, float* cost, float* pose_samples, float* logw,
                                float* const* peer_logw, float* const* peer_pose, int n_peers,
                                int B, int N, const EpnpParams* p, void* stream);

/* Backward of the differentiable outputs of monte_carlo_forward (epropnp.py:108-113: cost_init and the
 * Monte-Carlo costs inside pose_sample_logweights; proposal densities and samples carry no gradient,
 * epropnp.py:139-140,172-179) and of evaluate_pnp(out_cost=True) (common.py:67-100): for every object
 *   grad_x3d/x2d/w2d/delta = sum_p grad[p] * d cost(pose p) / d (x3d, x2d, w2d, delta)
 * over two pose sets given object-major: set a (B, PA, D) with grad_a (B, PA) -- e.g. the AMIS samples and
 * -dL/dlogw -- and [opt] set b (B, PB, D), grad_b (B, PB) -- e.g. pose_init and dL/dcost_init.
 * Differentiates what the reference's autograd sees: project_b (camera.py:21-30), the z / bound clamps
 * (zero gradient where clamped, :81-93), Huber (cost_fun.py:8-12).  Outputs [opt]: (B,N,3), (B,N,2), (B,N,2), (B). */
int epnp_cost_backward_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                           const float* lb, const float* ub, const float* delta,
                           const float* poses_a, const float* grad_a, int PA,
                           const float* poses_b, const float* grad_b, int PB,
                           float* grad_x3d, float* grad_x2d, float* grad_w2d, float* grad_delta,
                           int B, int N, int dof, float z_min, void* stream);

/* Epilogue on the AMIS outputs -- the step AFTER the path in every caller of monte_carlo_forward (one pass over the
 * object-major log-weights instead of a dozen torch ops on (M, B) views):
 *   lse (B)        = logsumexp_m logw[b, m]      -- `loss_pred` of MonteCarloPoseLoss.forward
 *                    (EPro-PnP-6DoF/lib/models/monte_carlo_pose_loss.py:27-28, EPro-PnP-Det/epropnp_det/models/losses/
 *                    monte_carlo_pose_loss.py:21-22)
 *   loss (B)       = cost_target[b] + lse[b], NaN replaced by 0 (same files :30-31 / :24-25); cost_target [opt]
 *   weights (B, M) = softmax_m logw[b, :]        -- deform_pnp_head.py:524
 *   score_te (B)   = sum_m weights[b, m] * clamp((2.5 - log2 ||(x, z)_{b,m} - (x, z)_opt,b||) / 4, 0, 1)
 *                    -- the Monte-Carlo 'te' score, deform_pnp_head.py:533-536; needs pose_samples (B, M, D), pose_opt (B, D)
 * Every output is [opt]; at least one must be given.                                                              */
int epnp_mc_epilogue_f32(const float* logw /*(B,M)*/, const float* pose_samples, const float* pose_opt,
                         const float* cost_target, float* lse, float* loss, float* weights, float* score_te,
                         int B, int M, int dof, void* stream);
/* Backward of lse: grad_logw (B, M) = grad_lse[b] * exp(logw[b, m] - lse[b]), exactly 0 where grad_lse[b] == 0.     */
int epnp_mc_lse_backward_f32(const float* logw, const float* lse, const float* grad_lse, float* grad_logw,
                             int B, int M, void* stream);

/* Same as epnp_lm_amis_fused_f32 with HOST buffers (pinned for full speed): copies the inputs to
 * the caller-provided device workspace, runs the fused kernel and copies the results back, all on
 * `stream`, in `n_chunks` object chunks through a copy-in / solve / copy-out pipeline (helper streams owned by
 * the calling host thread, created on first use -- the only resource the library keeps).  n_chunks = 0 cuts the
 * batch at whole waves of resident CTAs (SMs x CTAs per SM objects per chunk, as few waves per chunk as the limit of
 * 64 chunks allows); n_chunks >= 1 asks for that many equal chunks (8 for B = 4096, two calls in flight, is the measured
 * configuration).
 * workspace: device memory of at least epnp_fused_workspace_bytes(B, N, p) bytes.
 * Outputs [opt] as above (pose_samples_host may be NULL to skip the largest copy).              */
size_t epnp_fused_workspace_bytes(int B, int N, const EpnpParams* p);
int epnp_lm_amis_fused_host_f32(const float* x3d_host, const float* x2d_host, const float* w2d_host,
                                const float* cam_mats_host, const float* lb_host, const float* ub_host,
                                const float* delta_host, const float* pose_init_host,
                                uint64_t seed, uint32_t obj_offset,
                                float* pose_opt_host, float* pose_cov_host, float* cost_host,
                                float* pose_samples_host, float* logw_host,
                                void* workspace, size_t workspace_bytes, int n_chunks,
                                int B, int N, const EpnpParams* p, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EPROPNP_B200_H */
