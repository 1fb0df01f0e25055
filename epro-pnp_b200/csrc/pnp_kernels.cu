// pnp_kernels.cu -- sm_100a kernels of the EPro-PnP hot path and their C ABI (include/epropnp_b200.h).
//
//   lm_warp_kernel (pnp_lm.cuh)      Levenberg-Marquardt / Gauss-Newton pose solve, ONE WARP per object: raw correspondences
//                                    TMA-staged into the warp's shared memory, 16 points per lane, shuffle-only reduction,
//                                    6x6 damped Cholesky + SE(3) retraction + trust region on lane 0, no block barrier.
//   amis_kernel (pnp_amis.cuh)       the AMIS Monte-Carlo loop, ONE CTA per object: TMA ring -> packed pair records, one
//                                    thread per sample, packed fp32x2 cost sweep, refits as block reductions; five CTAs per SM.
//   epnp_lm_amis_fused_f32           = lm_warp_kernel, then amis_kernel, on the caller's stream (no host round trip); the
//                                    split is what a measurement asked for: as one kernel the LM half ran latency-bound at
//                                    4 points per thread between block barriers (DESIGN.md section 4).
//   cost_kernel, evaluate_full_kernel, rslm_draw_kernel, rslm_kernel, cost_backward_kernel, gn_plus_backward_kernel, adaptive_delta_kernel,
//   mc_epilogue_kernel, mc_lse_backward_kernel      the steps either side of the path (CTA per object).
//   epnp_init_kernel (pnp_epnp.cuh)  EPnP initial pose of the 6DoF evaluation flow, ONE CTA per object, fp64 solve.
// No tensor cores: the only contraction is 6-deep, the work is FP32-pipe + MUFU bound (DESIGN.md).
// Build options: EPNP_PHASE_TIMERS (profiling), EPNP_SIMT_EMUL (g++ build for the test-only CPU emulator).
#include <cuda_runtime.h>
#include <math_constants.h>

#include <cstdlib>

#include "pnp_device.cuh"
#include "pnp_lm.cuh"
#include "pnp_amis.cuh"
#include "pnp_epnp.cuh"

namespace {

thread_local int g_last_cuda_error = 0;

// Shared-memory image of the CTA-per-object kernels that are not the AMIS loop: head, TMA ring, packed pair records.
template <int DOF> struct ObjHead {
    uint64_t bar[2];
    float red[2 * NW * 32];
    float ev[32];                           // reduced evaluation: NV floats
    float pose[8];
    float step[2 * DOF];                    // gn_plus_backward: step, v
};
struct ObjPlan { int stage, pts, total_bytes; };
template <int DOF> __host__ __device__ inline ObjPlan plan_obj(int N) {
    ObjPlan s;
    int off = (int)((sizeof(ObjHead<DOF>) + 127) / 128 * 128 / 4);
    s.stage = off; off += 2 * STAGE_FLOATS;
    s.pts = off; off += 16 * ((N + 1) / 2);
    s.total_bytes = off * 4;
    return s;
}

// cost of S poses per object: poses (S, B, D) -> cost (S, B)
template <int DOF>
__global__ void __launch_bounds__(NT, 4) cost_kernel(const KArgs a) {
    EPNP_DYN_SMEM(unsigned char, smem_raw, 128);
    ObjHead<DOF>& sh = *reinterpret_cast<ObjHead<DOF>*>(smem_raw);
    float* dyn = reinterpret_cast<float*>(smem_raw);
    const ObjPlan pl = plan_obj<DOF>(a.N);
    float* pts4 = dyn + pl.pts;
    constexpr int PD = Dim<DOF>::POSE;
    const int obj = blockIdx.x;
    Loader ld(a, sh.bar, dyn + pl.stage);
    ld.load_object(obj, pts4);
    const Cam cam = load_cam(a, obj);
    const float delta = __ldg(a.delta + obj);
    for (int s = threadIdx.x; s < a.S_eval; s += NT) {
        float pose[PD];
#pragma unroll
        for (int k = 0; k < PD; ++k) pose[k] = __ldg(a.poses + ((size_t)s * a.B + obj) * PD + k);
        a.cost_out[(size_t)s * a.B + obj] = pose_cost<DOF>(pts4, a.N, pose, cam, delta);
    }
}

// ------------------------------------------------------------------------------------------------
// Random-sample LM initialiser (RSLMSolver.solve, levenberg_marquardt.py:300-353) for one object per CTA:
// thread <-> hypothesis.  A thread runs the whole LM / GN iteration of its hypothesis serially over that
// hypothesis' n sampled correspondences (read out of the object's resident pair records: the (P*B, n, .) gathered
// copies, the P-fold repeated cameras and the P*B tiny solves of the reference do not exist), scores the result
// on ALL N points with the same sweep the AMIS loop uses, and the CTA keeps the cheapest hypothesis.
struct RslmArgs {
    KArgs k;                    // correspondences, camera, bounds, delta, B, N, LM parameters
    const int* inds;            // (P, B, n) indices of the sampled correspondences, within the object
    const float* start;         // (P, B, D) starting poses
    float* pose_best;           // (B, D)
    float* cost_best;           // (B)
    float* pose_all;            // [opt] (P, B, D)
    float* cost_all;            // [opt] (P, B)
    int P, n;
};

// Order of torch.min over the hypotheses (levenberg_marquardt.py:350): a NaN cost wins (min propagates NaN), then the
// smaller cost, then the earlier hypothesis.
__device__ __forceinline__ bool cheaper_hypothesis(float c, int h, float wc, int wh) {
    const bool cn = (c != c), wn = (wc != wc);
    if (cn != wn) return cn;
    if (cn) return h < wh;
    return c < wc || (c == wc && h < wh);
}

template <int DOF, bool CLIP>
__device__ __forceinline__ void eval_subset(const float* pts, const int* idx, int n, const float* pose, const Cam& cam,
                                            float delta, float huber_eps, float* acc) {
    constexpr int NV = Dim<DOF>::NV;
    float R[9];
    pose_to_rot<DOF>(pose, R);
#pragma unroll
    for (int i = 0; i < NV; ++i) acc[i] = 0.f;
    for (int i = 0; i < n; ++i) {
        const int j = __ldg(idx + i);
        const float* q = pts + (j >> 1) * 16 + (j & 1);
        point_normal_eq<DOF, CLIP>(R, pose, cam, delta, huber_eps, q[0], q[2], q[4], -q[6], -q[8], q[10], q[12], acc);
    }
}

template <int DOF>
__global__ void __launch_bounds__(NT, 2) rslm_kernel(const RslmArgs r) {
    const KArgs& a = r.k;
    EPNP_DYN_SMEM(unsigned char, smem_raw, 128);
    ObjHead<DOF>& sh = *reinterpret_cast<ObjHead<DOF>*>(smem_raw);
    float* dyn = reinterpret_cast<float*>(smem_raw);
    const ObjPlan pl = plan_obj<DOF>(a.N);
    float* pts = dyn + pl.pts;
    constexpr int PD = Dim<DOF>::POSE;
    const Params& p = a.p;
    const int tid = threadIdx.x, obj = blockIdx.x;
    float* best_cost = sh.red;                                  // [NT]
    int* best_hyp = reinterpret_cast<int*>(sh.red + NT);        // [NT]
    Loader ld(a, sh.bar, dyn + pl.stage);
    ld.load_object(obj, pts);
    const Cam cam = load_cam(a, obj);
    const float delta = __ldg(a.delta + obj);
    float my_cost = CUDART_INF_F, my_pose[PD];
    int my_hyp = -1;
    for (int h = tid; h < r.P; h += NT) {
        const int* idx = r.inds + ((size_t)h * a.B + obj) * r.n;
        LMState<DOF> s;
#pragma unroll
        for (int i = 0; i < PD; ++i) s.pose[i] = __ldg(r.start + ((size_t)h * a.B + obj) * PD + i);
        s.radius = p.initial_radius;
        s.shrink = 2.0f;
        float acc[Dim<DOF>::NV];
        if (!p.fast_mode) {
            eval_subset<DOF, true>(pts, idx, r.n, s.pose, cam, delta, p.huber_eps, acc);
            lm_adopt<DOF>(s, acc);
            if (p.lm_iter > 0) lm_propose<DOF>(s, p);
            for (int k = 0; k < p.lm_iter; ++k) {
                eval_subset<DOF, true>(pts, idx, r.n, s.pose_new, cam, delta, p.huber_eps, acc);
                lm_update<DOF>(s, acc, p);
                if (k + 1 < p.lm_iter) lm_propose<DOF>(s, p);
            }
        } else {
            for (int k = 0; k < p.lm_iter; ++k) {
                eval_subset<DOF, false>(pts, idx, r.n, s.pose, cam, delta, p.huber_eps, acc);
                gn_advance<DOF>(s.pose, acc, p.eps, s.pose);
            }
        }
        const float c = pose_cost<DOF>(pts, a.N, s.pose, cam, delta);       // score on the full set
        if (r.pose_all) {
#pragma unroll
            for (int i = 0; i < PD; ++i) r.pose_all[((size_t)h * a.B + obj) * PD + i] = s.pose[i];
        }
        if (r.cost_all) r.cost_all[(size_t)h * a.B + obj] = c;
        if (my_hyp < 0 || cheaper_hypothesis(c, h, my_cost, my_hyp)) {
            my_cost = c; my_hyp = h;
#pragma unroll
            for (int i = 0; i < PD; ++i) my_pose[i] = s.pose[i];
        }
    }
    best_cost[tid] = my_cost;
    best_hyp[tid] = my_hyp;
    __syncthreads();
    if (tid == 0) {
        int w = -1;
        for (int t = 0; t < NT; ++t) {
            if (best_hyp[t] < 0) continue;
            if (w < 0 || cheaper_hypothesis(best_cost[t], best_hyp[t], best_cost[w], best_hyp[w])) w = t;
        }
        best_hyp[0] = w;                                    // the winning THREAD (it still holds the pose)
    }
    __syncthreads();
    if (tid == best_hyp[0]) {
#pragma unroll
        for (int i = 0; i < PD; ++i) r.pose_best[(size_t)obj * PD + i] = my_pose[i];
        r.cost_best[obj] = my_cost;
    }
}

// ------------------------------------------------------------------------------------------------
// Everything RSLMSolver.solve does before its solves (levenberg_marquardt.py:283-324), one CTA per object:
//   * the centre-based translation guess (center_based_init, :283-298): rays = K^-1 [u v 1] dehomogenised, direction =
//     (mean ray, 1), depth = spread of the 3D points over spread of the rays (unbiased standard deviations: y-extent
//     for 4DoF, sqrt(2/3) |std3d| / |std ray| for 6DoF) -- two block reductions over the N points; skipped when the
//     caller passes its own t_init;
//   * per hypothesis (thread <-> hypothesis) n DISTINCT correspondence indices, drawn without replacement with
//     probabilities proportional to wbar_i = mean(w2d[i, :]) -- torch.multinomial(wbar, n) (:306-312).  Same algorithm
//     as torch's: an exponential race, the n smallest of E_i / wbar_i with E_i ~ Exp(1) (Efraimidis-Spirakis); a weight
//     that is not positive is never drawn.  The race keeps its n current winners in shared memory ([slot][thread]:
//     conflict-free) with the position of the worst of them; once the list is full an element is rejected by one
//     multiply and compare (E >= 1 - u), and pays for a logarithm only when it might enter
//     (~ n (1 + ln(N / n)) times per hypothesis).  With fewer hypotheses than threads several lanes share one race;
//     the subset comes out in ascending key order (= the order of the draw);
//   * the starting pose: that translation with a uniformly random orientation -- a normalised Gaussian quaternion,
//     (1,0,0,0) when its norm is below eps (:318-324), or a yaw uniform on [0, 2 pi) (:316-317).
// Philox-4x32-10 keyed by (seed; global object index, hypothesis, block): independent of B, P tiling and launch shape.
struct RslmDrawArgs {
    const float *x3d, *x2d, *w2d, *cam;     // (B, N, 3), (B, N, 2), (B, N, 2), (B, 3, 3)
    const float* t_init;                    // [opt] (B, 3): overrides the centre-based guess
    int* inds;                              // (P, B, n)
    float* start;                           // (P, B, D)
    float* t_out;                           // [opt] (B, 3): the translation guess that was used
    uint64_t seed;
    uint32_t obj_offset;
    int P, n, B, N;
    float eps;
};

constexpr uint32_t RSLM_TAG_SUBSET = 0x52534c4du, RSLM_TAG_START = 0x52534c53u;

template <int DOF>
__global__ void __launch_bounds__(NT) rslm_draw_kernel(const RslmDrawArgs r) {
    EPNP_DYN_SMEM(unsigned char, smem_raw, 16);
    __shared__ float red[2 * NT];
    __shared__ float t0[3];
    __shared__ int counts[NT];
    float* wbar = reinterpret_cast<float*>(smem_raw);                       // [N]
    float* keys = wbar + ((r.N + 3) & ~3);                                  // [n][NT]
    int* slots = reinterpret_cast<int*>(keys + (size_t)r.n * NT);           // [n][NT]
    constexpr int PD = Dim<DOF>::POSE;
    const int tid = threadIdx.x, obj = blockIdx.x;
    const uint32_t gobj = r.obj_offset + (uint32_t)obj;
    for (int i = tid; i < r.N; i += NT) {
        const float2 w = *reinterpret_cast<const float2*>(r.w2d + ((size_t)obj * r.N + i) * 2);
        wbar[i] = 0.5f * (w.x + w.y);
    }
    if (r.t_init) {
        if (tid < 3) t0[tid] = __ldg(r.t_init + (size_t)obj * 3 + tid);
    } else {
        // K^-1 by the adjugate (general 3x3), then mean / unbiased variance of the two ray coordinates and of x3d
        float k[9], inv[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) k[i] = __ldg(r.cam + (size_t)obj * 9 + i);
        inv[0] = k[4] * k[8] - k[5] * k[7]; inv[1] = k[2] * k[7] - k[1] * k[8]; inv[2] = k[1] * k[5] - k[2] * k[4];
        inv[3] = k[5] * k[6] - k[3] * k[8]; inv[4] = k[0] * k[8] - k[2] * k[6]; inv[5] = k[2] * k[3] - k[0] * k[5];
        inv[6] = k[3] * k[7] - k[4] * k[6]; inv[7] = k[1] * k[6] - k[0] * k[7]; inv[8] = k[0] * k[4] - k[1] * k[3];
        const float idet = 1.0f / (k[0] * inv[0] + k[1] * inv[3] + k[2] * inv[6]);
#pragma unroll
        for (int i = 0; i < 9; ++i) inv[i] *= idet;
        const float* g2 = r.x2d + (size_t)obj * r.N * 2;
        const float* g3 = r.x3d + (size_t)obj * r.N * 3;
        auto ray = [&](int i, float& rx, float& ry) {
            const float u = __ldg(g2 + 2 * i), v = __ldg(g2 + 2 * i + 1);
            const float z = fmaxf(inv[6] * u + inv[7] * v + inv[8], 1e-6f);
            rx = (inv[0] * u + inv[1] * v + inv[2]) / z;
            ry = (inv[3] * u + inv[4] * v + inv[5]) / z;
        };
        float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        for (int i = tid; i < r.N; i += NT) {
            float rx, ry;
            ray(i, rx, ry);
            m[0] += rx; m[1] += ry; m[2] += __ldg(g3 + 3 * i); m[3] += __ldg(g3 + 3 * i + 1); m[4] += __ldg(g3 + 3 * i + 2);
        }
        block_sum<5>(m, red, 0);
        const float in = 1.0f / (float)r.N;
#pragma unroll
        for (int c = 0; c < 5; ++c) m[c] *= in;
        float v[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        for (int i = tid; i < r.N; i += NT) {
            float rx, ry;
            ray(i, rx, ry);
            const float d0 = rx - m[0], d1 = ry - m[1], d2 = __ldg(g3 + 3 * i) - m[2], d3 = __ldg(g3 + 3 * i + 1) - m[3],
                        d4 = __ldg(g3 + 3 * i + 2) - m[4];
            v[0] += d0 * d0; v[1] += d1 * d1; v[2] += d2 * d2; v[3] += d3 * d3; v[4] += d4 * d4;
        }
        block_sum<5>(v, red, 1);
        if (tid == 0) {
            const float iv = 1.0f / (float)max(r.N - 1, 1);             // unbiased (torch.std's default)
            float depth;
            if (DOF == 4) depth = sqrtf(v[3] * iv) / fmaxf(sqrtf(v[1] * iv), 1e-6f);
            else depth = 0.816496580927726f * sqrtf((v[2] + v[3] + v[4]) * iv) / fmaxf(sqrtf((v[0] + v[1]) * iv), 1e-6f);
            t0[0] = m[0] * depth; t0[1] = m[1] * depth; t0[2] = depth;
        }
    }
    __syncthreads();
    if (r.t_out && tid < 3) r.t_out[(size_t)obj * 3 + tid] = t0[tid];
    const Philox ph{(uint32_t)r.seed, (uint32_t)(r.seed >> 32)};
    // Fewer hypotheses than threads: G = 2, 4 or 8 lanes (of one warp) share a hypothesis.  Lane g races the Philox blocks
    // g, g + G, ... into its own list, then lane 0 folds the other lanes' winners into its list.  The n smallest keys of a
    // hypothesis do not depend on how the race was split, and the subset is written in ascending key order -- the order
    // in which a draw without replacement produces it -- so the output does not depend on G (or P, or the batch) either.
    int G = 1;
    while (G < 8 && r.P * (2 * G) <= NT) G *= 2;
    const int per_pass = NT / G, g = tid & (G - 1), nblk = (r.N + 3) >> 2;
    for (int h0 = 0; h0 < r.P; h0 += per_pass) {
        const int h = h0 + tid / G;
        const bool live = h < r.P;
        int cnt = 0, worst = 0;
        float thr = -1.0f;                                                  // the largest key in the list
        auto offer = [&](float key, int i) {
            if (cnt < r.n) {
                keys[cnt * NT + tid] = key; slots[cnt * NT + tid] = i;
                if (key > thr) { thr = key; worst = cnt; }
                ++cnt;
            } else if (key < thr) {
                keys[worst * NT + tid] = key; slots[worst * NT + tid] = i;
                thr = -1.0f;
                for (int s = 0; s < r.n; ++s) {
                    const float k = keys[s * NT + tid];
                    if (k > thr) { thr = k; worst = s; }
                }
            }
        };
        if (live) {
            for (int blk = g; blk < nblk; blk += G) {
                uint32_t u[4];
                ph(gobj, (uint32_t)h, (uint32_t)blk, RSLM_TAG_SUBSET, u);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int i = 4 * blk + j;
                    if (i >= r.N) break;
                    const float w = wbar[i];
                    if (!(w > 0.0f)) continue;
                    const float uu = u01(u[j]);
                    if (cnt == r.n && (1.0f - uu) >= thr * w) continue;    // E = -log u >= 1 - u: cannot beat the worst winner
                    offer(-fast_log(uu) / w, i);
                }
            }
        }
        if (G > 1) {
            counts[tid] = cnt;
            __syncwarp();
            if (live && g == 0) {
                for (int o = 1; o < G; ++o) {
                    const int c = counts[tid + o];
                    for (int s = 0; s < c; ++s) offer(keys[s * NT + tid + o], slots[s * NT + tid + o]);
                }
            }
        }
        if (live && g == 0) {
            // ascending (key, index): insertion sort of at most n entries
            for (int a = 1; a < cnt; ++a) {
                const float k = keys[a * NT + tid];
                const int i = slots[a * NT + tid];
                int bpos = a - 1;
                while (bpos >= 0 && (keys[bpos * NT + tid] > k || (keys[bpos * NT + tid] == k && slots[bpos * NT + tid] > i))) {
                    keys[(bpos + 1) * NT + tid] = keys[bpos * NT + tid]; slots[(bpos + 1) * NT + tid] = slots[bpos * NT + tid];
                    --bpos;
                }
                keys[(bpos + 1) * NT + tid] = k; slots[(bpos + 1) * NT + tid] = i;
            }
            // fewer than n positive weights (torch.multinomial raises): complete the subset with the first unused indices
            for (int i = 0; cnt < r.n && i < r.N; ++i) {
                if (wbar[i] > 0.0f) continue;
                slots[cnt * NT + tid] = i; ++cnt;
            }
            int* out = r.inds + ((size_t)h * r.B + obj) * r.n;
            for (int s = 0; s < r.n; ++s) out[s] = slots[s * NT + tid];
            float* st = r.start + ((size_t)h * r.B + obj) * PD;
            st[0] = t0[0]; st[1] = t0[1]; st[2] = t0[2];
            uint32_t v[4];
            ph(gobj, (uint32_t)h, 0u, RSLM_TAG_START, v);
            if (DOF == 4) {
                st[3] = u01(v[0]) * 6.283185307179586f;
            } else {
                float q[4];
                box_muller(v[0], v[1], q[0], q[1]);
                box_muller(v[2], v[3], q[2], q[3]);
                const float nrm = sqrtf(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
                const bool tiny = nrm < r.eps;
                const float inv = 1.0f / nrm;
                st[3] = tiny ? 1.0f : q[0] * inv; st[4] = tiny ? 0.0f : q[1] * inv;
                st[5] = tiny ? 0.0f : q[2] * inv; st[6] = tiny ? 0.0f : q[3] * inv;
            }
        }
        __syncwarp();                       // lane 0 has finished reading the other lanes' lists before they are reused
    }
}

// ------------------------------------------------------------------------------------------------
// Backward of pose_opt_plus = pose (+) gn_step(pose) w.r.t. the correspondences and the Huber delta (the
// derivative-regularisation branch of training, LMSolver.forward :66-68 with autograd on).  One CTA per object:
// re-evaluate the normal equations, let the serial lane form step, dL/dstep (through pose_add) and
// v = -(H + eps I)^-1 dL/dstep, then thread <-> correspondence with forward-mode duals (pnp::gn_step_point_backward).
struct GnBwArgs {
    KArgs k;                    // correspondences, camera, bounds, delta, poses = pose (B, D), p.eps / huber_eps / z_min
    const float* gplus;         // (B, D)  dL/d pose_opt_plus
    float *gx3d, *gx2d, *gw2d;  // [opt] (B, N, 3|2|2)
    float* gdelta;              // [opt] (B)
};

template <int DOF>
__global__ void __launch_bounds__(NT, 2) gn_plus_backward_kernel(const GnBwArgs g) {
    const KArgs& a = g.k;
    EPNP_DYN_SMEM(unsigned char, smem_raw, 128);
    ObjHead<DOF>& sh = *reinterpret_cast<ObjHead<DOF>*>(smem_raw);
    float* dyn = reinterpret_cast<float*>(smem_raw);
    const ObjPlan pl = plan_obj<DOF>(a.N);
    float* pts = dyn + pl.pts;
    constexpr int PD = Dim<DOF>::POSE, NA = Dim<DOF>::NA;
    const int tid = threadIdx.x, obj = blockIdx.x;
    Loader ld(a, sh.bar, dyn + pl.stage);
    ld.load_object(obj, pts);
    const Cam cam = load_cam(a, obj);
    const float delta = __ldg(a.delta + obj);
    if (tid < PD) sh.pose[tid] = __ldg(a.poses + (size_t)obj * PD + tid);
    __syncthreads();
    eval_normal_eq<DOF, true>(pts, a.N, sh.pose, cam, delta, a.p.huber_eps, sh.red, sh.ev);
    float* step = sh.step;              // [DOF]
    float* vvec = sh.step + DOF;        // [DOF]
    if (tid == 0) {
        float add[DOF], st[DOF], sbar[DOF], vv[DOF], gout[PD], pose[PD];
#pragma unroll
        for (int i = 0; i < DOF; ++i) add[i] = a.p.eps;
#pragma unroll
        for (int i = 0; i < PD; ++i) { pose[i] = sh.pose[i]; gout[i] = __ldg(g.gplus + (size_t)obj * PD + i); }
        damped_step_refined<DOF>(sh.ev, sh.ev + NA, add, st);
        pose_add_backward<DOF>(pose, st, gout, sbar);
        damped_step_refined<DOF>(sh.ev, sbar, add, vv);
#pragma unroll
        for (int i = 0; i < DOF; ++i) { step[i] = st[i]; vvec[i] = vv[i]; }
    }
    __syncthreads();
    float R[9], t[3], sv[DOF], vv[DOF];
    {
        float ps[PD];
#pragma unroll
        for (int i = 0; i < PD; ++i) ps[i] = sh.pose[i];
        pose_to_rot<DOF>(ps, R);
        t[0] = ps[0]; t[1] = ps[1]; t[2] = ps[2];
#pragma unroll
        for (int i = 0; i < DOF; ++i) { sv[i] = step[i]; vv[i] = vvec[i]; }
    }
    float gd[1] = {0.f};
    for (int n = tid; n < a.N; n += NT) {
        const float* q = pts + (n >> 1) * 16 + (n & 1);
        float gr[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        gn_step_point_backward<DOF>(R, t, cam, delta, a.p.huber_eps, q[0], q[2], q[4], -q[6], -q[8], q[10], q[12], vv, sv, gr);
        const size_t o = (size_t)obj * a.N + n;
        if (g.gx3d) { g.gx3d[o * 3] = gr[0]; g.gx3d[o * 3 + 1] = gr[1]; g.gx3d[o * 3 + 2] = gr[2]; }
        if (g.gx2d) { g.gx2d[o * 2] = gr[3]; g.gx2d[o * 2 + 1] = gr[4]; }
        if (g.gw2d) { g.gw2d[o * 2] = gr[5]; g.gw2d[o * 2 + 1] = gr[6]; }
        gd[0] += gr[7];
    }
    block_sum<1>(gd, sh.red, 0);
    if (tid == 0 && g.gdelta) g.gdelta[obj] = gd[0];
}

// residual / Jacobian / cost written out per point (API parity with evaluate_pnp's out_* tensors)
template <int DOF>
__global__ void __launch_bounds__(NT) evaluate_full_kernel(const KArgs a, float* residual, float* jac, float* cost,
                                                         int clip, float huber_eps) {
    __shared__ float red[NW];
    const int obj = blockIdx.x;
    constexpr int PD = Dim<DOF>::POSE;
    const Cam cam = load_cam(a, obj);
    const float delta = __ldg(a.delta + obj);
    float pose[PD], R[9];
#pragma unroll
    for (int k = 0; k < PD; ++k) pose[k] = __ldg(a.poses + (size_t)obj * PD + k);
    pose_to_rot<DOF>(pose, R);
    float csum = 0.f;
    for (int n = threadIdx.x; n < a.N; n += NT) {
        const size_t g = (size_t)obj * a.N + n;
        float r[2], j[2 * DOF];
        csum += point_residual_jac<DOF>(R, pose, cam, delta, huber_eps, clip != 0,
                                        a.x3d[g * 3], a.x3d[g * 3 + 1], a.x3d[g * 3 + 2],
                                        a.x2d[g * 2], a.x2d[g * 2 + 1], a.w2d[g * 2], a.w2d[g * 2 + 1], r, j);
        if (residual) { residual[g * 2] = r[0]; residual[g * 2 + 1] = r[1]; }
        if (jac) {
#pragma unroll
            for (int k = 0; k < 2 * DOF; ++k) jac[g * 2 * DOF + k] = j[k];
        }
    }
    if (cost) {
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) csum += __shfl_xor_sync(0xffffffffu, csum, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = csum;
        __syncthreads();
        if (threadIdx.x == 0) cost[obj] = (red[0] + red[1]) + (red[2] + red[3]);
    }
}

// ------------------------------------------------------------------------------------------------
// Backward of the Monte-Carlo cost: for every object, sum over its poses p (pose_init and all AMIS samples)
// of g[p] * d cost(pose p; x3d, x2d, w2d, delta) / d(x3d, x2d, w2d, delta).
// One CTA per object; thread <-> correspondence (up to BW_PPT per thread, accumulators in registers); the
// poses' pre-multiplied projections K[R|t] and upstream gradients are staged once in shared memory and read
// as broadcasts, so the (pose, point) loop touches no global memory.
constexpr int BW_PPT = 4;               // correspondences per thread and tile
constexpr int BW_POSE_TILE = 1024;      // poses staged per tile (13 floats each)

// Reverse mode of the cost for TWO correspondences at once (packed fp32x2; same math per half as
// pnp::point_cost_backward, with s = s2 * rsqrt(s2) and delta / s = delta * rsqrt(s2) from one MUFU.RSQ).
// g[0..2] += dL/d(X,Y,Z), g[3..4] += dL/d(u,v), g[5..6] += dL/d(wu,wv); gd += dL/d delta (both halves).
template <bool BOUNDED>
__device__ __forceinline__ void pair_cost_backward(const float (&P)[12], const Cam& cam, float delta, float gj,
                                                   float2 X, float2 Y, float2 Z, float2 nu, float2 nv, float2 wu,
                                                   float2 wv, float2 (&g)[7], float2& gd) {
    const float2 xh = __ffma2_rn(splat(P[0]), X, __ffma2_rn(splat(P[1]), Y, __ffma2_rn(splat(P[2]), Z, splat(P[3]))));
    const float2 yh = __ffma2_rn(splat(P[4]), X, __ffma2_rn(splat(P[5]), Y, __ffma2_rn(splat(P[6]), Z, splat(P[7]))));
    const float2 zh = __ffma2_rn(splat(P[8]), X, __ffma2_rn(splat(P[9]), Y, __ffma2_rn(splat(P[10]), Z, splat(P[11]))));
    const float2 iz = make_float2(FastRcp()(fmaxf(zh.x, cam.z_min)), FastRcp()(fmaxf(zh.y, cam.z_min)));
    const float2 px = __fmul2_rn(xh, iz), py = __fmul2_rn(yh, iz);
    float2 pxc = px, pyc = py;
    if (BOUNDED) {
        pxc.x = fminf(fmaxf(px.x, cam.lbx), cam.ubx); pxc.y = fminf(fmaxf(px.y, cam.lbx), cam.ubx);
        pyc.x = fminf(fmaxf(py.x, cam.lby), cam.uby); pyc.y = fminf(fmaxf(py.y, cam.lby), cam.uby);
    }
    const float2 ex = __fadd2_rn(pxc, nu), ey = __fadd2_rn(pyc, nv);
    const float2 rx = __fmul2_rn(ex, wu), ry = __fmul2_rn(ey, wv);
    const float2 s2 = __ffma2_rn(rx, rx, __fmul2_rn(ry, ry));
    const float2 rs = make_float2(FastRsqrt()(fmaxf(s2.x, 1e-30f)), FastRsqrt()(fmaxf(s2.y, 1e-30f)));
    const float2 s = __fmul2_rn(s2, rs);
    const bool in0 = s.x <= delta, in1 = s.y <= delta;
    const float2 ko = __fmul2_rn(splat(gj * delta), rs);                 // outlier: g * delta / s
    const float2 k = make_float2(in0 ? gj : ko.x, in1 ? gj : ko.y);
    const float2 grx = __fmul2_rn(k, rx), gry = __fmul2_rn(k, ry);
    g[5] = __ffma2_rn(grx, ex, g[5]);
    g[6] = __ffma2_rn(gry, ey, g[6]);
    const float2 gex = __fmul2_rn(grx, wu), gey = __fmul2_rn(gry, wv);
    g[3] = __ffma2_rn(gex, splat(-1.0f), g[3]);
    g[4] = __ffma2_rn(gey, splat(-1.0f), g[4]);
    float2 gpx = gex, gpy = gey;
    if (BOUNDED) {
        gpx.x = (pxc.x == px.x) ? gex.x : 0.f; gpx.y = (pxc.y == px.y) ? gex.y : 0.f;
        gpy.x = (pyc.x == py.x) ? gey.x : 0.f; gpy.y = (pyc.y == py.y) ? gey.y : 0.f;
    }
    const float2 gxh = __fmul2_rn(gpx, iz), gyh = __fmul2_rn(gpy, iz);
    const float2 tz = __ffma2_rn(gxh, px, __fmul2_rn(gyh, py));
    const float2 gzh = make_float2(zh.x >= cam.z_min ? -tz.x : 0.f, zh.y >= cam.z_min ? -tz.y : 0.f);
    g[0] = __ffma2_rn(splat(P[0]), gxh, __ffma2_rn(splat(P[4]), gyh, __ffma2_rn(splat(P[8]), gzh, g[0])));
    g[1] = __ffma2_rn(splat(P[1]), gxh, __ffma2_rn(splat(P[5]), gyh, __ffma2_rn(splat(P[9]), gzh, g[1])));
    g[2] = __ffma2_rn(splat(P[2]), gxh, __ffma2_rn(splat(P[6]), gyh, __ffma2_rn(splat(P[10]), gzh, g[2])));
    const float2 over = __fadd2_rn(s, splat(-delta));
    gd = __ffma2_rn(make_float2(in0 ? 0.f : over.x, in1 ? 0.f : over.y), splat(gj), gd);
}

struct BwArgs {
    const float *x3d, *x2d, *w2d, *cam, *lb, *ub, *delta;
    const float *poses_a, *grad_a;      // (B, PA, D), (B, PA)
    const float *poses_b, *grad_b;      // [opt] (B, PB, D), (B, PB)
    float *gx3d, *gx2d, *gw2d, *gdelta;
    int B, N, PA, PB;
    float z_min;
};

template <int DOF>
__global__ void __launch_bounds__(NT, 4) cost_backward_kernel(const BwArgs a) {
    EPNP_DYN_SMEM(float, bw_smem, 16);
    float* Pm = bw_smem;                                 // [tile][12]
    float* gs = bw_smem + BW_POSE_TILE * 12;             // [tile]
    float* red = gs + BW_POSE_TILE;                      // 2 * NW * 32
    constexpr int PD = Dim<DOF>::POSE;
    const int tid = threadIdx.x;
    const int P_total = a.PA + a.PB;
    for (int obj = blockIdx.x; obj < a.B; obj += gridDim.x) {
        KArgs ka{};
        ka.cam = a.cam; ka.lb = a.lb; ka.ub = a.ub; ka.p.z_min = a.z_min;
        const Cam cam = load_cam(ka, obj);
        const float delta = __ldg(a.delta + obj);
        float2 gd2 = make_float2(0.f, 0.f);
        for (int base = 0; base < a.N; base += NT * BW_PPT) {
            // BW_PPT = 4 correspondences per thread = 2 packed pairs: pair p holds points base + (2p)*NT + tid (.x)
            // and base + (2p+1)*NT + tid (.y); out-of-range slots get zero weights (exactly zero contribution)
            constexpr int NP = BW_PPT / 2;
            float2 X[NP], Y[NP], Z[NP], nu[NP], nv[NP], wu[NP], wv[NP], g[NP][7];
#pragma unroll
            for (int k = 0; k < NP; ++k) {
                float v7[2][7];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int n = base + (2 * k + h) * NT + tid;
                    const bool ok = n < a.N;
                    const size_t q = (size_t)obj * a.N + (ok ? n : 0);
                    v7[h][0] = __ldg(a.x3d + q * 3); v7[h][1] = __ldg(a.x3d + q * 3 + 1); v7[h][2] = __ldg(a.x3d + q * 3 + 2);
                    v7[h][3] = -__ldg(a.x2d + q * 2); v7[h][4] = -__ldg(a.x2d + q * 2 + 1);
                    v7[h][5] = ok ? __ldg(a.w2d + q * 2) : 0.f; v7[h][6] = ok ? __ldg(a.w2d + q * 2 + 1) : 0.f;
                }
                X[k] = make_float2(v7[0][0], v7[1][0]); Y[k] = make_float2(v7[0][1], v7[1][1]); Z[k] = make_float2(v7[0][2], v7[1][2]);
                nu[k] = make_float2(v7[0][3], v7[1][3]); nv[k] = make_float2(v7[0][4], v7[1][4]);
                wu[k] = make_float2(v7[0][5], v7[1][5]); wv[k] = make_float2(v7[0][6], v7[1][6]);
#pragma unroll
                for (int c = 0; c < 7; ++c) g[k][c] = make_float2(0.f, 0.f);
            }
            for (int p0 = 0; p0 < P_total; p0 += BW_POSE_TILE) {
                const int np = min(BW_POSE_TILE, P_total - p0);
                __syncthreads();                          // previous tile fully consumed
                for (int j = tid; j < np; j += NT) {
                    const int pi = p0 + j;
                    const bool in_a = pi < a.PA;
                    const float* src = in_a ? a.poses_a + ((size_t)obj * a.PA + pi) * PD
                                            : a.poses_b + ((size_t)obj * a.PB + (pi - a.PA)) * PD;
                    float pose[PD], R[9], Pj[12];
#pragma unroll
                    for (int c = 0; c < PD; ++c) pose[c] = __ldg(src + c);
                    pose_to_rot<DOF>(pose, R);
                    make_proj(cam.k, R, pose, Pj);
#pragma unroll
                    for (int c = 0; c < 12; ++c) Pm[j * 12 + c] = Pj[c];
                    gs[j] = in_a ? __ldg(a.grad_a + (size_t)obj * a.PA + pi) : __ldg(a.grad_b + (size_t)obj * a.PB + (pi - a.PA));
                }
                __syncthreads();
                for (int j = 0; j < np; ++j) {
                    const float4 r0 = reinterpret_cast<const float4*>(Pm)[3 * j];
                    const float4 r1 = reinterpret_cast<const float4*>(Pm)[3 * j + 1];
                    const float4 r2 = reinterpret_cast<const float4*>(Pm)[3 * j + 2];
                    const float Pj[12] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w};
                    const float gj = gs[j];
#pragma unroll
                    for (int k = 0; k < NP; ++k) {
                        if (cam.bounded) pair_cost_backward<true>(Pj, cam, delta, gj, X[k], Y[k], Z[k], nu[k], nv[k], wu[k], wv[k], g[k], gd2);
                        else pair_cost_backward<false>(Pj, cam, delta, gj, X[k], Y[k], Z[k], nu[k], nv[k], wu[k], wv[k], g[k], gd2);
                    }
                }
            }
#pragma unroll
            for (int k = 0; k < NP; ++k) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int n = base + (2 * k + h) * NT + tid;
                    if (n < a.N) {
                        const size_t q = (size_t)obj * a.N + n;
                        auto pick = [&](int c) { return h == 0 ? g[k][c].x : g[k][c].y; };
                        if (a.gx3d) { a.gx3d[q * 3] = pick(0); a.gx3d[q * 3 + 1] = pick(1); a.gx3d[q * 3 + 2] = pick(2); }
                        if (a.gx2d) { a.gx2d[q * 2] = pick(3); a.gx2d[q * 2 + 1] = pick(4); }
                        if (a.gw2d) { a.gw2d[q * 2] = pick(5); a.gw2d[q * 2 + 1] = pick(6); }
                    }
                }
            }
        }
        const float gdelta = gd2.x + gd2.y;
        // padded (n >= N) lanes carry zero weights: their residual is 0 -> inlier -> no delta contribution
        float gd[1] = {gdelta};
        __syncthreads();
        block_sum<1>(gd, red, 0);
        if (tid == 0 && a.gdelta) a.gdelta[obj] = gd[0];
    }
}

// AdaptiveHuberPnPCost.set_param: delta = mean(w2d) * sqrt(var_x + var_y) * relative_delta
__global__ void __launch_bounds__(NT) adaptive_delta_kernel(const float* x2d, const float* w2d, float rel,
                                                          float* delta, int N) {
    __shared__ float red[2 * NW * 32];
    const int obj = blockIdx.x;
    const float2* x = reinterpret_cast<const float2*>(x2d) + (size_t)obj * N;
    const float2* w = reinterpret_cast<const float2*>(w2d) + (size_t)obj * N;
    float s[3] = {0.f, 0.f, 0.f};
    for (int n = threadIdx.x; n < N; n += NT) {
        const float2 a = x[n], b = w[n];
        s[0] += a.x; s[1] += a.y; s[2] += b.x + b.y;
    }
    block_sum<3>(s, red, 0);
    const float mx = s[0] / N, my = s[1] / N, mw = s[2] / (2.f * N);
    float v[2] = {0.f, 0.f};
    for (int n = threadIdx.x; n < N; n += NT) {
        const float2 a = x[n];
        v[0] = fmaf(a.x - mx, a.x - mx, v[0]); v[1] = fmaf(a.y - my, a.y - my, v[1]);
    }
    block_sum<2>(v, red, 1);
    if (threadIdx.x == 0) delta[obj] = mw * sqrtf((v[0] + v[1]) / (float)(N - 1)) * rel;
}

// Epilogue on the AMIS outputs (the step after the path; SURVEY.md section 8 row f4).  One CTA per object reads the
// object's M log-weights (and, for the score, the x / z components of its M pose samples) once and writes
//   lse[b]      = logsumexp_m logw[b, m]                        (Monte-Carlo pose loss: loss_pred)
//   loss[b]     = cost_target[b] + lse[b], NaN -> 0              (the per-object loss before its mean)
//   weights     = softmax_m logw[b, :]                           (Det: pose_sample_logweights.softmax(dim=0))
//   score_te[b] = sum_m weights[m] * clamp((2.5 - log2 |(x,z)_m - (x,z)_opt|) / 4, 0, 1)   (Det 'te' MC score)
// with torch's conventions at the infinities (all -inf -> lse -inf, any NaN -> NaN).
template <int PD>
__global__ void __launch_bounds__(NT) mc_epilogue_kernel(const float* logw, const float* samples, const float* pose_opt,
                                                       const float* cost_target, float* lse_out, float* loss_out,
                                                       float* weights, float* score_out, int M) {
    __shared__ float red[2 * NW * 32];
    const int obj = blockIdx.x, tid = threadIdx.x;
    const float* l = logw + (size_t)obj * M;
    float mx = -CUDART_INF_F;
    bool any_nan = false;
    for (int m = tid; m < M; m += NT) { const float v = __ldg(l + m); mx = fmaxf(mx, v); any_nan |= (v != v); }
    mx = block_max(mx, red, 0);
    const float ref = (fabsf(mx) == CUDART_INF_F) ? 0.f : mx;          // torch.logsumexp: an infinite max is not subtracted
    const bool want_score = samples != nullptr && pose_opt != nullptr && score_out != nullptr;
    float ox = 0.f, oz = 0.f;
    if (want_score) { ox = __ldg(pose_opt + (size_t)obj * PD); oz = __ldg(pose_opt + (size_t)obj * PD + 2); }
    float acc[3] = {0.f, 0.f, any_nan ? 1.f : 0.f};                    // sum e, sum e * score, NaN seen
    for (int m = tid; m < M; m += NT) {
        const float e = expf(__ldg(l + m) - ref);
        acc[0] += e;
        if (want_score) {
            const float* sp = samples + ((size_t)obj * M + m) * PD;
            const float dx = __ldg(sp) - ox, dz = __ldg(sp + 2) - oz;
            const float dev = sqrtf(fmaf(dx, dx, dz * dz));
            const float sc = fminf(fmaxf((2.5f - log2f(dev)) * 0.25f, 0.f), 1.f);
            acc[1] = fmaf(e, sc, acc[1]);
        }
    }
    block_sum<3>(acc, red, 1);
    const float nan_in = acc[2] > 0.f ? CUDART_NAN_F : 0.f;            // fmaxf drops NaNs: put them back
    const float lse = logf(acc[0]) + ref + nan_in;
    const float inv = (mx == CUDART_INF_F) ? CUDART_NAN_F : 1.0f / acc[0];   // softmax: inf - inf poisons the whole object
    if (tid == 0) {
        if (lse_out) lse_out[obj] = lse;
        if (loss_out) {
            const float v = (cost_target ? __ldg(cost_target + obj) : 0.f) + lse;
            loss_out[obj] = (v != v) ? 0.f : v;
        }
        if (want_score) score_out[obj] = acc[1] * inv + nan_in;
    }
    if (weights) {
        float* w = weights + (size_t)obj * M;
        for (int m = tid; m < M; m += NT) w[m] = expf(__ldg(l + m) - ref) * inv;
    }
}

// Backward of lse (and of the NaN -> 0 mask): grad_logw[b, m] = g[b] * exp(logw[b, m] - lse[b]); g[b] == 0 gives exact zeros
// (masked objects have lse = NaN).
__global__ void __launch_bounds__(NT) mc_lse_backward_kernel(const float* logw, const float* lse, const float* g,
                                                           float* grad_logw, int M) {
    const int obj = blockIdx.x;
    const float gb = __ldg(g + obj), ls = __ldg(lse + obj);
    const float* l = logw + (size_t)obj * M;
    float* o = grad_logw + (size_t)obj * M;
    for (int m = threadIdx.x; m < M; m += NT) o[m] = (gb == 0.f) ? 0.f : gb * expf(__ldg(l + m) - ls);
}
// ------------------------------------------------------------------------------------------------
// Host side
int cuda_fail(cudaError_t e) { g_last_cuda_error = (int)e; return EPNP_ERR_CUDA; }

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

int check_common(const KArgs& a) {
    if (!a.x3d || !a.x2d || !a.w2d || !a.cam || !a.delta) return EPNP_ERR_BAD_ARG;
    if ((a.lb == nullptr) != (a.ub == nullptr)) return EPNP_ERR_BAD_ARG;
    if (a.B < 0 || a.N <= 0) return EPNP_ERR_BAD_ARG;
    if (a.p.dof != 4 && a.p.dof != 6) return EPNP_ERR_BAD_ARG;
    return EPNP_OK;
}

int device_sms(int* sms) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return cuda_fail(e);
    e = cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

bool tma_ok(const KArgs& a) { return (a.N % 4 == 0) && aligned16(a.x3d) && aligned16(a.x2d) && aligned16(a.w2d); }

// One CTA of NT threads per object (grid = B): the hardware scheduler hands CTAs to SMs as slots free up, the CTAs'
// serial and parallel phases de-synchronise and there is no lock-step tail (measured 5 % faster than a persistent grid).
template <int T = NT, class Kern, class... Extra>
int launch_cta_per_object(Kern kern, KArgs& a, int smem_bytes, cudaStream_t stream, Extra... extra) {
    if (a.B == 0) return EPNP_OK;
    if ((size_t)smem_bytes > SMEM_LIMIT) return EPNP_ERR_TOO_MANY_POINTS;
    a.use_tma = tma_ok(a);
    int rc = device_sms(&a.num_sms);
    if (rc != EPNP_OK) return rc;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
    if (e != cudaSuccess) return cuda_fail(e);
    // several resident CTAs need (nearly) the whole 228 KB of the SM as shared memory: ask for the full carve-out
    e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (e != cudaSuccess) return cuda_fail(e);
    EPNP_LAUNCH(kern, a.B, T, smem_bytes, stream, a, extra...);
    e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

// LM / GN solve: one CTA of WARPS warps per object (one warp unless the point set is long).  Outputs: a.pose_opt,
// a.pose_cov [opt] (stride a.cov_stride), a.cost [opt], a.pose_plus [opt], a.cost_init [opt].
template <int DOF, bool STAGED, int WARPS>
int launch_lm_as(KArgs& a, cudaStream_t stream) {
    const int smem_bytes = lm_smem_bytes<DOF, WARPS>(a.N, STAGED);
    cudaError_t e;
    if (STAGED) {
        e = cudaFuncSetAttribute(lm_warp_kernel<DOF, STAGED, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess) return cuda_fail(e);
        e = cudaFuncSetAttribute(lm_warp_kernel<DOF, STAGED, WARPS>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e != cudaSuccess) return cuda_fail(e);
    }
    EPNP_LAUNCH((lm_warp_kernel<DOF, STAGED, WARPS>), a.B, 32 * WARPS, smem_bytes, stream, a);
    e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

// Warps per object: a function of N ONLY, so that an object's result does not depend on how large a batch (or which
// shard of it) it is solved in -- the summation order of the 28 sums changes with the warp count.  Dense coordinate maps
// (N >= 2048: 16+ points per lane even with 8 warps) get 8 warps, everything else one.
int lm_warps_per_object(int N) { return N >= 2048 ? 8 : 1; }

template <int DOF>
int launch_lm(KArgs& a, cudaStream_t stream) {
    if (a.B == 0) return EPNP_OK;
    a.use_tma = tma_ok(a);
    int rc = device_sms(&a.num_sms);
    if (rc != EPNP_OK) return rc;
    const bool staged = a.N <= LM_STAGE_MAX_N;
    const int w = lm_warps_per_object(a.N);
    if (staged) {
        switch (w) {
            case 1: return launch_lm_as<DOF, true, 1>(a, stream);
            default: return launch_lm_as<DOF, true, 8>(a, stream);
        }
    }
    switch (w) {
        case 1: return launch_lm_as<DOF, false, 1>(a, stream);
        default: return launch_lm_as<DOF, false, 8>(a, stream);
    }
}

inline bool amis_dense(int N) { return N >= AMIS_DENSE_MIN_N; }
template <int DOF> int amis_smem_bytes(int N, int M) {
    return amis_dense(N) ? plan_amis<DOF, AMIS_T_DENSE>(N, M).total_bytes : plan_amis<DOF, NT>(N, M).total_bytes;
}

template <int DOF>
int launch_amis(KArgs& a, const PushArgs* push, cudaStream_t stream) {
    const int smem_bytes = amis_smem_bytes<DOF>(a.N, a.p.mc_samples);
    const PushArgs none{};
    if (amis_dense(a.N))
        return launch_cta_per_object<AMIS_T_DENSE>(amis_kernel<DOF, AMIS_T_DENSE>, a, smem_bytes, stream, push ? *push : none);
    return launch_cta_per_object<NT>(amis_kernel<DOF, NT>, a, smem_bytes, stream, push ? *push : none);
}

unsigned long long* g_prof_buffer = nullptr;     // set by epnp_debug_set_phase_buffer (profiling build)

// Objects the device works on at once in the AMIS kernel: SMs x resident CTAs per SM.  Used by the host-buffer entry
// point to cut the batch at whole waves.  0 when it cannot be determined.
template <int T, class Kern>
int resident_objects(Kern kern, int smem_bytes) {
    int sms = 0, occ = 0;
    if ((size_t)smem_bytes > SMEM_LIMIT) return 0;
    if (device_sms(&sms) != EPNP_OK) return 0;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes) != cudaSuccess) return 0;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100) != cudaSuccess) return 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, T, smem_bytes) != cudaSuccess) return 0;
    return sms * occ;
}

int check_amis_params(const Params& p) {
    if (p.mc_iter <= 0 || p.mc_iter > MAX_ITER || p.mc_samples <= 0 || p.mc_samples % p.mc_iter != 0) return EPNP_ERR_BAD_ARG;
    if (p.acg_mle_iter < 0) return EPNP_ERR_BAD_ARG;
    return EPNP_OK;
}

// LM kernel, then AMIS kernel, on `stream`.  The covariance travels through a.pose_cov (caller's buffer) or, when the
// caller did not ask for it, through the first dof^2 floats of each object's -- not yet written -- sample rows.
int run_lm_amis(KArgs& a, const PushArgs* push, cudaStream_t stream) {
    const int dof = a.p.dof, D = dof == 6 ? 7 : 4;
    if (a.pose_cov) a.cov_stride = dof * dof;
    else {
        if (a.p.mc_samples * D < dof * dof) return EPNP_ERR_BAD_ARG;
        a.pose_cov = a.pose_samples;
        a.cov_stride = a.p.mc_samples * D;
    }
    if ((size_t)(dof == 6 ? amis_smem_bytes<6>(a.N, a.p.mc_samples) : amis_smem_bytes<4>(a.N, a.p.mc_samples)) > SMEM_LIMIT)
        return EPNP_ERR_TOO_MANY_POINTS;        // before anything is launched
    int rc = dof == 6 ? launch_lm<6>(a, stream) : launch_lm<4>(a, stream);
    if (rc != EPNP_OK) return rc;
    a.pose_opt_in = a.pose_opt;
    a.pose_cov_in = a.pose_cov;
    return dof == 6 ? launch_amis<6>(a, push, stream) : launch_amis<4>(a, push, stream);
}

}  // namespace

// ================================================================================================
extern "C" {

#ifdef EPNP_PHASE_TIMERS
// profiling build only (not declared in the public header): device buffer of PH_COUNT uint64 counters
void epnp_debug_set_phase_buffer(unsigned long long* dev_buf) { g_prof_buffer = dev_buf; }
#endif

int epnp_abi_version(void) { return EPNP_ABI_VERSION; }

int epnp_last_cuda_error(void) { return g_last_cuda_error; }

const char* epnp_error_string(int code) {
    switch (code) {
        case EPNP_OK: return "ok";
        case EPNP_ERR_BAD_ARG: return "bad argument";
        case EPNP_ERR_TOO_MANY_POINTS: return "correspondence set (and sample buffers) exceed 227 KB of shared memory";
        case EPNP_ERR_UNSUPPORTED: return "combination not supported by this build";
        case EPNP_ERR_CUDA: return "CUDA runtime error (see epnp_last_cuda_error)";
        case EPNP_ERR_NO_DEVICE: return "no CUDA device";
        default: return "unknown error";
    }
}

void epnp_default_params(EpnpParams* p, int dof) {
    p->dof = dof; p->lm_iter = 10; p->fast_mode = 0; p->z_min = 0.1f;
    p->min_lm_diagonal = 1e-6f; p->max_lm_diagonal = 1e32f; p->min_relative_decrease = 1e-3f;
    p->initial_radius = 30.0f; p->max_radius = 1e16f; p->eps = 1e-5f; p->huber_eps = 1e-10f;
    p->mc_samples = 512; p->mc_iter = 4; p->amis_eps = 1e-5f; p->acg_mle_iter = 3; p->acg_dispersion = 1e-3f;
}

int epnp_max_points(int dof, int mc_samples, int mc_iter) {
    (void)mc_iter;
    const bool amis = mc_samples > 0;
    int lo = 0, hi = 1 << 16;
    while (lo + 4 <= hi) {                   // largest multiple of 4 that fits
        const int mid = ((lo + hi) / 2) / 4 * 4;
        if (mid == lo) break;
        int bytes;
        if (amis) bytes = (dof == 6) ? amis_smem_bytes<6>(mid, mc_samples) : amis_smem_bytes<4>(mid, mc_samples);
        else bytes = (dof == 6) ? plan_obj<6>(mid).total_bytes : plan_obj<4>(mid).total_bytes;
        if ((size_t)bytes <= SMEM_LIMIT) lo = mid; else hi = mid;
    }
    return lo;
}

int epnp_adaptive_delta_f32(const float* x2d, const float* w2d, float relative_delta, float* delta, int B, int N,
                            void* stream) {
    if (!x2d || !w2d || !delta || B < 0 || N <= 0) return EPNP_ERR_BAD_ARG;
    if (B == 0) return EPNP_OK;
    EPNP_LAUNCH(adaptive_delta_kernel, B, NT, 0, (cudaStream_t)stream, x2d, w2d, relative_delta, delta, N);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

int epnp_mc_epilogue_f32(const float* logw, const float* pose_samples, const float* pose_opt, const float* cost_target,
                         float* lse, float* loss, float* weights, float* score_te, int B, int M, int dof, void* stream) {
    if (!logw || B < 0 || M <= 0 || (dof != 4 && dof != 6)) return EPNP_ERR_BAD_ARG;
    if (!lse && !loss && !weights && !score_te) return EPNP_ERR_BAD_ARG;
    if (score_te && (!pose_samples || !pose_opt)) return EPNP_ERR_BAD_ARG;
    if (B == 0) return EPNP_OK;
    if (dof == 6)
        EPNP_LAUNCH(mc_epilogue_kernel<7>, B, NT, 0, (cudaStream_t)stream, logw, pose_samples, pose_opt, cost_target, lse, loss,
                    weights, score_te, M);
    else
        EPNP_LAUNCH(mc_epilogue_kernel<4>, B, NT, 0, (cudaStream_t)stream, logw, pose_samples, pose_opt, cost_target, lse, loss,
                    weights, score_te, M);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

int epnp_mc_lse_backward_f32(const float* logw, const float* lse, const float* grad_lse, float* grad_logw, int B, int M,
                             void* stream) {
    if (!logw || !lse || !grad_lse || !grad_logw || B < 0 || M <= 0) return EPNP_ERR_BAD_ARG;
    if (B == 0) return EPNP_OK;
    EPNP_LAUNCH(mc_lse_backward_kernel, B, NT, 0, (cudaStream_t)stream, logw, lse, grad_lse, grad_logw, M);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

int epnp_evaluate_cost_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                           const float* lb, const float* ub, const float* delta, const float* poses, float* cost,
                           int S, int B, int N, int dof, float z_min, void* stream) {
    KArgs a{};
    a.x3d = x3d; a.x2d = x2d; a.w2d = w2d; a.cam = cam_mats; a.lb = lb; a.ub = ub; a.delta = delta;
    a.poses = poses; a.cost_out = cost; a.S_eval = S; a.B = B; a.N = N;
    epnp_default_params(&a.p, dof);
    a.p.z_min = z_min;
    int rc = check_common(a);
    if (rc != EPNP_OK) return rc;
    if (!poses || !cost || S < 0) return EPNP_ERR_BAD_ARG;
    if (S == 0) return EPNP_OK;
    if (dof == 6) return launch_cta_per_object(cost_kernel<6>, a, plan_obj<6>(N).total_bytes, (cudaStream_t)stream);
    return launch_cta_per_object(cost_kernel<4>, a, plan_obj<4>(N).total_bytes, (cudaStream_t)stream);
}

int epnp_evaluate_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                      const float* lb, const float* ub, const float* delta, const float* pose,
                      float* residual, float* jac, float* cost, int clip_jac,
                      int B, int N, int dof, float z_min, float huber_eps, void* stream) {
    KArgs a{};
    a.x3d = x3d; a.x2d = x2d; a.w2d = w2d; a.cam = cam_mats; a.lb = lb; a.ub = ub; a.delta = delta;
    a.poses = pose; a.B = B; a.N = N;
    epnp_default_params(&a.p, dof);
    a.p.z_min = z_min;
    int rc = check_common(a);
    if (rc != EPNP_OK) return rc;
    if (!pose) return EPNP_ERR_BAD_ARG;
    if (B == 0) return EPNP_OK;
    if (dof == 6) EPNP_LAUNCH(evaluate_full_kernel<6>, B, NT, 0, (cudaStream_t)stream, a, residual, jac, cost, clip_jac, huber_eps);
    else EPNP_LAUNCH(evaluate_full_kernel<4>, B, NT, 0, (cudaStream_t)stream, a, residual, jac, cost, clip_jac, huber_eps);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

int epnp_lm_solve_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                      const float* lb, const float* ub, const float* delta, const float* pose_init,
                      float* pose_opt, float* pose_cov, float* cost, float* pose_opt_plus, float* cost_init,
                      int B, int N, const EpnpParams* p, void* stream) {
    if (!p) return EPNP_ERR_BAD_ARG;
    KArgs a{};
    a.x3d = x3d; a.x2d = x2d; a.w2d = w2d; a.cam = cam_mats; a.lb = lb; a.ub = ub; a.delta = delta;
    a.pose_init = pose_init; a.pose_opt = pose_opt; a.pose_cov = pose_cov; a.cost = cost;
    a.pose_plus = pose_opt_plus; a.cost_init = cost_init; a.B = B; a.N = N; a.p = *p;
    int rc = check_common(a);
    if (rc != EPNP_OK) return rc;
    if (!pose_init || !pose_opt || p->lm_iter < 0) return EPNP_ERR_BAD_ARG;
    a.cov_stride = p->dof * p->dof;
    return p->dof == 6 ? launch_lm<6>(a, (cudaStream_t)stream) : launch_lm<4>(a, (cudaStream_t)stream);
}

int epnp_gn_plus_backward_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                              const float* lb, const float* ub, const float* delta, const float* pose,
                              const float* grad_pose_plus, float* grad_x3d, float* grad_x2d, float* grad_w2d,
                              float* grad_delta, int B, int N, int dof, float z_min, float eps, float huber_eps,
                              void* stream) {
    GnBwArgs g{};
    KArgs& a = g.k;
    a.x3d = x3d; a.x2d = x2d; a.w2d = w2d; a.cam = cam_mats; a.lb = lb; a.ub = ub; a.delta = delta;
    a.poses = pose; a.B = B; a.N = N;
    epnp_default_params(&a.p, dof);
    a.p.z_min = z_min; a.p.eps = eps; a.p.huber_eps = huber_eps;
    g.gplus = grad_pose_plus; g.gx3d = grad_x3d; g.gx2d = grad_x2d; g.gw2d = grad_w2d; g.gdelta = grad_delta;
    int rc = check_common(a);
    if (rc != EPNP_OK) return rc;
    if (!pose || !grad_pose_plus) return EPNP_ERR_BAD_ARG;
    if (B == 0) return EPNP_OK;
    const int smem_bytes = (dof == 6) ? plan_obj<6>(N).total_bytes : plan_obj<4>(N).total_bytes;
    if ((size_t)smem_bytes > SMEM_LIMIT) return EPNP_ERR_TOO_MANY_POINTS;
    a.use_tma = tma_ok(a);
    rc = device_sms(&a.num_sms);
    if (rc != EPNP_OK) return rc;
    cudaError_t e;
    if (dof == 6) {
        e = cudaFuncSetAttribute(gn_plus_backward_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess) return cuda_fail(e);
        EPNP_LAUNCH(gn_plus_backward_kernel<6>, B, NT, smem_bytes, (cudaStream_t)stream, g);
    } else {
        e = cudaFuncSetAttribute(gn_plus_backward_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess) return cuda_fail(e);
        EPNP_LAUNCH(gn_plus_backward_kernel<4>, B, NT, smem_bytes, (cudaStream_t)stream, g);
    }
    e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

int epnp_rslm_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                  const float* lb, const float* ub, const float* delta, const int* inds, const float* start,
                  float* pose_best, float* cost_best, float* pose_all, float* cost_all,
                  int P, int n, int B, int N, const EpnpParams* p, void* stream) {
    if (!p) return EPNP_ERR_BAD_ARG;
    RslmArgs r{};
    KArgs& a = r.k;
    a.x3d = x3d; a.x2d = x2d; a.w2d = w2d; a.cam = cam_mats; a.lb = lb; a.ub = ub; a.delta = delta;
    a.B = B; a.N = N; a.p = *p;
    r.inds = inds; r.start = start; r.pose_best = pose_best; r.cost_best = cost_best;
    r.pose_all = pose_all; r.cost_all = cost_all; r.P = P; r.n = n;
    int rc = check_common(a);
    if (rc != EPNP_OK) return rc;
    if (!inds || !start || !pose_best || !cost_best || P <= 0 || n <= 0 || p->lm_iter < 0) return EPNP_ERR_BAD_ARG;
    if (B == 0) return EPNP_OK;
    const int smem_bytes = (p->dof == 6) ? plan_obj<6>(N).total_bytes : plan_obj<4>(N).total_bytes;
    if ((size_t)smem_bytes > SMEM_LIMIT) return EPNP_ERR_TOO_MANY_POINTS;
    a.use_tma = tma_ok(a);
    rc = device_sms(&a.num_sms);
    if (rc != EPNP_OK) return rc;
    cudaError_t e;
    if (p->dof == 6) {
        e = cudaFuncSetAttribute(rslm_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess) return cuda_fail(e);
        EPNP_LAUNCH(rslm_kernel<6>, B, NT, smem_bytes, (cudaStream_t)stream, r);
    } else {
        e = cudaFuncSetAttribute(rslm_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes);
        if (e != cudaSuccess) return cuda_fail(e);
        EPNP_LAUNCH(rslm_kernel<4>, B, NT, smem_bytes, (cudaStream_t)stream, r);
    }
    e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

int epnp_rslm_draw_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats, const float* t_init,
                       uint64_t seed, uint32_t obj_offset, int* inds, float* start, float* t_out,
                       int P, int n, int B, int N, int dof, float eps, void* stream) {
    if (!w2d || !inds || !start || (dof != 4 && dof != 6) || P <= 0 || n <= 0 || B < 0 || N <= 0 || n > N)
        return EPNP_ERR_BAD_ARG;
    if (!t_init && (!x3d || !x2d || !cam_mats)) return EPNP_ERR_BAD_ARG;
    if (B == 0) return EPNP_OK;
    const size_t smem = (size_t)((N + 3) & ~3) * sizeof(float) + (size_t)n * NT * (sizeof(float) + sizeof(int));
    if (smem + 2048 > SMEM_LIMIT) return EPNP_ERR_TOO_MANY_POINTS;
    RslmDrawArgs r{x3d, x2d, w2d, cam_mats, t_init, inds, start, t_out, seed, obj_offset, P, n, B, N, eps};
    cudaError_t e;
    if (dof == 6) {
        e = cudaFuncSetAttribute(rslm_draw_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e);
        EPNP_LAUNCH(rslm_draw_kernel<6>, B, NT, smem, (cudaStream_t)stream, r);
    } else {
        e = cudaFuncSetAttribute(rslm_draw_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return cuda_fail(e);
        EPNP_LAUNCH(rslm_draw_kernel<4>, B, NT, smem, (cudaStream_t)stream, r);
    }
    e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

int epnp_epnp_init_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                       float conf_quantile, float* pose, int* n_used, int B, int N, void* stream) {
    if (!x3d || !x2d || !w2d || !cam_mats || !pose || B < 0 || N <= 0) return EPNP_ERR_BAD_ARG;
    if (!(conf_quantile >= 0.0f && conf_quantile <= 1.0f)) return EPNP_ERR_BAD_ARG;
    if (N > EPNP_INIT_MAX_N) return EPNP_ERR_TOO_MANY_POINTS;
    // at least N - ceil(q (N - 1)) points are >= the quantile (the virtual index as numpy computes it, in fp32)
    const float h = conf_quantile * (float)(N - 1);
    if (N - (int)ceilf(h) < 4) return EPNP_ERR_BAD_ARG;
    if (B == 0) return EPNP_OK;
    const size_t smem = (size_t)N * sizeof(float);
    const EpnpInitArgs r{x3d, x2d, w2d, cam_mats, conf_quantile, pose, n_used, N};
    cudaError_t e = cudaFuncSetAttribute(epnp_init_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_fail(e);
    EPNP_LAUNCH(epnp_init_kernel, B, NT, smem, (cudaStream_t)stream, r);
    e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

int epnp_amis_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                  const float* lb, const float* ub, const float* delta, const float* pose_opt, const float* pose_cov,
                  const float* noise_normal, const float* noise_chi2, const float* noise_rot,
                  uint64_t seed, uint32_t obj_offset, float* pose_samples, float* logw, float* proposals,
                  int B, int N, const EpnpParams* p, void* stream) {
    if (!p) return EPNP_ERR_BAD_ARG;
    KArgs a{};
    a.x3d = x3d; a.x2d = x2d; a.w2d = w2d; a.cam = cam_mats; a.lb = lb; a.ub = ub; a.delta = delta;
    a.pose_opt_in = pose_opt; a.pose_cov_in = pose_cov;
    a.noise_n3 = noise_normal; a.noise_chi2 = noise_chi2; a.noise_rot = noise_rot;
    a.seed = seed; a.obj_offset = obj_offset;
    a.pose_samples = pose_samples; a.logw = logw; a.proposals = proposals; a.B = B; a.N = N; a.p = *p;
    a.prof = g_prof_buffer;
    int rc = check_common(a);
    if (rc != EPNP_OK) return rc;
    rc = check_amis_params(*p);
    if (rc != EPNP_OK) return rc;
    if (!pose_opt || !pose_cov || !pose_samples || !logw) return EPNP_ERR_BAD_ARG;
    const bool any = noise_normal || noise_chi2 || noise_rot, all = noise_normal && noise_chi2 && noise_rot;
    if (any && !all) return EPNP_ERR_BAD_ARG;
    a.cov_stride = p->dof * p->dof;
    return p->dof == 6 ? launch_amis<6>(a, nullptr, (cudaStream_t)stream) : launch_amis<4>(a, nullptr, (cudaStream_t)stream);
}

int epnp_lm_amis_fused_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                           const float* lb, const float* ub, const float* delta, const float* pose_init,
                           const float* noise_normal, const float* noise_chi2, const float* noise_rot,
                           uint64_t seed, uint32_t obj_offset,
                           float* pose_opt, float* pose_cov, float* cost, float* pose_opt_plus, float* cost_init,
                           float* pose_samples, float* logw, float* proposals,
                           int B, int N, const EpnpParams* p, void* stream) {
    if (!p) return EPNP_ERR_BAD_ARG;
    KArgs a{};
    a.x3d = x3d; a.x2d = x2d; a.w2d = w2d; a.cam = cam_mats; a.lb = lb; a.ub = ub; a.delta = delta;
    a.pose_init = pose_init;
    a.noise_n3 = noise_normal; a.noise_chi2 = noise_chi2; a.noise_rot = noise_rot;
    a.seed = seed; a.obj_offset = obj_offset;
    a.pose_opt = pose_opt; a.pose_cov = pose_cov; a.cost = cost; a.pose_plus = pose_opt_plus; a.cost_init = cost_init;
    a.pose_samples = pose_samples; a.logw = logw; a.proposals = proposals; a.B = B; a.N = N; a.p = *p;
    a.prof = g_prof_buffer;
    int rc = check_common(a);
    if (rc != EPNP_OK) return rc;
    rc = check_amis_params(*p);
    if (rc != EPNP_OK) return rc;
    if (!pose_init || !pose_opt || !pose_samples || !logw || p->lm_iter < 0) return EPNP_ERR_BAD_ARG;
    const bool any = noise_normal || noise_chi2 || noise_rot, all = noise_normal && noise_chi2 && noise_rot;
    if (any && !all) return EPNP_ERR_BAD_ARG;
    return run_lm_amis(a, nullptr, (cudaStream_t)stream);
}

int epnp_lm_amis_fused_push_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                                const float* lb, const float* ub, const float* delta, const float* pose_init,
                                uint64_t seed, uint32_t obj_offset,
                                float* pose_opt, float* pose_cov, float* cost, float* pose_samples, float* logw,
                                float* const* peer_logw, float* const* peer_pose, int n_peers,
                                int B, int N, const EpnpParams* p, void* stream) {
    if (!p) return EPNP_ERR_BAD_ARG;
    if (n_peers < 0 || n_peers > EPNP_MAX_PEERS || (n_peers > 0 && (!peer_logw || !peer_pose))) return EPNP_ERR_BAD_ARG;
    KArgs a{};
    a.x3d = x3d; a.x2d = x2d; a.w2d = w2d; a.cam = cam_mats; a.lb = lb; a.ub = ub; a.delta = delta;
    a.pose_init = pose_init;
    a.seed = seed; a.obj_offset = obj_offset;
    a.pose_opt = pose_opt; a.pose_cov = pose_cov; a.cost = cost;
    a.pose_samples = pose_samples; a.logw = logw; a.B = B; a.N = N; a.p = *p;
    a.prof = g_prof_buffer;
    int rc = check_common(a);
    if (rc != EPNP_OK) return rc;
    rc = check_amis_params(*p);
    if (rc != EPNP_OK) return rc;
    if (!pose_init || !pose_opt || !pose_samples || !logw || p->lm_iter < 0) return EPNP_ERR_BAD_ARG;
    PushArgs push{peer_logw, peer_pose, n_peers};
    return run_lm_amis(a, &push, (cudaStream_t)stream);
}

int epnp_cost_backward_f32(const float* x3d, const float* x2d, const float* w2d, const float* cam_mats,
                           const float* lb, const float* ub, const float* delta,
                           const float* poses_a, const float* grad_a, int PA,
                           const float* poses_b, const float* grad_b, int PB,
                           float* grad_x3d, float* grad_x2d, float* grad_w2d, float* grad_delta,
                           int B, int N, int dof, float z_min, void* stream) {
    if (!x3d || !x2d || !w2d || !cam_mats || !delta) return EPNP_ERR_BAD_ARG;
    if ((lb == nullptr) != (ub == nullptr)) return EPNP_ERR_BAD_ARG;
    if (B < 0 || N <= 0 || PA < 0 || PB < 0 || (dof != 4 && dof != 6)) return EPNP_ERR_BAD_ARG;
    if ((PA > 0 && (!poses_a || !grad_a)) || (PB > 0 && (!poses_b || !grad_b))) return EPNP_ERR_BAD_ARG;
    if (B == 0) return EPNP_OK;
    BwArgs a{};
    a.x3d = x3d; a.x2d = x2d; a.w2d = w2d; a.cam = cam_mats; a.lb = lb; a.ub = ub; a.delta = delta;
    a.poses_a = poses_a; a.grad_a = grad_a; a.poses_b = poses_b; a.grad_b = grad_b; a.PA = PA; a.PB = PB;
    a.gx3d = grad_x3d; a.gx2d = grad_x2d; a.gw2d = grad_w2d; a.gdelta = grad_delta;
    a.B = B; a.N = N; a.z_min = z_min;
    const int smem = (BW_POSE_TILE * 13 + 2 * NW * 32) * 4;
    cudaError_t e;
    int dev = 0, sms = 0;
    if ((e = cudaGetDevice(&dev)) != cudaSuccess) return cuda_fail(e);
    if ((e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess) return cuda_fail(e);
    const int grid = B < sms * 4 ? B : sms * 4;
    if (dof == 6) {
        if ((e = cudaFuncSetAttribute(cost_backward_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess) return cuda_fail(e);
        EPNP_LAUNCH(cost_backward_kernel<6>, grid, NT, smem, (cudaStream_t)stream, a);
    } else {
        if ((e = cudaFuncSetAttribute(cost_backward_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)) != cudaSuccess) return cuda_fail(e);
        EPNP_LAUNCH(cost_backward_kernel<4>, grid, NT, smem, (cudaStream_t)stream, a);
    }
    e = cudaGetLastError();
    return e == cudaSuccess ? EPNP_OK : cuda_fail(e);
}

// ---- host-buffer entry point: chunked H2D -> fused kernel -> D2H on two internal streams
static size_t align256(size_t x) { return (x + 255) / 256 * 256; }

struct WsLayout {
    size_t x3d, x2d, w2d, cam, lb, ub, delta, pose_init, pose_opt, pose_cov, cost, samples, logw, total;
};

static WsLayout ws_layout(int B, int N, const EpnpParams* p) {
    const size_t D = (p->dof == 6) ? 7 : 4, dof = p->dof, M = p->mc_samples;
    WsLayout w; size_t o = 0;
    w.x3d = o; o += align256((size_t)B * N * 3 * 4);
    w.x2d = o; o += align256((size_t)B * N * 2 * 4);
    w.w2d = o; o += align256((size_t)B * N * 2 * 4);
    w.cam = o; o += align256((size_t)B * 9 * 4);
    w.lb = o; o += align256((size_t)B * 2 * 4);
    w.ub = o; o += align256((size_t)B * 2 * 4);
    w.delta = o; o += align256((size_t)B * 4);
    w.pose_init = o; o += align256((size_t)B * D * 4);
    w.pose_opt = o; o += align256((size_t)B * D * 4);
    w.pose_cov = o; o += align256((size_t)B * dof * dof * 4);
    w.cost = o; o += align256((size_t)B * 4);
    w.samples = o; o += align256((size_t)B * M * D * 4);
    w.logw = o; o += align256((size_t)B * M * 4);
    w.total = o;
    return w;
}

size_t epnp_fused_workspace_bytes(int B, int N, const EpnpParams* p) {
    if (!p || B < 0 || N <= 0) return 0;
    return ws_layout(B, N, p).total;
}

// Helper streams of the host-buffer entry point: one copy-in, two compute, one copy-out stream per host
// thread, created on first use and kept for the life of the thread (the only resource the library owns;
// creating and destroying four streams per call costs more than a whole chunk of work).
struct HostPipe {
    cudaStream_t in = nullptr, k[2] = {nullptr, nullptr}, out = nullptr;
    int device = -1;
    cudaError_t ensure() {
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        if (dev == device && in) return cudaSuccess;
        if (in) { cudaStreamDestroy(in); cudaStreamDestroy(k[0]); cudaStreamDestroy(k[1]); cudaStreamDestroy(out); in = nullptr; }
        if ((e = cudaStreamCreateWithFlags(&in, cudaStreamNonBlocking)) != cudaSuccess) return e;
        if ((e = cudaStreamCreateWithFlags(&k[0], cudaStreamNonBlocking)) != cudaSuccess) return e;
        if ((e = cudaStreamCreateWithFlags(&k[1], cudaStreamNonBlocking)) != cudaSuccess) return e;
        if ((e = cudaStreamCreateWithFlags(&out, cudaStreamNonBlocking)) != cudaSuccess) return e;
        device = dev;
        return cudaSuccess;
    }
};
static thread_local HostPipe g_pipe;

int epnp_lm_amis_fused_host_f32(const float* x3d_host, const float* x2d_host, const float* w2d_host,
                                const float* cam_mats_host, const float* lb_host, const float* ub_host,
                                const float* delta_host, const float* pose_init_host,
                                uint64_t seed, uint32_t obj_offset,
                                float* pose_opt_host, float* pose_cov_host, float* cost_host,
                                float* pose_samples_host, float* logw_host,
                                void* workspace, size_t workspace_bytes, int n_chunks,
                                int B, int N, const EpnpParams* p, void* stream_) {
    if (!p || !workspace || !x3d_host || !x2d_host || !w2d_host || !cam_mats_host || !delta_host || !pose_init_host ||
        !pose_opt_host || !logw_host)
        return EPNP_ERR_BAD_ARG;
    if ((lb_host == nullptr) != (ub_host == nullptr)) return EPNP_ERR_BAD_ARG;
    if (B < 0 || N <= 0) return EPNP_ERR_BAD_ARG;
    if (B == 0) return EPNP_OK;
    const WsLayout w = ws_layout(B, N, p);
    if (workspace_bytes < w.total) return EPNP_ERR_BAD_ARG;
    // n_chunks = 0: cut the batch at whole waves of resident CTAs (a chunk of 1.7 waves costs 2), as few waves per chunk
    // as the 64-chunk limit allows; n_chunks >= 1: that many equal chunks
    int chunk_objects = 0;
    if (n_chunks == 0) {
        if (check_amis_params(*p) != EPNP_OK) return EPNP_ERR_BAD_ARG;
        const int wave = (p->dof == 6)
            ? (amis_dense(N) ? resident_objects<AMIS_T_DENSE>(amis_kernel<6, AMIS_T_DENSE>, amis_smem_bytes<6>(N, p->mc_samples))
                             : resident_objects<NT>(amis_kernel<6, NT>, amis_smem_bytes<6>(N, p->mc_samples)))
            : (amis_dense(N) ? resident_objects<AMIS_T_DENSE>(amis_kernel<4, AMIS_T_DENSE>, amis_smem_bytes<4>(N, p->mc_samples))
                             : resident_objects<NT>(amis_kernel<4, NT>, amis_smem_bytes<4>(N, p->mc_samples)));
        if (wave > 0) {
            const int waves_per_chunk = (B + 64 * wave - 1) / (64 * wave);
            chunk_objects = wave * waves_per_chunk;
            n_chunks = (B + chunk_objects - 1) / chunk_objects;
        }
    }
    if (n_chunks < 1) n_chunks = 1;
    if (n_chunks > B) n_chunks = B;
    if (n_chunks > 64) n_chunks = 64;
    cudaStream_t stream = (cudaStream_t)stream_;
    char* ws = (char*)workspace;
    const size_t D = (p->dof == 6) ? 7 : 4, dof = p->dof, M = p->mc_samples;
    // Three-stage pipeline over object chunks: copy-in stream -> {compute 0, compute 1} -> copy-out stream, chained
    // by per-chunk events, so all H2D copies run back to back on one DMA engine, all D2H copies on the other, and
    // the solve of chunk c overlaps both (and the tail of chunk c-1 on the other compute stream).
    cudaError_t e = cudaSuccess;
    int rc = EPNP_OK;
    cudaEvent_t fork = nullptr, ev_in[64], ev_k[64], done[3] = {nullptr, nullptr, nullptr};
    for (int i = 0; i < 64; ++i) { ev_in[i] = nullptr; ev_k[i] = nullptr; }
#define EPNP_TRY(x) do { e = (x); if (e != cudaSuccess) { rc = cuda_fail(e); goto done; } } while (0)
    EPNP_TRY(g_pipe.ensure());
    EPNP_TRY(cudaEventCreateWithFlags(&fork, cudaEventDisableTiming));
    EPNP_TRY(cudaEventRecord(fork, stream));
    EPNP_TRY(cudaStreamWaitEvent(g_pipe.in, fork, 0));
    EPNP_TRY(cudaStreamWaitEvent(g_pipe.k[0], fork, 0));
    EPNP_TRY(cudaStreamWaitEvent(g_pipe.k[1], fork, 0));
    EPNP_TRY(cudaStreamWaitEvent(g_pipe.out, fork, 0));
    for (int c = 0; c < n_chunks; ++c) {
        const int b0 = chunk_objects ? c * chunk_objects : (int)((long long)B * c / n_chunks);
        const int b1 = chunk_objects ? (b0 + chunk_objects < B ? b0 + chunk_objects : B) : (int)((long long)B * (c + 1) / n_chunks);
        const int nb = b1 - b0;
        if (nb <= 0) continue;
        cudaStream_t sk = g_pipe.k[c & 1];
#define H2D(field, host, per) EPNP_TRY(cudaMemcpyAsync(ws + w.field + (size_t)b0 * (per) * 4, (host) + (size_t)b0 * (per), (size_t)nb * (per) * 4, cudaMemcpyHostToDevice, g_pipe.in))
#define D2H(field, host, per) EPNP_TRY(cudaMemcpyAsync((host) + (size_t)b0 * (per), ws + w.field + (size_t)b0 * (per) * 4, (size_t)nb * (per) * 4, cudaMemcpyDeviceToHost, g_pipe.out))
        H2D(x3d, x3d_host, (size_t)N * 3); H2D(x2d, x2d_host, (size_t)N * 2); H2D(w2d, w2d_host, (size_t)N * 2);
        H2D(cam, cam_mats_host, 9); H2D(delta, delta_host, 1); H2D(pose_init, pose_init_host, D);
        if (lb_host) { H2D(lb, lb_host, 2); H2D(ub, ub_host, 2); }
        EPNP_TRY(cudaEventCreateWithFlags(&ev_in[c], cudaEventDisableTiming));
        EPNP_TRY(cudaEventRecord(ev_in[c], g_pipe.in));
        EPNP_TRY(cudaStreamWaitEvent(sk, ev_in[c], 0));
        rc = epnp_lm_amis_fused_f32(
            (float*)(ws + w.x3d) + (size_t)b0 * N * 3, (float*)(ws + w.x2d) + (size_t)b0 * N * 2,
            (float*)(ws + w.w2d) + (size_t)b0 * N * 2, (float*)(ws + w.cam) + (size_t)b0 * 9,
            lb_host ? (float*)(ws + w.lb) + (size_t)b0 * 2 : nullptr, lb_host ? (float*)(ws + w.ub) + (size_t)b0 * 2 : nullptr,
            (float*)(ws + w.delta) + b0, (float*)(ws + w.pose_init) + (size_t)b0 * D,
            nullptr, nullptr, nullptr, seed, obj_offset + (uint32_t)b0,
            (float*)(ws + w.pose_opt) + (size_t)b0 * D, (float*)(ws + w.pose_cov) + (size_t)b0 * dof * dof,
            (float*)(ws + w.cost) + b0, nullptr, nullptr,
            (float*)(ws + w.samples) + (size_t)b0 * M * D, (float*)(ws + w.logw) + (size_t)b0 * M, nullptr,
            nb, N, p, sk);
        if (rc != EPNP_OK) goto done;
        EPNP_TRY(cudaEventCreateWithFlags(&ev_k[c], cudaEventDisableTiming));
        EPNP_TRY(cudaEventRecord(ev_k[c], sk));
        EPNP_TRY(cudaStreamWaitEvent(g_pipe.out, ev_k[c], 0));
        D2H(pose_opt, pose_opt_host, D); D2H(logw, logw_host, M);
        if (pose_cov_host) D2H(pose_cov, pose_cov_host, dof * dof);
        if (cost_host) D2H(cost, cost_host, 1);
        if (pose_samples_host) D2H(samples, pose_samples_host, M * D);
#undef H2D
#undef D2H
    }
    {   // join: the caller's stream waits for everything the helpers were given
        cudaStream_t all[3] = {g_pipe.out, g_pipe.k[0], g_pipe.k[1]};
        for (int i = 0; i < 3; ++i) {
            EPNP_TRY(cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming));
            EPNP_TRY(cudaEventRecord(done[i], all[i]));
            EPNP_TRY(cudaStreamWaitEvent(stream, done[i], 0));
        }
    }
done:
#undef EPNP_TRY
    // events are released once recorded work has drained (cudaEventDestroy defers)
    for (int i = 0; i < 64; ++i) { if (ev_in[i]) cudaEventDestroy(ev_in[i]); if (ev_k[i]) cudaEventDestroy(ev_k[i]); }
    for (int i = 0; i < 3; ++i) if (done[i]) cudaEventDestroy(done[i]);
    if (fork) cudaEventDestroy(fork);
    return rc;
}

}  // extern "C"
