// pnp_epnp.cuh -- EPnP initial pose per object for the 6DoF evaluation flow (included from pnp_kernels.cu).
//
// What EPro-PnP-6DoF/lib/test.py:176-194 does on the host with numpy + cv2.solvePnP(SOLVEPNP_EPNP), one CTA per object:
//   1. conf[i] = 0.5 (w2d[i,0] + w2d[i,1]); threshold = numpy.quantile(conf, q) ('linear', evaluated in fp32 as numpy
//      does for a float32 array: virtual index q (N - 1), fraction and interpolation in fp32, a fraction >= 0.5
//      interpolated from above).  The two order statistics come from a bitwise binary search over the conf values'
//      order-preserving uint32 keys in shared memory (32 block counts each): exact, ties included.  conf >= threshold
//      selects the points.
//   2. EPnP (Lepetit, Moreno-Noguer, Fua, IJCV 2009) on the selected points, in fp64 from the first sum on:
//      control points = centroid + principal axes scaled by sqrt(lambda / n) (section 3.1), barycentric alphas (eq. 1-2),
//      M^T M (eq. 7-8, in pixels with fx fy cx cy; no skew, no distortion) from 40 per-thread moments,
//      its four smallest eigenvectors (cyclic Jacobi), L (6 x 10) and rho (eq. 13), the three beta approximations of
//      section 4.3, each refined by five Gauss-Newton steps (section 4.4, Householder least squares), the sign that puts
//      the first selected point in front of the camera, R and t by Procrustes, and the reprojection error (pixels); the
//      first approximation is kept unless a later one has a strictly smaller error.
//   3. pose = x y z w i j k with w >= 0.
// Serial linear algebra runs on thread 0 from shared memory; the per-point passes are block-wide with fp64 moments
// reduced by warp shuffles (deterministic order), so a result does not depend on the batch it is solved in.
namespace {

constexpr int EPNP_INIT_MAX_N = 16384;      // 128 x 128 map; conf values are resident in shared memory (64 KB)

struct EpnpInitArgs {
    const float *x3d, *x2d, *w2d, *cam;     // (B, N, 3), (B, N, 2), (B, N, 2), (B, 3, 3)
    float q;
    float* pose;                            // (B, 7)
    int* n_used;                            // [opt] (B)
    int N;
};

__device__ __forceinline__ uint32_t epnp_key(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float epnp_unkey(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

__device__ __forceinline__ double epnp_shfl_xor_d(double v, int m) {
#if defined(EPNP_SIMT_EMUL)
    uint64_t u;
    std::memcpy(&u, &v, 8);
    const uint32_t lo = __float_as_uint(__shfl_xor_sync(0xffffffffu, __uint_as_float((uint32_t)u), m));
    const uint32_t hi = __float_as_uint(__shfl_xor_sync(0xffffffffu, __uint_as_float((uint32_t)(u >> 32)), m));
    u = ((uint64_t)hi << 32) | lo;
    double r;
    std::memcpy(&r, &u, 8);
    return r;
#else
    return __shfl_xor_sync(0xffffffffu, v, m);
#endif
}

// Block sum of K doubles (every thread gets the totals); red holds NW * K doubles.  Fixed summation order.
template <int K> __device__ __forceinline__ void epnp_block_sum_d(double (&v)[K], double* red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double x = v[k];
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) x += epnp_shfl_xor_d(x, m);
        v[k] = x;
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) red[w * K + k] = v[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double s = red[k];
        for (int o = 1; o < NW; ++o) s += red[o * K + k];
        v[k] = s;
    }
    __syncthreads();
}

// Block sum of an integer count (exact: counts <= EPNP_INIT_MAX_N < 2^24 travel as floats).
__device__ __forceinline__ int epnp_block_count(int c, float* red) {
    float x = (float)c;
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) x += __shfl_xor_sync(0xffffffffu, x, m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = x;
    __syncthreads();
    float s = 0.f;
    for (int o = 0; o < NW; ++o) s += red[o];
    __syncthreads();
    return (int)s;
}

__device__ __forceinline__ float epnp_block_min(float x, float* red) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) x = fminf(x, __shfl_xor_sync(0xffffffffu, x, m));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = x;
    __syncthreads();
    float s = red[0];
    for (int o = 1; o < NW; ++o) s = fminf(s, red[o]);
    __syncthreads();
    return s;
}

// k-th smallest (0-based) of the n conf values: the largest key v with #{key < v} <= k, built from the top bit down.
__device__ __forceinline__ float epnp_kth(const float* conf, int n, int k, float* red) {
    uint32_t ans = 0;
    for (int bit = 31; bit >= 0; --bit) {
        const uint32_t cand = ans | (1u << bit);
        int c = 0;
        for (int i = threadIdx.x; i < n; i += NT) c += epnp_key(conf[i]) < cand;
        if (epnp_block_count(c, red) <= k) ans = cand;
    }
    return epnp_unkey(ans);
}

// Products in fp32 without contraction into an FMA (numpy rounds every step).
__device__ __forceinline__ float epnp_mul_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    volatile float r = a * b;
    return r;
#endif
}

// numpy.quantile(conf, q) for a float32 vector ('linear').
__device__ __forceinline__ float epnp_quantile(const float* conf, int n, float q, float* red) {
    const float h = epnp_mul_rn(q, (float)(n - 1));
    const int lo = (int)floorf(h), hi = min(lo + 1, n - 1);
    const float g = h - (float)lo;
    const float a = epnp_kth(conf, n, lo, red);
    const float b = hi == lo ? a : epnp_kth(conf, n, hi, red);
    const float d = b - a;
    return g >= 0.5f ? b - epnp_mul_rn(d, 1.0f - g) : a + epnp_mul_rn(d, g);
}

// Cyclic Jacobi eigen-decomposition of a symmetric n x n matrix (row-major, overwritten: eigenvalues on the diagonal);
// V receives the eigenvectors as columns.
__device__ inline void epnp_jacobi(double* A, double* V, int n) {
    for (int i = 0; i < n * n; ++i) V[i] = 0.0;
    for (int i = 0; i < n; ++i) V[i * n + i] = 1.0;
    for (int sweep = 0; sweep < 50; ++sweep) {
        double off = 0.0, dia = 0.0;
        for (int p = 0; p < n; ++p) {
            dia += A[p * n + p] * A[p * n + p];
            for (int q = p + 1; q < n; ++q) off += A[p * n + q] * A[p * n + q];
        }
        if (!(off > 1e-60 * dia)) break;
        for (int p = 0; p < n; ++p)
            for (int q = p + 1; q < n; ++q) {
                const double apq = A[p * n + q];
                if (apq == 0.0) continue;
                const double theta = (A[q * n + q] - A[p * n + p]) / (2.0 * apq);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                A[p * n + p] -= t * apq;
                A[q * n + q] += t * apq;
                A[p * n + q] = A[q * n + p] = 0.0;
                for (int r = 0; r < n; ++r) {
                    if (r != p && r != q) {
                        const double arp = A[r * n + p], arq = A[r * n + q];
                        A[r * n + p] = A[p * n + r] = c * arp - s * arq;
                        A[r * n + q] = A[q * n + r] = s * arp + c * arq;
                    }
                    const double vrp = V[r * n + p], vrq = V[r * n + q];
                    V[r * n + p] = c * vrp - s * vrq;
                    V[r * n + q] = s * vrp + c * vrq;
                }
            }
    }
}

// Principal axes of the 3 x 3 scatter S (overwritten: row k = axis k, unit length; lam = eigenvalues, decreasing) by
// one-sided (Hestenes) Jacobi on the rows of S: a pair of rows is rotated until orthogonal, by the rotation that leaves
// the larger norm in the lower index; then rows are ordered by decreasing norm (selection sort by swaps).  The axes'
// signs matter -- once the data are noisy EPnP is not invariant to which side of the centroid a control point sits --
// and this convention's are the ones the reference flow's EPnP gets.
__device__ inline void epnp_principal_axes(double* S, double* lam) {
    double W[3];
    for (int i = 0; i < 3; ++i) W[i] = S[i * 3] * S[i * 3] + S[i * 3 + 1] * S[i * 3 + 1] + S[i * 3 + 2] * S[i * 3 + 2];
    const double eps = 10.0 * 2.220446049250313e-16;
    for (int sweep = 0; sweep < 30; ++sweep) {
        bool changed = false;
        for (int i = 0; i < 2; ++i)
            for (int j = i + 1; j < 3; ++j) {
                const double a = W[i], b = W[j];
                double p = S[i * 3] * S[j * 3] + S[i * 3 + 1] * S[j * 3 + 1] + S[i * 3 + 2] * S[j * 3 + 2];
                if (fabs(p) <= eps * sqrt(a * b)) continue;
                p *= 2.0;
                const double beta = a - b, gamma = hypot(p, beta);
                double c, s;
                if (beta < 0.0) { s = sqrt((gamma - beta) * 0.5 / gamma); c = p / (gamma * s * 2.0); }
                else { c = sqrt((gamma + beta) / (gamma * 2.0)); s = p / (gamma * c * 2.0); }
                for (int k = 0; k < 3; ++k) {
                    const double ri = S[i * 3 + k], rj = S[j * 3 + k];
                    S[i * 3 + k] = c * ri + s * rj;
                    S[j * 3 + k] = -s * ri + c * rj;
                }
                W[i] = S[i * 3] * S[i * 3] + S[i * 3 + 1] * S[i * 3 + 1] + S[i * 3 + 2] * S[i * 3 + 2];
                W[j] = S[j * 3] * S[j * 3] + S[j * 3 + 1] * S[j * 3 + 1] + S[j * 3 + 2] * S[j * 3 + 2];
                changed = true;
            }
        if (!changed) break;
    }
    for (int i = 0; i < 3; ++i) lam[i] = sqrt(W[i]);
    for (int i = 0; i < 2; ++i) {
        int k = i;
        for (int j = i + 1; j < 3; ++j)
            if (lam[j] > lam[k]) k = j;
        if (k != i) {
            double t = lam[i]; lam[i] = lam[k]; lam[k] = t;
            for (int c = 0; c < 3; ++c) { t = S[i * 3 + c]; S[i * 3 + c] = S[k * 3 + c]; S[k * 3 + c] = t; }
        }
    }
    for (int i = 0; i < 3; ++i)
        for (int c = 0; c < 3; ++c) S[i * 3 + c] /= lam[i];
}

// min || A x - b || for A (6 x nc), nc <= 5, by Householder QR (A and b are overwritten).
__device__ inline void epnp_lsq6(double* A, double* b, int nc, double* x) {
    for (int k = 0; k < nc; ++k) {
        double nrm = 0.0;
        for (int i = k; i < 6; ++i) nrm += A[i * nc + k] * A[i * nc + k];
        nrm = sqrt(nrm);
        if (nrm == 0.0) continue;
        const double alpha = A[k * nc + k] > 0.0 ? -nrm : nrm;
        double v[6];
        for (int i = 0; i < 6; ++i) v[i] = i < k ? 0.0 : A[i * nc + k];
        v[k] -= alpha;
        double vv = 0.0;
        for (int i = k; i < 6; ++i) vv += v[i] * v[i];
        if (vv == 0.0) continue;
        for (int j = k; j < nc; ++j) {
            double s = 0.0;
            for (int i = k; i < 6; ++i) s += v[i] * A[i * nc + j];
            s = 2.0 * s / vv;
            for (int i = k; i < 6; ++i) A[i * nc + j] -= s * v[i];
        }
        double s = 0.0;
        for (int i = k; i < 6; ++i) s += v[i] * b[i];
        s = 2.0 * s / vv;
        for (int i = k; i < 6; ++i) b[i] -= s * v[i];
    }
    for (int k = nc - 1; k >= 0; --k) {
        double s = b[k];
        for (int j = k + 1; j < nc; ++j) s -= A[k * nc + j] * x[j];
        x[k] = A[k * nc + k] != 0.0 ? s / A[k * nc + k] : 0.0;
    }
}

// the ten products beta_a beta_b in L's column order: b11 b12 b22 b13 b23 b33 b14 b24 b34 b44
__device__ __forceinline__ void epnp_pair(int c, int& i, int& j) {
    const int I[10] = {0, 0, 1, 0, 1, 2, 0, 1, 2, 3}, J[10] = {0, 1, 1, 2, 2, 2, 3, 3, 3, 3};
    i = I[c]; j = J[c];
}

// Five Gauss-Newton steps on sum_r (L_r . b(beta) - rho_r)^2 (section 4.4).
__device__ inline void epnp_refine(const double* L, const double* rho, double* beta) {
    for (int it = 0; it < 5; ++it) {
        double J[24], r[6], dx[4];
        for (int row = 0; row < 6; ++row) {
            double lb = 0.0;
            for (int k = 0; k < 4; ++k) J[row * 4 + k] = 0.0;
            for (int c = 0; c < 10; ++c) {
                int i, j;
                epnp_pair(c, i, j);
                const double l = L[row * 10 + c];
                lb += l * beta[i] * beta[j];
                J[row * 4 + i] += l * beta[j];
                J[row * 4 + j] += l * beta[i];
            }
            r[row] = rho[row] - lb;
        }
        epnp_lsq6(J, r, 4, dx);
        for (int k = 0; k < 4; ++k) beta[k] += dx[k];
    }
}

__device__ inline void epnp_cross(const double* a, const double* b, double* c) {
    c[0] = a[1] * b[2] - a[2] * b[1]; c[1] = a[2] * b[0] - a[0] * b[2]; c[2] = a[0] * b[1] - a[1] * b[0];
}

// R maximising trace(R^T abt) (abt = sum (pc - pc0)(pw - pw0)^T): R = U V^T of the SVD abt = U D V^T; an improper
// result has its third row negated.  V and D^2 from the eigen-decomposition of abt^T abt; u_k = abt v_k / d_k for the two
// largest, u_3 = +-(u_1 x u_2) with the sign of abt v_3.
__device__ inline void epnp_procrustes(const double* abt, double* R) {
    double S[9], V[9];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double s = 0.0;
            for (int k = 0; k < 3; ++k) s += abt[k * 3 + i] * abt[k * 3 + j];
            S[i * 3 + j] = s;
        }
    epnp_jacobi(S, V, 3);
    int o[3] = {0, 1, 2};
    for (int a = 0; a < 3; ++a)
        for (int b = a + 1; b < 3; ++b)
            if (S[o[b] * 4] > S[o[a] * 4]) { const int t = o[a]; o[a] = o[b]; o[b] = t; }
    double v[3][3], u[3][3];
    for (int k = 0; k < 3; ++k)
        for (int i = 0; i < 3; ++i) v[k][i] = V[i * 3 + o[k]];
    for (int k = 0; k < 3; ++k) {
        for (int i = 0; i < 3; ++i) u[k][i] = abt[i * 3] * v[k][0] + abt[i * 3 + 1] * v[k][1] + abt[i * 3 + 2] * v[k][2];
    }
    const double av2[3] = {u[2][0], u[2][1], u[2][2]};
    for (int k = 0; k < 2; ++k) {
        const double nn = sqrt(u[k][0] * u[k][0] + u[k][1] * u[k][1] + u[k][2] * u[k][2]);
        for (int i = 0; i < 3; ++i) u[k][i] /= nn;
    }
    epnp_cross(u[0], u[1], u[2]);
    if (u[2][0] * av2[0] + u[2][1] * av2[1] + u[2][2] * av2[2] < 0.0)
        for (int i = 0; i < 3; ++i) u[2][i] = -u[2][i];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) R[i * 3 + j] = u[0][i] * v[0][j] + u[1][i] * v[1][j] + u[2][i] * v[2][j];
    const double det = R[0] * (R[4] * R[8] - R[5] * R[7]) - R[1] * (R[3] * R[8] - R[5] * R[6]) +
                       R[2] * (R[3] * R[7] - R[4] * R[6]);
    if (det < 0.0)
        for (int j = 0; j < 3; ++j) R[6 + j] = -R[6 + j];
}

// Shared state of one object's solve (thread 0 writes, all read after a barrier).
struct EpnpShared {
    double c0[3], cinv[9], K[4];            // centroid, inverse of the control-point basis, fx fy cx cy
    double A[144], V[144];                  // M^T M, eigenvectors
    double Rt[3][12];                       // candidate R (9) | t (3)
    double mom[40];
    double S[9], D[3];                      // scatter sum d d^T and sum d of d = pw - c0
    float thr;
    int n, first;
};

// Thread 0: everything between the M^T M moments and the reprojection errors (kept out of line so that its registers
// do not weigh on the per-point loops).
__device__ __noinline__ void epnp_solve_serial(EpnpShared& sh, const float* x3, int i0, int n)
{
    const double* m = sh.mom;
    const double* c0 = sh.c0;
    const double* ci = sh.cinv;
    const double* S = sh.S;
    const double* Dsum = sh.D;
        double* A = sh.A;
        const double fu = sh.K[0], fv = sh.K[1];
        for (int i = 0; i < 144; ++i) A[i] = 0.0;
        int c = 0;
        for (int kk = 0; kk < 4; ++kk)
            for (int j = 0; j <= kk; ++j, ++c)
                for (int sw = 0; sw < (j == kk ? 1 : 2); ++sw) {
                    const int r = sw ? kk : j, s = sw ? j : kk;
                    A[(3 * r) * 12 + 3 * s] = fu * fu * m[4 * c];
                    A[(3 * r + 1) * 12 + 3 * s + 1] = fv * fv * m[4 * c];
                    A[(3 * r) * 12 + 3 * s + 2] = fu * m[4 * c + 1];
                    A[(3 * r + 2) * 12 + 3 * s] = fu * m[4 * c + 1];
                    A[(3 * r + 1) * 12 + 3 * s + 2] = fv * m[4 * c + 2];
                    A[(3 * r + 2) * 12 + 3 * s + 1] = fv * m[4 * c + 2];
                    A[(3 * r + 2) * 12 + 3 * s + 2] = m[4 * c + 3];
                }
        epnp_jacobi(A, sh.V, 12);
        // the four eigenvectors of smallest eigenvalue, smallest first (eq. 8)
        int ord[12];
        for (int i = 0; i < 12; ++i) ord[i] = i;
        for (int x = 1; x < 12; ++x) {
            const int t = ord[x];
            int y = x - 1;
            while (y >= 0 && A[ord[y] * 13] > A[t * 13]) { ord[y + 1] = ord[y]; --y; }
            ord[y + 1] = t;
        }
        double v[4][12];
        for (int e = 0; e < 4; ++e)
            for (int i = 0; i < 12; ++i) v[e][i] = sh.V[i * 12 + ord[e]];
        // control points in the world frame and rho = their squared distances; L (eq. 13)
        double cw[4][3];
        for (int i = 0; i < 3; ++i) cw[0][i] = c0[i];
        {
            // c_{k+1} - c0 are the columns of cinv^-1; recover them from the stored inverse
            const double* q = sh.cinv;
            double inv[9] = {q[4] * q[8] - q[5] * q[7], q[2] * q[7] - q[1] * q[8], q[1] * q[5] - q[2] * q[4],
                             q[5] * q[6] - q[3] * q[8], q[0] * q[8] - q[2] * q[6], q[2] * q[3] - q[0] * q[5],
                             q[3] * q[7] - q[4] * q[6], q[1] * q[6] - q[0] * q[7], q[0] * q[4] - q[1] * q[3]};
            const double idet = 1.0 / (q[0] * inv[0] + q[1] * inv[3] + q[2] * inv[6]);
            for (int k = 1; k < 4; ++k)
                for (int i = 0; i < 3; ++i) cw[k][i] = c0[i] + inv[i * 3 + k - 1] * idet;
        }
        const int PA[6] = {0, 0, 0, 1, 1, 2}, PB[6] = {1, 2, 3, 2, 3, 3};
        double rho[6], L[60];
        for (int r = 0; r < 6; ++r) {
            double s = 0.0;
            for (int i = 0; i < 3; ++i) { const double d = cw[PA[r]][i] - cw[PB[r]][i]; s += d * d; }
            rho[r] = s;
            double dv[4][3];
            for (int e = 0; e < 4; ++e)
                for (int i = 0; i < 3; ++i) dv[e][i] = v[e][3 * PA[r] + i] - v[e][3 * PB[r] + i];
            for (int c = 0; c < 10; ++c) {
                int i, j;
                epnp_pair(c, i, j);
                L[r * 10 + c] = (i == j ? 1.0 : 2.0) * (dv[i][0] * dv[j][0] + dv[i][1] * dv[j][1] + dv[i][2] * dv[j][2]);
            }
        }
        // the three approximations (section 4.3)
        double beta[3][4];
        {
            double Ls[30], r6[6], b[5];
            const int cols1[4] = {0, 1, 3, 6};
            for (int r = 0; r < 6; ++r) { for (int c = 0; c < 4; ++c) Ls[r * 4 + c] = L[r * 10 + cols1[c]]; r6[r] = rho[r]; }
            epnp_lsq6(Ls, r6, 4, b);
            const double s = b[0] < 0.0 ? -1.0 : 1.0;
            beta[0][0] = sqrt(s * b[0]);
            for (int k = 1; k < 4; ++k) beta[0][k] = s * b[k] / beta[0][0];
            for (int approx = 2; approx <= 3; ++approx) {
                const int nc = approx == 2 ? 3 : 5;
                for (int r = 0; r < 6; ++r) { for (int c = 0; c < nc; ++c) Ls[r * nc + c] = L[r * 10 + c]; r6[r] = rho[r]; }
                epnp_lsq6(Ls, r6, nc, b);
                double b0, b1;
                if (b[0] < 0.0) { b0 = sqrt(-b[0]); b1 = b[2] < 0.0 ? sqrt(-b[2]) : 0.0; }
                else { b0 = sqrt(b[0]); b1 = b[2] > 0.0 ? sqrt(b[2]) : 0.0; }
                if (b[1] < 0.0) b0 = -b0;
                double* be = beta[approx - 1];
                be[0] = b0; be[1] = b1; be[2] = approx == 3 ? b[3] / b0 : 0.0; be[3] = 0.0;
            }
        }
        // the first selected point's alphas (its camera depth fixes the sign)
        double af[4];
        {
            const double d0 = (double)__ldg(x3 + 3 * i0) - c0[0], d1 = (double)__ldg(x3 + 3 * i0 + 1) - c0[1],
                         d2 = (double)__ldg(x3 + 3 * i0 + 2) - c0[2];
            af[1] = ci[0] * d0 + ci[1] * d1 + ci[2] * d2;
            af[2] = ci[3] * d0 + ci[4] * d1 + ci[5] * d2;
            af[3] = ci[6] * d0 + ci[7] * d1 + ci[8] * d2;
            af[0] = 1.0 - af[1] - af[2] - af[3];
        }
        // sums over the points of alpha_j (Asum) and alpha_j d (Q_j) follow from S and D: alpha_{1..3} = cinv d
        double Asum[4], Q[4][3];
        for (int j = 1; j < 4; ++j) {
            Asum[j] = ci[3 * (j - 1)] * Dsum[0] + ci[3 * (j - 1) + 1] * Dsum[1] + ci[3 * (j - 1) + 2] * Dsum[2];
            for (int c = 0; c < 3; ++c)
                Q[j][c] = ci[3 * (j - 1)] * S[c] + ci[3 * (j - 1) + 1] * S[3 + c] + ci[3 * (j - 1) + 2] * S[6 + c];
        }
        Asum[0] = (double)n - Asum[1] - Asum[2] - Asum[3];
        for (int c = 0; c < 3; ++c) Q[0][c] = Dsum[c] - Q[1][c] - Q[2][c] - Q[3][c];
        for (int e = 0; e < 3; ++e) {
            epnp_refine(L, rho, beta[e]);
            double cc[4][3];
            for (int j = 0; j < 4; ++j)
                for (int i = 0; i < 3; ++i)
                    cc[j][i] = beta[e][0] * v[0][3 * j + i] + beta[e][1] * v[1][3 * j + i] + beta[e][2] * v[2][3 * j + i] +
                               beta[e][3] * v[3][3 * j + i];
            const double zf = af[0] * cc[0][2] + af[1] * cc[1][2] + af[2] * cc[2][2] + af[3] * cc[3][2];
            if (zf < 0.0)
                for (int j = 0; j < 4; ++j)
                    for (int i = 0; i < 3; ++i) cc[j][i] = -cc[j][i];
            double pc0[3], abt[9];
            for (int i = 0; i < 3; ++i)
                pc0[i] = (Asum[0] * cc[0][i] + Asum[1] * cc[1][i] + Asum[2] * cc[2][i] + Asum[3] * cc[3][i]) / n;
            for (int i = 0; i < 3; ++i)
                for (int k = 0; k < 3; ++k)
                    abt[i * 3 + k] = cc[0][i] * Q[0][k] + cc[1][i] * Q[1][k] + cc[2][i] * Q[2][k] + cc[3][i] * Q[3][k] -
                                     pc0[i] * Dsum[k];
            double* R = sh.Rt[e];
            epnp_procrustes(abt, R);
            for (int i = 0; i < 3; ++i) {
                const double pw0 = c0[0] + Dsum[0] / n, pw1 = c0[1] + Dsum[1] / n, pw2 = c0[2] + Dsum[2] / n;
                R[9 + i] = pc0[i] - (R[i * 3] * pw0 + R[i * 3 + 1] * pw1 + R[i * 3 + 2] * pw2);
            }
        }
    }

__global__ void __launch_bounds__(NT) epnp_init_kernel(const EpnpInitArgs a) {
    // 128: the alignment the other kernels' first declaration of this extern array gives it (this one precedes them)
    EPNP_DYN_SMEM(unsigned char, smem_raw, 128);
    __shared__ EpnpShared sh;
    __shared__ double redd[NW * 40];
    __shared__ float redf[NW];
    float* conf = reinterpret_cast<float*>(smem_raw);
    const int tid = threadIdx.x, obj = blockIdx.x, N = a.N;
    const float* x3 = a.x3d + (size_t)obj * N * 3;
    const float* x2 = a.x2d + (size_t)obj * N * 2;
    for (int i = tid; i < N; i += NT) {
        const float2 w = *reinterpret_cast<const float2*>(a.w2d + ((size_t)obj * N + i) * 2);
        conf[i] = 0.5f * (w.x + w.y);
    }
    __syncthreads();
    const float thr = epnp_quantile(conf, N, a.q, redf);
    int cnt = 0;
    float first = (float)N;
    for (int i = tid; i < N; i += NT)
        if (conf[i] >= thr) { ++cnt; first = fminf(first, (float)i); }
    const int n = epnp_block_count(cnt, redf);
    const int i0 = (int)epnp_block_min(first, redf);
    if (tid == 0 && a.n_used) a.n_used[obj] = n;
    // centroid, then the scatter S = sum d d^T and D = sum d of d = pw - c0 (two passes, fp64)
    double s3[3] = {0.0, 0.0, 0.0};
    for (int i = tid; i < N; i += NT)
        if (conf[i] >= thr)
            for (int k = 0; k < 3; ++k) s3[k] += (double)__ldg(x3 + 3 * i + k);
    epnp_block_sum_d<3>(s3, redd);
    const double c0[3] = {s3[0] / n, s3[1] / n, s3[2] / n};
    double s9[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = tid; i < N; i += NT)
        if (conf[i] >= thr) {
            const double d0 = (double)__ldg(x3 + 3 * i) - c0[0], d1 = (double)__ldg(x3 + 3 * i + 1) - c0[1],
                         d2 = (double)__ldg(x3 + 3 * i + 2) - c0[2];
            s9[0] += d0 * d0; s9[1] += d0 * d1; s9[2] += d0 * d2; s9[3] += d1 * d1; s9[4] += d1 * d2; s9[5] += d2 * d2;
            s9[6] += d0; s9[7] += d1; s9[8] += d2;
        }
    epnp_block_sum_d<9>(s9, redd);
    const double S[9] = {s9[0], s9[1], s9[2], s9[1], s9[3], s9[4], s9[2], s9[4], s9[5]}, Dsum[3] = {s9[6], s9[7], s9[8]};
    if (tid == 0) {
        // control points (section 3.1): c_{k+1} = c0 + sqrt(lambda_k / n) e_k, principal axes by decreasing variance
        double P[9], lam[3];
        for (int i = 0; i < 9; ++i) P[i] = S[i];
        epnp_principal_axes(P, lam);
        double C[9];                                     // columns: c_{k+1} - c0
        for (int k = 0; k < 3; ++k) {
            const double sc = sqrt(lam[k] / n);
            for (int i = 0; i < 3; ++i) C[i * 3 + k] = sc * P[k * 3 + i];
        }
        const double inv[9] = {C[4] * C[8] - C[5] * C[7], C[2] * C[7] - C[1] * C[8], C[1] * C[5] - C[2] * C[4],
                               C[5] * C[6] - C[3] * C[8], C[0] * C[8] - C[2] * C[6], C[2] * C[3] - C[0] * C[5],
                               C[3] * C[7] - C[4] * C[6], C[1] * C[6] - C[0] * C[7], C[0] * C[4] - C[1] * C[3]};
        const double idet = 1.0 / (C[0] * inv[0] + C[1] * inv[3] + C[2] * inv[6]);
        for (int i = 0; i < 9; ++i) sh.cinv[i] = inv[i] * idet;
        for (int i = 0; i < 3; ++i) { sh.c0[i] = c0[i]; sh.D[i] = Dsum[i]; }
        for (int i = 0; i < 9; ++i) sh.S[i] = S[i];
        const float* k = a.cam + (size_t)obj * 9;
        sh.K[0] = __ldg(k); sh.K[1] = __ldg(k + 4); sh.K[2] = __ldg(k + 2); sh.K[3] = __ldg(k + 5);
    }
    __syncthreads();
    // M^T M moments (eq. 7): for each pair j <= k of control points sum a_j a_k {1, x, y, x^2 + y^2}
    double m[40];
#pragma unroll
    for (int c = 0; c < 40; ++c) m[c] = 0.0;
    const double fx = sh.K[0], fy = sh.K[1], cx = sh.K[2], cy = sh.K[3];
    const double* ci = sh.cinv;                          // broadcast shared loads: registers go to the 40 moments
    for (int i = tid; i < N; i += NT) {
        if (!(conf[i] >= thr)) continue;
        const double d0 = (double)__ldg(x3 + 3 * i) - sh.c0[0], d1 = (double)__ldg(x3 + 3 * i + 1) - sh.c0[1],
                     d2 = (double)__ldg(x3 + 3 * i + 2) - sh.c0[2];
        double al[4];
        al[1] = ci[0] * d0 + ci[1] * d1 + ci[2] * d2;
        al[2] = ci[3] * d0 + ci[4] * d1 + ci[5] * d2;
        al[3] = ci[6] * d0 + ci[7] * d1 + ci[8] * d2;
        al[0] = 1.0 - al[1] - al[2] - al[3];
        const double x = cx - (double)__ldg(x2 + 2 * i), y = cy - (double)__ldg(x2 + 2 * i + 1);
        const double r2 = x * x + y * y;
        int c = 0;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
#pragma unroll
            for (int j = 0; j <= kk; ++j, ++c) {
                const double p = al[j] * al[kk];
                m[4 * c] += p; m[4 * c + 1] += p * x; m[4 * c + 2] += p * y; m[4 * c + 3] += p * r2;
            }
    }
    epnp_block_sum_d<40>(m, redd);
    if (tid == 0) {
        for (int c = 0; c < 40; ++c) sh.mom[c] = m[c];
        epnp_solve_serial(sh, x3, i0, n);
    }
    __syncthreads();
    // reprojection error of the three candidates (pixels; summed, the comparison does not need the mean)
    double err[3] = {0.0, 0.0, 0.0};
    for (int i = tid; i < N; i += NT) {
        if (!(conf[i] >= thr)) continue;
        const double p0 = __ldg(x3 + 3 * i), p1 = __ldg(x3 + 3 * i + 1), p2 = __ldg(x3 + 3 * i + 2);
        const double u = __ldg(x2 + 2 * i), v = __ldg(x2 + 2 * i + 1);
#pragma unroll
        for (int e = 0; e < 3; ++e) {
            const double* R = sh.Rt[e];
            const double X = R[0] * p0 + R[1] * p1 + R[2] * p2 + R[9], Y = R[3] * p0 + R[4] * p1 + R[5] * p2 + R[10],
                         Z = R[6] * p0 + R[7] * p1 + R[8] * p2 + R[11];
            const double ex = u - cx - fx * X / Z, ey = v - cy - fy * Y / Z;
            err[e] += sqrt(ex * ex + ey * ey);
        }
    }
    epnp_block_sum_d<3>(err, redd);
    if (tid == 0) {
        int best = 0;
        if (err[1] < err[best]) best = 1;
        if (err[2] < err[best]) best = 2;
        const double* R = sh.Rt[best];
        // R -> unit quaternion (Shepperd), w >= 0
        const double tr = R[0] + R[4] + R[8];
        double q[4];
        if (tr >= R[0] && tr >= R[4] && tr >= R[8]) {
            const double w = 0.5 * sqrt(1.0 + tr), f = 0.25 / w;
            q[0] = w; q[1] = (R[7] - R[5]) * f; q[2] = (R[2] - R[6]) * f; q[3] = (R[3] - R[1]) * f;
        } else if (R[0] >= R[4] && R[0] >= R[8]) {
            const double x = 0.5 * sqrt(1.0 + 2.0 * R[0] - tr), f = 0.25 / x;
            q[0] = (R[7] - R[5]) * f; q[1] = x; q[2] = (R[1] + R[3]) * f; q[3] = (R[2] + R[6]) * f;
        } else if (R[4] >= R[8]) {
            const double y = 0.5 * sqrt(1.0 + 2.0 * R[4] - tr), f = 0.25 / y;
            q[0] = (R[2] - R[6]) * f; q[1] = (R[1] + R[3]) * f; q[2] = y; q[3] = (R[5] + R[7]) * f;
        } else {
            const double z = 0.5 * sqrt(1.0 + 2.0 * R[8] - tr), f = 0.25 / z;
            q[0] = (R[3] - R[1]) * f; q[1] = (R[2] + R[6]) * f; q[2] = (R[5] + R[7]) * f; q[3] = z;
        }
        double nq = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
        if (q[0] < 0.0) nq = -nq;
        float* out = a.pose + (size_t)obj * 7;
        out[0] = (float)R[9]; out[1] = (float)R[10]; out[2] = (float)R[11];
        for (int k = 0; k < 4; ++k) out[3 + k] = (float)(q[k] / nq);
    }
}

}  // namespace
