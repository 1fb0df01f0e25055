"""Float64 restatement of the EPnP initialiser of the 6DoF evaluation flow (test infrastructure, not a product path).

The reference evaluation loop (EPro-PnP-6DoF/lib/test.py:176-194) keeps each object's correspondences whose confidence
mean(w2d, -1) is at or above the object's `conf_quantile` quantile (numpy, 'linear') and runs EPnP on them.  EPnP is
Lepetit, Moreno-Noguer, Fua, "EPnP: An Accurate O(n) Solution to the PnP Problem", IJCV 81(2), 2009; equation numbers
below are that paper's.  It works in pixels with the camera's fx, fy, cx, cy (eq. 7; no skew, no distortion), and the
reprojection error that picks among the three approximations is in pixels too.

    select(w2d, q)                -> boolean mask (B, N), count (B)
    epnp(x3d, x2d, K)             -> R (3, 3), t (3)    one object, float64
    epnp_pose_init(x3d, x2d, w2d, cam_mats, q) -> pose (B, 7) = x y z w i j k, w >= 0
"""
import numpy as np

# the ten products beta_a beta_b in the order of L's columns (eq. 13): b11 b12 b22 b13 b23 b33 b14 b24 b34 b44
_PAIRS = [(0, 0), (0, 1), (1, 1), (0, 2), (1, 2), (2, 2), (0, 3), (1, 3), (2, 3), (3, 3)]
_CP_PAIRS = [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]


def quantile_threshold(conf, q):
    """numpy.quantile(conf, q) of one fp32 vector ('linear'), as numpy evaluates it for a float32 array: the virtual
    index q (N - 1), its fraction and the interpolation are all fp32; a fraction >= 0.5 interpolates from above."""
    conf = np.asarray(conf, np.float32)
    n = conf.shape[0]
    h = np.float32(q) * np.float32(n - 1)
    lo = int(np.floor(h))
    hi = min(lo + 1, n - 1)
    g = np.float32(h - np.float32(lo))
    s = np.sort(conf)
    a, b = s[lo], s[hi]
    d = np.float32(b - a)
    return np.float32(b - d * (np.float32(1) - g)) if g >= 0.5 else np.float32(a + d * g)


def select(w2d, q):
    w2d = np.asarray(w2d, np.float32)
    conf = (np.float32(0.5) * (w2d[..., 0] + w2d[..., 1])).astype(np.float32)
    mask = np.stack([c >= quantile_threshold(c, q) for c in conf])
    return mask, mask.sum(1).astype(np.int32)


def _sym_eig_desc(a):
    w, v = np.linalg.eigh(a)
    order = np.argsort(w)[::-1]
    return w[order], v[:, order]


def principal_axes(S, eps=10 * np.finfo(np.float64).eps):
    """Eigen-decomposition of the 3 x 3 scatter S by one-sided (Hestenes) Jacobi on its rows: each pair of rows is
    rotated until orthogonal, by the rotation that leaves the larger norm in the lower index; V^T (started at I) takes
    the same rotations; then rows are ordered by decreasing norm.  -> eigenvalues (desc), axes as columns.

    The signs of the axes matter: EPnP's least-squares steps are not invariant to which side of the centroid a control
    point sits once the data are noisy.  This is the convention whose axes the reference flow's EPnP uses."""
    A = np.array(S, np.float64)
    n = A.shape[0]
    W = [A[i] @ A[i] for i in range(n)]
    for _ in range(30):
        changed = False
        for i in range(n - 1):
            for j in range(i + 1, n):
                a, b, p = W[i], W[j], A[i] @ A[j]
                if abs(p) <= eps * np.sqrt(a * b):
                    continue
                p *= 2.0
                beta = a - b
                gamma = np.hypot(p, beta)
                if beta < 0:
                    s = np.sqrt((gamma - beta) * 0.5 / gamma)
                    c = p / (gamma * s * 2)
                else:
                    c = np.sqrt((gamma + beta) / (gamma * 2))
                    s = p / (gamma * c * 2)
                A[i], A[j] = c * A[i] + s * A[j], -s * A[i] + c * A[j]
                W[i], W[j] = A[i] @ A[i], A[j] @ A[j]
                changed = True
        if not changed:
            break
    w = np.sqrt(np.array(W))
    for i in range(n - 1):              # selection sort by swaps, decreasing norm
        k = i + int(np.argmax(w[i:]))
        if k != i:
            w[[i, k]] = w[[k, i]]
            A[[i, k]] = A[[k, i]]
    return w, (A / w[:, None]).T


def _lstsq(a, b):
    return np.linalg.lstsq(a, b, rcond=None)[0]


def epnp(x3d, x2d, K):
    """One object: x3d (n, 3), x2d (n, 2) pixel coordinates, K (3, 3) -> R, t (float64)."""
    pw = np.asarray(x3d, np.float64)
    uv = np.asarray(x2d, np.float64)
    K = np.asarray(K, np.float64)
    n = pw.shape[0]
    fu, fv, uc, vc = K[0, 0], K[1, 1], K[0, 2], K[1, 2]
    # control points (section 3.1): centroid + principal directions scaled by sqrt(lambda / n)
    c0 = pw.mean(0)
    d = pw - c0
    lam, axes = principal_axes(d.T @ d)
    cws = np.stack([c0] + [c0 + np.sqrt(lam[i] / n) * axes[:, i] for i in range(3)])
    # barycentric coordinates (eq. 1-2)
    cc = (cws[1:] - c0).T
    alpha123 = d @ np.linalg.inv(cc).T
    alphas = np.concatenate([1.0 - alpha123.sum(1, keepdims=True), alpha123], 1)
    # M (eq. 7), M^T M and its null-space basis (eq. 8): the four eigenvectors of smallest eigenvalue
    M = np.zeros((2 * n, 12))
    for j in range(4):
        M[0::2, 3 * j] = alphas[:, j] * fu
        M[0::2, 3 * j + 2] = alphas[:, j] * (uc - uv[:, 0])
        M[1::2, 3 * j + 1] = alphas[:, j] * fv
        M[1::2, 3 * j + 2] = alphas[:, j] * (vc - uv[:, 1])
    _, ev = _sym_eig_desc(M.T @ M)
    v = [ev[:, 11 - i] for i in range(4)]
    # L (6 x 10) and rho (eq. 13): squared control-point distances, invariant to the camera frame
    rho = np.array([np.sum((cws[a] - cws[b]) ** 2) for a, b in _CP_PAIRS])
    dv = [[v[i][3 * a:3 * a + 3] - v[i][3 * b:3 * b + 3] for a, b in _CP_PAIRS] for i in range(4)]
    L = np.array([[(1.0 if i == j else 2.0) * dv[i][r] @ dv[j][r] for i, j in _PAIRS] for r in range(6)])

    def refine(betas):          # section 4.4: Gauss-Newton on sum (L b(beta) - rho)^2, five steps
        betas = betas.copy()
        for _ in range(5):
            bb = np.array([betas[i] * betas[j] for i, j in _PAIRS])
            res = rho - L @ bb
            J = np.zeros((6, 4))
            for c, (i, j) in enumerate(_PAIRS):
                J[:, i] += L[:, c] * betas[j]
                J[:, j] += L[:, c] * betas[i]
            betas = betas + _lstsq(J, res)
        return betas

    # the three approximations of section 4.3 (N = 1, 2, 3 via linearisation)
    b4 = _lstsq(L[:, [0, 1, 3, 6]], rho)
    if b4[0] < 0:
        be1 = np.array([np.sqrt(-b4[0]), -b4[1], -b4[2], -b4[3]])
        be1[1:] /= be1[0]
    else:
        be1 = np.array([np.sqrt(b4[0]), b4[1], b4[2], b4[3]])
        be1[1:] /= be1[0]

    def first_two(b):
        if b[0] < 0:
            b0, b1 = np.sqrt(-b[0]), (np.sqrt(-b[2]) if b[2] < 0 else 0.0)
        else:
            b0, b1 = np.sqrt(b[0]), (np.sqrt(b[2]) if b[2] > 0 else 0.0)
        if b[1] < 0:
            b0 = -b0
        return b0, b1

    b3 = _lstsq(L[:, [0, 1, 2]], rho)
    be2 = np.array([*first_two(b3), 0.0, 0.0])
    b5 = _lstsq(L[:, [0, 1, 2, 3, 4]], rho)
    p0, p1 = first_two(b5)
    be3 = np.array([p0, p1, b5[3] / p0, 0.0])

    def pose_of(betas):
        ccs = sum(betas[i] * v[i] for i in range(4)).reshape(4, 3)
        pcs = alphas @ ccs
        if pcs[0, 2] < 0:                    # the points must be in front of the camera
            ccs, pcs = -ccs, -pcs
        # absolute orientation (Procrustes) between pcs and pws
        pc0, pw0 = pcs.mean(0), pw.mean(0)
        abt = (pcs - pc0).T @ (pw - pw0)
        U, _, Vt = np.linalg.svd(abt)
        R = U @ Vt
        if np.linalg.det(R) < 0:
            R[2] = -R[2]
        t = pc0 - R @ pw0
        cam = pw @ R.T + t
        err = np.mean(np.hypot(uv[:, 0] - uc - fu * cam[:, 0] / cam[:, 2], uv[:, 1] - vc - fv * cam[:, 1] / cam[:, 2]))
        return R, t, err

    best = pose_of(refine(be1))
    for be in (be2, be3):
        cand = pose_of(refine(be))
        if cand[2] < best[2]:
            best = cand
    return best[0], best[1]


def mat_to_quat(R):
    """Rotation matrix -> unit quaternion (w, i, j, k) with w >= 0 (Shepperd's method)."""
    tr = np.trace(R)
    m = [tr, R[0, 0], R[1, 1], R[2, 2]]
    k = int(np.argmax(m))
    if k == 0:
        w = 0.5 * np.sqrt(1 + tr)
        q = np.array([w, (R[2, 1] - R[1, 2]) / (4 * w), (R[0, 2] - R[2, 0]) / (4 * w), (R[1, 0] - R[0, 1]) / (4 * w)])
    elif k == 1:
        x = 0.5 * np.sqrt(1 + 2 * R[0, 0] - tr)
        q = np.array([(R[2, 1] - R[1, 2]) / (4 * x), x, (R[0, 1] + R[1, 0]) / (4 * x), (R[0, 2] + R[2, 0]) / (4 * x)])
    elif k == 2:
        y = 0.5 * np.sqrt(1 + 2 * R[1, 1] - tr)
        q = np.array([(R[0, 2] - R[2, 0]) / (4 * y), (R[0, 1] + R[1, 0]) / (4 * y), y, (R[1, 2] + R[2, 1]) / (4 * y)])
    else:
        z = 0.5 * np.sqrt(1 + 2 * R[2, 2] - tr)
        q = np.array([(R[1, 0] - R[0, 1]) / (4 * z), (R[0, 2] + R[2, 0]) / (4 * z), (R[1, 2] + R[2, 1]) / (4 * z), z])
    q /= np.linalg.norm(q)
    return -q if q[0] < 0 else q


def epnp_pose_init(x3d, x2d, w2d, cam_mats, q=0.8):
    x3d, x2d, w2d = (np.asarray(t) for t in (x3d, x2d, w2d))
    B = x3d.shape[0]
    K = np.broadcast_to(np.asarray(cam_mats, np.float64), (B, 3, 3))
    mask, count = select(w2d, q)
    out = np.zeros((B, 7))
    for b in range(B):
        R, t = epnp(x3d[b][mask[b]], x2d[b][mask[b]], K[b])
        out[b, :3] = t
        out[b, 3:] = mat_to_quat(R)
    return out, mask, count
