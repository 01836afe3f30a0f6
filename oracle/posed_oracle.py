"""CPU restatement of the posed-view evaluation (evaluations/posed_evaluation.py, include/spn_posed.h), numpy fp64, for
the tests: the reprojection chain of spn_posed_reproject in its operation order, visibility, brute-force
nearest-neighbour repeatability, match correctness, relative-pose error and AUC.

Every step is one numpy ufunc (a separately rounded IEEE operation, element by element) in the order the header
documents, so positions and flags equal the kernel's bit for bit.  Test infrastructure only.
"""
import numpy as np


def inverse3x3(m):
    """Adjugate / determinant of a 3x3 fp32 matrix in fp64, in the kernel's order -> (9,) float64."""
    a, b, c, d, e, f, g, h, i = (float(v) for v in np.asarray(m, np.float32).reshape(9))
    c00, c01, c02 = e * i - f * h, f * g - d * i, d * h - e * g
    det = (a * c00 + b * c01) + c * c02
    return np.array([c00 / det, (c * h - b * i) / det, (b * f - c * e) / det,
                     c01 / det, (a * i - c * g) / det, (c * d - a * f) / det,
                     c02 / det, (b * g - a * h) / det, (a * e - b * d) / det], np.float64)


def _row(m, k, x, y, z):
    return (m[3 * k] * x + m[3 * k + 1] * y) + m[3 * k + 2] * z


def reproject_points(rc, depth_src, depth_dst, K_src, R_src, t_src, K_dst, R_dst, t_dst, depth_tol):
    """Keypoints rc (n,2) int (row, col) of the source view into the destination view -> (proj (n,2) float64 with NaN
    where undefined, visible (n,) bool)."""
    rc = np.asarray(rc, np.int64).reshape(-1, 2)
    H, W = depth_src.shape
    n = len(rc)
    proj = np.full((n, 2), np.nan)
    vis = np.zeros(n, bool)
    inside = (rc[:, 0] >= 0) & (rc[:, 0] < H) & (rc[:, 1] >= 0) & (rc[:, 1] < W)
    if not inside.any():
        return proj, vis
    r, c = rc[inside, 0], rc[inside, 1]
    Ki, Rinv = inverse3x3(K_src), inverse3x3(R_dst)
    Ks = np.asarray(K_dst, np.float32).reshape(9).astype(np.float64)
    Rs = np.asarray(R_src, np.float32).reshape(9).astype(np.float64)
    ts = np.asarray(t_src, np.float32).reshape(3).astype(np.float64)
    td = np.asarray(t_dst, np.float32).reshape(3).astype(np.float64)
    d = np.asarray(depth_src, np.float32)[r, c].astype(np.float64)
    x, y = c.astype(np.float64), r.astype(np.float64)
    with np.errstate(all="ignore"):
        ray = [(Ki[3 * k] * x + Ki[3 * k + 1] * y) + Ki[3 * k + 2] for k in range(3)]
        nrm = np.sqrt((ray[0] * ray[0] + ray[1] * ray[1]) + ray[2] * ray[2])
        X = [(ray[k] / nrm) * d for k in range(3)]
        w = [(_row(Rs, k, *X) + ts[k]) - td[k] for k in range(3)]
        Y = [_row(Rinv, k, *w) for k in range(3)]
        p = [_row(Ks, k, *Y) for k in range(3)]
        row, col = p[1] / p[2], p[0] / p[2]
        ok = np.isfinite(row) & np.isfinite(col)
        row, col = np.where(ok, row, np.nan), np.where(ok, col, np.nan)
        v = np.isfinite(d) & (d > 0) & (Y[2] > 0) & (row >= 0) & (row <= H - 1) & (col >= 0) & (col <= W - 1)
        nr = np.where(v, np.floor(row + 0.5), 0).astype(np.int64)
        nc = np.where(v, np.floor(col + 0.5), 0).astype(np.int64)
        db = np.asarray(depth_dst, np.float32)[nr, nc].astype(np.float64)
        nY = np.sqrt((Y[0] * Y[0] + Y[1] * Y[1]) + Y[2] * Y[2])
        v &= np.isfinite(db) & (db > 0) & (np.abs(nY - db) <= depth_tol * db)
    proj[inside, 0], proj[inside, 1] = row, col
    vis[inside] = v
    return proj, vis


def posed_reproject(kp, kp_count, depth, K, R, t, pairs, depth_tol):
    """What spn_posed_reproject writes, for numpy inputs of its layout -> dict(proj, vis, set1, set2, set_count)."""
    kp, depth = np.asarray(kp), np.asarray(depth, np.float32)
    V, max_kp = kp.shape[:2]
    K, R, t = (np.asarray(x, np.float32).reshape(V, -1) for x in (K, R, t))
    P = len(pairs)
    out = {"proj": np.full((P, max_kp, 2), np.nan), "vis": np.zeros((P, 2, max_kp), np.int32),
           "set1": np.full((P, max_kp, 2), np.nan), "set2": np.full((P, max_kp, 2), np.nan),
           "set_count": np.zeros((P, 2), np.int32)}
    for q, (a, b) in enumerate(pairs):
        for direction, (s, d) in enumerate(((a, b), (b, a))):
            n = min(max(int(kp_count[s]), 0), max_kp)
            proj, vis = reproject_points(kp[s, :n], depth[s], depth[d], K[s], R[s], t[s], K[d], R[d], t[d], depth_tol)
            out["vis"][q, direction, :n] = vis
            pts = proj[vis] if direction == 0 else kp[s, :n][vis].astype(np.float64)
            out["set1" if direction == 0 else "set2"][q, :len(pts)] = pts
            out["set_count"][q, direction] = len(pts)
            if direction == 0:
                out["proj"][q, :n] = proj
    return out


def repeatability_counts(set1, n1, set2, n2, thresh):
    """Brute-force nearest neighbours per pair -> (P,4) {N1, N2, count1, count2}."""
    out = np.zeros((len(n1), 4), np.int64)
    for q in range(len(n1)):
        a, b = set1[q, :n1[q]], set2[q, :n2[q]]
        c1 = c2 = 0
        if len(a) and len(b):
            dist = np.sqrt(((a[:, None, :] - b[None, :, :]) ** 2).sum(-1))
            c1, c2 = int((dist.min(1) <= thresh).sum()), int((dist.min(0) <= thresh).sum())
        out[q] = (len(a), len(b), c1, c2)
    return out


def match_correct(proj, vis, kp_b, match, thresh):
    """Per query keypoint i with match[i] = j >= 0: vis[i] and |proj[i] - kp_b[j]| <= thresh -> (n_matches, n_correct)."""
    i = np.nonzero(match >= 0)[0]
    j = match[i]
    dy = proj[i, 0] - kp_b[j, 0].astype(np.float64)
    dx = proj[i, 1] - kp_b[j, 1].astype(np.float64)
    with np.errstate(invalid="ignore"):
        ok = (vis[i] != 0) & (np.sqrt(dy * dy + dx * dx) <= thresh)
    return len(i), int(ok.sum())


def relative_pose(R_a, t_a, R_b, t_b):
    """Ground-truth motion from camera a to camera b of camera-to-world poses: X_b = R_ab X_a + t_ab."""
    R_a, R_b = np.asarray(R_a, np.float64).reshape(3, 3), np.asarray(R_b, np.float64).reshape(3, 3)
    Rb_inv = np.linalg.inv(R_b)
    return Rb_inv @ R_a, Rb_inv @ (np.asarray(t_a, np.float64).reshape(3) - np.asarray(t_b, np.float64).reshape(3))


def pose_error(R_est, t_est, R_gt, t_gt):
    """(rotation error, translation direction error) in degrees."""
    cos = (np.trace(np.asarray(R_est).T @ R_gt) - 1.0) / 2.0
    err_r = np.degrees(np.arccos(np.clip(cos, -1.0, 1.0)))
    t_est, t_gt = np.asarray(t_est, np.float64).reshape(3), np.asarray(t_gt, np.float64).reshape(3)
    cos = t_est @ t_gt / (np.linalg.norm(t_est) * np.linalg.norm(t_gt))
    err_t = np.degrees(np.arccos(np.clip(cos, -1.0, 1.0)))
    return float(err_r), float(min(err_t, 180.0 - err_t))


def pose_auc(errors, thresholds):
    """Area under the recall-vs-error curve up to each threshold, over the threshold: the points (0, 0) and
    (e_k, k / n) for the sorted errors below the threshold, joined by straight lines, then flat up to the threshold."""
    e = np.sort(np.asarray(errors, np.float64))
    out = []
    for th in thresholds:
        area, prev_e, prev_r = 0.0, 0.0, 0.0
        for k, ek in enumerate(e):
            if not ek < th:
                break
            r = (k + 1) / len(e)
            area += (ek - prev_e) * (prev_r + r) / 2.0
            prev_e, prev_r = ek, r
        area += (th - prev_e) * prev_r
        out.append(area / th)
    return out
