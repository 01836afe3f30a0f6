"""Planted two-view scenes for the geometric verification tests and tools/bench_verify.py: matches with integer
keypoint coordinates, a known fraction of true correspondences and uniform outliers.  numpy RandomState only."""
import numpy as np

W, H = 640, 480


def _rot(rng, scale):
    w = rng.uniform(-scale, scale, 3)
    th = np.linalg.norm(w)
    k = w / th
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K


def camera_pair(rng):
    """-> (K, R, t): camera a at the origin, b = (R, t); F_true = K^-T [t]x R K^-1 maps a to b."""
    K = np.array([[500.0, 0, W / 2], [0, 500.0, H / 2], [0, 0, 1]])
    R = _rot(rng, 0.15)
    t = rng.uniform(-1, 1, 3)
    t[2] *= 0.3
    return K, R, t / np.linalg.norm(t)


def true_fundamental(K, R, t):
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    Ki = np.linalg.inv(K)
    F = Ki.T @ tx @ R @ Ki
    return F / np.linalg.norm(F)


def true_homography(rng):
    """A homography of a plane seen from two views, with moderate perspective."""
    K, R, t = camera_pair(rng)
    n = np.array([0.1, -0.2, 1.0])
    n /= np.linalg.norm(n)
    d = 5.0
    Hm = K @ (R - np.outer(t * 0.5, n) / d) @ np.linalg.inv(K)
    return Hm / Hm[2, 2]


def scene(rng, n, inlier_ratio, kind, noise=0.5):
    """n matches (xa, xb) (n, 2) int (col, row), is_true (n,) bool, and the true model (F or H).  True matches are
    projections of random 3-D points (F) or of a plane (H) with Gaussian noise, rounded; outliers are uniform."""
    n_in = int(round(n * inlier_ratio))
    if kind == "fundamental":
        K, R, t = camera_pair(rng)
        model = true_fundamental(K, R, t)
        xa, xb = [], []
        while len(xa) < n_in:
            X = np.c_[rng.uniform(-4, 4, 2 * n_in + 8), rng.uniform(-3, 3, 2 * n_in + 8), rng.uniform(4, 12, 2 * n_in + 8)]
            pa = (K @ X.T).T
            pb = (K @ (R @ X.T + t[:, None])).T
            ok = (pb[:, 2] > 0)
            pa, pb = pa[:, :2] / pa[:, 2:], pb[:, :2] / np.where(ok, pb[:, 2], 1)[:, None]
            inside = ok & (pa >= 0).all(1) & (pa[:, 0] < W) & (pa[:, 1] < H) & (pb >= 0).all(1) & (pb[:, 0] < W) & (pb[:, 1] < H)
            xa.extend(pa[inside].tolist())
            xb.extend(pb[inside].tolist())
        xa, xb = np.array(xa[:n_in]).reshape(-1, 2), np.array(xb[:n_in]).reshape(-1, 2)
    else:
        model = true_homography(rng)
        xa = np.c_[rng.uniform(0, W, 4 * n_in + 8), rng.uniform(0, H, 4 * n_in + 8)]
        p = (model @ np.c_[xa, np.ones(len(xa))].T).T
        xb = p[:, :2] / p[:, 2:]
        inside = (p[:, 2] > 0) & (xb >= 0).all(1) & (xb[:, 0] < W) & (xb[:, 1] < H)
        xa, xb = xa[inside][:n_in], xb[inside][:n_in]
    xa = np.clip(np.rint(xa + noise * rng.randn(*xa.shape)), 0, [W - 1, H - 1])
    xb = np.clip(np.rint(xb + noise * rng.randn(*xb.shape)), 0, [W - 1, H - 1])
    n_out = n - len(xa)
    oa = np.c_[rng.randint(0, W, n_out), rng.randint(0, H, n_out)]
    ob = np.c_[rng.randint(0, W, n_out), rng.randint(0, H, n_out)]
    perm = rng.permutation(n)
    xa = np.concatenate([xa, oa]).astype(np.int64)[perm]
    xb = np.concatenate([xb, ob]).astype(np.int64)[perm]
    is_true = np.r_[np.ones(n - n_out, bool), np.zeros(n_out, bool)][perm]
    return xa, xb, is_true, model


def pool(pair_matches, cap):
    """Keypoint pool, pairs, offsets and matches for a list of (xa, xb) match sets, one image pair (2p, 2p+1) each,
    every match its own keypoint: -> kp (N, cap, 2) int32 (row, col), pairs (P, 2), offsets (P+1,) int64, matches (M, 2)
    int32."""
    P = len(pair_matches)
    kp = np.zeros((2 * P, cap, 2), np.int32)
    pairs, offsets, matches = [], [0], []
    for p, (xa, xb) in enumerate(pair_matches):
        n = len(xa)
        assert n <= cap
        kp[2 * p, :n] = np.asarray(xa)[:, ::-1]
        kp[2 * p + 1, :n] = np.asarray(xb)[:, ::-1]
        pairs.append((2 * p, 2 * p + 1))
        offsets.append(offsets[-1] + n)
        matches.append(np.c_[np.arange(n), np.arange(n)])
    m = np.concatenate(matches).astype(np.int32) if matches else np.zeros((0, 2), np.int32)
    return kp, np.array(pairs, np.int64).reshape(-1, 2), np.array(offsets, np.int64), m.reshape(-1, 2)
