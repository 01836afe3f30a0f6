"""fp64 numpy restatement of spn_verify_pairs (include/spn_verify.h): the integer sampler, Householder 7-point F and
4-point H solvers, scoring, selection, the stopping rule and the refits, one round of 256 hypotheses at a time.

The sampler is integer-exact and the decisions follow the same formulas as the kernel, so the GPU and this oracle
take the same decisions except where fp64 rounding could flip one.  ``ransac`` returns a margin flag for those pairs:
  - a match whose inlier test lies within 1e-9 (relative) of the threshold for a model that competes for the best
    model, is the best model or one of its refits (its count or mask could change);
  - a minimal sample near a solver decision (Householder pivot within [1e-12, 1e-6], cubic leading coefficient within
    [1e-15, 1e-9] relative, cubic discriminant within 1e-9 relative of 0, |H22| within [1e-15, 1e-9] relative) whose
    models could compete with the best;
  - counts of competing models within the number of such borderline matches, a stopping bound within 1e-9 of the
    hypotheses drawn, a refit decision within the borderline matches, or a normal matrix whose two smallest
    eigenvalues are within 1e-9 (relative) of each other."""
import numpy as np

ROUND = 256
MAX_DRAWS = 1024
PIVOT_TOL, LEAD_TOL, H22_TOL = 1e-9, 1e-12, 1e-12
NEAR = 1e3          # decision bands: a factor NEAR either side of the tolerance
REL = 1e-9          # relative margin of inlier tests, discriminants, stopping bounds and eigengaps
MAX_REFITS = 3
SAMPLE = {"fundamental": 7, "homography": 4}
MIN_MATCHES = {"fundamental": 8, "homography": 4}
_U = np.uint64


def splitmix64(x):
    """SplitMix64 finaliser on uint64 arrays (wrapping arithmetic)."""
    x = np.asarray(x, dtype=np.uint64)
    with np.errstate(over="ignore"):
        x = x + _U(0x9E3779B97F4A7C15)
        x = (x ^ (x >> _U(30))) * _U(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> _U(27))) * _U(0x94D049BB133111EB)
        return x ^ (x >> _U(31))


def pair_key(seed, a, b):
    return splitmix64(_U(seed) ^ splitmix64(_U((int(a) << 32) | int(b))))


def samples(key, hyps, n, s):
    """Minimal samples of hypotheses ``hyps`` -> (len(hyps), s) int64 indices and a bool 'complete' flag per row."""
    hyps = np.asarray(hyps, dtype=np.uint64)
    out = np.zeros((len(hyps), s), np.int64)
    ok = np.zeros(len(hyps), bool)
    width = s + 8
    draws = None
    for row, h in enumerate(hyps):
        got = []
        j0 = 0
        while len(got) < s and j0 < MAX_DRAWS:
            j = np.arange(j0, min(j0 + width, MAX_DRAWS), dtype=np.uint64)
            r = splitmix64(_U(key) ^ splitmix64((h << _U(32)) | j))
            draws = ((r >> _U(32)) * _U(n)) >> _U(32)
            for k in draws.astype(np.int64):
                if k not in got:
                    got.append(int(k))
                    if len(got) == s:
                        break
            j0 += width
        if len(got) == s:
            out[row], ok[row] = got, True
    return out, ok


def sample(seed, a, b, h, n, s):
    """The minimal sample of hypothesis h of pair (a, b) over n matches -> list of s indices (None: incomplete)."""
    idx, ok = samples(pair_key(seed, a, b), [h], n, s)
    return idx[0].tolist() if ok[0] else None


# ------------------------------------------------------------------------------------------------ normalisation
def normalisation(xa, xb):
    """Hartley transform per image -> (sa, cxa, cya, sb, cxb, cyb); None when the points of a or b all coincide."""
    xa, xb = np.asarray(xa, np.float64), np.asarray(xb, np.float64)
    ca, cb = xa.mean(0), xb.mean(0)
    da, db = np.sqrt(((xa - ca) ** 2).sum(1)).mean(), np.sqrt(((xb - cb) ** 2).sum(1)).mean()
    if not (da > 0 and db > 0):
        return None
    return (np.sqrt(2.0) / da, ca[0], ca[1], np.sqrt(2.0) / db, cb[0], cb[1])


def _apply(T, xa, xb):
    sa, cxa, cya, sb, cxb, cyb = T
    return sa * (xa[..., 0] - cxa), sa * (xa[..., 1] - cya), sb * (xb[..., 0] - cxb), sb * (xb[..., 1] - cyb)


def _mats(T):
    sa, cxa, cya, sb, cxb, cyb = T
    Ta = np.array([[sa, 0, -sa * cxa], [0, sa, -sa * cya], [0, 0, 1.0]])
    Tb = np.array([[sb, 0, -sb * cxb], [0, sb, -sb * cyb], [0, 0, 1.0]])
    return Ta, Tb


def denorm_f(f, T):
    Ta, Tb = _mats(T)
    return Tb.T @ f.reshape(-1, 3, 3) @ Ta


def denorm_h(h, T):
    """-> (H scaled to H22 = 1, ok, near) for a batch of normalised 3x3 homographies."""
    Ta, Tb = _mats(T)
    with np.errstate(all="ignore"):
        H = np.linalg.inv(Tb) @ h.reshape(-1, 3, 3) @ Ta
        mx = np.abs(H).reshape(-1, 9).max(1)
        h22 = np.abs(H[:, 2, 2])
        ok = (h22 >= H22_TOL * mx) & (h22 != 0)
        near = (h22 >= H22_TOL / NEAR * mx) & (h22 <= H22_TOL * NEAR * mx)
        H = H / H[:, 2, 2][:, None, None]
    ok &= np.isfinite(H).reshape(-1, 9).all(1)
    return H, ok, near


# ------------------------------------------------------------------------------------------------ solvers
def _householder(A, ncols, rhs_cols=()):
    """Householder QR over the first ncols columns of the batch A (B, m, k), in place.  -> (betas (B, ncols), diag
    (B, ncols) = R_kk, ok, near)."""
    B, m, _ = A.shape
    betas = np.zeros((B, ncols))
    diag = np.zeros((B, ncols))
    ok = np.ones(B, bool)
    near = np.zeros(B, bool)
    for k in range(ncols):
        nrm = np.sqrt((A[:, k:, k] ** 2).sum(1))
        ok &= nrm > PIVOT_TOL
        near |= (nrm >= PIVOT_TOL / NEAR) & (nrm <= PIVOT_TOL * NEAR)
        alpha = np.where(A[:, k, k] >= 0, -nrm, nrm)
        A[:, k, k] -= alpha
        vv = (A[:, k:, k] ** 2).sum(1)
        with np.errstate(all="ignore"):
            betas[:, k] = 2.0 / vv
            for j in range(k + 1, A.shape[2]):
                dot = (A[:, k:, k] * A[:, k:, j]).sum(1) * betas[:, k]
                A[:, k:, j] -= dot[:, None] * A[:, k:, k]
        diag[:, k] = alpha
    return betas, diag, ok, near


def _cofactors(A):
    a = A.reshape(-1, 9)
    c = np.stack([a[:, 4] * a[:, 8] - a[:, 5] * a[:, 7], a[:, 5] * a[:, 6] - a[:, 3] * a[:, 8], a[:, 3] * a[:, 7] - a[:, 4] * a[:, 6],
                  a[:, 2] * a[:, 7] - a[:, 1] * a[:, 8], a[:, 0] * a[:, 8] - a[:, 2] * a[:, 6], a[:, 1] * a[:, 6] - a[:, 0] * a[:, 7],
                  a[:, 1] * a[:, 5] - a[:, 2] * a[:, 4], a[:, 2] * a[:, 3] - a[:, 0] * a[:, 5], a[:, 0] * a[:, 4] - a[:, 1] * a[:, 3]], 1)
    return c


def cubic_roots(c3, c2, c1, c0):
    """Real roots of the batch of cubics (closed form, two Newton steps, ascending).  -> (roots (B, 4), nominal (B, 4)
    bool, any (B, 4) bool, near (B,)): slots 0-2 the roots, slot 3 the real part of a complex pair (a candidate only
    where the discriminant is near 0)."""
    with np.errstate(all="ignore"):
        mx = np.maximum(np.maximum(np.abs(c0), np.abs(c1)), np.maximum(np.abs(c2), np.abs(c3)))
        lead_ok = np.abs(c3) > LEAD_TOL * mx
        near = (np.abs(c3) >= LEAD_TOL / NEAR * mx) & (np.abs(c3) <= LEAD_TOL * NEAR * mx)
        b, c, d = c2 / c3, c1 / c3, c0 / c3
        Q = (b * b - 3.0 * c) / 9.0
        R = (2.0 * b * b * b - 9.0 * b * c + 27.0 * d) / 54.0
        Q3 = Q * Q * Q
        three = R * R < Q3
        near |= np.abs(R * R - Q3) <= REL * np.maximum(R * R, np.abs(Q3))
        th = np.arccos(np.clip(R / np.sqrt(np.where(three, Q3, 1.0)), -1, 1))
        sq = -2.0 * np.sqrt(np.where(three, Q, 0.0))
        tp = 6.283185307179586
        t3 = np.stack([sq * np.cos(th / 3.0) - b / 3.0, sq * np.cos((th + tp) / 3.0) - b / 3.0, sq * np.cos((th - tp) / 3.0) - b / 3.0], 1)
        A = -np.copysign(np.cbrt(np.abs(R) + np.sqrt(np.maximum(R * R - Q3, 0.0))), R)
        Bv = np.where(A != 0.0, Q / np.where(A != 0.0, A, 1.0), 0.0)
        one = A + Bv - b / 3.0
        pair_re = -(A + Bv) / 2.0 - b / 3.0
        x = np.where(three[:, None], t3, np.stack([one, np.zeros_like(one), np.zeros_like(one)], 1))
        x = np.concatenate([x, pair_re[:, None]], 1)
        for _ in range(2):
            v = ((c3[:, None] * x + c2[:, None]) * x + c1[:, None]) * x + c0[:, None]
            dv = (3.0 * c3[:, None] * x + 2.0 * c2[:, None]) * x + c1[:, None]
            x = np.where(dv != 0.0, x - v / np.where(dv != 0.0, dv, 1.0), x)
    x[:, :3] = np.where(three[:, None], np.sort(x[:, :3], axis=1), x[:, :3])
    nominal = np.zeros(x.shape, bool)
    nominal[:, 0] = lead_ok
    nominal[:, 1:3] = (lead_ok & three)[:, None]
    anyv = np.ones(x.shape, bool)
    anyv[:, 3] = ~three
    return x, nominal, anyv, near


def solve7(xa, xb, T):
    """7-point F of a batch of samples xa, xb (B, 7, 2) pixels -> (models (B, 4, 3, 3) pixels, nominal (B, 4), any
    (B, 4), near (B,)); see cubic_roots for the slots."""
    x1, y1, x2, y2 = _apply(T, np.asarray(xa, np.float64), np.asarray(xb, np.float64))
    A = np.stack([x2 * x1, x2 * y1, x2, y2 * x1, y2 * y1, y2, x1, y1, np.ones_like(x1)], 1)   # (B, 9, 7)
    betas, _, ok, near = _householder(A, 7)
    B = len(A)
    null = np.zeros((B, 9, 2))
    null[:, 7, 0] = 1.0
    null[:, 8, 1] = 1.0
    with np.errstate(all="ignore"):
        for k in range(6, -1, -1):
            d = (A[:, k:, k][:, :, None] * null[:, k:, :]).sum(1) * betas[:, k][:, None]
            null[:, k:, :] -= d[:, None, :] * A[:, k:, k][:, :, None]
        f1, f2 = null[:, :, 0], null[:, :, 1]
        D = f1 - f2
        cA, cD = _cofactors(f2), _cofactors(D)
        c0 = (f2[:, :3] * cA[:, :3]).sum(1)
        c3 = (D[:, :3] * cD[:, :3]).sum(1)
        c1 = (cA * D).sum(1)
        c2 = (cD * f2).sum(1)
        x, nominal, anyv, cnear = cubic_roots(c3, c2, c1, c0)
        f = x[:, :, None] * f1[:, None, :] + (1.0 - x[:, :, None]) * f2[:, None, :]
    models = denorm_f(f.reshape(-1, 9), T).reshape(B, 4, 3, 3)
    # a pivot inside the band keeps its models as candidates; one below the band is degenerate on both sides
    nominal &= ok[:, None]
    anyv &= (ok | near)[:, None] & np.isfinite(models).reshape(B, 4, 9).all(2)
    nominal &= anyv
    return models, nominal, anyv, near | cnear


def _collinear(p):
    """(B, 4, 2) integer points -> any three collinear (exact)."""
    p = np.asarray(p, np.int64)
    out = np.zeros(len(p), bool)
    for u in range(4):
        i0, i1, i2 = [i for i in range(4) if i != u]
        d = (p[:, i1, 0] - p[:, i0, 0]) * (p[:, i2, 1] - p[:, i0, 1]) - (p[:, i1, 1] - p[:, i0, 1]) * (p[:, i2, 0] - p[:, i0, 0])
        out |= d == 0
    return out


def solve4(xa, xb, T):
    """4-point H of a batch of samples (B, 4, 2) pixels -> (models (B, 4, 3, 3) pixels, nominal, any, near) with the
    model in slot 0 (the other slots are never set)."""
    B = len(xa)
    x1, y1, x2, y2 = _apply(T, np.asarray(xa, np.float64), np.asarray(xb, np.float64))
    z, o = np.zeros_like(x1), np.ones_like(x1)
    r0 = np.stack([x1, y1, o, z, z, z, -x1 * x2, -y1 * x2, x2], 2)
    r1 = np.stack([z, z, z, x1, y1, o, -x1 * y2, -y1 * y2, y2], 2)
    A = np.stack([r0, r1], 2).reshape(B, 8, 9)
    _, diag, ok, near = _householder(A, 8)
    h = np.ones((B, 9))
    with np.errstate(all="ignore"):
        for k in range(7, -1, -1):
            s = A[:, k, 8] - (A[:, k, k + 1:8] * h[:, k + 1:8]).sum(1)
            h[:, k] = s / diag[:, k]
    H, hok, hnear = denorm_h(h, T)
    coll = _collinear(xa) | _collinear(xb)
    models = np.zeros((B, 4, 3, 3))
    models[:, 0] = H
    nominal = np.zeros((B, 4), bool)
    anyv = np.zeros((B, 4), bool)
    anyv[:, 0] = ~coll & (ok | near) & (hok | hnear) & np.isfinite(H).reshape(B, 9).all(1)
    nominal[:, 0] = anyv[:, 0] & ok & hok
    return models, nominal, anyv, (near | hnear) & ~coll


# ------------------------------------------------------------------------------------------------ scoring
def test_terms(models, xa, xb, kind):
    """Both sides of the division-free inlier test of every model (K, 3, 3) on every match -> (lhs, rhs_over_t2) (K, n)."""
    F = np.asarray(models, np.float64).reshape(-1, 9)[:, :, None]
    xa, ya = np.asarray(xa, np.float64)[:, 0][None], np.asarray(xa, np.float64)[:, 1][None]
    xb, yb = np.asarray(xb, np.float64)[:, 0][None], np.asarray(xb, np.float64)[:, 1][None]
    with np.errstate(all="ignore"):
        if kind == "fundamental":
            l0, l1, l2 = F[:, 0] * xa + F[:, 1] * ya + F[:, 2], F[:, 3] * xa + F[:, 4] * ya + F[:, 5], F[:, 6] * xa + F[:, 7] * ya + F[:, 8]
            m0, m1 = F[:, 0] * xb + F[:, 3] * yb + F[:, 6], F[:, 1] * xb + F[:, 4] * yb + F[:, 7]
            e = xb * l0 + yb * l1 + l2
            return e * e, l0 * l0 + l1 * l1 + m0 * m0 + m1 * m1
        p0, p1, p2 = F[:, 0] * xa + F[:, 1] * ya + F[:, 2], F[:, 3] * xa + F[:, 4] * ya + F[:, 5], F[:, 6] * xa + F[:, 7] * ya + F[:, 8]
        u, v = p0 - xb * p2, p1 - yb * p2
        return u * u + v * v, p2 * p2


def errors(model, xa, xb, kind):
    """Sampson (F) or forward transfer (H) error in pixels of every match under one model."""
    lhs, den = test_terms(np.asarray(model)[None], xa, xb, kind)
    with np.errstate(all="ignore"):
        return np.sqrt(lhs[0] / den[0])


def score(models, xa, xb, kind, t2):
    """-> (inlier (K, n) bool, borderline (K, n) bool)."""
    lhs, den = test_terms(models, xa, xb, kind)
    rhs = t2 * den
    with np.errstate(all="ignore"):
        return lhs <= rhs, np.abs(lhs - rhs) <= REL * np.abs(rhs)


# ------------------------------------------------------------------------------------------------ refinement
def refit(xa, xb, mask, T, kind):
    """Normalised 8-point (rank 2) / DLT on the matches in mask -> (model (3, 3) pixels or None, eigengap flag)."""
    x1, y1, x2, y2 = _apply(T, np.asarray(xa, np.float64)[mask], np.asarray(xb, np.float64)[mask])
    o, z = np.ones_like(x1), np.zeros_like(x1)
    if kind == "fundamental":
        rows = np.stack([x2 * x1, x2 * y1, x2, y2 * x1, y2 * y1, y2, x1, y1, o], 1)
    else:
        rows = np.concatenate([np.stack([-x1, -y1, -o, z, z, z, x2 * x1, x2 * y1, x2], 1),
                               np.stack([z, z, z, -x1, -y1, -o, y2 * x1, y2 * y1, y2], 1)])
    ata = rows.T @ rows
    w, V = np.linalg.eigh(ata)
    gap_near = (w[1] - w[0]) <= REL * max(abs(w[-1]), 1e-300)
    v = V[:, 0].reshape(3, 3)
    if kind == "fundamental":
        w3, U = np.linalg.eigh(v.T @ v)
        u = U[:, 0]
        gap_near |= (w3[1] - w3[0]) <= REL * max(abs(w3[-1]), 1e-300)
        f = v @ (np.eye(3) - np.outer(u, u))
        return denorm_f(f.reshape(1, 9), T)[0], gap_near
    H, ok, near = denorm_h(v.reshape(1, 9), T)
    return (H[0] if ok[0] else None), bool(gap_near or near[0])


def canonical(model, kind):
    """The output scaling of include/spn_verify.h: ||F||_F = 1 with the largest-magnitude element positive; H22 = 1."""
    m = np.asarray(model, np.float64).reshape(9).copy()
    if kind == "fundamental":
        im = 0
        for k in range(9):
            if abs(m[k]) > abs(m[im]):
                im = k
        m *= (-1.0 if m[im] < 0 else 1.0) / np.sqrt((m * m).sum())
    return m.reshape(3, 3)


# ------------------------------------------------------------------------------------------------ RANSAC
def _stop(best_cnt, n, s, drawn, max_hyp, log1mc):
    """-> (stop, bound near drawn)"""
    if drawn >= max_hyp:
        return True, False
    if best_cnt <= 0:
        return False, False
    w = best_cnt / n
    ws = w
    for _ in range(s - 1):
        ws *= w
    with np.errstate(all="ignore"):
        l = np.log(1.0 - ws)
        if not l < 0.0:
            return False, False
        x = log1mc / l
    return bool(drawn >= x), bool(abs(drawn - x) <= REL * max(x, 1.0))


def ransac(xa, xb, a, b, kind, threshold=3.0, confidence=0.999, max_iters=10000, seed=0):
    """The rule of include/spn_verify.h on one pair: xa, xb (n, 2) integer pixel coordinates (col, row) of the matches
    in match order.  -> dict(model (3, 3) canonical, zeros without one; num_inliers; hypotheses; best; inliers (n,)
    bool; margin bool: a decision of this pair could flip under rounding)."""
    xa, xb = np.asarray(xa, np.int64).reshape(-1, 2), np.asarray(xb, np.int64).reshape(-1, 2)
    n, s = len(xa), SAMPLE[kind]
    t2 = float(threshold) * float(threshold)
    none = dict(model=np.zeros((3, 3)), num_inliers=0, hypotheses=0, best=-1, inliers=np.zeros(n, bool), margin=False)
    if n < MIN_MATCHES[kind]:
        return none
    T = normalisation(xa, xb)
    if T is None:
        return none
    key = pair_key(seed, a, b)
    max_hyp = -(-int(max_iters) // ROUND) * ROUND
    log1mc = float(np.log(1.0 - confidence))
    solver = solve7 if kind == "fundamental" else solve4
    margin = False
    best_cnt, best_h, best_model, best_b = -1, -1, None, 0
    hist_c, hist_b = [], []          # count and borderline count of every nominal model drawn, except the best
    unc_hi = []                      # count + borderline of candidate models of samples near a solver decision
    drawn = 0
    for r in range(max_hyp // ROUND):
        hyps = np.arange(r * ROUND, (r + 1) * ROUND)
        idx, ok = samples(key, hyps, n, s)
        models, nominal, anyv, near = solver(xa[idx], xb[idx], T)
        nominal &= ok[:, None]
        anyv &= ok[:, None]
        cand = anyv.reshape(-1)
        cnt = np.full(cand.shape, -1, np.int64)
        bord = np.zeros(cand.shape, np.int64)
        if cand.any():
            inl, bl = score(models.reshape(-1, 3, 3)[cand], xa, xb, kind, t2)
            cnt[cand], bord[cand] = inl.sum(1), bl.sum(1)
        cnt, bord = cnt.reshape(ROUND, 4), bord.reshape(ROUND, 4)
        nom_cnt = np.where(nominal, cnt, -1)
        unc = near[:, None] & anyv
        if unc.any():
            unc_hi.append(int((cnt + bord)[unc].max()))
        # thread best: count desc, root asc; round best: count desc, hypothesis asc
        tk = np.argmax(nom_cnt[:, :3], axis=1)
        tc = nom_cnt[np.arange(ROUND), tk]
        wt = int(np.argmax(tc))
        wc = int(tc[wt])
        keep = nominal.copy()
        if wc > best_cnt:
            if best_model is not None:
                hist_c.append(best_cnt)
                hist_b.append(best_b)
            best_cnt, best_h = wc, r * ROUND + wt
            best_model, best_b = models[wt, tk[wt]], int(bord[wt, tk[wt]])
            keep[wt, tk[wt]] = False
        hist_c.extend(cnt[keep].tolist())
        hist_b.extend(bord[keep].tolist())
        drawn = (r + 1) * ROUND
        # selection margin against every other model drawn so far, and near-degenerate candidates
        if best_cnt >= 0:
            hc, hb = np.asarray(hist_c, np.int64), np.asarray(hist_b, np.int64)
            thr = best_cnt - best_b
            if len(hc) and (((hb > 0) | (best_b > 0)) & (hc + hb >= thr)).any():
                margin = True
            if unc_hi and max(unc_hi) >= thr:
                margin = True
        stop, bound_near = _stop(best_cnt, n, s, drawn, max_hyp, log1mc)
        margin |= bound_near
        if best_b and best_cnt > 0:
            lo = _stop(max(best_cnt - best_b, 0), n, s, drawn, max_hyp, log1mc)[0]
            hi = _stop(min(best_cnt + best_b, n), n, s, drawn, max_hyp, log1mc)[0]
            margin |= lo != stop or hi != stop
        if stop:
            break
    if best_cnt < 0:
        return dict(none, hypotheses=drawn, margin=margin or bool(unc_hi))
    inl, bl = score(best_model[None], xa, xb, kind, t2)
    mask, cur, cur_b = inl[0], int(inl[0].sum()), int(bl[0].sum())
    model = best_model
    for _ in range(MAX_REFITS):
        if cur < MIN_MATCHES[kind]:
            margin |= cur + cur_b >= MIN_MATCHES[kind]
            break
        margin |= cur_b > 0                      # the refit's inlier set itself is uncertain
        fit, gap_near = refit(xa, xb, mask, T, kind)
        margin |= gap_near
        if fit is None:
            break
        inl2, bl2 = score(fit[None], xa, xb, kind, t2)
        c2, b2 = int(inl2[0].sum()), int(bl2[0].sum())
        if abs(c2 - cur) <= b2 + cur_b and (b2 or cur_b):
            margin = True
        if c2 < cur:
            break
        rising = c2 > cur
        model, mask, cur, cur_b = fit, inl2[0], c2, b2
        if not rising:
            break
    margin |= cur_b > 0
    return dict(model=canonical(model, kind), num_inliers=cur, hypotheses=drawn, best=best_h, inliers=mask.copy(),
                margin=bool(margin))
