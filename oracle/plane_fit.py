"""numpy restatement of l3d_fit_plane (include/l3d.h, DESIGN.md section 4f).  TEST INFRASTRUCTURE ONLY.

The RANSAC stage follows the kernel's exact f64 contract: every operation is one element-wise numpy operation (IEEE
round-to-nearest, no fused multiply-add; never `@` or a BLAS call, which may fuse or reorder), so the hypothesis planes,
their inlier counts and the winner are bit-identical to the GPU's.  The refinement is the float64 reference the GPU's
least-squares fits are compared against (numpy's eigh, pairwise sums: equal within rounding, not bit for bit).
"""
import numpy as np

GOLDEN = 0x9E3779B97F4A7C15
M64 = (1 << 64) - 1


def splitmix64(z):
    """The splitmix64 finaliser on a uint64 array (wrapping arithmetic)."""
    z = np.asarray(z, np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def hypothesis_indices(n, hypotheses, seed):
    """(hypotheses, 3) int64: i_k of hypothesis h = splitmix64(seed + (3h + k + 1) * GOLDEN mod 2^64) mod n."""
    j = np.arange(1, 3 * hypotheses + 1, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(int(seed) & M64) + j * np.uint64(GOLDEN)
    return (splitmix64(z) % np.uint64(n)).astype(np.int64).reshape(hypotheses, 3)


def hypothesis_planes(pts, hypotheses, seed):
    """(planes (hypotheses, 4) [nx, ny, nz, d], valid (hypotheses,) bool) in the kernel's operation order."""
    pts = np.asarray(pts, np.float64)
    idx = hypothesis_indices(len(pts), hypotheses, seed)
    p0, p1, p2 = pts[idx[:, 0]], pts[idx[:, 1]], pts[idx[:, 2]]
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        u, v = p1 - p0, p2 - p0
        nx = u[:, 1] * v[:, 2] - u[:, 2] * v[:, 1]
        ny = u[:, 2] * v[:, 0] - u[:, 0] * v[:, 2]
        nz = u[:, 0] * v[:, 1] - u[:, 1] * v[:, 0]
        s = np.sqrt((nx * nx + ny * ny) + nz * nz)
        valid = np.isfinite(p0).all(1) & np.isfinite(p1).all(1) & np.isfinite(p2).all(1) & (s > 0) & (s < np.inf)
        nx, ny, nz = nx / s, ny / s, nz / s
        d = -((nx * p0[:, 0] + ny * p0[:, 1]) + nz * p0[:, 2])
    return np.stack([nx, ny, nz, d], 1), valid


def residuals(pts, plane):
    """((nx*x + ny*y) + nz*z) + d per point, element-wise."""
    pts = np.asarray(pts, np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        return ((plane[0] * pts[:, 0] + plane[1] * pts[:, 1]) + plane[2] * pts[:, 2]) + plane[3]


def inliers(pts, plane, threshold):
    with np.errstate(invalid="ignore"):
        return np.abs(residuals(pts, plane)) <= threshold  # NaN: never


def ransac(pts, threshold, hypotheses, seed):
    """-> (winner h, its inlier count, counts per hypothesis (-1 invalid)).  Ties go to the lowest h."""
    pts = np.asarray(pts, np.float64)
    planes, valid = hypothesis_planes(pts, hypotheses, seed)
    counts = np.full(hypotheses, -1, np.int64)
    block = max(1, 4_000_000 // max(len(pts), 1))  # hypotheses per step: bounded temporaries
    X, Y, Z = pts[:, 0][None, :], pts[:, 1][None, :], pts[:, 2][None, :]
    for h0 in range(0, hypotheses, block):
        pl = planes[h0:h0 + block]
        with np.errstate(invalid="ignore", over="ignore"):
            r = ((pl[:, 0:1] * X + pl[:, 1:2] * Y) + pl[:, 2:3] * Z) + pl[:, 3:4]
            c = (np.abs(r) <= threshold).sum(1)
        counts[h0:h0 + block] = np.where(valid[h0:h0 + block], c, -1)
    if counts.max() < 0:
        raise ValueError("no valid hypothesis")
    win = int(np.argmax(counts))
    return win, int(counts[win]), counts


def lsq_plane(pts):
    """Least-squares plane of the rows of pts: centroid, covariance divided by the count, eigh.
    -> (plane [n, d] with d = -n.c, ascending eigenvalues)"""
    c = pts.mean(0)
    q = pts - c
    cov = np.empty((3, 3))
    for a in range(3):
        for b in range(3):
            cov[a, b] = np.mean(q[:, a] * q[:, b])
    w, v = np.linalg.eigh(cov)
    nrm = v[:, 0]
    return np.r_[nrm, -((nrm[0] * c[0] + nrm[1] * c[1]) + nrm[2] * c[2])], w


def refine(pts, plane, threshold, max_fits=10):
    """The refinement from a start plane: S = its inliers; fit, reselect, stop when the set repeats.
    -> dict(plane (d >= 0), mask, inliers, rms, eig, refits)"""
    pts = np.asarray(pts, np.float64)
    S = inliers(pts, plane, threshold)
    fits = 0
    while True:
        if S.sum() < 3:
            raise ValueError("fewer than 3 inliers")
        pl, w = lsq_plane(pts[S])
        S2 = inliers(pts, pl, threshold)
        fits += 1
        same = np.array_equal(S, S2)
        S = S2
        if same or fits == max_fits:
            break
    if S.sum() < 3:
        raise ValueError("fewer than 3 inliers")
    if pl[3] < 0:
        pl = -pl
    r = residuals(pts[S], pl)
    return dict(plane=pl, mask=S, inliers=int(S.sum()), rms=float(np.sqrt(np.mean(r * r))), eig=w, refits=fits)


def fit_plane(pts, threshold, hypotheses, seed):
    """RANSAC + refinement: dict of refine() plus hypothesis / hypothesis_inliers."""
    win, cnt, _ = ransac(pts, threshold, hypotheses, seed)
    planes, _ = hypothesis_planes(pts, hypotheses, seed)
    out = refine(pts, planes[win], threshold)
    out.update(hypothesis=win, hypothesis_inliers=cnt)
    return out
