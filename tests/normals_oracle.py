"""CPU restatement of attributes.estimate_normals (fpcc_knn_normals, DESIGN 3.8), test infrastructure only: numpy,
Python integers and scipy's cKDTree, never imported by the product.

N(p) = every row of p's cloud at squared distance <= d_K, the K-th least distance from p (p itself counts); M = n sum
d d^T - (sum d)(sum d)^T over the offsets d = q - p, formed in Python integers and rounded once to double (the rounding
of float(int)); the normal = numpy.linalg.eigh's eigenvector of the least eigenvalue; zero when n < 3 or rank M <= 1
(exact 2 x 2 principal minors of the integer M); orientation as the docstring of estimate_normals states it.
Parity with MPEG pc_error's normals file is unpinned.
"""
import numpy as np
from scipy.spatial import cKDTree

BRUTE_MAX_PAIRS = 1 << 24   # below this many (row, row) pairs of one cloud: brute force
CHUNK = 1 << 15


def _moments(x, K):
    """one cloud x int64 [n, 3] -> (count n [n], S1 [n, 3] int64, S2 [n, 6] int64: xx, yy, zz, xy, xz, yz)"""
    n = x.shape[0]
    cnt = np.zeros(n, np.int64)
    s1 = np.zeros((n, 3), np.int64)
    s2 = np.zeros((n, 6), object)   # Python integers where int64 would overflow (|c| >= 2^26)
    if n == 0:
        return cnt, s1, s2
    kk = min(K, n)

    wide = np.abs(x).max() >= (1 << 26)   # sums of products could pass int64: Python integers

    def add(rows, idx, keep):
        d = x[idx] - x[rows][:, None, :]                          # [r, m, 3] offsets q - p
        d = d * keep[:, :, None]
        if wide:
            d = d.astype(object)
        cnt[rows] = keep.sum(1)
        s1[rows] = d.sum(1)
        s2[rows] = np.stack([(d[:, :, a] * d[:, :, b]).sum(1) for a, b in
                             ((0, 0), (1, 1), (2, 2), (0, 1), (0, 2), (1, 2))], 1)

    def brute(rows):
        step = max(1, (1 << 20) // n)
        for c in range(0, rows.size, step):
            r = rows[c:c + step]
            d2 = ((x[r][:, None, :] - x[None, :, :]) ** 2).sum(2)
            dk = np.partition(d2, kk - 1, axis=1)[:, kk - 1] if kk < n else np.full(r.size, np.iinfo(np.int64).max)
            add(r, np.broadcast_to(np.arange(n), d2.shape), (d2 <= dk[:, None]).astype(np.int64))

    if n * n <= BRUTE_MAX_PAIRS:
        brute(np.arange(n))
        return cnt, s1, s2
    assert np.abs(x).max() < (1 << 21)  # squared distances exact in float64
    tree = cKDTree(x.astype(np.float64))
    m = min(n, 2 * K + 8)               # the K-th distance and the ties past it, for most rows
    for c in range(0, n, CHUNK):
        rows = np.arange(c, min(n, c + CHUNK))
        idx = tree.query(x[rows].astype(np.float64), k=m)[1].reshape(rows.size, m)
        d2 = ((x[idx] - x[rows][:, None, :]) ** 2).sum(2)
        d2s = np.sort(d2, 1)
        dk = d2s[:, kk - 1] if kk < n else np.full(rows.size, np.iinfo(np.int64).max)
        keep = d2 <= dk[:, None]
        add(rows, idx, keep.astype(np.int64))
        full = np.nonzero(keep.all(1) & (m < n))[0]             # the m-th row still inside: ties may lie beyond
        for i in full:
            p = rows[i]
            ball = np.array(tree.query_ball_point(x[p].astype(np.float64), np.sqrt(float(dk[i])) + 0.5))
            bd = ((x[ball] - x[p]) ** 2).sum(1)
            add(np.array([p]), ball[None, :], (bd <= dk[i]).astype(np.int64)[None, :])
    return cnt, s1, s2


def scatter(points, K, n_batch=None):
    """-> (count [n], M [n, 6] Python-int object array: xx, yy, zz, xy, xz, yz) over [n, 3] or [n, 4] rows"""
    pts = np.asarray(points, np.int64)
    n = pts.shape[0]
    cnt, s1, s2 = np.zeros(n, np.int64), np.zeros((n, 3), np.int64), np.zeros((n, 6), object)
    if pts.shape[1] == 3:
        cnt, s1, s2 = _moments(pts, K)
    else:
        nb = (int(pts[:, 0].max()) + 1 if n else 1) if n_batch is None else n_batch
        for b in np.unique(pts[:, 0]):
            if not 0 <= b < nb:
                continue                                        # rows outside [0, n_batch): zero
            r = np.nonzero(pts[:, 0] == b)[0]
            cnt[r], s1[r], s2[r] = _moments(pts[r, 1:], K)
    c = cnt.astype(object)
    S1, S2 = s1.astype(object), s2.astype(object)
    M = np.empty((n, 6), object)
    for j, (a, b) in enumerate(((0, 0), (1, 1), (2, 2), (0, 1), (0, 2), (1, 2))):
        M[:, j] = c * S2[:, j] - S1[:, a] * S1[:, b]
    return cnt, M


def normals(points, K, n_batch=None, viewpoint=None, details=False):
    """estimate_normals' definition: float32 [n, 3]; details: also (eigenvalues [n, 3] ascending, M double [n, 3, 3],
    the orientation margin [n]: |the deciding quantity|, 0 where a tie or none)"""
    pts = np.asarray(points, np.int64)
    n = pts.shape[0]
    cnt, M = scatter(pts, K, n_batch)
    flat = (cnt < 3) | ((M[:, 0] * M[:, 1] == M[:, 3] ** 2) & (M[:, 0] * M[:, 2] == M[:, 4] ** 2) &
                        (M[:, 1] * M[:, 2] == M[:, 5] ** 2)).astype(bool)
    Md = np.array([[float(v) for v in row] for row in M], np.float64).reshape(n, 6)  # float(int): one rounding
    A = np.stack([Md[:, [0, 3, 4]], Md[:, [3, 1, 5]], Md[:, [4, 5, 2]]], 1)
    w, V = np.linalg.eigh(A) if n else (np.zeros((0, 3)), np.zeros((0, 3, 3)))
    v = V[:, :, 0]
    v = v / np.linalg.norm(v, axis=1, keepdims=True)
    if viewpoint is None:
        top = np.argmax(np.abs(v), 1)                          # first maximum: the lowest axis on a tie
        dec = v[np.arange(n), top]
        mags = np.sort(np.abs(v), 1)
        margin = np.where(mags[:, 2] - mags[:, 1] > 1e-9, np.abs(dec), 0.0)  # near-tie in magnitude: undecided
    else:
        dec = (v * (np.asarray(viewpoint, np.float64)[None, :] - pts[:, -3:].astype(np.float64))).sum(1)
        margin = np.abs(dec)
    v = np.where((dec < 0)[:, None], -v, v)
    v[flat] = 0.0
    out = v.astype(np.float32)
    return (out, w, A, margin, flat) if details else out
