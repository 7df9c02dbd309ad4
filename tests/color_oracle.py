"""CPU restatement of the colour pieces (fastpcc_b200.attributes, the colour keys of metrics.pc_error), test
infrastructure only: numpy int64 and scipy's cKDTree, never imported by the product.

Parity with MPEG pc_error's colour figures is unpinned (its source is not in the reference repository): this restates
the definitions written in metrics.pc_error, in double, with every reference row at the least distance counted once.
"""
import math

import numpy as np
from scipy.spatial import cKDTree

BRUTE_MAX_PAIRS = 1 << 26   # below this many (query, reference) pairs: brute force


def _ties_one(q, r, rgb, k=32):
    """one cloud: (d2, count, sums [nq, 3], lowest row at d2) over int64 [n, 3] rows"""
    nq, nr = q.shape[0], r.shape[0]
    d_out = np.zeros(nq, np.int64)
    n_out = np.zeros(nq, np.int64)
    s_out = np.zeros((nq, 3), np.int64)
    i_out = np.full(nq, -1, np.int64)
    if nr == 0 or nq == 0:
        return d_out, n_out, s_out, i_out
    rgb = rgb.astype(np.int64)

    def brute(rows):
        step = max(1, (1 << 22) // nr)
        for s in range(0, rows.size, step):
            sel = rows[s:s + step]
            d = ((q[sel, None, :] - r[None, :, :]) ** 2).sum(2)
            m = d.min(1)
            at = d == m[:, None]
            d_out[sel], n_out[sel] = m, at.sum(1)
            s_out[sel] = at.astype(np.int64) @ rgb
            i_out[sel] = at.argmax(1)

    if nq * nr <= BRUTE_MAX_PAIRS:
        brute(np.arange(nq))
        return d_out, n_out, s_out, i_out
    assert np.abs(q).max() < (1 << 21) and np.abs(r).max() < (1 << 21)  # squared distances exact in float64
    kk = min(k, nr)
    tree = cKDTree(r.astype(np.float64))
    for c in range(0, nq, 1 << 17):
        qc = q[c:c + (1 << 17)]
        idx = tree.query(qc.astype(np.float64), k=kk)[1].reshape(qc.shape[0], kk)
        d = ((qc[:, None, :] - r[idx]) ** 2).sum(2)
        m = d.min(1)
        at = d == m[:, None]
        d_out[c:c + qc.shape[0]], n_out[c:c + qc.shape[0]] = m, at.sum(1)
        s_out[c:c + qc.shape[0]] = (rgb[idx] * at[:, :, None]).sum(1)
        i_out[c:c + qc.shape[0]] = np.where(at, idx, np.iinfo(np.int64).max).min(1)
        # the k-th neighbour still at the least distance: more ties may lie beyond k
        full = np.nonzero(at[:, -1] & (kk < nr))[0]
        if full.size:
            brute(c + full)
    return d_out, n_out, s_out, i_out


def ties(query, ref, rgb):
    """all-ties nearest neighbour of every query row: (d2, count, sums [nq, 3], lowest ref row at d2); rows are
    [n, 3] xyz of one cloud or [n, 4] (batch, x, y, z), never across batches; -1 / 0 where a batch has no ref row"""
    query, ref = np.asarray(query, np.int64), np.asarray(ref, np.int64)
    if query.shape[1] == 3:
        return _ties_one(query, ref, rgb)
    nq = query.shape[0]
    d, n, s, i = np.zeros(nq, np.int64), np.zeros(nq, np.int64), np.zeros((nq, 3), np.int64), np.full(nq, -1, np.int64)
    for b in np.unique(query[:, 0]):
        qm, rm = np.nonzero(query[:, 0] == b)[0], np.nonzero(ref[:, 0] == b)[0]
        bd, bn, bs, bi = _ties_one(query[qm, 1:], ref[rm, 1:], rgb[rm])
        d[qm], n[qm], s[qm] = bd, bn, bs
        i[qm] = np.where(bi >= 0, rm[np.maximum(bi, 0)] if rm.size else -1, -1)
    return d, n, s, i


def recolor(org, org_rgb, rec, two_way=True, forward=None):
    """attributes.recolor's rule in numpy int64; forward: ties(rec, org, org_rgb) when already computed"""
    _, n_f, s_f, _ = forward if forward is not None else ties(rec, org, org_rgb)
    n_f = n_f[:, None]
    out = (2 * s_f + n_f) // np.maximum(2 * n_f, 1)
    if two_way:
        _, _, _, near = ties(org, rec, np.zeros((np.asarray(rec).shape[0], 3), np.uint8))
        hit = near >= 0
        s_b = np.zeros_like(s_f)
        n_b = np.zeros_like(n_f)
        np.add.at(s_b, near[hit], org_rgb[hit].astype(np.int64))
        np.add.at(n_b, near[hit], 1)
        num = s_f * n_b + s_b * n_f
        den = 2 * n_f * n_b
        out = np.where(n_b > 0, (2 * num + den) // np.maximum(2 * den, 1), out)
    return out.astype(np.uint8)


def yuv(rgb):
    """BT.709, normalised to [0, 1], double"""
    r, g, b = (np.asarray(rgb, np.float64)[:, a] for a in range(3))
    return np.stack([(0.2126 * r + 0.7152 * g + 0.0722 * b) / 255,
                     (-0.1146 * r - 0.3854 * g + 0.5 * b) / 255 + 0.5,
                     (0.5 * r - 0.4542 * g - 0.0458 * b) / 255 + 0.5], 1)


def color_keys(org, org_rgb, rec, rec_rgb):
    """the colour keys of metrics.pc_error (one cloud: a batch column is ignored)"""
    org, rec = np.asarray(org)[:, -3:], np.asarray(rec)[:, -3:]

    def mse(a, a_rgb, b, b_rgb):
        _, n, s, _ = ties(a, b, b_rgb)
        return list(((yuv(a_rgb) - yuv(s / n[:, None])) ** 2).mean(0))

    c1, c2 = mse(org, org_rgb, rec, rec_rgb), mse(rec, rec_rgb, org, org_rgb)
    out = {}
    for tag, m in (('1', c1), ('2', c2), ('F', [max(x, y) for x, y in zip(c1, c2)])):
        for i, v in enumerate(m):
            out[f'c[{i}],    {tag}'] = float(v)
            out[f'c[{i}],PSNR{tag}'] = float('inf') if v == 0 else 10.0 * math.log10(1.0 / v)
    return out
