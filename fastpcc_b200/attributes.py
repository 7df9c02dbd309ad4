"""Attributes of voxel clouds on the device, colour and geometric.

Colour: the all-ties nearest-neighbour search fpcc_nn_tie_attr and the recolouring of decoded geometry built on it.
Lossy geometry decodes to points that are not in the original cloud; `recolor` gives each of them a colour taken
from the original, the step before colours can be coded or scored (and how the training targets of
models/convolutional/lossy_coord_lossy_color are built, layers.py:269-333).  `metrics.pc_error` uses the same search
for its colour figures, and `rgb_to_yuv` for its colour space (as does the colour loss of `train.LossyColorNet`).

The rule of `recolor` is this project's own definition, a forward / backward transfer in the spirit of MPEG's
recolouring; the reference's layers.py:269-333 was not available when this module was written, and parity with it
or with TMC13's distance-weighted recolour is NOT claimed.  Every step is integer arithmetic, so the result is exact
and deterministic.

Geometry: `estimate_normals`, point normals from all-ties K-neighbourhoods (fpcc_knn_normals, one fused search and
3 x 3 eigen solve per point), which give `metrics.pc_error` its point-to-plane (D2) figures for any voxel cloud.
The definition is the project's own (DESIGN 3.8), PCA over a K-neighbourhood in the family of Open3D's
`estimate_normals(KDTreeSearchParamKNN)`; parity with the normals MPEG pc_error reads from a file is unpinned.
"""
import ctypes as C
import math
import numbers
from typing import Optional

import torch

from . import _lib
from .knn3d import search_rows
from .ops import _p, _s

NORMALS_MAX_K = 32
COORD_LIMIT = 1 << 30  # |coordinates| < 2^30: the K-NN grid and the exact 128-bit moments of fpcc_knn_normals


def _rows(query: torch.Tensor, ref: torch.Tensor, n_batch: Optional[int]):
    """knn3d.knn_voxels' row conventions -> (contiguous query, ref, n_batch, xyz column, batch column)"""
    for t in (query, ref):
        if t.dtype != torch.int32 or t.dim() != 2 or t.shape[1] not in (3, 4) or not t.is_cuda:
            raise RuntimeError('nn_tie_attr: expected int32 CUDA tensors [N,3] or [N,4]')
    if query.shape[1] != ref.shape[1]:
        raise RuntimeError('nn_tie_attr: query and ref must both carry a batch column or both not')
    if query.shape[1] == 3:
        return query.contiguous(), ref.contiguous(), 1, 0, -1
    if n_batch is None:
        tops = [int(t[:, 0].max().item()) for t in (query, ref) if t.shape[0]]
        n_batch = max([0] + tops) + 1
    return query.contiguous(), ref.contiguous(), n_batch, 1, 0


def rgb_to_yuv(rgb: torch.Tensor) -> torch.Tensor:
    """[n, 3] RGB in 0..255 (any dtype) -> BT.709 YUV normalised to [0, 1], double (pc_error's colour space)"""
    r, g, b = rgb.double().unbind(1)
    return torch.stack([(0.2126 * r + 0.7152 * g + 0.0722 * b) / 255,
                        (-0.1146 * r - 0.3854 * g + 0.5 * b) / 255 + 0.5,
                        (0.5 * r - 0.4542 * g - 0.0458 * b) / 255 + 0.5], 1)


def nearest_tie_attr(query: torch.Tensor, ref: torch.Tensor, ref_rgb: torch.Tensor, n_batch: Optional[int] = None):
    """Every reference row at the least distance from each query row.  query [nq, 4], ref [nr, 4] int32 CUDA
    (batch, x, y, z) rows (never across batches), or [n, 3] (x, y, z) rows of one cloud; |coordinates| < 2^30;
    ref_rgb [nr, 3] uint8.  n_batch: as knn3d.knn_voxels (None reads max id + 1, which synchronises).
    -> (d2 int64 [nq] = d*, the least squared distance; count int32 [nq] = the reference rows at exactly d*;
    sums int64 [nq, 3] = the channel sums of their ref_rgb rows).  A query whose batch has no reference row gets
    d2 0, count 0, sums 0."""
    query, ref, n_batch, col, bcol = _rows(query, ref, n_batch)
    if ref_rgb.dtype != torch.uint8 or tuple(ref_rgb.shape) != (ref.shape[0], 3) or ref_rgb.device != ref.device:
        raise RuntimeError('nn_tie_attr: ref_rgb must be uint8 [nr,3] on the device of ref')
    ref_rgb = ref_rgb.contiguous()
    nq, nr = query.shape[0], ref.shape[0]
    ws = int(_lib.load().fpcc_knn_workspace(nr, n_batch))
    work = torch.empty(ws, dtype=torch.uint8, device=query.device)
    d2 = torch.empty(nq, dtype=torch.int64, device=query.device)
    count = torch.empty(nq, dtype=torch.int32, device=query.device)
    sums = torch.empty((nq, 3), dtype=torch.int64, device=query.device)
    _lib.call('fpcc_nn_tie_attr', n_batch, _p(query), nq, query.shape[1], col, bcol,
              _p(ref), nr, ref.shape[1], col, bcol, _p(ref_rgb), _p(d2), _p(count), _p(sums), _p(work), ws, _s())
    return d2, count, sums


def recolor(org: torch.Tensor, org_rgb: torch.Tensor, rec: torch.Tensor, two_way: bool = True,
            n_batch: Optional[int] = None) -> torch.Tensor:
    """Colours for the reconstructed rows `rec` from the original rows `org` and their colours `org_rgb` [n_org, 3]
    uint8.  org / rec: int32 CUDA rows as in `nearest_tie_attr` ((batch, x, y, z) or (x, y, z)); colours never cross
    batches.  -> uint8 [n_rec, 3].

    For a reconstructed row r:
      forward set F(r): the original rows at the least distance from r (all of them: nearest_tie_attr with
        query = rec, ref = org), channel sums S_f over n_f rows;
      backward set B(r): the original rows o whose nearest reconstructed row is r (knn3d at K = 1, the lowest row of
        rec winning a tie), channel sums S_b over n_b rows.
      two_way False, or n_b = 0: colour = (2 S_f + n_f) // (2 n_f), the forward mean rounded half up;
      otherwise: colour = (2 num + den) // (2 den) with num = S_f n_b + S_b n_f and den = 2 n_f n_b, the mean of the
        forward and the backward mean rounded half up, evaluated exactly in int64.
      A reconstructed row whose batch has no original row gets colour 0.
    int64 holds 2 num + den <= 1022 n_f n_b exactly while n_f n_b < 2^53 (any cloud of fewer than 2^26 rows).

    This rule is the project's own definition; parity with the reference's recolour (lossy_coord_lossy_color
    layers.py:269-333, not available when this module was written) or TMC13's distance-weighted recolour is NOT
    claimed."""
    rec, org, n_batch, col, bcol = _rows(rec, org, n_batch)
    _, n_f, s_f = nearest_tie_attr(rec, org, org_rgb, n_batch)
    n_f = n_f.long()[:, None]
    out = (2 * s_f + n_f) // (2 * n_f).clamp(min=1)
    if two_way:
        idx = search_rows(org, rec, 1, n_batch, col=col, batch_col=bcol)[1].view(-1)
        hit = idx >= 0
        src = torch.nonzero(hit).view(-1)
        dst = idx[hit].long()
        s_b = torch.zeros_like(s_f).index_add_(0, dst, org_rgb[src].long())
        n_b = torch.zeros_like(n_f).index_add_(0, dst, torch.ones_like(dst)[:, None])
        num = s_f * n_b + s_b * n_f
        den = 2 * n_f * n_b
        out = torch.where(n_b > 0, (2 * num + den) // (2 * den).clamp(min=1), out)
    return out.to(torch.uint8)


def estimate_normals(points: torch.Tensor, K: int = 16, n_batch: Optional[int] = None,
                     viewpoint=None) -> torch.Tensor:
    """Unit normals of int32 CUDA rows `points`: [n, 4] (batch, x, y, z) rows (neighbourhoods never cross batches) or
    [n, 3] (x, y, z) rows of one cloud, |coordinates| < 2^30 (checked, which synchronises).  n_batch: as
    knn3d.knn_voxels (None reads max id + 1, which synchronises).  -> float32 [n, 3].

    For a row p (the project's own definition, DESIGN 3.8):
      N(p) = every row of its cloud at squared distance <= d_K, the K-th least distance from p (p itself counts, at
        0; all ties are kept, so N(p) may hold more than K rows; a cloud of fewer than K rows is N(p) entire);
      M = n sum d d^T - (sum d)(sum d)^T over the offsets d = q - p of N(p), n = |N(p)|, exact in integers, rounded once
        to double;
      normal = the unit eigenvector of M's least eigenvalue (double, stored as float32); the zero vector when n < 3,
        when M has rank <= 1 (duplicates, collinear rows; decided exactly), or when the batch id lies outside
        [0, n_batch).
    Orientation: viewpoint None: the component of largest magnitude is positive (the lowest axis on a tie);
    viewpoint = three numbers in the cloud's coordinates (e.g. the sensor position after voxelisation):
    normal . (viewpoint - p) >= 0.  Point-to-plane errors square the projection, so orientation never changes a metric.
    The result depends on the point set only, not on the row order.

    Parity unpinned: MPEG pc_error reads normals from a file, and how the reference's evaluator produces it could not
    be checked.  This is PCA over a K-neighbourhood, the family of Open3D's estimate_normals(KDTreeSearchParamKNN),
    with a tie rule of the project's own."""
    if isinstance(K, bool) or not isinstance(K, numbers.Integral) or not 3 <= K <= NORMALS_MAX_K:
        raise RuntimeError(f'estimate_normals: K must be an int in 3..{NORMALS_MAX_K}, got {K!r}')
    vp = None
    if viewpoint is not None:
        try:
            v = [float(x) for x in (viewpoint.tolist() if hasattr(viewpoint, 'tolist') else viewpoint)]
        except (TypeError, ValueError):
            v = []
        if len(v) != 3 or not all(math.isfinite(x) for x in v):
            raise RuntimeError('estimate_normals: viewpoint must be three finite numbers')
        vp = (C.c_double * 3)(*v)
    if points.dtype != torch.int32 or points.dim() != 2 or points.shape[1] not in (3, 4) or not points.is_cuda:
        raise RuntimeError('estimate_normals: expected an int32 CUDA tensor [N,3] or [N,4]')
    pts = points.contiguous()
    n = pts.shape[0]
    if n:
        lo, hi = torch.stack(torch.aminmax(pts[:, -3:])).tolist()
        if lo <= -COORD_LIMIT or hi >= COORD_LIMIT:
            raise RuntimeError('estimate_normals: coordinates must satisfy |c| < 2^30')
    col, bcol = (0, -1) if pts.shape[1] == 3 else (1, 0)
    if bcol < 0:
        n_batch = 1
    elif n_batch is None:
        n_batch = int(pts[:, 0].max().item()) + 1 if n else 1
    out = torch.empty((n, 3), dtype=torch.float32, device=pts.device)
    ws = int(_lib.load().fpcc_knn_workspace(n, n_batch))
    work = torch.empty(ws, dtype=torch.uint8, device=pts.device)
    _lib.call('fpcc_knn_normals', int(K), n_batch, _p(pts), n, pts.shape[1], col, bcol, vp, _p(out), _p(work), ws, _s())
    return out
