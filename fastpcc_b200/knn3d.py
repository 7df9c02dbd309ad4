"""Exact K nearest neighbours in 3-D on the device (fpcc_knn_search: a cell grid built per call, O(N*K) for voxel
clouds instead of brute force).

The surface follows PyTorch3D's `knn_points` / `knn_gather`, which the reference's `lib/knn3d` (a float32, D = 3
brute-force K-NN, lib/knn3d/src/knn3d.cu:25,75,165) is adapted from.  The reference's Python wrapper
(lib/knn3d/__init__.py) was not available when this module was written, so parity of function names or argument
order with that wrapper is NOT claimed; parity with PyTorch3D's documented `knn_points(p1, p2, lengths1, lengths2, K,
return_nn)` is the intent.

Results are exact and deterministic: neighbours ascend by (distance, row) with the lowest row winning a tie, float32
distances are ((dx*dx + dy*dy) + dz*dz) rounded per operation as NumPy float32 evaluates it, int32 distances are exact
int64.  Missing neighbours (a cloud with fewer than K points) are idx -1, distance 0.
"""
from collections import namedtuple
from typing import Optional

import torch

from . import _lib
from .ops import _p, _s

MAX_K = 32
MAX_BATCH = 1023  # batch ids are a 10-bit field of the cell keys

_KNN = namedtuple('KNN', 'dists idx knn')


def search_rows(query: torch.Tensor, ref: torch.Tensor, k: int, n_batch: int = 1, col: int = 0, batch_col: int = -1):
    """Raw entry: query [nq, ld], ref [nr, ld] int32 or float32 CUDA rows, xyz at `col`, batch id at `batch_col`
    (-1: one cloud, n_batch must be 1).  -> (dist [nq, k] int64 | float32, idx [nq, k] int32 rows of `ref`)."""
    if query.dtype != ref.dtype or query.dtype not in (torch.int32, torch.float32):
        raise RuntimeError('knn: query and ref must both be int32 or both float32')
    for t in (query, ref):
        if not t.is_cuda or t.dim() != 2:
            raise RuntimeError('knn: expected 2-D CUDA tensors of rows')
    query, ref = query.contiguous(), ref.contiguous()
    nq, nr = query.shape[0], ref.shape[0]
    ws = int(_lib.load().fpcc_knn_workspace(nr, n_batch))
    work = torch.empty(ws, dtype=torch.uint8, device=query.device)
    ddt = torch.int64 if query.dtype == torch.int32 else torch.float32
    dist = torch.empty((nq, k), dtype=ddt, device=query.device)
    idx = torch.empty((nq, k), dtype=torch.int32, device=query.device)
    _lib.call('fpcc_knn_search', 0 if query.dtype == torch.int32 else 1, k, n_batch,
              _p(query), nq, query.shape[1], col, batch_col, _p(ref), nr, ref.shape[1], col, batch_col,
              _p(dist), _p(idx), _p(work), ws, _s())
    return dist, idx


def knn_voxels(query: torch.Tensor, ref: torch.Tensor, K: int = 1, n_batch: Optional[int] = None):
    """K nearest reference voxels of every query voxel.  query [nq, 4], ref [nr, 4] int32 CUDA (batch, x, y, z) rows
    (neighbours never cross batches), or [n, 3] (x, y, z) rows of one cloud; |coordinates| < 2^30.
    n_batch: number of batch ids (rows with ids outside [0, n_batch) are ignored); None reads max id + 1 from the
    tensors, which synchronises.  -> (d2 int64 [nq, K], idx int32 [nq, K] rows of `ref`)."""
    for t in (query, ref):
        if t.dtype != torch.int32 or t.dim() != 2 or t.shape[1] not in (3, 4):
            raise RuntimeError('knn_voxels: expected int32 tensors [N,3] or [N,4]')
    if query.shape[1] != ref.shape[1]:
        raise RuntimeError('knn_voxels: query and ref must both carry a batch column or both not')
    if query.shape[1] == 3:
        return search_rows(query, ref, K)
    if n_batch is None:
        tops = [int(t[:, 0].max().item()) for t in (query, ref) if t.shape[0]]
        n_batch = max([0] + tops) + 1
    return search_rows(query, ref, K, n_batch, col=1, batch_col=0)


def _cloud_rows(p: torch.Tensor, lengths: Optional[torch.Tensor]):
    """[N, P, 3] -> [N*P, 4] float32 rows (x, y, z, batch); rows past a cloud's length get batch -1 (ignored)."""
    n, m, _ = p.shape
    pos = torch.arange(m, device=p.device)
    b = torch.arange(n, device=p.device, dtype=torch.float32)[:, None].expand(n, m)
    if lengths is not None:
        b = torch.where(pos[None, :] < lengths.to(p.device)[:, None], b, torch.full_like(b, -1.0))
    return torch.cat([p.detach().reshape(n * m, 3).float(), b.reshape(n * m, 1)], 1)


class _KnnDists(torch.autograd.Function):
    """dists = |p1 - p2[idx]|^2 with the neighbours fixed: d/dp1 = 2 (p1 - p2[idx]), scattered with the opposite sign
    into p2."""

    @staticmethod
    def forward(ctx, p1, p2, idx, dists):
        ctx.save_for_backward(p1, p2, idx)
        return dists.clone()

    @staticmethod
    def backward(ctx, grad):
        p1, p2, idx = ctx.saved_tensors
        n, p1n, k = idx.shape
        valid = (idx >= 0).unsqueeze(-1)
        ic = idx.clamp(min=0)
        nn = knn_gather(p2, ic)
        g = 2.0 * grad.unsqueeze(-1) * (p1.unsqueeze(2) - nn) * valid
        g1 = g.sum(2) if ctx.needs_input_grad[0] else None
        g2 = None
        if ctx.needs_input_grad[1]:
            g2 = torch.zeros_like(p2).scatter_add_(1, ic.reshape(n, p1n * k, 1).expand(-1, -1, 3),
                                                   -g.reshape(n, p1n * k, 3))
        return g1, g2, None, None


def knn_points(p1: torch.Tensor, p2: torch.Tensor, lengths1: Optional[torch.Tensor] = None,
               lengths2: Optional[torch.Tensor] = None, K: int = 1, return_nn: bool = False):
    """K nearest points of p2 for every point of p1, cloud by cloud (PyTorch3D's knn_points).
    p1 [N, P1, 3], p2 [N, P2, 3] float32 CUDA; lengths1 / lengths2 [N]: points in use per cloud (padding after).
    -> (dists [N, P1, K] float32 squared distances, differentiable w.r.t. p1 and p2; idx [N, P1, K] int64 indices
    into each cloud of p2, -1 where a cloud has fewer than K points or the query is padding;
    knn [N, P1, K, 3] = p2 gathered at idx when return_nn, else None)."""
    if not 1 <= K <= MAX_K:
        raise RuntimeError(f'knn_points: K must be in 1..{MAX_K}')
    if p1.dim() != 3 or p2.dim() != 3 or p1.shape[2] != 3 or p2.shape[2] != 3 or p1.shape[0] != p2.shape[0]:
        raise RuntimeError('knn_points: expected p1 [N,P1,3] and p2 [N,P2,3]')
    if p1.dtype != torch.float32 or p2.dtype != torch.float32 or not p1.is_cuda or not p2.is_cuda:
        raise RuntimeError('knn_points: float32 CUDA tensors required')
    n, n1, n2 = p1.shape[0], p1.shape[1], p2.shape[1]
    r1, r2 = _cloud_rows(p1, lengths1), _cloud_rows(p2, lengths2)
    dists = torch.zeros((n, n1, K), dtype=torch.float32, device=p1.device)
    idx = torch.full((n, n1, K), -1, dtype=torch.int64, device=p1.device)
    for b0 in range(0, n, MAX_BATCH):  # one call covers up to 1023 clouds
        b1 = min(n, b0 + MAX_BATCH)
        q, r = r1[b0 * n1:b1 * n1], r2[b0 * n2:b1 * n2]
        if b0:
            q, r = q.clone(), r.clone()
            q[:, 3] -= torch.where(q[:, 3] >= 0, float(b0), 0.0)
            r[:, 3] -= torch.where(r[:, 3] >= 0, float(b0), 0.0)
        d, i = search_rows(q, r, K, b1 - b0, col=0, batch_col=3)
        i = i.long()
        dists[b0:b1] = d.view(b1 - b0, n1, K)
        idx[b0:b1] = torch.where(i >= 0, i % max(n2, 1), i).view(b1 - b0, n1, K)
    if p1.requires_grad or p2.requires_grad:
        dists = _KnnDists.apply(p1, p2, idx, dists)
    nn = knn_gather(p2, idx, lengths2) if return_nn else None
    return _KNN(dists, idx, nn)


def knn_gather(x: torch.Tensor, idx: torch.Tensor, lengths: Optional[torch.Tensor] = None):
    """x [N, M, D], idx [N, L, K] int -> [N, L, K, D] = x[n, idx[n, l, k]]; zeros where idx is -1 (or >= lengths[n])."""
    n, m, dd = x.shape
    _, l, k = idx.shape
    idx = idx.long()
    if m == 0:
        return x.new_zeros((n, l, k, dd))
    bad = idx < 0
    if lengths is not None:
        bad = bad | (idx >= lengths.to(idx.device).view(n, 1, 1))
    ic = idx.masked_fill(bad, 0)
    out = x.gather(1, ic.reshape(n, l * k, 1).expand(-1, -1, dd)).view(n, l, k, dd)
    return out.masked_fill(bad.unsqueeze(-1), 0)
