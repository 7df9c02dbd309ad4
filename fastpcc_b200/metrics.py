"""Geometry distortion and rate on the device: D1 (point-to-point) and D2 (point-to-plane) MSE / PSNR as the MPEG
`pc_error` tool reports them, and bits per point.  Replaces the subprocess + PLY round trip of
lib/metrics/pc_error_wrapper.py:40-106 as used by lib/evaluators.py:49-124; result keys are pc_error's own
(the ones the reference's evaluator reads).  Nearest neighbours come from the cell-grid search fpcc_knn_search at
K = 1 (exact, O(N)); the brute-force fpcc_nn_search stays available as `nn_search_bruteforce`, the on-device
reference of the tests and the workspace-free C entry point.  The colour figures (pc_error's `-c 1`) run on the
all-ties search fpcc_nn_tie_attr (attributes.nearest_tie_attr)."""
import math
from typing import Callable, Dict, Optional

import torch

from . import _lib, attributes, knn3d
from .ops import _p, _s


def _check_clouds(query: torch.Tensor, ref: torch.Tensor):
    for t in (query, ref):
        if not t.is_cuda or t.dtype != torch.int32 or t.dim() != 2 or t.shape[1] not in (3, 4):
            raise RuntimeError('nn_search: expected int32 CUDA tensors [N,3] or [N,4]')
    if query.shape[0] == 0 or ref.shape[0] == 0:
        raise RuntimeError('nn_search: empty cloud')


def nn_search(query: torch.Tensor, ref: torch.Tensor, want_index: bool = True):
    """query [nq,3|4], ref [nr,3|4] int32 CUDA ((batch,x,y,z) rows when 4 columns) -> (d2 int64 [nq], idx int32 [nq]).
    One cloud: the batch column is ignored.  Exact squared distances, the lowest ref row among equidistant ones;
    |coordinates| < 2^30."""
    _check_clouds(query, ref)
    lim = int(max(query[:, -3:].abs().max().item(), ref[:, -3:].abs().max().item()))
    if lim.bit_length() > 30:
        raise RuntimeError('nn_search: coordinates must satisfy |c| < 2^30')
    d2, idx = knn3d.search_rows(query, ref, 1, col=query.shape[1] - 3) if query.shape[1] == ref.shape[1] else \
        knn3d.search_rows(query[:, -3:], ref[:, -3:], 1)
    return d2.view(-1), (idx.view(-1) if want_index else None)


def nn_search_bruteforce(query: torch.Tensor, ref: torch.Tensor, want_index: bool = True):
    """nn_search by brute force (fpcc_nn_search, O(nq * nr)): same arguments and results."""
    for t in (query, ref):
        if not t.is_cuda or t.dtype != torch.int32 or t.dim() != 2 or t.shape[1] not in (3, 4):
            raise RuntimeError('nn_search: expected int32 CUDA tensors [N,3] or [N,4]')
    query, ref = query.contiguous(), ref.contiguous()
    if query.shape[0] == 0 or ref.shape[0] == 0:
        raise RuntimeError('nn_search: empty cloud')
    lim = int(max(query[:, -3:].abs().max().item(), ref[:, -3:].abs().max().item()))
    bits = max(1, lim.bit_length())
    d2 = torch.empty(query.shape[0], dtype=torch.int64, device=query.device)
    idx = torch.empty(query.shape[0], dtype=torch.int32, device=query.device) if want_index else None
    _lib.call('fpcc_nn_search', _p(query), query.shape[0], query.shape[1], query.shape[1] - 3,
              _p(ref), ref.shape[0], ref.shape[1], ref.shape[1] - 3, bits, _p(d2), _p(idx), _s())
    return d2, idx


def _psnr(mse: float, peak: float) -> float:
    return float('inf') if mse == 0 else 10.0 * math.log10(3.0 * peak * peak / mse)


_yuv = attributes.rgb_to_yuv


def _color_mse(a: torch.Tensor, a_rgb: torch.Tensor, b: torch.Tensor, b_rgb: torch.Tensor):
    """per-channel YUV MSE over the points of a against the colour of b at each of them: the mean colour of every
    point of b at the least distance"""
    _, n, s = attributes.nearest_tie_attr(a[:, -3:], b[:, -3:], b_rgb)
    return (_yuv(a_rgb) - _yuv(s.double() / n.double()[:, None])).square().mean(0).tolist()


def _check_colors(rgb: torch.Tensor, xyz: torch.Tensor, what: str):
    if rgb.dtype != torch.uint8 or tuple(rgb.shape) != (xyz.shape[0], 3) or rgb.device != xyz.device:
        raise RuntimeError(f'pc_error: {what} must be uint8 [n,3] rows of the cloud, on its device')


def pc_error(org: torch.Tensor, rec: torch.Tensor, resolution: float, org_normals: Optional[torch.Tensor] = None,
             hausdorff: bool = False, search: Optional[Callable] = None, org_colors: Optional[torch.Tensor] = None,
             rec_colors: Optional[torch.Tensor] = None, normals_k: Optional[int] = None) -> Dict[str, float]:
    """`mpeg_pc_error(infile1=org, infile2=rec, resolution)` for geometry: peak = resolution - 1
    (pc_error_wrapper.py:50).  1 = loop over org (A->B), 2 = loop over rec (B->A), F = symmetric = max of both.
    With `org_normals` (float [n_org,3]) the point-to-plane figures are added: the error vector of a pair is
    projected on the normal of its ORIGINAL point (for B->A: the normal of the nearest original point).
    With `normals_k` (3..32) instead, those normals are estimated on the device from org itself:
    attributes.estimate_normals(org[:, -3:], normals_k) (one cloud, as everywhere here; all-ties K-neighbourhood PCA,
    the project's own definition, DESIGN 3.8; parity with the normals file MPEG pc_error reads is unpinned).  Passing
    both raises.
    `search`: the nearest-neighbour function, nn_search (cell grid) by default; nn_search_bruteforce gives the same
    results by brute force.
    With `org_colors` and `rec_colors` (uint8 [n,3] RGB rows of org / rec) pc_error's colour figures (`-c 1`) are
    added: 1 = for every original point a, its colour against the colour of rec at a (the mean colour of all rec
    points at the least distance from a), 2 = the mirror image, both in BT.709 YUV normalised to [0, 1]; per channel
    'c[i],    1' = MSE and 'c[i],PSNR1' = 10 log10(1 / MSE), F = the larger MSE of 1 and 2.  Parity unpinned: the
    pc_error source is not in the reference repository; pc_error keeps YUV in float32 where this keeps double, and by
    default merges duplicate coordinates before averaging where this counts every row at the least distance once
    (the same on duplicate-free clouds, such as everything frontend.voxelize and the decoders produce)."""
    if (org_colors is None) != (rec_colors is None):
        raise RuntimeError('pc_error: colours need both org_colors and rec_colors')
    if org_colors is not None:
        _check_colors(org_colors, org, 'org_colors')
        _check_colors(rec_colors, rec, 'rec_colors')
    if normals_k is not None:
        if org_normals is not None:
            raise RuntimeError('pc_error: pass org_normals or normals_k, not both')
        org_normals = attributes.estimate_normals(org[:, -3:], normals_k)  # one cloud, as the searches
    search = search or nn_search
    peak = float(resolution) - 1.0
    d_ab, i_ab = search(org, rec)
    d_ba, i_ba = search(rec, org)
    out = {'org points num': int(org.shape[0])}
    m1, m2 = d_ab.double().mean().item(), d_ba.double().mean().item()
    mf = max(m1, m2)
    out['mse1      (p2point)'], out['mse1,PSNR (p2point)'] = m1, _psnr(m1, peak)
    out['mse2      (p2point)'], out['mse2,PSNR (p2point)'] = m2, _psnr(m2, peak)
    out['mseF      (p2point)'], out['mseF,PSNR (p2point)'] = mf, _psnr(mf, peak)
    if hausdorff:
        h1, h2 = float(d_ab.max().item()), float(d_ba.max().item())
        out['h.       1(p2point)'], out['h.,PSNR  1(p2point)'] = h1, _psnr(h1, peak)
        out['h.       2(p2point)'], out['h.,PSNR  2(p2point)'] = h2, _psnr(h2, peak)
        out['h.        (p2point)'], out['h.,PSNR   (p2point)'] = max(h1, h2), _psnr(max(h1, h2), peak)
    if org_normals is not None:
        a, b, nrm = org[:, -3:].double(), rec[:, -3:].double(), org_normals.double()
        e1 = ((a - b[i_ab.long()]) * nrm).sum(1).square().mean().item()
        e2 = ((b - a[i_ba.long()]) * nrm[i_ba.long()]).sum(1).square().mean().item()
        ef = max(e1, e2)
        out['mse1      (p2plane)'], out['mse1,PSNR (p2plane)'] = e1, _psnr(e1, peak)
        out['mse2      (p2plane)'], out['mse2,PSNR (p2plane)'] = e2, _psnr(e2, peak)
        out['mseF      (p2plane)'], out['mseF,PSNR (p2plane)'] = ef, _psnr(ef, peak)
    out['mse1+mse2 (p2point)'] = m1 + m2              # pc_error_wrapper.py:97-98
    out['mse1+mse2/2(p2point)'] = (m1 + m2) / 2
    if org_colors is not None:
        c1 = _color_mse(org, org_colors, rec, rec_colors)
        c2 = _color_mse(rec, rec_colors, org, org_colors)
        for tag, mse in (('1', c1), ('2', c2), ('F', [max(x, y) for x, y in zip(c1, c2)])):
            for i, m in enumerate(mse):
                psnr = float('inf') if m == 0 else 10.0 * math.log10(1.0 / m)
                out[f'c[{i}],    {tag}'], out[f'c[{i}],PSNR{tag}'] = m, psnr
    return out


def bpp(compressed_bytes, org_points_num: int) -> float:
    """bits per input point (lib/evaluators.py: `len(compressed_bytes) * 8 / org_points_num`)"""
    n = len(compressed_bytes) if not isinstance(compressed_bytes, int) else compressed_bytes
    return n * 8 / org_points_num
