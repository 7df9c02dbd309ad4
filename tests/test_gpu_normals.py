"""fpcc_knn_normals (attributes.estimate_normals) and metrics.pc_error(normals_k=) against the CPU oracle
(tests/normals_oracle.py): components within 1e-6 where the eigenproblem is well separated, eigen-residuals elsewhere,
zero vectors exactly where the oracle has them; bitwise reproducible across calls, row orders and batching."""
import math

import numpy as np
import pytest
import torch

from fastpcc_b200 import attributes, metrics, synth
from tests import normals_oracle as NO

pytestmark = pytest.mark.gpu


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check(pts, K, n_batch=None, viewpoint=None):
    got = attributes.estimate_normals(_cuda(pts), K, n_batch, viewpoint)
    assert got.dtype == torch.float32 and tuple(got.shape) == (pts.shape[0], 3)
    got = got.cpu().numpy()
    want, w, A, margin, flat = NO.normals(pts, K, n_batch, viewpoint, details=True)
    # zero vectors exactly where the oracle has them
    assert ((got == 0).all(1) == flat).all()
    live = ~flat
    g, v = got.astype(np.float64), want.astype(np.float64)
    gap = (w[:, 1] - w[:, 0]) / np.maximum(np.abs(w[:, 2]), np.finfo(np.float64).tiny)
    sep = live & (gap >= 1e-6)
    # well separated: every component within 1e-6, up to sign; the sign itself unless the decision is a near tie
    err = np.minimum(np.abs(g - v).max(1), np.abs(g + v).max(1))
    assert err[sep].max(initial=0) <= 1e-6, err[sep].max()
    signed = sep & (margin > 1e-9)
    assert np.abs(g - v).max(1)[signed].max(initial=0) <= 1e-6
    # elsewhere: a unit eigenvector of the least eigenvalue
    rest = live & ~sep
    if rest.any():
        gr = g[rest]
        assert np.abs(np.linalg.norm(gr, axis=1) - 1).max() <= 1e-6
        res = np.linalg.norm(np.einsum('nij,nj->ni', A[rest], gr) - w[rest, :1] * gr, axis=1)
        assert (res <= 1e-6 * np.linalg.norm(A[rest], axis=(1, 2))).all()
    return got, flat, sep


@pytest.fixture(scope='module')
def clouds():
    surface = synth.surface_cloud(1, bits=10, n_target=220000)
    assert surface.shape[0] >= 200000
    lidar = synth.lidar_frame(2)
    frames = [synth.lidar_frame(10 + i, azimuths=1024) for i in range(3)]
    batch = np.concatenate([synth.with_batch(f, i) for i, f in enumerate(frames)])
    return {'surface': surface, 'lidar': lidar, 'batch3': batch, 'frames': frames}


@pytest.mark.parametrize('K', [3, 8, 16, 32])
@pytest.mark.parametrize('name', ['surface', 'lidar', 'batch3'])
def test_equal_to_oracle(clouds, name, K):
    got, flat, sep = _check(clouds[name], K)
    assert sep.mean() > 0.5            # most rows are compared component by component
    if name != 'lidar' or K > 3:
        assert flat.mean() < 0.2


def test_viewpoint_orientation_matches_oracle(clouds):
    lidar = clouds['lidar']
    vp = lidar.mean(0).tolist()        # inside the scan, as a sensor position is
    got, _, _ = _check(lidar, 16, viewpoint=vp)
    dots = (got * (np.asarray(vp)[None, :] - lidar)).sum(1)
    assert (dots >= 0).all()


def test_bitwise_reproducible_across_calls_orders_and_batching(clouds):
    surface = clouds['surface']
    a = attributes.estimate_normals(_cuda(surface), 16)
    assert torch.equal(a, attributes.estimate_normals(_cuda(surface), 16))
    perm = np.random.default_rng(3).permutation(surface.shape[0])
    b = attributes.estimate_normals(_cuda(surface[perm]), 16)
    back = torch.empty_like(b)
    back[torch.from_numpy(perm).cuda()] = b
    assert torch.equal(a, back)
    # batched rows, shuffled, against each frame alone
    batch = clouds['batch3']
    perm = np.random.default_rng(4).permutation(batch.shape[0])
    nb = attributes.estimate_normals(_cuda(batch[perm]), 16, n_batch=3).cpu().numpy()
    whole = np.empty_like(nb)
    whole[perm] = nb
    start = 0
    for f in clouds['frames']:
        alone = attributes.estimate_normals(_cuda(f), 16).cpu().numpy()
        assert (whole[start:start + f.shape[0]] == alone).all()
        start += f.shape[0]


def test_small_clouds_bounds_and_empty_input():
    two = _cuda(np.array([[0, 0, 0], [1, 2, 3]], np.int32))
    assert (attributes.estimate_normals(two, 3) == 0).all()
    tri = _cuda(np.array([[5, 5, 5], [6, 5, 5], [5, 6, 5]], np.int32))   # fewer rows than K: the whole cloud
    assert attributes.estimate_normals(tri, 32).cpu().tolist() == [[0.0, 0.0, 1.0]] * 3
    # a row whose batch id lies outside [0, n_batch) gets zero
    rows = _cuda(np.array([[0, 5, 5, 5], [0, 6, 5, 5], [0, 5, 6, 5], [7, 0, 0, 0]], np.int32))
    assert attributes.estimate_normals(rows, 3, n_batch=1).cpu().tolist() == [[0.0, 0.0, 1.0]] * 3 + [[0.0] * 3]
    assert tuple(attributes.estimate_normals(torch.zeros((0, 3), dtype=torch.int32, device='cuda')).shape) == (0, 3)
    for bad in (1 << 30, -(1 << 30)):
        with pytest.raises(RuntimeError, match=r'\|c\| < 2\^30'):
            attributes.estimate_normals(_cuda(np.array([[0, 0, 0], [bad, 0, 0], [0, 1, 0]], np.int32)))
    # 16-bit coordinates far apart: the exact 128-bit moments; rows along x and y: normal z
    big = _cuda(np.array([[0, 0, 0], [65535, 0, 0], [0, 65535, 0], [65535, 65535, 0]], np.int32))
    assert attributes.estimate_normals(big, 3).cpu().tolist() == [[0.0, 0.0, 1.0]] * 4


def test_large_coordinates_take_the_wide_integer_paths():
    # a sparse cloud spanning |c| < 2^30: from K = 16 on, entries of M pass 2^64 (the two-word rounding to double) and
    # the rank test's products pass 2^128 (the high words of the 256-bit comparison); 100 rows: past the grid's scan
    # threshold, small enough for the oracle's brute force
    lim = (1 << 30) - 1
    pts = np.random.default_rng(8).integers(-lim, lim + 1, (100, 3)).astype(np.int32)
    for K in (3, 16, 32):
        _, M = NO.scatter(pts, K)
        if K >= 16:
            assert max(abs(int(v)) for v in M.ravel()) >= 1 << 64
        got, flat, sep = _check(pts, K)
        assert not flat.any() and sep.mean() > 0.9
    # 30 rows on a line with every step near 2^25: rank 1, decided exactly on minors past 2^128, the zero vector
    t = np.arange(-15, 15)[:, None]
    line = (t * np.array([[(1 << 26) + 1, (1 << 25) + 3, -(1 << 25) + 5]]) + np.array([[5, -7, 11]])).astype(np.int32)
    _, M = NO.scatter(line, 32)
    assert max(abs(int(r[0]) * int(r[1])) for r in M) >= 1 << 128
    got, flat, _ = _check(line, 32)
    assert flat.all() and (got == 0).all()
    # one row off that line: every neighbourhood is then a plane
    got, flat, _ = _check(np.concatenate([line, [[5, 1 << 28, 11]]]).astype(np.int32), 32)
    assert not flat.any()


def _p2plane(out):
    return {k: v for k, v in out.items() if 'p2plane' in k}


def test_pc_error_normals_k_equals_explicit_normals(clouds):
    org = clouds['surface']
    rng = np.random.default_rng(6)
    rec = np.unique(np.clip(org + rng.integers(-1, 2, org.shape), 0, 1023).astype(np.int32), axis=0)
    o, r = _cuda(org), _cuda(rec)
    plain = metrics.pc_error(o, r, 1024)
    assert not _p2plane(plain)
    for K in (3, 16):
        got = metrics.pc_error(o, r, 1024, normals_k=K)
        want = metrics.pc_error(o, r, 1024, org_normals=attributes.estimate_normals(o, K))
        assert got == want and len(_p2plane(got)) == 6
        for key, v in plain.items():
            assert got[key] == v, key


@pytest.fixture(scope='module')
def big():
    org = synth.surface_cloud(3, bits=11, n_target=800000)
    rng = np.random.default_rng(4)
    rec = np.unique(np.clip(org + rng.integers(-2, 3, org.shape), 0, 2047).astype(np.int32)
                    [rng.random(org.shape[0]) < 0.8], axis=0)
    return org, rec


def test_pc_error_800k_against_oracle_normals(big):
    org, rec = big
    assert org.shape[0] >= 790000
    K = 16
    o, r = _cuda(org), _cuda(rec)
    got = metrics.pc_error(o, r, 2048, normals_k=K)
    ref = metrics.pc_error(o, r, 2048, org_normals=_cuda(NO.normals(org, K)))
    for tag in ('1', '2', 'F'):
        key = f'mse{tag}      (p2plane)'
        assert math.isclose(got[key], ref[key], rel_tol=1e-6), (key, got[key], ref[key])
        pkey = f'mse{tag},PSNR (p2plane)'
        assert abs(got[pkey] - ref[pkey]) < 5e-4, (pkey, got[pkey], ref[pkey])
        assert got[pkey] > got[f'mse{tag},PSNR (p2point)']   # projected errors are smaller
