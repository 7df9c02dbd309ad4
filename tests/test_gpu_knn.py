"""fpcc_knn_search (fastpcc_b200.knn3d, metrics.nn_search) against exact oracles: numpy brute force (int64 and the
same float32 expression), scipy's cKDTree, and the on-device brute force fpcc_nn_search at sizes numpy cannot reach."""
import numpy as np
import pytest
import torch

from fastpcc_b200 import knn3d, metrics, synth

pytestmark = pytest.mark.gpu


def _brute(q, r, k, dtype=np.int64):
    """exact K-NN by (distance, row): int64 squared distances, or float32 ((dx*dx + dy*dy) + dz*dz); -1 / 0 padding"""
    nq, nr = q.shape[0], r.shape[0]
    d_out = np.zeros((nq, k), dtype)
    i_out = np.full((nq, k), -1, np.int64)
    if nr == 0:
        return d_out, i_out
    kk = min(k, nr)
    step = max(1, (1 << 24) // nr)
    q, r = q.astype(dtype), r.astype(dtype)
    for s in range(0, nq, step):
        dx, dy, dz = (q[s:s + step, None, a] - r[None, :, a] for a in range(3))
        d = (dx * dx + dy * dy) + dz * dz
        o = np.argsort(d, axis=1, kind='stable')[:, :kk]  # stable: equal distances keep ascending rows
        d_out[s:s + step, :kk] = np.take_along_axis(d, o, 1)
        i_out[s:s + step, :kk] = o
    return d_out, i_out


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


_INT_CASES = {6: (3000, 1500), 10: (8000, 3000), 16: (5000, 5000), 20: (20000, 5000)}
_int_cache = {}


def _int_case(bits):
    if bits not in _int_cache:
        nq, nr = _INT_CASES[bits]
        rng = np.random.default_rng(100 + bits)
        half = 1 << (bits - 1)
        q = rng.integers(-half, half, (nq, 3)).astype(np.int32)
        r = rng.integers(-half, half, (nr, 3)).astype(np.int32)
        _int_cache[bits] = (q, r, _brute(q, r, 32))
    return _int_cache[bits]


@pytest.mark.parametrize('k', [1, 4, 16, 32])
@pytest.mark.parametrize('bits', [6, 10, 16, 20])
def test_int32_matches_brute_force_exactly(bits, k):
    q, r, (want_d, want_i) = _int_case(bits)
    d, i = knn3d.knn_voxels(_cuda(q), _cuda(r), k)
    assert d.dtype == torch.int64 and i.dtype == torch.int32 and tuple(d.shape) == (q.shape[0], k)
    assert (d.cpu().numpy() == want_d[:, :k]).all()
    assert (i.cpu().numpy() == want_i[:, :k]).all()
    # the same through (batch, x, y, z) rows of one batch
    d4, i4 = knn3d.knn_voxels(_cuda(synth.with_batch(q)), _cuda(synth.with_batch(r)), k)
    assert torch.equal(d4, d) and torch.equal(i4, i)


def _jittered(xyz, seed, keep=0.8, hi=None):
    rng = np.random.default_rng(seed)
    out = xyz + rng.integers(-2, 3, xyz.shape)
    if hi is not None:
        out = np.clip(out, 0, hi)
    return np.unique(out.astype(np.int32)[rng.random(xyz.shape[0]) < keep], axis=0)


@pytest.fixture(scope='module')
def big_clouds():
    org = synth.surface_cloud(3, bits=11, n_target=800000)
    rec = _jittered(org, 4, hi=2047)
    lidar = synth.lidar_frame(5)
    return org, rec, lidar, _jittered(lidar, 6)


def test_large_k1_matches_device_brute_force(big_clouds):
    org, rec, lidar, lidar_rec = big_clouds
    assert org.shape[0] >= 790000
    for q, r in ((rec, org), (org, rec), (lidar_rec, lidar)):
        qt, rt = _cuda(synth.with_batch(q)), _cuda(synth.with_batch(r))
        d, i = metrics.nn_search(qt, rt)
        bd, bi = metrics.nn_search_bruteforce(qt, rt)
        assert torch.equal(d, bd) and torch.equal(i, bi)


def test_large_k16_matches_ckdtree(big_clouds):
    from scipy.spatial import cKDTree
    org, rec, _, _ = big_clouds
    q = rec[np.random.default_rng(7).choice(rec.shape[0], 100000, replace=False)]
    d, i = knn3d.knn_voxels(_cuda(q), _cuda(org), 16)
    d, i = d.cpu().numpy(), i.cpu().numpy().astype(np.int64)
    kd, ki = cKDTree(org.astype(np.float64)).query(q.astype(np.float64), k=16)
    want = np.rint(kd * kd).astype(np.int64)
    assert (d == want).all()
    real = ((org[i].astype(np.int64) - q[:, None, :]) ** 2).sum(2)
    assert (real == d).all()                                   # every index realises its distance
    assert (np.diff(d, axis=1) >= 0).all()
    for a, b, da, db in zip(i, ki, d, want):                   # beyond the ties at the K-th distance, same sets
        assert set(a[da < da[-1]]) == set(b[db < db[-1]])


def _float_case(seed, n_q, n_r, scale, grid=None):
    rng = np.random.default_rng(seed)
    if grid is None:
        q = (rng.random((n_q, 3)) * scale - scale / 3).astype(np.float32)
        r = (rng.random((n_r, 3)) * scale - scale / 3).astype(np.float32)
    else:  # coordinates on a grid of `grid` units: many points exactly on cell faces, many equal distances
        q = (rng.integers(-40, 40, (n_q, 3)) * grid).astype(np.float32)
        r = (rng.integers(-40, 40, (n_r, 3)) * grid).astype(np.float32)
    return q, r


@pytest.mark.parametrize('k', [1, 8, 32])
@pytest.mark.parametrize('case', [(1, 4000, 3000, 37.3, None), (2, 3000, 4000, 1e-3, None), (3, 3000, 3000, 5000.0, None),
                                  (4, 3000, 2000, None, 0.25), (5, 2000, 3000, None, 1.0), (6, 2000, 2000, None, 0.3)])
def test_float32_bit_identical_to_numpy(case, k):
    seed, nq, nr, scale, grid = case
    q, r = _float_case(seed, nq, nr, scale, grid)
    want_d, want_i = _brute(q, r, k, np.float32)
    d, i = knn3d.search_rows(_cuda(q), _cuda(r), k)
    assert d.dtype == torch.float32
    assert (d.cpu().numpy().view(np.uint32) == want_d.view(np.uint32)).all()
    assert (i.cpu().numpy() == want_i).all()
    # knn_points: one cloud as a batch of one
    res = knn3d.knn_points(_cuda(q)[None], _cuda(r)[None], K=k)
    assert (res.dists[0].cpu().numpy().view(np.uint32) == want_d.view(np.uint32)).all()
    assert (res.idx[0].cpu().numpy() == want_i).all()


def test_ragged_batches_never_cross_and_pad():
    rng = np.random.default_rng(11)
    sizes_r = [3000, 5, 0, 700]   # batch 1 has fewer than K points, batch 2 has none
    sizes_q = [1000, 40, 30, 500]
    qs, rs = [], []
    for b, (nq, nr) in enumerate(zip(sizes_q, sizes_r)):
        qs.append(synth.with_batch(rng.integers(0, 512, (nq, 3)).astype(np.int32), b))
        rs.append(synth.with_batch(rng.integers(0, 512, (nr, 3)).astype(np.int32), b))
    perm_q, perm_r = rng.permutation(sum(sizes_q)), rng.permutation(sum(sizes_r))  # batches interleaved in the rows
    q, r = np.concatenate(qs)[perm_q], np.concatenate(rs)[perm_r]
    k = 8
    d, i = knn3d.knn_voxels(_cuda(q), _cuda(r), k)
    d, i = d.cpu().numpy(), i.cpu().numpy()
    valid = i >= 0
    assert (r[i[valid], 0] == np.broadcast_to(q[:, :1], i.shape)[valid]).all()  # same batch only
    for b in range(len(sizes_q)):
        qm, rm = q[:, 0] == b, np.nonzero(r[:, 0] == b)[0]
        wd, wi = _brute(q[qm, 1:], r[rm, 1:], k)
        if rm.size:  # brute-force indices within the batch -> rows of r
            wi = np.where(wi >= 0, rm[np.maximum(wi, 0)], -1)
        assert (d[qm] == wd).all() and (i[qm] == wi).all(), b
    assert (i[q[:, 0] == 1][:, 5:] == -1).all() and (d[q[:, 0] == 1][:, 5:] == 0).all()
    assert (i[q[:, 0] == 2] == -1).all() and (d[q[:, 0] == 2] == 0).all()


@pytest.mark.parametrize('name', ['single_ref', 'one_cell_duplicates', 'far_query', 'sparse_2p20'])
def test_degenerate_inputs(name):
    rng = np.random.default_rng(12)
    k = 16
    if name == 'single_ref':
        q, r = rng.integers(0, 1000, (500, 3)), np.array([[7, -3, 12]])
    elif name == 'one_cell_duplicates':  # 600 points on 8 positions: the tie order is by row
        q, r = rng.integers(0, 2, (300, 3)), rng.integers(0, 2, (600, 3))
        k = 32
    elif name == 'far_query':
        r = rng.integers(0, 256, (5000, 3))
        q = np.concatenate([rng.integers(0, 256, (100, 3)), [[1 << 29, -(1 << 29), 5], [-(1 << 29) + 1, 0, 0]]])
    else:  # 1 k points in a 2^20 cube
        r = rng.integers(0, 1 << 20, (1000, 3))
        q = rng.integers(0, 1 << 20, (1000, 3))
    q, r = q.astype(np.int32), r.astype(np.int32)
    want_d, want_i = _brute(q, r, k)
    d, i = knn3d.knn_voxels(_cuda(q), _cuda(r), k)
    assert (d.cpu().numpy() == want_d).all() and (i.cpu().numpy() == want_i).all()
    # the float path on the same points
    fd, fi = _brute(q.astype(np.float32), r.astype(np.float32), k, np.float32)
    d, i = knn3d.search_rows(_cuda(q.astype(np.float32)), _cuda(r.astype(np.float32)), k)
    assert (d.cpu().numpy().view(np.uint32) == fd.view(np.uint32)).all() and (i.cpu().numpy() == fi).all()


def test_knn_points_gradients_and_gather():
    g = torch.Generator().manual_seed(13)
    p1 = (torch.rand(2, 300, 3, generator=g) * 10).cuda().requires_grad_()
    p2 = (torch.rand(2, 400, 3, generator=g) * 10).cuda().requires_grad_()
    l1, l2 = torch.tensor([300, 120]).cuda(), torch.tensor([400, 3]).cuda()
    res = knn3d.knn_points(p1, p2, l1, l2, K=4, return_nn=True)
    idx = res.idx
    assert idx.dtype == torch.int64
    assert (idx[1, 120:] == -1).all() and (res.dists[1, 120:] == 0).all()   # padded queries
    assert (idx[1, :120, 3] == -1).all() and (idx[1, :120, :3] >= 0).all()  # cloud 1 has 3 points
    assert (idx[1, :120, :3] < 3).all() and (res.knn[1, :120, 3] == 0).all()
    w = torch.rand(res.dists.shape, generator=g).cuda()
    (res.dists * w).sum().backward()
    g1, g2 = p1.grad.clone(), p2.grad.clone()
    # autograd of the brute-force formula on the same neighbours
    a1, a2 = p1.detach().clone().requires_grad_(), p2.detach().clone().requires_grad_()
    valid = (idx >= 0).unsqueeze(-1)
    nn = knn3d.knn_gather(a2, idx)
    ref = (((a1.unsqueeze(2) - nn) ** 2) * valid).sum(-1)
    assert torch.allclose(ref, res.dists.detach(), rtol=1e-5, atol=1e-5)
    (ref * w).sum().backward()
    assert torch.allclose(g1, a1.grad, rtol=1e-5, atol=1e-5) and torch.allclose(g2, a2.grad, rtol=1e-5, atol=1e-5)
    # knn_gather with padding
    x = torch.arange(24, dtype=torch.float32).view(2, 4, 3).cuda()
    gi = torch.tensor([[[0, -1], [3, 1]], [[2, 2], [-1, 0]]]).cuda()
    out = knn3d.knn_gather(x, gi, torch.tensor([4, 2]).cuda())
    assert out.shape == (2, 2, 2, 3)
    assert torch.equal(out[0, 0, 0], x[0, 0]) and (out[0, 0, 1] == 0).all() and torch.equal(out[0, 1, 0], x[0, 3])
    assert (out[1, 0] == 0).all() and (out[1, 1, 0] == 0).all() and torch.equal(out[1, 1, 1], x[1, 0])


def test_pc_error_800k_equals_brute_force(big_clouds):
    org, rec, _, _ = big_clouds
    rng = np.random.default_rng(14)
    nrm = rng.normal(size=org.shape)
    nrm = torch.from_numpy(nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).float().cuda()
    o, r = _cuda(org), _cuda(rec)
    got = metrics.pc_error(o, r, 2048, org_normals=nrm, hausdorff=True)
    want = metrics.pc_error(o, r, 2048, org_normals=nrm, hausdorff=True, search=metrics.nn_search_bruteforce)
    assert set(got) == set(want) and 'mseF      (p2plane)' in got and 'h.        (p2point)' in got
    for key, v in want.items():
        assert got[key] == v, key
