"""Host-side pieces of the point normals: the argument checks of fpcc_knn_normals (every bad call comes back as an error
code and a message before any CUDA work), the checks of attributes.estimate_normals and metrics.pc_error(normals_k=),
and hand-computed cases of the CPU oracle's definition (tests/normals_oracle.py), so these run without a device."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from tests import normals_oracle as NO


@pytest.fixture(scope='module')
def lib():
    from fastpcc_b200 import _lib
    return _lib.load()


@pytest.fixture(scope='module')
def buf():
    b = (C.c_uint8 * 4096)()
    return b, (C.addressof(b) + 15) & ~15


def _call(lib, p, ws=2048, k=8, n_batch=1, n=8, ld=3, col=0, b=-1, pts=True, out=True, work=True, align=0,
          viewpoint=None):
    return lib.fpcc_knn_normals(k, n_batch, p if pts else None, n, ld, col, b, viewpoint, p if out else None,
                                (p + align) if work else None, ws, None)


def _fails(lib, rc, text):
    assert rc != 0
    msg = lib.fpcc_last_error()
    assert msg and text in msg.decode(), msg
    assert msg.decode().startswith('knn_normals: '), msg


def test_k_outside_3_to_32_is_rejected(lib, buf):
    _, p = buf
    for k in (-1, 0, 1, 2, 33):
        _fails(lib, _call(lib, p, k=k), 'k must be in 3..32')


def test_bad_row_layouts_are_rejected(lib, buf):
    _, p = buf
    _fails(lib, _call(lib, p, ld=2), 'bad row layout')             # xyz does not fit the row
    _fails(lib, _call(lib, p, ld=4, col=2), 'bad row layout')      # columns 2..4 of a 4-wide row
    _fails(lib, _call(lib, p, col=-1), 'bad row layout')
    _fails(lib, _call(lib, p, ld=4, col=1, b=1), 'bad row layout')  # batch inside xyz
    _fails(lib, _call(lib, p, ld=4, col=1, b=4), 'bad row layout')  # batch past the row


def test_batch_count_is_checked(lib, buf):
    _, p = buf
    kw = dict(ld=4, col=1, b=0)
    _fails(lib, _call(lib, p, n_batch=1024, **kw), 'n_batch must be in 1..1023')
    _fails(lib, _call(lib, p, n_batch=0, **kw), 'n_batch must be in 1..1023')
    _fails(lib, _call(lib, p, n_batch=2), 'one cloud')  # no batch column but several batches


def test_workspace_size_pointers_and_viewpoint_are_checked(lib, buf):
    _, p = buf
    need = lib.fpcc_knn_workspace(8, 1)   # the workspace of fpcc_knn_search
    assert need <= 4096 - 16
    _fails(lib, _call(lib, p, ws=need - 1), 'workspace too small')
    _fails(lib, _call(lib, p, ws=16), 'workspace too small')
    _fails(lib, _call(lib, p, align=4), '16-byte aligned')
    for missing in ('pts', 'out', 'work'):
        _fails(lib, _call(lib, p, **{missing: False}), 'NULL pointer')
    _fails(lib, _call(lib, p, n=-1), 'row counts')
    _fails(lib, _call(lib, p, n=1 << 31), 'row counts')
    for bad in ((0.0, float('nan'), 1.0), (float('inf'), 0.0, 0.0)):
        _fails(lib, _call(lib, p, ws=need, viewpoint=(C.c_double * 3)(*bad)), 'viewpoint must be three finite numbers')


def test_python_layer_raises_with_the_message():
    from fastpcc_b200 import attributes, metrics
    q = torch.zeros(4, 3, dtype=torch.int32)
    with pytest.raises(RuntimeError, match='int32 CUDA'):
        attributes.estimate_normals(q)                      # host tensor
    with pytest.raises(RuntimeError, match='int32 CUDA'):
        attributes.estimate_normals(q.float())              # float rows
    for k in (2, 33, 8.0, True):
        with pytest.raises(RuntimeError, match='K must be an int in 3..32'):
            attributes.estimate_normals(q, K=k)
    with pytest.raises(RuntimeError, match='int32 CUDA'):   # numpy integers are accepted as K
        attributes.estimate_normals(q, K=np.int64(16))
    for vp in ((0, 0), (0, 0, float('nan')), 'abc', (0, 0, 0, 0)):
        with pytest.raises(RuntimeError, match='viewpoint must be three finite numbers'):
            attributes.estimate_normals(q, viewpoint=vp)
    with pytest.raises(RuntimeError, match='org_normals or normals_k, not both'):  # before any search
        metrics.pc_error(q, q, 1024, org_normals=torch.zeros(4, 3), normals_k=8)


def _grid(nx, ny):
    return np.stack(np.meshgrid(np.arange(nx), np.arange(ny), indexing='ij'), -1).reshape(-1, 2)


def test_plane_z_const_gives_z():
    g = _grid(10, 10)
    pts = np.concatenate([g, np.full((g.shape[0], 1), 7)], 1)
    for k in (3, 8, 16, 32):
        assert (NO.normals(pts, k) == np.array([0, 0, 1], np.float32)).all(), k
    # the same plane seen from below: every normal points down
    assert (NO.normals(pts, 8, viewpoint=(4.5, 4.5, -10.0)) == np.array([0, 0, -1], np.float32)).all()


def test_voxelised_diagonal_plane():
    # x + y = 9 on a voxel grid: rows (x, 9 - x, z)
    x, z = _grid(10, 6).T
    pts = np.stack([x, 9 - x, z], 1)
    want = np.float32(1 / math.sqrt(2))
    # K = 3: a row off the z ends sees itself and its two z neighbours (d2 = 1; the in-plane steps are at d2 = 2),
    # a collinear neighbourhood: the zero vector
    got = NO.normals(pts, 3)
    inner = (z > 0) & (z < 5)
    assert (got[inner] == 0).all() and (got[~inner] != 0).any()
    for k in (8, 16):
        got = NO.normals(pts, k)
        np.testing.assert_allclose(got, np.broadcast_to([want, want, 0], got.shape), rtol=0, atol=1e-7)
        assert (got[:, 0] > 0).all() and (got[:, 1] > 0).all()   # a tie in magnitude: the x axis decides, + + 0
    got = NO.normals(pts, 8, viewpoint=(0.0, 0.0, 3.0))         # the origin side of the plane: - - 0
    np.testing.assert_allclose(got, np.broadcast_to([-want, -want, 0], got.shape), rtol=0, atol=1e-7)


def test_k3_on_a_plane_takes_the_whole_unit_shell():
    # an interior row of a planar grid: itself at 0, four rows at d2 = 1; K = 3 ends inside that shell, and all of it
    # is N(p): n = 5, sum d = 0, sum d d^T = diag(2, 2, 0), M = diag(10, 10, 0)
    g = _grid(5, 5)
    pts = np.concatenate([g, np.zeros((25, 1), np.int64)], 1)
    cnt, M = NO.scatter(pts, 3)
    centre = 12
    assert (pts[centre] == [2, 2, 0]).all()
    assert cnt[centre] == 5 and list(M[centre]) == [10, 10, 0, 0, 0, 0]
    corner = 0  # itself and two rows at d2 = 1: n = 3, M = 3 diag(1, 1, 0) - (1, 1, 0)(1, 1, 0)^T
    assert cnt[corner] == 3 and list(M[corner]) == [2, 2, 0, -1, 0, 0]
    assert (NO.normals(pts, 3) == np.array([0, 0, 1], np.float32)).all()
    # batch rows: the same plane as batch 1 next to another batch's rows changes nothing
    other = np.concatenate([np.zeros((25, 1), np.int64), pts + [0, 0, 1]], 1)
    both = np.concatenate([other, np.concatenate([np.ones((25, 1), np.int64), pts], 1)])
    cnt4, M4 = NO.scatter(both, 3)
    assert (cnt4[25:] == cnt).all() and (M4[25:] == M).all()


def test_lines_duplicates_and_tiny_clouds_give_zero():
    line = np.stack([np.arange(20), 2 * np.arange(20), np.full(20, 5)], 1)
    assert (NO.normals(line, 8) == 0).all()                     # rank 1
    assert (NO.normals(np.array([[0, 0, 0], [3, 1, 2]]), 3) == 0).all()  # n = 2 < 3
    dup = np.array([[1, 1, 1]] * 6 + [[4, 4, 4]] * 3)           # duplicates on two positions: collinear
    assert (NO.normals(dup, 4) == 0).all()
    # a row whose batch id lies outside [0, n_batch) gets zero; its own batch's rows are unaffected
    tri = np.array([[0, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, 0], [5, 0, 0, 0]])
    got = NO.normals(tri, 3, n_batch=2)
    assert (got[:3] == np.array([0, 0, 1], np.float32)).all() and (got[3] == 0).all()


def test_orientation_rules():
    # a tilted plane z = 2x: normal +-(-2, 0, 1)/sqrt 5; the x component is the largest in magnitude, made positive
    x, y = _grid(8, 8).T
    pts = np.stack([x, y, 2 * x], 1)
    want = np.array([2, 0, -1]) / math.sqrt(5)
    np.testing.assert_allclose(NO.normals(pts, 8), np.broadcast_to(want, (64, 3)), rtol=0, atol=1e-7)
    # with a viewpoint above the plane (z larger than 2x): the normal points to it
    np.testing.assert_allclose(NO.normals(pts, 8, viewpoint=(0.0, 0.0, 100.0)), np.broadcast_to(-want, (64, 3)),
                               rtol=0, atol=1e-7)
