"""Host-side argument checks of fpcc_knn_search / fpcc_knn_workspace: every bad call comes back as an error code and a
message before any CUDA work, so these run without a device."""
import ctypes as C

import pytest


@pytest.fixture(scope='module')
def lib():
    from fastpcc_b200 import _lib
    return _lib.load()


@pytest.fixture(scope='module')
def buf():
    b = (C.c_uint8 * 4096)()
    return b, (C.addressof(b) + 15) & ~15


def _call(lib, p, ws=2048, coord_type=0, k=4, n_batch=1, nq=8, q_ld=3, q_col=0, q_b=-1, nr=8, r_ld=3, r_col=0, r_b=-1,
          query=True, ref=True, dist=True, idx=True, work=True, align=0):
    return lib.fpcc_knn_search(coord_type, k, n_batch, p if query else None, nq, q_ld, q_col, q_b, p if ref else None,
                               nr, r_ld, r_col, r_b, p if dist else None, p if idx else None,
                               (p + align) if work else None, ws, None)


def _fails(lib, rc, text):
    assert rc != 0
    msg = lib.fpcc_last_error()
    assert msg and text in msg.decode(), msg


def test_k_outside_1_to_32_is_rejected(lib, buf):
    _, p = buf
    _fails(lib, _call(lib, p, k=0), 'k must be in 1..32')
    _fails(lib, _call(lib, p, k=33), 'k must be in 1..32')
    _fails(lib, _call(lib, p, k=-1), 'k must be in 1..32')


def test_bad_row_layouts_are_rejected(lib, buf):
    _, p = buf
    _fails(lib, _call(lib, p, q_ld=2), 'bad row layout')                    # xyz does not fit the row
    _fails(lib, _call(lib, p, r_ld=4, r_col=2), 'bad row layout')           # columns 2..4 of a 4-wide row
    _fails(lib, _call(lib, p, q_col=-1), 'bad row layout')
    _fails(lib, _call(lib, p, q_ld=4, q_col=1, q_b=1, r_ld=4, r_col=1, r_b=0), 'bad row layout')  # batch inside xyz
    _fails(lib, _call(lib, p, q_ld=4, q_col=1, q_b=4, r_ld=4, r_col=1, r_b=0), 'bad row layout')  # batch past the row
    _fails(lib, _call(lib, p, q_ld=4, q_col=1, q_b=0), 'on both sides or on neither')  # batch column on one side only
    _fails(lib, _call(lib, p, coord_type=2), 'coord_type')


def test_batch_count_is_checked(lib, buf):
    _, p = buf
    kw = dict(q_ld=4, q_col=1, q_b=0, r_ld=4, r_col=1, r_b=0)
    _fails(lib, _call(lib, p, n_batch=1024, **kw), 'n_batch must be in 1..1023')
    _fails(lib, _call(lib, p, n_batch=0, **kw), 'n_batch must be in 1..1023')
    _fails(lib, _call(lib, p, n_batch=2), 'one cloud')  # no batch column but several batches


def test_workspace_size_and_pointers_are_checked(lib, buf):
    _, p = buf
    need = lib.fpcc_knn_workspace(8, 1)
    assert need > 8 * 16
    _fails(lib, _call(lib, p, ws=need - 1), 'workspace too small')
    _fails(lib, _call(lib, p, ws=16), 'workspace too small')
    _fails(lib, _call(lib, p, align=4), '16-byte aligned')
    for missing in ('query', 'ref', 'dist', 'idx', 'work'):
        _fails(lib, _call(lib, p, **{missing: False}), 'NULL pointer')
    _fails(lib, _call(lib, p, nq=-1), 'row counts')
    _fails(lib, _call(lib, p, nr=1 << 31), 'row counts')
    # workspace grows with the reference rows and the batch count
    assert lib.fpcc_knn_workspace(1 << 20, 1) > lib.fpcc_knn_workspace(1 << 10, 1)
    assert lib.fpcc_knn_workspace(1 << 10, 1023) > lib.fpcc_knn_workspace(1 << 10, 1)


def test_python_layer_raises_with_the_message():
    import torch
    from fastpcc_b200 import knn3d
    with pytest.raises(RuntimeError, match='K must be in 1..32'):
        knn3d.knn_points(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3), K=33)
    with pytest.raises(RuntimeError, match='int32'):
        knn3d.knn_voxels(torch.zeros(4, 4), torch.zeros(4, 4))
