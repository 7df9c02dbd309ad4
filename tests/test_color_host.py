"""Host-side pieces of the colour attributes: the argument checks of fpcc_nn_tie_attr (every bad call comes back as an
error code and a message before any CUDA work) and hand-computed cases of the CPU oracle's definitions (YUV, tie sets,
the rounding of recolouring), so these run without a device."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import color_oracle as CO


@pytest.fixture(scope='module')
def lib():
    from fastpcc_b200 import _lib
    return _lib.load()


@pytest.fixture(scope='module')
def buf():
    b = (C.c_uint8 * 4096)()
    return b, (C.addressof(b) + 15) & ~15


def _call(lib, p, ws=2048, n_batch=1, nq=8, q_ld=3, q_col=0, q_b=-1, nr=8, r_ld=3, r_col=0, r_b=-1,
          query=True, ref=True, rgb=True, d2=True, count=True, sums=True, work=True, align=0):
    return lib.fpcc_nn_tie_attr(n_batch, p if query else None, nq, q_ld, q_col, q_b, p if ref else None, nr, r_ld,
                                r_col, r_b, p if rgb else None, p if d2 else None, p if count else None,
                                p if sums else None, (p + align) if work else None, ws, None)


def _fails(lib, rc, text):
    assert rc != 0
    msg = lib.fpcc_last_error()
    assert msg and text in msg.decode(), msg
    assert msg.decode().startswith('nn_tie_attr: '), msg


def test_bad_row_layouts_are_rejected(lib, buf):
    _, p = buf
    _fails(lib, _call(lib, p, q_ld=2), 'bad row layout')                    # xyz does not fit the row
    _fails(lib, _call(lib, p, r_ld=4, r_col=2), 'bad row layout')           # columns 2..4 of a 4-wide row
    _fails(lib, _call(lib, p, q_col=-1), 'bad row layout')
    _fails(lib, _call(lib, p, q_ld=4, q_col=1, q_b=1, r_ld=4, r_col=1, r_b=0), 'bad row layout')  # batch inside xyz
    _fails(lib, _call(lib, p, q_ld=4, q_col=1, q_b=4, r_ld=4, r_col=1, r_b=0), 'bad row layout')  # batch past the row
    _fails(lib, _call(lib, p, q_ld=4, q_col=1, q_b=0), 'on both sides or on neither')  # batch column on one side only


def test_batch_count_is_checked(lib, buf):
    _, p = buf
    kw = dict(q_ld=4, q_col=1, q_b=0, r_ld=4, r_col=1, r_b=0)
    _fails(lib, _call(lib, p, n_batch=1024, **kw), 'n_batch must be in 1..1023')
    _fails(lib, _call(lib, p, n_batch=0, **kw), 'n_batch must be in 1..1023')
    _fails(lib, _call(lib, p, n_batch=2), 'one cloud')  # no batch column but several batches


def test_workspace_size_and_pointers_are_checked(lib, buf):
    _, p = buf
    need = lib.fpcc_knn_workspace(8, 1)   # the workspace of fpcc_knn_search
    _fails(lib, _call(lib, p, ws=need - 1), 'workspace too small')
    _fails(lib, _call(lib, p, ws=16), 'workspace too small')
    _fails(lib, _call(lib, p, align=4), '16-byte aligned')
    for missing in ('query', 'ref', 'rgb', 'd2', 'count', 'sums', 'work'):
        _fails(lib, _call(lib, p, **{missing: False}), 'NULL pointer')
    _fails(lib, _call(lib, p, nq=-1), 'row counts')
    _fails(lib, _call(lib, p, nr=1 << 31), 'row counts')


def test_python_layer_raises_with_the_message():
    from fastpcc_b200 import attributes
    q = torch.zeros(4, 3, dtype=torch.int32)
    with pytest.raises(RuntimeError, match='int32 CUDA'):
        attributes.nearest_tie_attr(q, q, torch.zeros(4, 3, dtype=torch.uint8))      # host tensors
    with pytest.raises(RuntimeError, match='int32 CUDA'):
        attributes.recolor(q.float(), torch.zeros(4, 3, dtype=torch.uint8), q)
    from fastpcc_b200 import metrics
    with pytest.raises(RuntimeError, match='both org_colors and rec_colors'):
        metrics.pc_error(q, q, 1024, org_colors=torch.zeros(4, 3, dtype=torch.uint8))
    with pytest.raises(RuntimeError, match='rec_colors must be uint8'):  # before any search
        metrics.pc_error(q, q, 1024, org_colors=torch.zeros(4, 3, dtype=torch.uint8),
                         rec_colors=torch.zeros(4, 3, dtype=torch.int32))


def test_yuv_of_black_white_and_primaries():
    from fastpcc_b200 import metrics
    rgb = np.array([[0, 0, 0], [255, 255, 255], [255, 0, 0], [0, 255, 0], [0, 0, 255]])
    want = np.array([[0.0, 0.5, 0.5],
                     [1.0, 0.5, 0.5],
                     [0.2126, 0.5 - 0.1146, 1.0],
                     [0.7152, 0.5 - 0.3854, 0.5 - 0.4542],
                     [0.0722, 1.0, 0.5 - 0.0458]])
    np.testing.assert_allclose(CO.yuv(rgb), want, rtol=0, atol=1e-15)
    # the product's conversion (double torch ops, no device needed) is the same expression
    np.testing.assert_array_equal(metrics._yuv(torch.from_numpy(rgb)).numpy(), CO.yuv(rgb))


def test_six_face_neighbours_are_one_tie_set():
    # a voxel at the origin of a 3^3 block: 6 neighbours at d2 = 1, 12 at 2, 8 at 3
    g = np.stack(np.meshgrid(*[np.arange(-1, 2)] * 3, indexing='ij'), -1).reshape(-1, 3)
    ref = g[np.abs(g).sum(1) > 0]                       # the block without its centre
    rgb = np.zeros((ref.shape[0], 3), np.uint8)
    face = np.abs(ref).sum(1) == 1
    rgb[face] = np.array([[10, 20, 30], [11, 21, 31], [12, 22, 32], [13, 23, 33], [14, 24, 34], [15, 25, 35]])
    rgb[~face] = 255                                    # farther rows must not count
    d, n, s, i = CO.ties(np.zeros((1, 3), np.int32), ref, rgb)
    assert d[0] == 1 and n[0] == 6 and (s[0] == [75, 135, 195]).all() and i[0] == np.nonzero(face)[0][0]
    assert (s[0] / n[0] == [12.5, 22.5, 32.5]).all()
    # the same with batch rows: another batch's nearer point is invisible
    q4 = np.array([[1, 0, 0, 0]])
    r4 = np.concatenate([np.concatenate([np.ones((ref.shape[0], 1), int), ref], 1), [[0, 0, 0, 0]]])
    rgb4 = np.concatenate([rgb, [[0, 0, 0]]]).astype(np.uint8)
    d4, n4, s4, _ = CO.ties(q4, r4, rgb4)
    assert d4[0] == 1 and n4[0] == 6 and (s4[0] == s[0]).all()


def test_two_way_blend_rounds_half_up():
    # one reconstructed point: its forward set is the nearest original (colour 10), its backward set is every
    # original point (mean (10 + 12) / 2 = 11): the blend 10.5 rounds up to 11, the forward mean alone is 10
    org = np.array([[1, 0, 0], [5, 0, 0]])
    org_rgb = np.array([[10, 10, 10], [12, 12, 12]], np.uint8)
    rec = np.array([[0, 0, 0]])
    assert (CO.recolor(org, org_rgb, rec) == 11).all()
    assert (CO.recolor(org, org_rgb, rec, two_way=False) == 10).all()
    # forward tie (10 and 11 at the same distance): 10.5 rounds up to 11 in one-way mode too
    org = np.array([[1, 0, 0], [-1, 0, 0]])
    org_rgb = np.array([[10, 0, 255], [11, 1, 254]], np.uint8)
    assert (CO.recolor(org, org_rgb, rec, two_way=False) == [[11, 1, 255]]).all()
    # a reconstructed point whose batch has no original point gets colour 0
    got = CO.recolor(np.array([[0, 1, 0, 0]]), np.array([[9, 9, 9]], np.uint8), np.array([[0, 0, 0, 0], [1, 0, 0, 0]]))
    assert (got == [[9, 9, 9], [0, 0, 0]]).all()
