"""fpcc_nn_tie_attr (attributes.nearest_tie_attr), attributes.recolor and the colour keys of metrics.pc_error against
the CPU oracle (tests/color_oracle.py): the search exactly (d2, count, sums), recolouring byte for byte, the colour
figures within 1e-12 relative."""
import math

import numpy as np
import pytest
import torch

from fastpcc_b200 import attributes, metrics, synth
from tests import color_oracle as CO

pytestmark = pytest.mark.gpu


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _rgb(rng, n):
    return rng.integers(0, 256, (n, 3)).astype(np.uint8)


def _check(q, r, rgb, n_batch=None):
    d, n, s = attributes.nearest_tie_attr(_cuda(q), _cuda(r), _cuda(rgb), n_batch)
    assert d.dtype == torch.int64 and n.dtype == torch.int32 and s.dtype == torch.int64 and tuple(s.shape) == (q.shape[0], 3)
    wd, wn, ws, _ = CO.ties(q, r, rgb)
    assert (d.cpu().numpy() == wd).all()
    assert (n.cpu().numpy() == wn).all()
    assert (s.cpu().numpy() == ws).all()
    return wn


_INT_CASES = {6: (3000, 1500), 10: (8000, 3000), 16: (5000, 5000), 20: (20000, 5000)}


@pytest.mark.parametrize('bits', [6, 10, 16, 20])
def test_random_clouds_match_oracle_exactly(bits):
    nq, nr = _INT_CASES[bits]
    rng = np.random.default_rng(200 + bits)
    half = 1 << (bits - 1)
    q = rng.integers(-half, half, (nq, 3)).astype(np.int32)
    r = rng.integers(-half, half, (nr, 3)).astype(np.int32)
    rgb = _rgb(rng, nr)
    _check(q, r, rgb)
    _check(synth.with_batch(q), synth.with_batch(r), rgb)   # (batch, x, y, z) rows of one batch


def test_ragged_interleaved_batches():
    rng = np.random.default_rng(21)
    sizes_r = [3000, 40, 0, 700]   # batch 1 is scanned (<= 64 points), batch 2 has none
    sizes_q = [1000, 50, 30, 500]
    qs, rs = [], []
    for b, (nq, nr) in enumerate(zip(sizes_q, sizes_r)):
        qs.append(synth.with_batch(rng.integers(0, 64, (nq, 3)).astype(np.int32), b))
        rs.append(synth.with_batch(rng.integers(0, 64, (nr, 3)).astype(np.int32), b))
    q = np.concatenate(qs)[rng.permutation(sum(sizes_q))]
    r = np.concatenate(rs)[rng.permutation(sum(sizes_r))]
    rgb = _rgb(rng, r.shape[0])
    wn = _check(q, r, rgb)
    assert (wn[q[:, 0] == 2] == 0).all() and (wn[q[:, 0] != 2] > 0).all()
    _check(q, r, rgb, n_batch=4)


@pytest.mark.parametrize('name', ['single_ref', 'one_cell_duplicates', 'far_query', 'sparse_2p20', 'lattice'])
def test_degenerate_inputs(name):
    rng = np.random.default_rng(22)
    if name == 'single_ref':
        q, r = rng.integers(0, 1000, (500, 3)), np.array([[7, -3, 12]])
    elif name == 'one_cell_duplicates':  # 600 points on 8 positions: tie sets of about 75 rows
        q, r = rng.integers(0, 2, (300, 3)), rng.integers(0, 2, (600, 3))
    elif name == 'far_query':            # the last two queries take the batch scan
        r = rng.integers(0, 256, (5000, 3))
        q = np.concatenate([rng.integers(0, 256, (100, 3)), [[1 << 29, -(1 << 29), 5], [-(1 << 29) + 1, 0, 0]]])
    elif name == 'sparse_2p20':          # 1 k points in a 2^20 cube
        r = rng.integers(0, 1 << 20, (1000, 3))
        q = rng.integers(0, 1 << 20, (1000, 3))
    else:                                # even lattice: 1, 2, 4 or 8 equidistant neighbours per query
        g = np.stack(np.meshgrid(*[np.arange(16)] * 3, indexing='ij'), -1).reshape(-1, 3)
        q, r = g, g[(g % 2 == 0).all(1)]
    q, r = q.astype(np.int32), r.astype(np.int32)
    wn = _check(q, r, _rgb(rng, r.shape[0]))
    if name == 'lattice':
        assert set(np.unique(wn)) == {1, 2, 4, 8}
    if name == 'one_cell_duplicates':
        assert wn.min() > 30


@pytest.fixture(scope='module')
def big_colored():
    org, org_rgb = synth.colored_surface(3, bits=11, n_target=800000)
    rng = np.random.default_rng(4)
    rec = org + rng.integers(-2, 3, org.shape)
    rec = np.unique(np.clip(rec, 0, 2047).astype(np.int32)[rng.random(org.shape[0]) < 0.8], axis=0)
    return org, org_rgb, rec, CO.ties(rec, org, org_rgb)


def test_800k_search_matches_nn_search_and_oracle(big_colored):
    org, org_rgb, rec, (wd, wn, ws, _) = big_colored
    assert org.shape[0] >= 790000
    d, n, s = attributes.nearest_tie_attr(_cuda(rec), _cuda(org), _cuda(org_rgb))
    d1, _ = metrics.nn_search(_cuda(rec), _cuda(org))
    assert torch.equal(d, d1)
    assert (d.cpu().numpy() == wd).all() and (n.cpu().numpy() == wn).all() and (s.cpu().numpy() == ws).all()
    assert wn.max() > 1   # jittered geometry has ties


def test_recolor_of_a_permutation_returns_the_colours():
    org, rgb = synth.colored_surface(5, bits=10, n_target=50000)
    perm = np.random.default_rng(5).permutation(org.shape[0])
    for two_way in (True, False):
        got = attributes.recolor(_cuda(org), _cuda(rgb), _cuda(org[perm]), two_way=two_way)
        assert got.dtype == torch.uint8 and (got.cpu().numpy() == rgb[perm]).all()


@pytest.mark.parametrize('two_way', [True, False])
def test_recolor_of_jittered_geometry_matches_oracle(big_colored, two_way):
    org, org_rgb, rec, fwd = big_colored
    got = attributes.recolor(_cuda(org), _cuda(org_rgb), _cuda(rec), two_way=two_way).cpu().numpy()
    want = CO.recolor(org, org_rgb, rec, two_way=two_way, forward=fwd)
    assert (got == want).all()


def test_recolor_rounds_half_up():
    # the constructed cases of test_color_host.py::test_two_way_blend_rounds_half_up, on the device
    rec = _cuda(np.array([[0, 0, 0]], np.int32))
    org, org_rgb = _cuda(np.array([[1, 0, 0], [5, 0, 0]], np.int32)), _cuda(np.array([[10] * 3, [12] * 3], np.uint8))
    assert (attributes.recolor(org, org_rgb, rec).cpu() == 11).all()
    assert (attributes.recolor(org, org_rgb, rec, two_way=False).cpu() == 10).all()
    org, org_rgb = _cuda(np.array([[1, 0, 0], [-1, 0, 0]], np.int32)), _cuda(np.array([[10, 0, 255], [11, 1, 254]], np.uint8))
    assert attributes.recolor(org, org_rgb, rec, two_way=False).cpu().tolist() == [[11, 1, 255]]


def test_recolor_never_crosses_batches():
    rng = np.random.default_rng(7)
    org0, rgb0 = synth.colored_surface(8, bits=8, n_target=5000)
    org1 = org0 + 1                       # batch 1 sits next to batch 0, with colours no batch-0 point has
    rgb0 = np.minimum(rgb0, 100).astype(np.uint8)
    rgb1 = np.full_like(rgb0, 200)
    org = np.concatenate([synth.with_batch(org0, 0), synth.with_batch(org1, 1)])
    rgb = np.concatenate([rgb0, rgb1])
    rec = np.concatenate([synth.with_batch(org1, 0), synth.with_batch(org0, 1), synth.with_batch(org0[:10], 2)])
    perm = rng.permutation(org.shape[0])
    for two_way in (True, False):
        got = attributes.recolor(_cuda(org[perm]), _cuda(rgb[perm]), _cuda(rec), two_way=two_way).cpu().numpy()
        b = rec[:, 0]
        assert (got[b == 0] <= 100).all() and (got[b == 1] == 200).all() and (got[b == 2] == 0).all()
        assert (got == CO.recolor(org[perm], rgb[perm], rec, two_way=two_way)).all()


def _color_keys(out):
    return {k: v for k, v in out.items() if k.startswith('c[')}


def test_pc_error_colours_match_oracle():
    org, org_rgb = synth.colored_surface(9, bits=10, n_target=60000)
    rng = np.random.default_rng(9)
    rec = np.unique(np.clip(org + rng.integers(-1, 2, org.shape), 0, 1023).astype(np.int32), axis=0)
    rec_rgb = CO.recolor(org, org_rgb, rec)
    rec_rgb = np.clip(rec_rgb.astype(int) + rng.integers(-6, 7, rec_rgb.shape), 0, 255).astype(np.uint8)
    o, r = _cuda(org), _cuda(rec)
    plain = metrics.pc_error(o, r, 1024, hausdorff=True)
    got = metrics.pc_error(o, r, 1024, hausdorff=True, org_colors=_cuda(org_rgb), rec_colors=_cuda(rec_rgb))
    for key, v in plain.items():      # the geometry keys are untouched
        assert got[key] == v, key
    want = CO.color_keys(org, org_rgb, rec, rec_rgb)
    assert set(got) == set(plain) | set(want) and len(want) == 18
    for key, v in want.items():
        assert math.isclose(got[key], v, rel_tol=1e-12), (key, got[key], v)
    assert all(0 < want[f'c[{i}],    F'] for i in range(3))
    # the batch column is ignored, as for the geometry keys
    got4 = metrics.pc_error(_cuda(synth.with_batch(org)), _cuda(synth.with_batch(rec)), 1024,
                            org_colors=_cuda(org_rgb), rec_colors=_cuda(rec_rgb))
    assert _color_keys(got4) == _color_keys(got)


def test_pc_error_identical_clouds_give_inf_colour_psnr():
    org, rgb = synth.colored_surface(10, bits=10, n_target=30000)
    perm = np.random.default_rng(10).permutation(org.shape[0])
    out = metrics.pc_error(_cuda(org), _cuda(org[perm]), 1024, org_colors=_cuda(rgb), rec_colors=_cuda(rgb[perm]))
    for tag in ('1', '2', 'F'):
        for i in range(3):
            assert out[f'c[{i}],    {tag}'] == 0 and out[f'c[{i}],PSNR{tag}'] == float('inf')


def test_pc_error_colours_800k(big_colored):
    org, org_rgb, rec, _ = big_colored
    rec_rgb = attributes.recolor(_cuda(org), _cuda(org_rgb), _cuda(rec))
    out = metrics.pc_error(_cuda(org), _cuda(rec), 2048, org_colors=_cuda(org_rgb), rec_colors=rec_rgb)
    assert len(_color_keys(out)) == 18
    assert all(math.isfinite(out[f'c[{i}],PSNR{t}']) and out[f'c[{i}],PSNR{t}'] > 20 for i in range(3) for t in '12F')
