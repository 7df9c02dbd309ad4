"""Host-side pieces of the fp16 / bf16 tensor-core GEMMs: every argument check of fpcc_spconv_f16 and fpcc_linear_f16
comes back as an error code and its message before any CUDA work, and hand-computed cases of the fp64 oracle
(tests/f16_gemm_oracle.py), its table builders and its covering design, so these run without a device.  Every call
below has exactly one bad argument: a call that passed the checks would launch on the dummy buffer."""
import ctypes as C

import pytest
import torch

from tests import f16_gemm_oracle as FO


@pytest.fixture(scope='module')
def lib():
    from fastpcc_b200 import _lib
    return _lib.load()


_BUF = (C.c_uint8 * 4096)()


@pytest.fixture(scope='module')
def p():
    return (C.addressof(_BUF) + 15) & ~15


def _fails(lib, rc, prefix, text):
    assert rc != 0
    msg = lib.fpcc_last_error().decode()
    assert msg.startswith(prefix + ': ') and text in msg, msg


def _conv(lib, p, feats=0, dtype=0, n_in=4, c_in=16, weight=512, kvol=27, c_out=16, table=1024, ld=4, n_out=4,
          act=0, post_act=0, out=2048, out_type=2):
    ptr = lambda off: None if off is None else p + off  # noqa: E731
    return lib.fpcc_spconv_f16(ptr(feats), dtype, n_in, c_in, ptr(weight), kvol, c_out, ptr(table), ld, n_out, None, None,
                               act, 0.0, None, post_act, 0.0, ptr(out), out_type, None)


def _lin(lib, p, a=0, dtype=0, m=4, k=16, w=512, n=16, sel=False, sel_out=1024, offsets=1040, n_groups=2, n_sel=4,
         act=0, post_act=0, out=2048, out_type=2):
    ptr = lambda off: None if off is None else p + off  # noqa: E731
    if sel:
        return lib.fpcc_linear_f16(ptr(a), dtype, m, k, ptr(w), n, p + 1008, ptr(sel_out), ptr(offsets), n_groups, n_sel,
                                   None, act, 0.0, None, post_act, 0.0, ptr(out), out_type, None)
    return lib.fpcc_linear_f16(ptr(a), dtype, m, k, ptr(w), n, None, None, None, 1, 0, None, act, 0.0, None, post_act, 0.0,
                               ptr(out), out_type, None)


def test_spconv_f16_rejects_bad_arguments(lib, p):
    name = 'spconv_f16'
    for kw in ({'feats': None}, {'weight': None}, {'table': None}, {'out': None}):
        _fails(lib, _conv(lib, p, **kw), name, 'NULL pointer')
    for kw in ({'kvol': 0}, {'kvol': 33}, {'kvol': -1}, {'ld': 3}, {'n_out': 0}, {'n_out': -5, 'ld': 0}, {'n_in': 0}):
        _fails(lib, _conv(lib, p, **kw), name, 'bad sizes')


@pytest.mark.parametrize('entry', ['conv', 'linear', 'linear_sel'])
def test_common_checks_of_both_entry_points(lib, p, entry):
    if entry == 'conv':
        call = lambda **kw: _conv(lib, p, **{('c_in' if k == 'k' else 'c_out' if k == 'n' else k): v for k, v in kw.items()})  # noqa: E731
    else:
        call = lambda **kw: _lin(lib, p, sel=entry == 'linear_sel', **{('a' if k == 'feats' else k): v for k, v in kw.items()})  # noqa: E731
    g = 'f16 GEMM'
    for dt in (-1, 2):
        _fails(lib, call(dtype=dt), g, 'dtype must be 0 (fp16) or 1 (bf16)')
    for ot in (-1, 3):
        _fails(lib, call(out_type=ot), g, 'out_type must be')
    for kw in ({'act': -1}, {'act': 3}, {'post_act': -1}, {'post_act': 3}):
        _fails(lib, call(**kw), g, 'bad activation code')
    for kw in ({'k': 8}, {'k': 0}, {'k': 20}, {'k': 36}, {'n': 15}, {'n': 1}, {'n': 0}):
        _fails(lib, call(**kw), g, 'needs C_in % 8 == 0, C_in >= 16, C_out >= 16')
    for kw in ({'feats': 2}, {'feats': 8}, {'w': 516} if entry != 'conv' else {'weight': 516}, {'out': 2052}):
        _fails(lib, call(**kw), g, 'pointers must be 16-byte aligned')


def test_linear_f16_rejects_bad_arguments(lib, p):
    name = 'linear_f16'
    for kw in ({'a': None}, {'w': None}, {'out': None}, {'m': 0}, {'m': -3}):
        _fails(lib, _lin(lib, p, **kw), name, 'bad arguments')
        _fails(lib, _lin(lib, p, sel=True, **kw), name, 'bad arguments')
    for kw in ({'sel_out': None}, {'offsets': None}, {'n_groups': 0}, {'n_groups': -1}, {'n_sel': 0}, {'n_sel': -2}):
        _fails(lib, _lin(lib, p, sel=True, **kw), name, 'incomplete selection')


# ---- the oracle by hand -------------------------------------------------------------------------------------------------
def test_oracle_spconv_by_hand():
    f = torch.tensor([[1.0, 2.0], [3.0, 4.0], [5.0, 6.0]])
    w_t = torch.tensor([[[1.0, 0.0], [0.0, 1.0]], [[1.0, 1.0], [2.0, -1.0]]])       # [kvol 2, C_out 2, C_in 2]
    t = torch.tensor([[3, 0, 1], [2, 1, 0]], dtype=torch.int32)                       # k-major, input row + 1
    # out 0 = f2 w0^T + f1 w1^T = (5, 6) + (7, 2);  out 1 = f0 w1^T = (3, 0);  out 2 = f0 w0^T = (1, 2)
    assert FO.spconv(f, w_t, t).tolist() == [[12.0, 8.0], [3.0, 0.0], [1.0, 2.0]]
    b = torch.tensor([-4.0, -1.0])
    assert FO.spconv(f, w_t, t, b, FO.ACT_RELU).tolist() == [[8.0, 7.0], [0.0, 0.0], [0.0, 1.0]]
    assert FO.spconv(f, w_t, t, b, FO.ACT_LEAKY, 0.25).tolist() == [[8.0, 7.0], [-0.25, -0.25], [-0.75, 1.0]]
    res = torch.tensor([[0.0, -10.0], [1.0, 0.0], [0.5, -4.0]])
    got = FO.spconv(f, w_t, t, b, FO.ACT_LEAKY, 0.25, res, FO.ACT_LEAKY, 0.5)
    assert got.tolist() == [[8.0, -1.5], [0.75, -0.125], [-0.125, -1.5]]
    # post_act applies without a residual too (the kernel's epilogue does)
    assert FO.spconv(f, w_t, t, b, post_act=FO.ACT_RELU).tolist() == [[8.0, 7.0], [0.0, 0.0], [0.0, 1.0]]
    # a table with no neighbour gives act(bias) on every row
    assert FO.spconv(f, w_t, torch.zeros((2, 2), dtype=torch.int32), b, FO.ACT_LEAKY, 0.5).tolist() == [[-2.0, -0.5]] * 2


def test_oracle_linear_and_selection_by_hand():
    a = torch.tensor([[1.0, 2.0], [3.0, -1.0]])
    w = torch.tensor([[1.0, 1.0], [0.0, 2.0], [1.0, -1.0], [2.0, 0.0]])              # 2 groups of n = 2
    assert FO.linear(a, w[:2], torch.tensor([0.5, 0.0])).tolist() == [[3.5, 4.0], [2.5, -2.0]]
    out = torch.full((4, 2), -7.0)
    # group 0 empty, group 1: a1 -> out row 3, a0 -> out row 0
    got = FO.linear_sel(a, w, torch.tensor([1, 0]), torch.tensor([3, 0]), [0, 0, 2], out, torch.tensor([1.0, -1.0]))
    assert got.tolist() == [[0.0, 1.0], [-7.0, -7.0], [-7.0, -7.0], [5.0, 5.0]]
    res = torch.tensor([[1.0, 1.0], [0.0, 0.0], [0.0, 0.0], [-10.0, 2.0]])             # residual row = OUTPUT row
    got = FO.linear_sel(a, w, torch.tensor([1, 0]), torch.tensor([3, 0]), [0, 0, 2], out, None, FO.ACT_NONE, 0.0, res,
                        FO.ACT_RELU)
    assert got.tolist() == [[0.0, 3.0], [-7.0, -7.0], [-7.0, -7.0], [0.0, 8.0]]
    assert out.tolist() == [[-7.0, -7.0]] * 4                                          # the input is not written


def test_oracle_wgrad_by_hand():
    x = torch.tensor([[1.0, 2.0], [3.0, 4.0]])
    dy = torch.tensor([[1.0], [-1.0], [2.0]])
    # offset 0: pairs (0 -> 2), (1 -> 0); offset 1: none; offset 2: (1 -> 1)
    dw = FO.wgrad(x, dy, torch.tensor([0, 1, 1]), torch.tensor([2, 0, 1]), [0, 2, 2, 3])
    assert dw.shape == (3, 2, 1)
    assert dw.reshape(3, 2).tolist() == [[2.0 + 3.0, 4.0 + 4.0], [0.0, 0.0], [-3.0, -4.0]]


def test_oracle_bound_and_exact_premise():
    f = torch.tensor([[1.0, -2.0]])
    w_t = torch.tensor([[[3.0, 4.0]]])
    t = torch.tensor([[1]], dtype=torch.int32)
    s = FO.abs_sum(f, w_t, t, torch.tensor([-5.0]), torch.tensor([[2.0]]))
    assert s.tolist() == [[3.0 + 8.0 + 5.0 + 2.0]]
    assert FO.bound(s, 2).tolist() == [[2.0 * 5 * 2.0 ** -24 * 18.0]]
    FO.assert_exact_premise(torch.tensor([FO.EXACT_LIMIT - 1.0]))
    with pytest.raises(AssertionError, match='premise'):
        FO.assert_exact_premise(torch.tensor([0.0, float(FO.EXACT_LIMIT)]))


# ---- table builders -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n_out', [1, 127, 128, 129, 1000])
def test_table_builders(n_out):
    kv, n_in = 27, 300
    for kind in FO.BUILDERS:
        t = FO.build_table(kind, kv, n_out, n_in, seed=n_out)
        assert t.shape == (kv, n_out) and t.dtype == torch.int32
        assert int(t.min()) >= 0 and int(t.max()) <= n_in
        assert torch.equal(t, FO.build_table(kind, kv, n_out, n_in, seed=n_out))       # deterministic
    n_tiles = (n_out + 127) // 128
    e = FO.empty_tile_table(kv, n_out, n_in, 0.9, 1)
    empty = [i for i in range(n_tiles) if not e[:, i * 128:(i + 1) * 128].any()]
    assert empty == list(range(min(1, n_tiles - 1), n_tiles, 7))
    o = FO.one_row_per_offset_table(kv, n_out, n_in, 2)
    for tile in range(n_tiles):
        blk = o[:, tile * 128:(tile + 1) * 128]
        assert ((blk != 0).sum(1) == 1).all()                                            # one row per offset
        if blk.shape[1] == 128:
            warps = {int(torch.nonzero(blk[k])[0]) // 32 for k in range(kv)}
            assert warps == {0, 1, 2, 3}
            masks = [int(((blk[:, w * 32:(w + 1) * 32] != 0).any(1)).sum()) for w in range(4)]
            assert all(0 < m < kv for m in masks)                                        # no warp sees the whole mask
    d = FO.edge_source_table(kv, n_out, n_in, 0.3, 3)
    for k in range(kv):
        assert (d[k] == 1).any() and (n_out == 1 or (d[k] == n_in).any())


def test_permute_rows_follows_the_row_perm_contract():
    t = FO.random_table(4, 300, 50, 0.5, 0)
    tp, perm = FO.permute_rows(t, 1)
    assert perm.dtype == torch.int32 and sorted(perm.tolist()) == list(range(300)) and perm.tolist() != list(range(300))
    for j in (0, 17, 299):
        assert torch.equal(tp[:, j], t[:, int(perm[j])])


def test_pairwise_design_covers_every_pair():
    factors = [(1, 2, 3), ('a', 'b', 'c', 'd'), (True, False), tuple(range(5))]
    cases = FO.pairwise(factors, seed=3)
    assert FO.covers_all_pairs(factors, cases)
    assert len(cases) < 3 * 4 * 2 * 5 // 3                                               # far fewer than the product
    assert cases == FO.pairwise(factors, seed=3)
    assert not FO.covers_all_pairs(factors, [c for c in cases if c[1] != 'd'])
