"""Host-side pieces of the MinkowskiEngine-shim training path: every bad argument of fpcc_kmap_transpose and
fpcc_act_grad_f16 comes back as an error code and a message prefixed with the entry point's name before any CUDA work,
and hand-computed cases of the gradient oracle (tests/me_grad_oracle.py), so these run without a device."""
import ctypes as C

import pytest
import torch

from tests import me_grad_oracle as MO


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


def _kt(lib, p, table=True, kvol=8, n_out=4, ld=4, n_in=4, tt=True, ld_t=4):
    return lib.fpcc_kmap_transpose(p if table else None, kvol, n_out, ld, n_in, p + 512 if tt else None, ld_t, None)


def test_kmap_transpose_rejects_bad_arguments(lib, p):
    _fails(lib, _kt(lib, p, table=False), 'kmap_transpose', 'NULL pointer')
    _fails(lib, _kt(lib, p, tt=False), 'kmap_transpose', 'NULL pointer')
    for kv in (0, -1, 65536):
        _fails(lib, _kt(lib, p, kvol=kv), 'kmap_transpose', 'kvol')
    _fails(lib, _kt(lib, p, n_out=-1), 'kmap_transpose', 'negative row count')
    _fails(lib, _kt(lib, p, n_in=-1), 'kmap_transpose', 'negative row count')
    _fails(lib, _kt(lib, p, ld=3), 'kmap_transpose', 'row pitch')
    _fails(lib, _kt(lib, p, ld_t=3), 'kmap_transpose', 'row pitch')


def test_kmap_transpose_of_nothing_is_a_no_op(lib, p):
    assert _kt(lib, p, n_in=0, n_out=0, ld=0, ld_t=0) == 0


def _ag(lib, p, dy=True, dy_type=0, ld_dy=8, y=True, y_type=0, ld_y=8, n=4, c=8, act=1, slope=0.0, dz=True, dz_type=0,
        c_pad=16, dbias=True, ws=True, ws_bytes=None):
    if ws_bytes is None:
        ws_bytes = lib.fpcc_act_grad_workspace(n, c)
    return lib.fpcc_act_grad_f16(p if dy else None, dy_type, ld_dy, p if y else None, y_type, ld_y, n, c, act, slope,
                                 p + 1024 if dz else None, dz_type, c_pad, p + 2048 if dbias else None,
                                 p + 3072 if ws else None, ws_bytes, None)


def test_act_grad_rejects_bad_arguments(lib, p):
    name = 'act_grad_f16'
    _fails(lib, _ag(lib, p, dy=False), name, 'NULL pointer')
    _fails(lib, _ag(lib, p, dz=False), name, 'NULL pointer')
    for a in (-1, 3):
        _fails(lib, _ag(lib, p, act=a), name, 'unknown activation')
    _fails(lib, _ag(lib, p, y=False, act=1), name, 'forward output')
    _fails(lib, _ag(lib, p, act=2, slope=-0.1), name, 'slope')
    _fails(lib, _ag(lib, p, act=2, slope=float('nan')), name, 'slope')
    _fails(lib, _ag(lib, p, act=2, slope=float('inf')), name, 'slope')
    for t in (-1, 3):
        _fails(lib, _ag(lib, p, dy_type=t), name, 'dy / y types')
        _fails(lib, _ag(lib, p, y_type=t), name, 'dy / y types')
    for t in (-1, 2):
        _fails(lib, _ag(lib, p, dz_type=t), name, 'dz type')
    _fails(lib, _ag(lib, p, n=-1), name, 'bad row count')
    _fails(lib, _ag(lib, p, c=0), name, 'c <= c_pad')
    _fails(lib, _ag(lib, p, c_pad=4), name, 'c <= c_pad')
    _fails(lib, _ag(lib, p, c_pad=1 << 17), name, 'c <= c_pad')
    _fails(lib, _ag(lib, p, ld_dy=7), name, 'row pitch')
    _fails(lib, _ag(lib, p, ld_y=7), name, 'row pitch')
    _fails(lib, _ag(lib, p, ws=False), name, 'workspace')
    _fails(lib, _ag(lib, p, ws_bytes=8), name, 'workspace')


def test_act_grad_needs_no_y_or_workspace_when_unused(lib, p):
    # ACT_NONE reads no y; without dbias no workspace: both pass the checks (n = 0 launches nothing)
    assert _ag(lib, p, y=False, act=0, n=0, dbias=False, ws=False) == 0


def test_act_grad_workspace_holds_one_fp64_row_per_256_rows(lib):
    assert lib.fpcc_act_grad_workspace(1, 8) == 256
    assert lib.fpcc_act_grad_workspace(257, 40) == 768  # 2 partial rows x 40 doubles, rounded up to 256 bytes


def test_oracle_transpose_table_by_hand():
    t = torch.tensor([[2, 0, 1], [0, 3, 0]], dtype=torch.int32)   # offset 0: out 0 <- in 1, out 2 <- in 0; offset 1: out 1 <- in 2
    assert MO.transpose_table(t, 4).tolist() == [[3, 1, 0, 0], [0, 0, 2, 0]]


def test_oracle_act_grad_by_hand():
    dy = torch.tensor([[1.0, -2.0, 3.0], [0.5, 0.25, -1.0]])
    y = torch.tensor([[0.5, 0.0, -1.0], [2.0, -0.5, 1.0]])
    dz, db = MO.act_grad(dy, y, MO.ACT_LEAKY, 0.5, 8, torch.float16)
    assert dz.shape == (2, 8) and dz[:, 3:].abs().sum() == 0
    assert dz[:, :3].float().tolist() == [[1.0, -1.0, 1.5], [0.5, 0.125, -1.0]]
    assert db.tolist() == [1.5, -0.875, 0.5]
    dz, _ = MO.act_grad(dy, y, MO.ACT_RELU, 0.0, 8, torch.bfloat16)
    assert dz[:, :3].float().tolist() == [[1.0, 0.0, 0.0], [0.5, 0.0, -1.0]]


def test_oracle_layers_by_hand():
    f = torch.tensor([[1.0], [2.0]], dtype=torch.float64)
    w = torch.tensor([[[10.0]], [[100.0]]], dtype=torch.float64)           # K = 2, 1 -> 1
    t = torch.tensor([[1, 2], [2, 0]])                                      # out 0 = f0 w0 + f1 w1, out 1 = f1 w0
    assert MO.conv(f, w, torch.tensor([1.0], dtype=torch.float64), t).reshape(-1).tolist() == [211.0, 21.0]
    g = MO.gen(f, torch.arange(8, dtype=torch.float64).reshape(8, 1, 1), None)
    assert g.reshape(-1).tolist() == [float(k) for k in range(8)] + [2.0 * k for k in range(8)]
    # one parent at stride 2, children at slot 1 (x + 1) and slot 6 (y + 1, z + 1), and an orphan in another cell
    pc = torch.tensor([[0, 0, 0, 0]], dtype=torch.int32)
    oc = torch.tensor([[0, 1, 0, 0], [0, 0, 1, 1], [0, 2, 0, 0]], dtype=torch.int32)
    w8 = torch.arange(8, dtype=torch.float64).reshape(8, 1, 1)
    out = MO.tconv(torch.tensor([[3.0]], dtype=torch.float64), w8, torch.tensor([-1.0], dtype=torch.float64), pc, oc, 2, MO.ACT_RELU)
    assert out.reshape(-1).tolist() == [2.0, 17.0, 0.0]


def test_oracle_gradients_are_the_transposed_products():
    f = torch.tensor([[1.0, 2.0], [3.0, 4.0]], dtype=torch.float64, requires_grad=True)
    w = torch.tensor([[[1.0], [0.0]], [[0.0], [1.0]]], dtype=torch.float64, requires_grad=True)
    t = torch.tensor([[1, 2], [2, 0]])
    out = MO.conv(f, w, None, t)                                            # [[1 + 4], [3]]
    out.sum().backward()
    assert f.grad.tolist() == [[1.0, 0.0], [1.0, 1.0]]                      # dgrad on the transposed map
    assert w.grad.reshape(-1).tolist() == [4.0, 6.0, 3.0, 4.0]              # wgrad: sum of the gathered input rows
