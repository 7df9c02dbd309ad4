"""Host-side pieces of the deep-factorized entropy model: every bad argument of fpcc_factorized_bits / _grad / _pmf comes
back as an error code and a message prefixed with the entry point's name before any CUDA work, and hand-computed cases
of the fp64 oracle (tests/entropy_model_oracle.py), so these run without a device."""
import ctypes as C
import math

import pytest
import torch

from tests import entropy_model_oracle as EO


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


def _bits(lib, p, y=True, ld=8, n=4, c=8, params=True, bound=1e-9, out=True):
    return lib.fpcc_factorized_bits(p if y else None, ld, n, c, p + 1024 if params else None, bound, p + 2048 if out else None, None)


def test_bits_rejects_bad_arguments(lib, p):
    name = 'factorized_bits'
    for kw in ({'y': False}, {'params': False}, {'out': False}):
        _fails(lib, _bits(lib, p, **kw), name, 'NULL pointer')
    for c in (0, -1, (1 << 24) + 1):
        _fails(lib, _bits(lib, p, c=c), name, 'C ')
    _fails(lib, _bits(lib, p, n=-1), name, 'bad row count')
    _fails(lib, _bits(lib, p, ld=7), name, 'row pitch')
    for b in (0.0, -1e-9, 1.0, float('nan'), float('inf')):
        _fails(lib, _bits(lib, p, bound=b), name, 'bound')


def test_bits_of_no_rows_is_a_no_op(lib, p):
    assert _bits(lib, p, n=0) == 0


def _grad(lib, p, y=True, ld=8, db=True, ld_db=8, n=4, c=8, params=True, bound=1e-9, dy=True, dp=True, ws=True, ws_bytes=None):
    if ws_bytes is None:
        ws_bytes = lib.fpcc_factorized_grad_workspace(n, c)
    return lib.fpcc_factorized_grad(p if y else None, ld, p + 512 if db else None, ld_db, n, c, p + 1024 if params else None,
                                    bound, p + 2048 if dy else None, p + 2560 if dp else None, p + 3072 if ws else None,
                                    ws_bytes, None)


def test_grad_rejects_bad_arguments(lib, p):
    name = 'factorized_grad'
    for kw in ({'y': False}, {'db': False}, {'params': False}, {'dy': False}, {'dp': False}):
        _fails(lib, _grad(lib, p, **kw), name, 'NULL pointer')
    for c in (0, -3):
        _fails(lib, _grad(lib, p, c=c), name, 'C ')
    _fails(lib, _grad(lib, p, n=-1), name, 'bad row count')
    _fails(lib, _grad(lib, p, ld=7), name, 'row pitch')
    _fails(lib, _grad(lib, p, ld_db=7), name, 'row pitch')
    _fails(lib, _grad(lib, p, bound=0.0), name, 'bound')
    _fails(lib, _grad(lib, p, ws=False), name, 'workspace')
    _fails(lib, _grad(lib, p, ws_bytes=8), name, 'workspace')


def test_grad_workspace_holds_fp64_partial_rows(lib):
    assert lib.fpcc_factorized_grad_workspace(1, 8) == (8 * 43 * 8 + 255) // 256 * 256         # one part
    assert lib.fpcc_factorized_grad_workspace(1000, 2) == (4 * 2 * 43 * 8 + 255) // 256 * 256   # 4 parts of 256 rows
    assert lib.fpcc_factorized_grad_workspace(10 ** 7, 1) == (296 * 43 * 8 + 255) // 256 * 256   # at most 296 parts


def test_pmf_rejects_bad_arguments(lib, p):
    name = 'factorized_pmf'
    _fails(lib, lib.fpcc_factorized_pmf(None, 4, -64, 129, p, None), name, 'NULL pointer')
    _fails(lib, lib.fpcc_factorized_pmf(p, 4, -64, 129, None, None), name, 'NULL pointer')
    _fails(lib, lib.fpcc_factorized_pmf(p, 0, -64, 129, p, None), name, 'C ')
    for ns in (0, -1, (1 << 16) + 1):
        _fails(lib, lib.fpcc_factorized_pmf(p, 4, -64, ns, p, None), name, 'n_sym')
    _fails(lib, lib.fpcc_factorized_pmf(p, 4, -(1 << 24) - 1, 129, p, None), name, '2^24')
    _fails(lib, lib.fpcc_factorized_pmf(p, 4, (1 << 24) - 10, 129, p, None), name, '2^24')


# ---------------------------------------------------------------------------------------------------------------------
# the oracle by hand
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_zero_params_is_linear_with_the_closed_form_slope():
    """H = b = a = 0: softplus(0) = ln 2 per weight, 3 inputs summed in layers 1-3 -> f(x) = 27 ln(2)^4 x"""
    params = torch.zeros((1, 43), dtype=torch.float64)
    k = 27 * math.log(2.0) ** 4
    x = torch.tensor([[-3.0], [0.0], [0.25], [7.0]], dtype=torch.float64)
    assert torch.allclose(EO.logits(params, x), k * x, rtol=1e-14, atol=0)
    y = 1.5
    u, l = k * (y + 0.5), k * (y - 0.5)                         # u + l > 0 -> s = -1
    want = -math.log2(1 / (1 + math.exp(l)) - 1 / (1 + math.exp(u)))   # sigmoid(-l) - sigmoid(-u)
    got = float(EO.bits(params, torch.tensor([[y]], dtype=torch.float64)))
    assert abs(got - want) < 1e-12, (got, want)


def test_oracle_logits_are_monotone():
    gen = torch.Generator().manual_seed(5)
    params = EO.random_params(16, gen, spread=2.0)
    x = torch.linspace(-300, 300, 4001, dtype=torch.float64)[:, None].expand(-1, 16)
    f = EO.logits(params, x)
    assert bool((f[1:] >= f[:-1]).all())


def test_oracle_bound_and_its_gradient_rule():
    params = torch.zeros((1, 43), dtype=torch.float64, requires_grad=True)
    y = torch.tensor([[5.0]], dtype=torch.float64, requires_grad=True)      # tail: L ~ 1e-12, below the bound
    assert float(EO.likelihood(params.detach(), y.detach())) < 1e-11
    b = EO.bits(params, y, 1e-9)
    assert abs(float(b.detach()) + math.log2(1e-9)) < 1e-12
    b.sum().backward()
    # dbits > 0 asks to raise L: the gradient passes, and a descent step moves y back towards the centre
    assert float(y.grad) > 0
    # an upstream gradient that would lower L below the bound is stopped
    y2 = torch.tensor([[5.0]], dtype=torch.float64, requires_grad=True)
    (-EO.bits(params.detach(), y2, 1e-9)).sum().backward()
    assert float(y2.grad) == 0.0
    # above the bound the gradient passes either way
    y3 = torch.tensor([[0.7]], dtype=torch.float64, requires_grad=True)
    (-EO.bits(params.detach(), y3, 1e-9)).sum().backward()
    assert float(y3.grad) != 0.0


def test_oracle_sign_choice_at_u_plus_l_zero():
    """y = 0 with zero params: u = -l, u + l = 0 -> s = +1; the likelihood is the same as with s = -1 by symmetry and
    never 0 (the -sign() choice would multiply by 0)"""
    params = torch.zeros((1, 43), dtype=torch.float64)
    y = torch.zeros((1, 1), dtype=torch.float64)
    u, l = EO.logits(params, y + 0.5), EO.logits(params, y - 0.5)
    assert float(u + l) == 0.0
    L = float(EO.likelihood(params, y))
    assert L > 0 and abs(L - (torch.sigmoid(u) - torch.sigmoid(l)).item()) < 1e-15
