"""Host-side pieces of the Gaussian conditional entropy model: every bad argument of fpcc_gaussian_bits / _grad / _pmf /
_indexes and of their ops wrappers comes back as an error before any CUDA work, and hand-computed cases of the fp64
oracle (tests/gaussian_oracle.py), so these run without a device."""
import ctypes as C
import math

import pytest
import torch

from tests import gaussian_oracle as GO


@pytest.fixture(scope='module')
def lib():
    from fastpcc_b200 import _lib
    return _lib.load()


_BUF = (C.c_uint8 * 8192)()


@pytest.fixture(scope='module')
def p():
    return (C.addressof(_BUF) + 15) & ~15


def _fails(lib, rc, prefix, text):
    assert rc != 0
    msg = lib.fpcc_last_error().decode()
    assert msg.startswith(prefix + ': ') and text in msg, msg


def _bits(lib, p, y=True, ld_y=8, mu=True, ld_mu=16, s=True, ld_s=16, n=4, c=8, sb=0.11, bound=1e-9, out=True):
    return lib.fpcc_gaussian_bits(p if y else None, ld_y, p + 1024 if mu else None, ld_mu, p + 1056 if s else None, ld_s, n, c,
                                  sb, bound, p + 2048 if out else None, None)


def test_bits_rejects_bad_arguments(lib, p):
    name = 'gaussian_bits'
    for kw in ({'y': False}, {'s': False}, {'out': False}):
        _fails(lib, _bits(lib, p, **kw), name, 'NULL pointer')
    for c in (0, -1, (1 << 22) + 1):
        _fails(lib, _bits(lib, p, c=c), name, 'C ')
    _fails(lib, _bits(lib, p, n=-1), name, 'bad row count')
    for kw in ({'ld_y': 7}, {'ld_mu': 7}, {'ld_s': 7}):
        _fails(lib, _bits(lib, p, **kw), name, 'row pitch')
    for sb in (0.0, -0.11, float('nan'), float('inf')):
        _fails(lib, _bits(lib, p, sb=sb), name, 'scale bound')
    for b in (0.0, -1e-9, 1.0, float('nan')):
        _fails(lib, _bits(lib, p, bound=b), name, 'likelihood bound')


def test_no_mean_and_no_rows(lib, p):
    assert _bits(lib, p, n=0) == 0
    assert _bits(lib, p, mu=False, ld_mu=0, n=0) == 0          # without mu its pitch is not looked at


def _grad(lib, p, y=True, mu=True, s=True, db=True, ld=8, ld_db=8, n=4, c=8, sb=0.11, bound=1e-9, dy=True, dmu=True, ds=True):
    return lib.fpcc_gaussian_grad(p if y else None, ld, p + 256 if mu else None, ld, p + 512 if s else None, ld,
                                  p + 768 if db else None, ld_db, n, c, sb, bound, p + 2048 if dy else None,
                                  p + 2560 if dmu else None, p + 3072 if ds else None, None)


def test_grad_rejects_bad_arguments(lib, p):
    name = 'gaussian_grad'
    for kw in ({'y': False}, {'s': False}, {'db': False}, {'dy': False}, {'ds': False}):
        _fails(lib, _grad(lib, p, **kw), name, 'NULL pointer')
    _fails(lib, _grad(lib, p, mu=False), name, 'dmu needs mu')
    assert _grad(lib, p, mu=False, dmu=False, n=0) == 0
    for c in (0, -3):
        _fails(lib, _grad(lib, p, c=c), name, 'C ')
    _fails(lib, _grad(lib, p, n=-1), name, 'bad row count')
    _fails(lib, _grad(lib, p, ld=7), name, 'row pitch')
    _fails(lib, _grad(lib, p, ld_db=7), name, 'row pitch')
    _fails(lib, _grad(lib, p, sb=0.0), name, 'scale bound')
    _fails(lib, _grad(lib, p, bound=1.5), name, 'likelihood bound')


def test_pmf_rejects_bad_arguments(lib, p):
    name = 'gaussian_pmf'
    _fails(lib, lib.fpcc_gaussian_pmf(None, 4, 1e-9, 99, p, p + 4096, None), name, 'NULL pointer')
    _fails(lib, lib.fpcc_gaussian_pmf(p, 4, 1e-9, 99, None, p + 4096, None), name, 'NULL pointer')
    _fails(lib, lib.fpcc_gaussian_pmf(p, 4, 1e-9, 99, p, None, None), name, 'NULL pointer')
    for T in (0, -1, (1 << 16) + 1):
        _fails(lib, lib.fpcc_gaussian_pmf(p, T, 1e-9, 99, p, p + 4096, None), name, 'T ')
    for tm in (0.0, -1e-9, 1.0, 2.0, float('nan')):
        _fails(lib, lib.fpcc_gaussian_pmf(p, 4, tm, 99, p, p + 4096, None), name, 'tail mass')
    for S in (0, -1, (1 << 20) + 1):
        _fails(lib, lib.fpcc_gaussian_pmf(p, 4, 1e-9, S, p, p + 4096, None), name, 'S ')


def _idx(lib, p, y=True, mu=True, s=True, ld=8, n=4, c=8, sb=0.11, table=True, T=64, sym=True, idx=True):
    return lib.fpcc_gaussian_indexes(p if y else None, ld, p + 256 if mu else None, ld, p + 512 if s else None, ld, n, c, sb,
                                     p + 1024 if table else None, T, p + 2048 if sym else None, p + 3072 if idx else None, None)


def test_indexes_reject_bad_arguments(lib, p):
    name = 'gaussian_indexes'
    for kw in ({'s': False}, {'table': False}, {'idx': False}):
        _fails(lib, _idx(lib, p, **kw), name, 'NULL pointer')
    _fails(lib, _idx(lib, p, sym=False), name, 'both or neither')
    _fails(lib, _idx(lib, p, y=False), name, 'both or neither')
    assert _idx(lib, p, y=False, sym=False, n=0) == 0          # the decoder's call
    for c in (0, -1):
        _fails(lib, _idx(lib, p, c=c), name, 'C ')
    _fails(lib, _idx(lib, p, n=-1), name, 'bad row count')
    _fails(lib, _idx(lib, p, ld=7), name, 'row pitch')
    _fails(lib, _idx(lib, p, sb=float('nan')), name, 'scale bound')
    for T in (0, -2):
        _fails(lib, _idx(lib, p, T=T), name, 'T ')


def test_tail_multiplier_is_the_normal_quantile(lib):
    for tm in (1e-9, 1e-3, 0.5, 0.999):
        assert abs(lib.fpcc_gaussian_tail_multiplier(tm) - GO.tail_multiplier(tm)) < 1e-12 * max(1.0, GO.tail_multiplier(tm))
    assert abs(GO.tail_multiplier(1e-9) - 6.109410204869) < 1e-9
    for tm in (0.0, 1.0, -1.0, float('nan')):
        assert math.isnan(lib.fpcc_gaussian_tail_multiplier(tm))


# ---------------------------------------------------------------------------------------------------------------------
# the ops wrappers (checks that come before any device work)
# ---------------------------------------------------------------------------------------------------------------------
def test_ops_wrappers_reject_bad_arguments():
    from fastpcc_b200 import ops
    s = torch.ones((4, 8))
    y = torch.zeros((4, 8))
    for tbl, text in ((torch.tensor([0.11, 0.11, 1.0]), 'strictly increasing'), (torch.tensor([1.0, 0.5]), 'strictly increasing'),
                      (torch.tensor([0.0, 1.0]), 'positive'), (torch.tensor([-1.0, 1.0]), 'positive'),
                      (torch.tensor([0.11, float('inf')]), 'positive'), (torch.tensor([]), 'non-empty'),
                      (torch.tensor([0.11, 1.0], dtype=torch.float64), '1-D fp32')):
        with pytest.raises(RuntimeError, match=text):
            ops.gaussian_pmf(tbl)
        with pytest.raises(RuntimeError, match=text):
            ops.gaussian_indexes(tbl, s)
    with pytest.raises(RuntimeError, match='CUDA'):                     # a good table, but on the host
        ops.gaussian_pmf(torch.tensor([0.11, 1.0]))
    for tm in (0.0, 1.0, -0.5):
        with pytest.raises(RuntimeError, match='tail_mass'):
            ops.gaussian_tail_multiplier(tm)
    with pytest.raises(RuntimeError, match='scale_bound'):
        ops.gaussian_bits(y, s, scale_bound=0.0)
    with pytest.raises(RuntimeError, match='likelihood bound'):
        ops.gaussian_bits(y, s, bound=1.0)
    with pytest.raises(RuntimeError, match='scales must be a 2-D fp32'):
        ops.gaussian_bits(y, s.double())
    with pytest.raises(RuntimeError, match=r'scales must be a 2-D fp32 CUDA tensor \[4, 8\]'):
        ops.gaussian_bits(y, s)                                          # host tensors
    with pytest.raises(RuntimeError, match=r'\[4, 8\]'):
        ops.gaussian_grad(torch.zeros((4, 7)), s, y)
    with pytest.raises(RuntimeError, match=r'\[4, 8\]'):
        ops.gaussian_bits(torch.zeros((5, 8)), s)


# ---------------------------------------------------------------------------------------------------------------------
# the oracle by hand
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_wide_scale_costs_the_gaussian_density():
    """sigma >> 1: L = erf(1 / (2 sqrt(2) s)) = (1 - 1 / (24 s^2) + ...) / (s sqrt(2 pi)), so at v = 0
    bits -> log2 s + log2(2 pi) / 2, within 1 / (24 s^2 ln 2)"""
    for s in (50.0, 300.0, 3000.0):
        got = float(GO.bits(torch.zeros(1, 1, dtype=torch.float64), torch.full((1, 1), s, dtype=torch.float64)))
        want = math.log2(s) + 0.5 * math.log2(2 * math.pi)
        assert 0 < got - want < 1.01 / (24 * s * s * math.log(2)), (s, got, want)


def test_oracle_slope_vanishes_at_the_mean():
    y = torch.zeros((1, 1), dtype=torch.float64, requires_grad=True)
    mu = torch.zeros((1, 1), dtype=torch.float64, requires_grad=True)
    s = torch.full((1, 1), 2.0, dtype=torch.float64, requires_grad=True)
    GO.bits(y, s, mu).sum().backward()
    assert float(y.grad) == 0.0 and float(mu.grad) == 0.0
    # the closed form of dL/ds at v = 0: (l phi(l) - u phi(u)) / s with u = -l = 1 / (2 s)
    u = 0.25
    phi = math.exp(-u * u / 2) / math.sqrt(2 * math.pi)
    L = math.erf(u / math.sqrt(2))
    dLds = (-u * phi - u * phi) / 2.0
    assert abs(float(s.grad) - (-dLds / (L * math.log(2)))) < 1e-12


def test_oracle_mean_shift_and_symmetry():
    y = torch.tensor([[3.7, -1.2]], dtype=torch.float64)
    mu = torch.tensor([[1.2, 0.3]], dtype=torch.float64)
    s = torch.tensor([[0.8, 4.0]], dtype=torch.float64)
    assert torch.allclose(GO.bits(y, s, mu), GO.bits(y - mu, s), rtol=0, atol=1e-14)
    assert torch.allclose(GO.bits(y - mu, s), GO.bits(mu - y, s), rtol=0, atol=0)


def test_oracle_both_bounds_and_their_gradient_rule():
    s = torch.full((1, 1), 0.5, dtype=torch.float64)
    y = torch.full((1, 1), 8.0, dtype=torch.float64, requires_grad=True)     # L ~ 1e-50: below the likelihood bound
    b = GO.bits(y, s)
    assert abs(float(b.detach()) + math.log2(1e-9)) < 1e-12
    b.sum().backward()
    assert float(y.grad) > 0                                                  # raising L passes: descent moves y in
    y2 = torch.full((1, 1), 8.0, dtype=torch.float64, requires_grad=True)
    (-GO.bits(y2, s)).sum().backward()
    assert float(y2.grad) == 0.0                                              # lowering it further is stopped
    # the scale bound: below it the value is the bound's
    lo = torch.full((1, 1), 0.01, dtype=torch.float64, requires_grad=True)
    at = torch.full((1, 1), 0.11, dtype=torch.float64)
    y3 = torch.full((1, 1), 1.0, dtype=torch.float64)
    assert float(GO.bits(y3, lo.detach())) == float(GO.bits(y3, at))
    GO.bits(y3, lo).sum().backward()
    assert float(lo.grad) < 0                   # |y| = 1 wants a wider scale: the step raises sigma, so it passes
    lo2 = torch.full((1, 1), 0.01, dtype=torch.float64, requires_grad=True)
    GO.bits(torch.zeros((1, 1), dtype=torch.float64), lo2).sum().backward()
    assert float(lo2.grad) == 0.0               # at the mean a narrower scale is better: the step would lower it


def test_oracle_index_rule_at_and_around_table_entries():
    table = torch.tensor([0.11, 0.5, 1.0, 4.0], dtype=torch.float32)
    nxt = lambda x, d: float(torch.nextafter(torch.tensor(x, dtype=torch.float32), torch.tensor(d, dtype=torch.float32)))  # noqa: E731
    cases = [(0.0, 0), (-5.0, 0), (0.05, 0), (0.11, 0), (nxt(0.11, 1), 1), (nxt(0.5, 0), 1), (0.5, 1), (nxt(0.5, 1), 2),
             (1.0, 2), (nxt(1.0, 2), 3), (4.0, 3), (nxt(4.0, 5), 3), (1e6, 3)]
    s = torch.tensor([[c[0] for c in cases]], dtype=torch.float32)
    assert GO.indexes(s, table).reshape(-1).tolist() == [c[1] for c in cases]


def test_oracle_default_table_rule():
    from fastpcc_b200.entropy_models import default_scale_table
    t = default_scale_table()
    assert t.dtype == torch.float32 and t.numel() == 64
    assert abs(float(t[0]) - 0.11) < 1e-7 and abs(float(t[-1]) - 256.0) < 1e-4 and bool((t[1:] > t[:-1]).all())
    ratio = (t[1:] / t[:-1]).double()
    assert float(ratio.max() - ratio.min()) < 1e-5 and abs(float(ratio.mean()) - 1.1312) < 1e-3
    m = GO.tail_multiplier(1e-9)
    centers = [math.ceil(float(v) * m) for v in t.double()]
    assert centers[0] == 1 and centers[-1] == 1565 and 2 * max(centers) + 1 == 3131
    pmf = GO.pmf_rows(t.double(), centers)
    mass = pmf.sum(1)
    assert float((1 - mass).max()) < 2e-9 and float((1 - mass).min()) > -1e-12   # tail mass <= 1e-9 (+ rounding)


def test_default_lossy_color_net_keeps_its_state_dict():
    """prior='factorized' (the default) builds the same modules in the same order: the state-dict keys and the seeded
    initial values hash as they did before the hyperprior option existed"""
    import hashlib
    from fastpcc_b200 import train
    torch.manual_seed(0)
    sd = train.LossyColorNet().state_dict()
    keys = sorted(sd)
    assert hashlib.sha256('\n'.join(keys).encode()).hexdigest() == '0157173d2eddf33abf03c5e9030537542a0ec4bca16cca81e01d0f52fd9efca5'
    h = hashlib.sha256()
    for k in keys:
        if torch.is_tensor(sd[k]):
            h.update(k.encode())
            h.update(sd[k].detach().float().contiguous().numpy().tobytes())
    assert h.hexdigest() == '4714b51486253197f5b979a484dee239fbe1802a321d410f605c96148e2b9441'
    hp = train.LossyColorNet(32, prior='hyperprior').state_dict()
    assert 'entropy_model.conditional.scale_table' in hp and 'entropy_model.hyper_prior.matrices.0' in hp
    with pytest.raises(ValueError, match='prior'):
        train.LossyColorNet(prior='gaussian')
